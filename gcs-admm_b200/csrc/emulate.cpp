// TEST-ONLY host emulation of kernel K1 (the per-vertex warp solve).  Compiles the same
// vertex_ipm.cuh / vertex_update.cuh sources with GCS_EMULATE so the CPU test suite can check the
// kernel's arithmetic against the oracle without a GPU.  It is never linked into libgcsadmm.so
// and nothing in the product path loads it.
#define GCS_EMULATE 1
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "vertex_update.cuh"
#include "vertex_perf.cuh"

extern "C" int gcsemu_vertex_update_all(int nV, int nE, const int *poly_off, const double *polyA, const double *polyb,
                                        const int *he_off, const int *he_edge, const unsigned char *he_flags,
                                        const unsigned char *vtype, const double *cent, double *xc, const double *mu,
                                        const double *z, double *x_v, double *z_v, double *y_v, double rho, double mu_scale,
                                        double tol, int max_iter, int dcap, int mcap, long *total_iters, double *ws, double theta) {
    GcsGraphView G = {nV, nE, poly_off, polyA, polyb, he_off, he_edge, he_flags, vtype, cent};
    GcsStateView St = {xc, mu, z, x_v, z_v, y_v, ws, theta, 0.0};
    GcsScratchLayout L = gcs_scratch_layout(dcap, mcap);
    double *S = (double *)malloc(sizeof(double) * L.total);
    int fails = 0;
    long iters = 0;
    for (int v = 0; v < nV; ++v) {
        int status = 0;
        memset(S, getenv("GCSEMU_POISON") ? 0xFF : 0, sizeof(double) * L.total);
        iters += gcs_vertex_update(G, St, v, rho, mu_scale, tol, max_iter, L, S, 0, &status);
        if (status > 0 && status != 5) { fails++; if (getenv("GCSEMU_VERBOSE")) fprintf(stderr, "emu: vertex %d status %d\n", v, status); }
    }
    free(S);
    *total_iters = iters;
    return fails;
}
extern "C" int gcsemu_scratch_doubles(int dcap, int mcap) { return gcs_scratch_layout(dcap, mcap).total; }
extern "C" int gcsemu_ws_stride(int dcap, int mcap) { return gcs_ws_stride(gcs_scratch_layout(dcap, mcap)); }

// perf-mode K1 (vertex_perf.cuh), emulated: one host thread plays each thread block (tile) in turn.
// INNER: the variant that also measures the inner residual; each tile's share goes to rin_tile[t] (summed by the caller in
// tile order, so the result does not depend on the OpenMP schedule)
template <bool INNER>
static int perf_all(int nV, int nE, const int *poly_off, const double *polyA, const double *polyb,
                    const int *he_off, const int *he_edge, const unsigned char *he_flags,
                    const unsigned char *vtype, const double *cent, double *xc, const double *mu,
                    const double *z, double *x_v, double *z_v, double *y_v, double rho, double mu_scale,
                    const int *vclass, const double *cls_tab, const int *cone_off, const double *cone,
                    const int *blk_off, const int *blk_he, const int *blk_edge, const int *blk_info, const int *tile_voff, int ntiles,
                    int cap_blocks, int cap_verts, int cap_cone, double *tstate, double *tn,
                    int inner_iters, double alpha, double kappa, double theta, const double *edge_delta, double *rin_tile) {
    GcsGraphView G = {nV, nE, poly_off, polyA, polyb, he_off, he_edge, he_flags, vtype, cent};
    GcsStateView St = {xc, mu, z, x_v, z_v, y_v, 0, 0.0, 0.0};
    GcsPerfLayout L = gcs_perf_layout(cap_blocks, cap_verts, cap_cone);
    // the packed descriptors gcsadmm_enable_perf builds on the host (same rules)
    const int nB = blk_off[nV];
    int *brec = (int *)calloc(4 * (size_t)(nB ? nB : 1), sizeof(int)), *vrec = (int *)calloc(GCS_VI_N * (size_t)nV, sizeof(int)), *trec = (int *)calloc(8 * (size_t)ntiles, sizeof(int));
    for (int b = 0; b < nB; ++b) { brec[4 * b] = blk_he[b]; brec[4 * b + 1] = blk_info[b]; brec[4 * b + 2] = blk_edge[b]; }
    for (int t = 0; t < ntiles; ++t) {
        const int a = tile_voff[t], b = tile_voff[t + 1];
        int *r = trec + 8 * t;
        r[0] = a; r[1] = b - a; r[2] = blk_off[a]; r[3] = blk_off[b] - blk_off[a]; r[4] = cone_off[a]; r[5] = cone_off[b] - cone_off[a];
        r[6] = he_off[a]; r[7] = he_off[b] - he_off[a];
        for (int hh = he_off[a]; hh < he_off[b]; ++hh) if (he_flags[hh] & GCS_HE_ZERO) r[7] |= 1 << 30;
        for (int v = a; v < b; ++v) {
            int *w = vrec + GCS_VI_N * v;
            w[GCS_VI_CONE] = cone_off[v] - cone_off[a]; w[GCS_VI_NV] = cone_off[v + 1] - cone_off[v]; w[GCS_VI_CLS] = vclass[v];
            int nin = 0;
            for (int bb = blk_off[v]; bb < blk_off[v + 1]; ++bb) nin += ((blk_info[bb] >> 8) & 3) == 0;
            w[GCS_VI_TERM] = (vtype[v] != GCS_VT_GENERIC) | (nin << 1); w[GCS_VI_BLK] = blk_off[v] - blk_off[a]; w[GCS_VI_NB] = blk_off[v + 1] - blk_off[v];
            w[GCS_VI_ACTIVE] = 0; w[GCS_VI_HE] = he_off[v] - he_off[a];
        }
    }
    GcsPerfTables T = {vclass, cls_tab, cone_off, cone, blk_off, brec, vrec, trec, ntiles, tstate, tn, inner_iters, alpha, kappa, theta, edge_delta};
    Ctrl ctrl;
    memset(&ctrl, 0, sizeof ctrl);
    ctrl.rho = rho; ctrl.mu_scale = mu_scale;
    const int poison = getenv("GCSEMU_POISON") ? 0xFF : 0;     // 0xFF: NaN doubles / -1 ints expose uninitialised reads
#pragma omp parallel
    {
        double *S = (double *)malloc(sizeof(double) * L.total);
#pragma omp for schedule(dynamic, 16)
        for (int t = 0; t < ntiles; ++t) {
            memset(S, poison, sizeof(double) * L.total);
            Ctrl local = ctrl;
            double rin = 0.0;
            gcs_perf_tile<INNER, false>(G, St, T, L, S, S + L.work, t, &local, rin, nullptr, 0, nullptr);
            if (rin_tile) rin_tile[t] = rin;
        }
        free(S);
    }
    free(brec); free(vrec); free(trec);
    for (int v = 0; v < nV; ++v)      // what perf_init_dead_kernel writes once on the device
        if (vtype[v] == GCS_VT_DEAD) { for (int k = 0; k < 4; ++k) { z_v[4 * v + k] = 0.0; x_v[4 * v + k] = cent[2 * v + (k & 1)]; } y_v[v] = 0.0; }
    return ntiles;
}

extern "C" int gcsemu_vertex_update_perf_all(int nV, int nE, const int *poly_off, const double *polyA, const double *polyb,
                                             const int *he_off, const int *he_edge, const unsigned char *he_flags,
                                             const unsigned char *vtype, const double *cent, double *xc, const double *mu,
                                             const double *z, double *x_v, double *z_v, double *y_v, double rho, double mu_scale,
                                             const int *vclass, const double *cls_tab, const int *cone_off, const double *cone,
                                             const int *blk_off, const int *blk_he, const int *blk_edge, const int *blk_info, const int *tile_voff, int ntiles,
                                             int cap_blocks, int cap_verts, int cap_cone, double *tstate, double *tn,
                                             int inner_iters, double alpha, double kappa, double theta, const double *edge_delta) {
    return perf_all<false>(nV, nE, poly_off, polyA, polyb, he_off, he_edge, he_flags, vtype, cent, xc, mu, z, x_v, z_v, y_v, rho, mu_scale,
                           vclass, cls_tab, cone_off, cone, blk_off, blk_he, blk_edge, blk_info, tile_voff, ntiles, cap_blocks, cap_verts,
                           cap_cone, tstate, tn, inner_iters, alpha, kappa, theta, edge_delta, nullptr);
}

// the INNER variant of K1 (what the device runs once the run is near its absolute tolerance): the same update, plus
// *inner_sq = the squared inner residual |(M u + m0) - c|^2 over every pair and path-length item of the last pass
extern "C" int gcsemu_vertex_update_perf_inner(int nV, int nE, const int *poly_off, const double *polyA, const double *polyb,
                                               const int *he_off, const int *he_edge, const unsigned char *he_flags,
                                               const unsigned char *vtype, const double *cent, double *xc, const double *mu,
                                               const double *z, double *x_v, double *z_v, double *y_v, double rho, double mu_scale,
                                               const int *vclass, const double *cls_tab, const int *cone_off, const double *cone,
                                               const int *blk_off, const int *blk_he, const int *blk_edge, const int *blk_info, const int *tile_voff, int ntiles,
                                               int cap_blocks, int cap_verts, int cap_cone, double *tstate, double *tn,
                                               int inner_iters, double alpha, double kappa, double theta, const double *edge_delta, double *inner_sq) {
    double *rin = (double *)calloc((size_t)(ntiles > 0 ? ntiles : 1), sizeof(double));
    const int r = perf_all<true>(nV, nE, poly_off, polyA, polyb, he_off, he_edge, he_flags, vtype, cent, xc, mu, z, x_v, z_v, y_v, rho, mu_scale,
                                 vclass, cls_tab, cone_off, cone, blk_off, blk_he, blk_edge, blk_info, tile_voff, ntiles, cap_blocks, cap_verts,
                                 cap_cone, tstate, tn, inner_iters, alpha, kappa, theta, edge_delta, rin);
    double s = 0.0;
    for (int t = 0; t < ntiles; ++t) s += rin[t];       // tile order: independent of the OpenMP schedule
    *inner_sq = s;
    free(rin);
    return r;
}

// gcs_cone_project on n points (pts, out: n x 3) against one cone of nv records (GCS_CONE_REC doubles each)
extern "C" void gcsemu_cone_project(const double *cone, int nv, const double *pts, int n, double *out) {
    for (int i = 0; i < n; ++i) gcs_cone_project(cone, nv, pts[3 * i], pts[3 * i + 1], pts[3 * i + 2], out[3 * i], out[3 * i + 1], out[3 * i + 2]);
}
// gcs_cone_project2 on the point pairs (pts[2 i], pts[2 i + 1]), i < n / 2, against one cone (n even; out as for gcsemu_cone_project)
extern "C" void gcsemu_cone_project2(const double *cone, int nv, const double *pts, int n, double *out) {
    for (int i = 0; i + 1 < n; i += 2) {
        const double *c = pts + 3 * i;
        double *q = out + 3 * i;
        gcs_cone_project2(cone, nv, c[0], c[1], c[2], c[3], c[4], c[5], q[0], q[1], q[2], q[3], q[4], q[5]);
    }
}
