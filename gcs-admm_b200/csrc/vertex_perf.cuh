// K1 in `perf` mode — the x-update of the full-vertex-split ADMM (reference admm_solver_v3.py:352-540) done INEXACTLY by
// K warm-started iterations of an operator-splitting scheme whose steps are all closed-form (north_star:
// "fixed-iteration inner projection / primal-dual scheme").
//
// Every inequality of the vertex program (:416-440) says that a (point, flow) pair lies in the perspective cone of the
// vertex's polygon,  K_P = {(p, h) in R^3 : A p <= h b}:
//     C3: (a_i, y_e)        C4: (x_i - a_i, 1 - y_e)        C1: (z_i, y_v)        C2: (x_i - z_i, 1 - y_v)
// and the pairs are 0/+-1 linear images  pv = M u + m0  of the variables u = (x, z_v, y_v, (a_1, a_2, y) per live half-edge).
// Splitting  c in prod K_P  from u, with one vector  t = c + lam  per pair kept in HBM between ADMM iterations
// (Moreau: c = Proj_K(t), lam = t - c), one inner iteration is
//     c-step : c = Proj_{K_P}(t), lam = t - c        exact 3-D cone projection, O(#polygon vertices); the path-length term
//              |z_1 - z_2| (:380-384) is a block soft-threshold with threshold 1 / sigma  (sigma = kappa rho)
//     v-step : u = argmin  rho/2 |S u - T|^2 + eps'y + sigma/2 |M u + m0 - (c - lam)|^2   over the equalities C6 / C7 (:450-464)
//     t-step : t = alpha (M u + m0) + (1 - alpha) c + lam
// The v-step is an equality-constrained quadratic whose matrix depends only on the vertex CLASS (type, #in, #out).  Its
// solution has the structure  u[b, tau] = dinv[g, tau] r[b, tau] + beta[g, tau]  for the five variables tau of a
// half-edge block b in group g (in / out), with the 19-vector (x, z_v, y_v, beta_in, beta_out) a class-constant linear
// map of (r_x, r_z, r_yv, sum_in r, sum_out r): O(d) work per vertex instead of a dense (5d)^2 product
// (tables: gcs-admm_b200/perf.py class_tables).
//
// Mapping: a thread block works on one TILE of consecutive vertices at a time (<= 64 blocks = 256 pairs; the kernel's blocks are
// persistent and walk tiles, staging the next one while they compute — gcsadmm.cu vertex_perf_kernel); every phase is a flat loop
// over (pair | block variable | vertex) items of the whole tile, so lanes stay busy whatever the degrees are; phases
// exchange data through shared memory only.  The per-tile state t, the cone records and the path-length state are
// contiguous in HBM and move with 1-D bulk async copies (cp.async.bulk + mbarrier).
//
// The fixed point of the outer ADMM is unchanged (an exact minimiser of the vertex program is a fixed point of the
// inner iteration); the trajectory is not the reference's, so this mode is validated at convergence against the
// classic relaxation optimum and gated by tests/test_gpu_perf.py.
//
// The file compiles two ways, like vertex_ipm.cuh: nvcc (device) and g++ with GCS_EMULATE (tests only: one host
// thread plays the whole thread block, loops run serially, barriers are no-ops, bulk copies are memcpy).
#pragma once
#include <string.h>
#include "gcs_ctrl.h"
#include "vertex_update.cuh"

#define GCS_CONE_REC 12   // doubles per polygon vertex in the cone table
#define GCS_NCX 19        // extended core of the v-step: x(4) z(4) y_v | beta_in(5) | beta_out(5)
#define GCS_CLS_G0 361    // class table: G transposed (19 x 19) | g0 (19) | dinv (2 x 5) | pad
#define GCS_CLS_DINV 380
#define GCS_CLS_STRIDE 392
#define GCS_PERF_THREADS 256

#ifdef GCS_EMULATE
#define GCS_CTA_LOOP(i, n) for (int i = 0; i < (n); ++i)
#define GCS_CTA_SYNC() ((void)0)
#else
#define GCS_CTA_LOOP(i, n) for (int i = threadIdx.x; i < (n); i += blockDim.x)
#define GCS_CTA_SYNC() __syncthreads()
#endif

struct GcsPerfTables {
    const int *vclass;         // [nV] class id (-1: dead vertex)
    const double *cls_tab;     // [ncls][GCS_CLS_STRIDE]
    const int *cone_off;       // [nV+1] polygon vertices of vertex v: cone_off[v]..cone_off[v+1]
    const double *cone;        // GCS_CONE_REC doubles per polygon vertex (see gcs_cone_project)
    const int *blk_off;        // [nV+1] blocks of vertex v: its live half-edges in half-edge order (in-half-edges first), then (z_v, y_v)
    const int *blk_rec;        // [B][4]: half-edge of the block (-1 for the (z_v, y_v) block) | descriptor: bits 0-7 vertex index inside its
                               //         tile, bits 8-9 group (0 in, 1 out, 2 z-block), bit 10 's' / 't' | edge of the half-edge | 0
    const int *vrec;           // [nV][GCS_VI_N]: the per-vertex descriptor the kernel keeps in shared memory (offsets relative to the tile)
    const int *tile_rec;       // [ntiles][8]: first vertex, #vertices, first block, #blocks, first cone record, #records, first half-edge,
                               //              #half-edges | bit 30 of #half-edges: the tile has forced-zero half-edges
    int ntiles;
    double *tstate;            // [B][4 pairs][3]  t = c + lam of every (point, flow) pair
    double *tn;                // [nV][2]          the same for the path-length item z_1 - z_2
    int inner_iters;           // K
    double alpha, kappa;
    double theta;              // penalty of the flow scalars = theta * rho (1: the reference's single rho; see GcsPerfConfig)
    const double *edge_delta;  // [nE][2] or null.  Non-null = LOCAL FRAMES: every vertex program works in coordinates centred on its
                               // own region (polytopes / cones shifted by cent[v]); the two copies of an edge e = (u, w) then agree through
                               // x_head = z_e,  x_tail = B_e z_e  with  B_e (p1, p2, y) = (p1, p2 - y delta_e, y),  delta_e = cent[u] - cent[w]
    double *tile_res;          // [grid] or null (host emulation); out: squared INNER residual summed over the tiles a thread block walked (INNER kernel variant)
};

// shared memory of one tile (offsets in doubles).  Two regions: the STAGED arrays that arrive by bulk copies (state t, cone
// records, path-length state, per-vertex and per-block descriptors; offsets relative to the stage base — the kernel keeps two
// stage buffers and fills one while it works on the other) and the WORK arrays (offsets relative to the work base).
struct GcsPerfLayout { int nb_cap, nvt_cap, cone_cap, tS, cone, tnS, vi, bi, tr, stage, eS, enS, T, r, cin, cout, vd, rin, work, total; };
#define GCS_VI_N 8        // ints per vertex of the tile
#define GCS_VI_CONE 0     // first cone record, relative to the tile's
#define GCS_VI_NV 1       // polygon vertices
#define GCS_VI_CLS 2
#define GCS_VI_TERM 3     // bit 0: 's' / 't' vertex | bits 1-: live in-half-edges (its blocks hold all of them before any out-half-edge)
#define GCS_VI_BLK 4      // first block, relative to the tile's
#define GCS_VI_NB 5       // blocks (0: dead vertex)
#define GCS_VI_ACTIVE 6   // its problem is still iterating (the table holds the vertex's problem index here)
#define GCS_VI_HE 7       // first half-edge, relative to the tile's
#if defined(__CUDACC__)
__host__ __device__
#endif
static inline GcsPerfLayout gcs_perf_layout(int nb_cap, int nvt_cap, int cone_cap) {
    GcsPerfLayout L;
    if (nb_cap < 1) nb_cap = 1;
    if (nvt_cap < 1) nvt_cap = 1;
    if (cone_cap < 1) cone_cap = 1;
    L.nb_cap = nb_cap; L.nvt_cap = nvt_cap; L.cone_cap = cone_cap;
    int o = 0;
    L.tS = o; o += 12 * nb_cap;              // every staged array starts at a 16-byte aligned offset and is a multiple of 16 bytes long
    L.cone = o; o += GCS_CONE_REC * cone_cap;
    L.tnS = o; o += 2 * nvt_cap;
    L.vi = o; o += (GCS_VI_N * nvt_cap) / 2;
    L.bi = o; o += 2 * nb_cap;                // 4 ints per block: half-edge, descriptor, edge, pad
    L.tr = o; o += 4;                         // the tile's own record (8 ints)
    L.stage = o;
    o = 0;
    L.eS = o; o += 12 * nb_cap;
    L.enS = o; o += 2 * nvt_cap;
    L.T = o; o += 5 * nb_cap;
    L.r = o; o += 5 * nb_cap;
    L.cin = o; o += GCS_NCX * nvt_cap;
    L.cout = o; o += GCS_NCX * nvt_cap;
    L.vd = o; o += 2 * nvt_cap;
    L.rin = o; o += GCS_PERF_THREADS / 32;     // per-warp partial sums of the inner residual
    L.work = o + (o & 1);
    L.total = L.work + L.stage;               // single-buffered (host emulation); the kernel uses work + 2 stage
    return L;
}

// exact projection of c onto the cone spanned by the rays r_k = (V_k, 1), k = 0..nv-1 (counter-clockwise).
// record k: V_k (2) | unit outward normal n_k of the face between rays k and k+1 (3) | 1/|r_k|^2 | sector normals ma, mb (3 + 3)
// The projection is c itself (inside), lies on a face (then c is outside that face and its foot point is inside the
// face's sector: unique, and no other candidate can be nearer), on a ray (the one with the largest reduction
// tau^2 / |r|^2 of the squared distance), or is the apex.  ma, mb are orthogonal to n_k, so the sector test of the foot
// point  c - dist n_k  is a test on c itself.
// record k: ray and face (read for every record); the sector normals are read only when a point is outside face k
struct GcsConeRay { double vx, vy, nx, ny, nh, inv; };
#if defined(GCS_EMULATE)
GCS_DEV GcsConeRay gcs_cone_ray(const double *cone, int k) { const double *r = cone + GCS_CONE_REC * k; return GcsConeRay{r[0], r[1], r[2], r[3], r[4], r[5]}; }
#else
// records are 96 bytes, 16-byte aligned: 3 LDS.128 for the ray and the face, 2 + 2 for the sector normals
GCS_DEV GcsConeRay gcs_cone_ray(const double *cone, int k) {
    const double2 *r = reinterpret_cast<const double2 *>(cone + GCS_CONE_REC * k);
    const double2 r0 = r[0], r1 = r[1], r2 = r[2];
    return GcsConeRay{r0.x, r0.y, r1.x, r1.y, r2.x, r2.y};
}
#endif
// sector normal ma (s = 0) or mb (s = 1) of record k dotted with the point c
GCS_DEV double gcs_cone_sector_dot(const double *cone, int k, int s, double c0, double c1, double c2) {
    const double *m = cone + GCS_CONE_REC * k + 6 + 3 * s;
    return c0 * m[0] + c1 * m[1] + c2 * m[2];
}
// candidate ray k for the point c (code: -1 apex | 2k ray k | 2k+1 face k); returns the signed distance of c from face k
GCS_DEV double gcs_cone_test_ray(const GcsConeRay &R, int k, double c0, double c1, double c2, double &best, int &code) {
    const double tau = c0 * R.vx + c1 * R.vy + c2;
    const double dist = R.nx * c0 + R.ny * c1 + R.nh * c2;
    if (tau > 0.0) {
        const double red = tau * tau * R.inv;
        if (red > best) { best = red; code = 2 * k; }
    }
    return dist;
}
// face k is the candidate for a point c outside it (dist > 0) whose dot products with both sector normals are >= 0
GCS_DEV void gcs_cone_take_face(bool sector, int k, double &best, int &code, bool &inside) {
    inside = false;
    if (sector) { best = 1e300; code = 2 * k + 1; }
}
GCS_DEV void gcs_cone_pick(const double *cone, int code, bool inside, double c0, double c1, double c2, double &q0, double &q1, double &q2) {
    if (inside) { q0 = c0; q1 = c1; q2 = c2; return; }
    q0 = 0.0; q1 = 0.0; q2 = 0.0;
    if (code < 0) return;
    const double *ck = cone + GCS_CONE_REC * (code >> 1);
    if (code & 1) {
        const double dist = ck[2] * c0 + ck[3] * c1 + ck[4] * c2;
        q0 = c0 - dist * ck[2]; q1 = c1 - dist * ck[3]; q2 = c2 - dist * ck[4];
    } else {
        const double tau = (c0 * ck[0] + c1 * ck[1] + c2) * ck[5];
        q0 = tau * ck[0]; q1 = tau * ck[1]; q2 = tau;
    }
}
GCS_DEV void gcs_cone_project(const double *cone, int nv, double c0, double c1, double c2, double &q0, double &q1, double &q2) {
    double best = 0.0;
    int code = -1;
    bool inside = true;
#pragma unroll 1
    for (int k = 0; k < nv; ++k) {
        const double dist = gcs_cone_test_ray(gcs_cone_ray(cone, k), k, c0, c1, c2, best, code);
        if (dist > 0.0) gcs_cone_take_face(gcs_cone_sector_dot(cone, k, 0, c0, c1, c2) >= 0.0 && gcs_cone_sector_dot(cone, k, 1, c0, c1, c2) >= 0.0, k, best, code, inside);
    }
    gcs_cone_pick(cone, code, inside, c0, c1, c2, q0, q1, q2);
}
// the same projection of two points onto one cone: each record is loaded once for both points (two independent dependency
// chains); every point sees exactly the expressions of gcs_cone_project in the same order, so the results are bit-identical to
// two calls
GCS_DEV void gcs_cone_project2(const double *cone, int nv, double c0, double c1, double c2, double d0, double d1, double d2,
                               double &q0, double &q1, double &q2, double &s0, double &s1, double &s2) {
    double best_c = 0.0, best_d = 0.0;
    int code_c = -1, code_d = -1;
    bool inside_c = true, inside_d = true;
#pragma unroll 1
    for (int k = 0; k < nv; ++k) {
        const GcsConeRay R = gcs_cone_ray(cone, k);
        const double dist_c = gcs_cone_test_ray(R, k, c0, c1, c2, best_c, code_c);
        const double dist_d = gcs_cone_test_ray(R, k, d0, d1, d2, best_d, code_d);
        if (dist_c > 0.0 || dist_d > 0.0) {      // the sector normals one at a time: fewer registers live
            const bool ma_c = gcs_cone_sector_dot(cone, k, 0, c0, c1, c2) >= 0.0, ma_d = gcs_cone_sector_dot(cone, k, 0, d0, d1, d2) >= 0.0;
            const bool mb_c = gcs_cone_sector_dot(cone, k, 1, c0, c1, c2) >= 0.0, mb_d = gcs_cone_sector_dot(cone, k, 1, d0, d1, d2) >= 0.0;
            if (dist_c > 0.0) gcs_cone_take_face(ma_c && mb_c, k, best_c, code_c, inside_c);
            if (dist_d > 0.0) gcs_cone_take_face(ma_d && mb_d, k, best_d, code_d, inside_d);
        }
    }
    gcs_cone_pick(cone, code_c, inside_c, c0, c1, c2, q0, q1, q2);
    gcs_cone_pick(cone, code_d, inside_d, d0, d1, d2, s0, s1, s2);
}

#if !defined(GCS_EMULATE) && defined(__CUDACC__)
// 1-D bulk async copies (TMA unit, SASS UBLKCP) with an mbarrier for the loads and a bulk group for the stores
__device__ __forceinline__ unsigned gcs_smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void gcs_mbar_init(unsigned long long *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(gcs_smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void gcs_mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(gcs_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void gcs_bulk_g2s(void *dst, const void *src, unsigned bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(gcs_smem_u32(dst)), "l"(src), "r"(bytes), "r"(gcs_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void gcs_mbar_wait(unsigned long long *bar, unsigned parity) {
    unsigned done = 0;
    while (!done) {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(done) : "r"(gcs_smem_u32(bar)), "r"(parity) : "memory");
    }
}
__device__ __forceinline__ void gcs_bulk_s2g(void *dst, const void *src, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(gcs_smem_u32(src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void gcs_bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void gcs_bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void gcs_fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
#endif

#define GCS_PF 3   // consensus targets a thread keeps in registers between issuing their loads and using them (device build)

// input k of the extended core of vertex vl:  r_x (4) | r_z, r_yv (5) | sum of r over the in-blocks (5) | over the out-blocks (5)
GCS_DEV double gcs_core_input(const double *tS, const double *rS, const int *w, int k, double kappa) {
    const int bl = w[GCS_VI_BLK], zb = bl + w[GCS_VI_NB] - 1;
    double s = 0.0;
    if (k < 4) {
        if (!(w[GCS_VI_TERM] & 1)) { for (int b = bl; b <= zb; ++b) s += tS[12 * b + 6 * (k >> 1) + 3 + (k & 1)]; s *= kappa; }
    } else if (k < 9) s = rS[5 * zb + k - 4];
    else {      // the in-blocks are bl .. bl + nin - 1, the out-blocks follow up to the z-block
        const int g = k >= 14, tau = k - 9 - 5 * g, bin = bl + (w[GCS_VI_TERM] >> 1);
        for (int b = g ? bin : bl; b < (g ? zb : bin); ++b) s += rS[5 * b + tau];
    }
    return s;
}
// output k of the extended core:  (x, z_v, y_v, beta_in, beta_out)[k] = g0[k] + G[k, :] . in
GCS_DEV double gcs_core_output(const double *tab, const double *in, int k) {
    // G is stored TRANSPOSED (tab[19 j + k] = G[k, j]): the 19 lanes that evaluate the 19 outputs of a vertex read 19 consecutive
    // doubles per step (2 cache lines) instead of 19 doubles 152 bytes apart (19 lines)
    const double *gk = tab + k;
    double s0 = tab[GCS_CLS_G0 + k], s1 = 0.0;
#pragma unroll
    for (int j = 0; j + 1 < GCS_NCX; j += 2) { s0 += gk[GCS_NCX * j] * in[j]; s1 += gk[GCS_NCX * (j + 1)] * in[j + 1]; }
    return s0 + s1 + gk[GCS_NCX * (GCS_NCX - 1)] * in[GCS_NCX - 1];
}

// right-hand side r[q] of block-variable q = 5 b + tau of vertex vl (see P3 in gcs_perf_tile); d = c - lam of the block's pairs
GCS_DEV double gcs_rhs(const GcsPerfTables &T, const double *tS, const double *TS, const double *tnS, const int *brec, int q, int vl, double rho, double kappa) {
    const int b = q / 5, tau = q - 5 * b, info = brec[4 * b + 1], grp = (info >> 8) & 3;
    const bool term = (info >> 10) & 1;
    const double *d = tS + 12 * b;                                    // pair (i, fam) at 3 (2 i + fam)
    double val;
    if (tau < 4) {
        const int i = tau >> 1, c = tau & 1;
        val = d[6 * i + c];
        if (!term) val -= d[6 * i + 3 + c];
        val *= kappa;
        if (grp == 1) val += TS[q];                                    // out-edge: both points carry the rho-quadratic
        else if (grp == 0) { if (tau < 2) val += TS[q + 2]; }          // in-edge: own first point (edge-canonical slots 2, 3)
        else val += (i ? -kappa : kappa) * tnS[2 * vl + c];            // (z_v, y_v) block: the path-length item
    } else {
        val = d[2] + d[8];
        if (!term) val += (1.0 - d[5]) + (1.0 - d[11]);
        val *= kappa;
        if (grp < 2) val += T.theta * TS[q] - GCS_EDGE_PENALTY / rho;
    }
    return val;
}
// block variable tau of block b after the v-step:  u = dinv r + beta  (edge blocks),  (z_v, y_v) itself for the vertex's own block
GCS_DEV double gcs_block_u(const double *rS, const double *co, const double *tab, int info, int b, int tau) {
    const int grp = (info >> 8) & 3;
    return grp == 2 ? co[4 + tau] : tab[GCS_CLS_DINV + 5 * grp + tau] * rS[5 * b + tau] + co[9 + 5 * grp + tau];
}

// consensus target of scalar c of half-edge h (block descriptor `info`) before the dual is added:  (B z_e)[c]
GCS_DEV double gcs_target_z(const GcsStateView &St, const GcsPerfTables &T, int e, int c, int info) {
    double zc = St.z[5 * (size_t)e + c];
    if (T.edge_delta && ((info >> 8) & 3) == 1 && (c == 2 || c == 3))      // tail side, second point: p2 - y delta_e
        zc -= T.edge_delta[2 * (size_t)e + c - 2] * St.z[5 * (size_t)e + 4];
    return zc;
}


#if !defined(GCS_EMULATE) && defined(__CUDACC__)
// the thread that issues and waits for the bulk copies of the tiles after the first (bulk groups belong to the thread that
// commits them): lane 0 of the last warp, which has no vertex in P3 - P5 when a tile has fewer vertices than the block has warps
#define GCS_COPY_THREAD (blockDim.x - 32)
// P0 (one thread): the bulk copies that stage tile `tile` into the stage buffer B; completion is signalled on `bar`
__device__ __forceinline__ void gcs_perf_stage(const GcsPerfTables &T, const GcsPerfLayout &L, double *B, int tile, unsigned long long *bar) {
    const int *tr = T.tile_rec + 8 * (size_t)tile;
    const int v0 = tr[0], nvt = tr[1], b0 = tr[2], nb = tr[3], c0 = tr[4], ncone = tr[5];
    gcs_mbar_expect_tx(bar, (unsigned)(sizeof(double) * (12 * nb + 2 * nvt + GCS_CONE_REC * ncone) + sizeof(int) * (GCS_VI_N * nvt + 4 * nb + 8)));
    gcs_bulk_g2s(B + L.tr, tr, (unsigned)(sizeof(int) * 8), bar);
    gcs_bulk_g2s(B + L.vi, T.vrec + GCS_VI_N * (size_t)v0, (unsigned)(sizeof(int) * GCS_VI_N * nvt), bar);
    if (nb) gcs_bulk_g2s(B + L.bi, T.blk_rec + 4 * (size_t)b0, (unsigned)(sizeof(int) * 4 * nb), bar);
    if (nb) gcs_bulk_g2s(B + L.tS, T.tstate + 12 * (size_t)b0, (unsigned)(sizeof(double) * 12 * nb), bar);
    gcs_bulk_g2s(B + L.tnS, T.tn + 2 * (size_t)v0, (unsigned)(sizeof(double) * 2 * nvt), bar);
    if (ncone) gcs_bulk_g2s(B + L.cone, T.cone + GCS_CONE_REC * (size_t)c0, (unsigned)(sizeof(double) * GCS_CONE_REC * ncone), bar);
}
#endif

// c-step of one pair from its projection q:  d = c - lam replaces t in place, e = (1 - alpha) c + lam waits for the t-step
GCS_DEV void gcs_cstep_store(double *t, double *e, double t0, double t1, double t2, double q0, double q1, double q2, double ms, double alpha) {
    const double l0 = ms * (t0 - q0), l1 = ms * (t1 - q1), l2 = ms * (t2 - q2);
    t[0] = q0 - l0; t[1] = q1 - l1; t[2] = q2 - l2;
    e[0] = (1.0 - alpha) * q0 + l0; e[1] = (1.0 - alpha) * q1 + l1; e[2] = (1.0 - alpha) * q2 + l2;
}

// x-update of one tile of vertices in perf mode.  S: work arrays, B: the tile's staged arrays (device build: already filled by
// gcs_perf_stage and waited for; the new state leaves B by bulk stores of GCS_COPY_THREAD).  Device build: after the tile's first
// barrier GCS_COPY_THREAD waits until the stores of the previous tile have read Bn and stages tile `next` into it (signalled on
// bar_next): the stores drain during P1 - P2 and the loads land during P3 - P8, without holding the block at a barrier.
// INNER: also accumulate (into `rin`, per thread) the squared inner residual  |(M u + m0) - c|^2  of the tile's pairs after the
// last pass — compiled in only for the kernel variant the host switches to near convergence (gcsadmm_run), so the throughput
// path carries none of it.
// BATCH: the tile's vertices belong to several problems, each with its own control block ctrl_all[GCS_VI_ACTIVE of the vertex]
// (rho, mu_scale, stop flag per vertex); otherwise one problem, ctrl_all.
template <bool INNER, bool BATCH>
GCS_DEV void gcs_perf_tile(const GcsGraphView &G, const GcsStateView &St, const GcsPerfTables &T, const GcsPerfLayout &L,
                           double *S, double *B, int tile, Ctrl *ctrl_all, double &rin,
                           double *Bn, int next, unsigned long long *bar_next) {
    // single problem: rho / mu_scale are uniform — loaded once into registers here
    // (batched problems: per vertex, from its problem's control block)
    const double rho_u = ctrl_all->rho, ms_u = ctrl_all->mu_scale;
#define RHO(vl) (BATCH ? vd[2 * (vl)] : rho_u)
#define MSC(vl) (BATCH ? vd[2 * (vl) + 1] : ms_u)
#define ACT(vl) (!BATCH || vi[GCS_VI_N * (vl) + GCS_VI_ACTIVE])
#define ACT_W (!BATCH || w[GCS_VI_ACTIVE])
#if defined(GCS_EMULATE)
    const int *tr = T.tile_rec + 8 * (size_t)tile;
#else
    const int *tr = (const int *)(B + L.tr);       // staged with the rest of the tile
#endif
    const int v0 = tr[0], nvt = tr[1], b0 = tr[2], nb = tr[3], h0 = tr[6], nhe = tr[7] & 0x3fffffff;
    const bool has_zero = (tr[7] >> 30) & 1;
    double *tS = B + L.tS, *eS = S + L.eS, *coneS = B + L.cone, *tnS = B + L.tnS, *enS = S + L.enS, *TS = S + L.T, *rS = S + L.r;
    double *cin = S + L.cin, *cout = S + L.cout, *vd = S + L.vd;
    int *vi = (int *)(B + L.vi), *brec = (int *)(B + L.bi);
#define bhe(b) brec[4 * (b)]
#define binfo(b) brec[4 * (b) + 1]
#define bedge(b) brec[4 * (b) + 2]
#if defined(GCS_EMULATE)
    {   // ---- P0 on the host: the tile's contiguous state, cone records and descriptors
        const int c0 = tr[4], ncone = tr[5];
        memcpy(tS, T.tstate + 12 * (size_t)b0, sizeof(double) * 12 * nb);
        memcpy(tnS, T.tn + 2 * (size_t)v0, sizeof(double) * 2 * nvt);
        memcpy(coneS, T.cone + GCS_CONE_REC * (size_t)c0, sizeof(double) * GCS_CONE_REC * ncone);
        memcpy(vi, T.vrec + GCS_VI_N * (size_t)v0, sizeof(int) * GCS_VI_N * nvt);
        memcpy(brec, T.blk_rec + 4 * (size_t)b0, sizeof(int) * 4 * nb);
    }
#endif
    // Until the first barrier of a pass the block works as two groups: the first half of the warps does the c-step, two pairs per
    // thread; the others issue the gathers of the consensus targets, answer the forced-zero half-edges and do the path-length item
    // meanwhile.  A one-warp block does both, one after the other.
#if defined(GCS_EMULATE)
    const bool cgrp = true, ggrp = true;
    const int cid = 0, cn = 1, gid0 = 0, gn = 1;
#else
    const int nw = blockDim.x >> 5, cn = 32 * ((nw + 1) >> 1);
    const bool cgrp = (int)threadIdx.x < cn, ggrp = !cgrp || nw == 1;
    const int cid = threadIdx.x, gid0 = nw == 1 ? (int)threadIdx.x : (int)threadIdx.x - cn, gn = nw == 1 ? cn : (int)blockDim.x - cn;
#endif
    if (BATCH) {
        GCS_CTA_LOOP(i, nvt) {     // rho, mu_scale and the stop flag of the vertex's problem
            int *w = vi + GCS_VI_N * i;
            Ctrl *c = ctrl_all + w[GCS_VI_ACTIVE];
            w[GCS_VI_ACTIVE] = !(c->stop && !c->ignore_stop);
            vd[2 * i] = c->rho; vd[2 * i + 1] = c->mu_scale;
            if (w[GCS_VI_ACTIVE] && w[GCS_VI_NB]) {
#if defined(GCS_EMULATE)
                c->inner_iters += (unsigned long long)T.inner_iters;
#else
                atomicAdd(&c->inner_iters, (unsigned long long)T.inner_iters);
#endif
            }
        }
        GCS_CTA_SYNC();     // vd / ACTIVE of every vertex of the tile are in shared memory
    }
    const double alpha = T.alpha, kappa = T.kappa;
    for (int it = 0; it < T.inner_iters; ++it) {
        const bool last = it + 1 == T.inner_iters;
        if (ggrp) {
#if defined(GCS_EMULATE)
            const int gid = gid0;
#else
            // opaque inside the pass: otherwise the gather slots' block / scalar indices are hoisted out of the tile and pass
            // loops and held in registers through every phase (spills at 64 registers)
            int gid = gid0;
            asm volatile("" : "+r"(gid));
#endif
            if (it == 0 && has_zero) for (int q = gid; q < 5 * nhe; q += gn) {
                const int hl = q / 5, c = q - 5 * hl, h = h0 + hl, f = G.he_flags[h];
                if (!(f & GCS_HE_ZERO)) continue;
                int vl = 0;
                while (vl + 1 < nvt && vi[GCS_VI_N * (vl + 1) + GCS_VI_HE] <= hl) ++vl;
                if (!ACT(vl)) continue;
                // own copy and flow are 0; an incoming edge's "other copy" first point is unconstrained and sits on its target
                double x = 0.0;
                if (c < 2 && !(f & GCS_HE_OUT)) x = St.z[5 * (size_t)G.he_edge[h] + c] + MSC(vl) * St.mu[5 * (size_t)h + c];
                St.xc[5 * (size_t)h + c] = x;
            }
            for (int i = gid; i < nvt; i += gn) {                           // path-length item: block soft-threshold, threshold 1 / sigma
                const int *w = vi + GCS_VI_N * i;
                if (!ACT_W || !w[GCS_VI_NB]) continue;
                const double ms = it ? 1.0 : MSC(i);
                const double sigma = kappa * RHO(i) * ms;                      // the threshold of the pass that produced t (rho before its rescale)
                const double a0 = tnS[2 * i], a1 = tnS[2 * i + 1], nrm = hypot(a0, a1);
                const double sc = nrm > 0.0 ? fmax(0.0, 1.0 - 1.0 / (sigma * nrm)) : 0.0;
                const double q0 = sc * a0, q1 = sc * a1, l0 = ms * (a0 - q0), l1 = ms * (a1 - q1);
                tnS[2 * i] = q0 - l0; tnS[2 * i + 1] = q1 - l1;
                enS[2 * i] = (1.0 - alpha) * q0 + l0; enS[2 * i + 1] = (1.0 - alpha) * q1 + l1;
            }
            // ---- P1 (first pass): consensus targets  T = z_e + mu_h  of the live half-edges.  Device build: the GCS_PF gathers of a
            // thread are all issued before the first is used (their DRAM / L2 latency overlaps), while the other warps project
#if !defined(GCS_EMULATE)
            double pz[GCS_PF], pm[GCS_PF];
            if (it == 0) {
#pragma unroll
                for (int j = 0; j < GCS_PF; ++j) {
                    const int q = gid + j * gn;
                    pz[j] = 0.0; pm[j] = 0.0;
                    if (q < 5 * nb) {
                        const int b = q / 5, c = q - 5 * b, h = bhe(b);
                        if (h >= 0) { pz[j] = gcs_target_z(St, T, bedge(b), c, binfo(b)); pm[j] = St.mu[5 * (size_t)h + c]; }
                    }
                }
            }
#endif
            if (it == 0) {
#if !defined(GCS_EMULATE)
#pragma unroll
                for (int j = 0; j < GCS_PF; ++j) {
                    const int q = gid + j * gn;
                    if (q < 5 * nb) TS[q] = pz[j] + MSC(binfo(q / 5) & 255) * pm[j];
                }
                for (int q = gid + GCS_PF * gn; q < 5 * nb; q += gn) {     // small blocks: the targets beyond the prefetched ones
#else
                for (int q = 0; q < 5 * nb; ++q) {
#endif
                    const int b = q / 5, c = q - 5 * b, h = bhe(b), vl = binfo(b) & 255;
                    if (h < 0 || !ACT(vl)) continue;
                    TS[q] = gcs_target_z(St, T, bedge(b), c, binfo(b)) + MSC(vl) * St.mu[5 * (size_t)h + c];
                }
            }
        }
        // ---- P2: c-step.  Item j = point i of block b (j = 2 b + i): its fam-0 and fam-1 pairs p = 2 j, 2 j + 1 belong to one vertex
        // and are projected onto its cone in one pass over the records ('s' / 't' blocks have no fam-1 pair: no C2 / C4)
        if (cgrp) for (int j = cid; j < 2 * nb; j += cn) {
            const int b = j >> 1, info = binfo(b), vl = info & 255;
            const int *w = vi + GCS_VI_N * vl;
            if (!ACT_W) continue;
            const double ms = it ? 1.0 : MSC(vl);                      // sigma = kappa rho: lam rescales with mu (:705 / :708)
            const double *cone = coneS + GCS_CONE_REC * w[GCS_VI_CONE];
            double *t = tS + 6 * j, *e = eS + 6 * j;
            const double t0 = t[0], t1 = t[1], t2 = t[2];
            double q0, q1, q2;
            if ((info >> 10) & 1) gcs_cone_project(cone, w[GCS_VI_NV], t0, t1, t2, q0, q1, q2);
            else {
                const double t3 = t[3], t4 = t[4], t5 = t[5];
                double q3, q4, q5;
                gcs_cone_project2(cone, w[GCS_VI_NV], t0, t1, t2, t3, t4, t5, q0, q1, q2, q3, q4, q5);
                gcs_cstep_store(t + 3, e + 3, t3, t4, t5, q3, q4, q5, ms, alpha);
            }
            gcs_cstep_store(t, e, t0, t1, t2, q0, q1, q2, ms, alpha);
        }
        GCS_CTA_SYNC();
#if !defined(GCS_EMULATE)
        if (it == 0 && threadIdx.x == GCS_COPY_THREAD && next < T.ntiles) {
            gcs_bulk_wait_read();      // the stores of the previous tile have finished reading Bn
            gcs_perf_stage(T, L, Bn, next, bar_next);
        }
#endif
        // ---- P3 + P4 + P5, one warp per vertex (device build), so that only warp barriers separate them:
        //   P3  right-hand side of the v-step in units of rho,  r = S'T - (eps / rho) e_y + kappa M'(d - m0),  for the vertex's blocks
        //   P4  the 19 inputs of its extended core (r_x, r_z, r_yv, sums of r over the in- and the out-blocks)
        //   P5  (x, z_v, y_v, beta_in, beta_out) = G (inputs) + g0
#if defined(GCS_EMULATE)
        for (int vl = 0; vl < nvt; ++vl) {
            const int *w = vi + GCS_VI_N * vl;
            if (!ACT_W || !w[GCS_VI_NB]) continue;
            for (int q = 5 * w[GCS_VI_BLK]; q < 5 * (w[GCS_VI_BLK] + w[GCS_VI_NB]); ++q) rS[q] = gcs_rhs(T, tS, TS, tnS, brec, q, vl, RHO(vl), kappa);
            for (int k = 0; k < GCS_NCX; ++k) cin[GCS_NCX * vl + k] = gcs_core_input(tS, rS, w, k, kappa);
            for (int k = 0; k < GCS_NCX; ++k) cout[GCS_NCX * vl + k] = gcs_core_output(T.cls_tab + (size_t)GCS_CLS_STRIDE * w[GCS_VI_CLS], cin + GCS_NCX * vl, k);
        }
#else
        for (int vl = threadIdx.x >> 5; vl < nvt; vl += blockDim.x >> 5) {
            const int *w = vi + GCS_VI_N * vl;
            const int k = threadIdx.x & 31;
            if (!ACT_W || !w[GCS_VI_NB]) continue;                    // warp-uniform
            for (int q = 5 * w[GCS_VI_BLK] + k; q < 5 * (w[GCS_VI_BLK] + w[GCS_VI_NB]); q += 32) rS[q] = gcs_rhs(T, tS, TS, tnS, brec, q, vl, RHO(vl), kappa);
            __syncwarp();
            if (k < GCS_NCX) cin[GCS_NCX * vl + k] = gcs_core_input(tS, rS, w, k, kappa);
            __syncwarp();
            if (k < GCS_NCX) cout[GCS_NCX * vl + k] = gcs_core_output(T.cls_tab + (size_t)GCS_CLS_STRIDE * w[GCS_VI_CLS], cin + GCS_NCX * vl, k);
        }
#endif
        GCS_CTA_SYNC();
        // ---- P7: block variables  u = dinv r + beta  (evaluated where they are used), t-step  t = alpha (M u + m0) + e;  on the
        // last pass the vertex outputs and the consensus copies xc in edge-canonical order (:492-522)
        GCS_CTA_LOOP(p, 4 * nb) {
            const int b = p >> 2, i = (p >> 1) & 1, fam = p & 1, info = binfo(b), vl = info & 255;
            const int *w = vi + GCS_VI_N * vl;
            if (!ACT_W || ((info >> 10) & fam)) continue;
            const double *co = cout + GCS_NCX * vl, *tab = T.cls_tab + (size_t)GCS_CLS_STRIDE * w[GCS_VI_CLS], *e = eS + 3 * p;
            double p0 = gcs_block_u(rS, co, tab, info, b, 2 * i), p1 = gcs_block_u(rS, co, tab, info, b, 2 * i + 1), p2 = gcs_block_u(rS, co, tab, info, b, 4);
            if (fam) { p0 = co[2 * i] - p0; p1 = co[2 * i + 1] - p1; p2 = 1.0 - p2; }
            double *t = tS + 3 * p;
            if (INNER && last) {      // inner residual  (M u + m0) - c  of the pair:  t holds d = c - lam, e = (1 - alpha) c + lam  =>  c = (d + e) / (2 - alpha)
                const double ic = 1.0 / (2.0 - alpha), r0 = p0 - ic * (t[0] + e[0]), r1 = p1 - ic * (t[1] + e[1]), r2_ = p2 - ic * (t[2] + e[2]);
                rin += r0 * r0 + r1 * r1 + r2_ * r2_;
            }
            t[0] = alpha * p0 + e[0]; t[1] = alpha * p1 + e[1]; t[2] = alpha * p2 + e[2];
        }
        GCS_CTA_LOOP(i, nvt) {
            const int *w = vi + GCS_VI_N * i;
            if (!ACT_W || !w[GCS_VI_NB]) continue;
            const double *zz = cout + GCS_NCX * i + 4;
            if (INNER && last) {
                const double ic = 1.0 / (2.0 - alpha), r0 = (zz[0] - zz[2]) - ic * (tnS[2 * i] + enS[2 * i]), r1 = (zz[1] - zz[3]) - ic * (tnS[2 * i + 1] + enS[2 * i + 1]);
                rin += r0 * r0 + r1 * r1;
            }
            tnS[2 * i] = alpha * (zz[0] - zz[2]) + enS[2 * i]; tnS[2 * i + 1] = alpha * (zz[1] - zz[3]) + enS[2 * i + 1];
        }
        if (last) {
            GCS_CTA_LOOP(q, 9 * nvt) {
                const int vl = q / 9, k = q - 9 * vl;
                const int *w = vi + GCS_VI_N * vl;
                if (!ACT_W || !w[GCS_VI_NB]) continue;
                double val = cout[GCS_NCX * vl + k];
                const size_t v = (size_t)(v0 + vl);
                if (T.edge_delta && k < 8)          // local frames: back to global coordinates  x = x' + c_v,  z_v = z_v' + y_v c_v
                    val += (k < 4 ? 1.0 : cout[GCS_NCX * vl + 8]) * G.cent[2 * v + (k & 1)];
                if (k < 4) St.x_v[4 * v + k] = val; else if (k < 8) St.z_v[4 * v + k - 4] = val; else St.y_v[v] = val;
            }
            GCS_CTA_LOOP(q, 5 * nb) {
                const int b = q / 5, c = q - 5 * b, h = bhe(b), info = binfo(b), vl = info & 255;
                const int *w = vi + GCS_VI_N * vl;
                if (h < 0 || !ACT_W) continue;
                const double *co = cout + GCS_NCX * vl, *tab = T.cls_tab + (size_t)GCS_CLS_STRIDE * w[GCS_VI_CLS];
                double x;
                if ((info >> 8) & 1) x = gcs_block_u(rS, co, tab, info, b, c);      // out-edge: own first point | other's first point == own second point (C5)
                else x = c < 2 ? TS[q] : gcs_block_u(rS, co, tab, info, b, c < 4 ? c - 2 : 4);   // in-edge: other's first point is free -> its target | own first point
                St.xc[5 * (size_t)h + c] = x;
            }
        }
        if (!last) GCS_CTA_SYNC();     // (after the last pass P8's barrier follows)
    }
    // ---- P8: the new state goes back with bulk stores (GCS_COPY_THREAD waits for them before it restages B)
#if defined(GCS_EMULATE)
    memcpy(T.tstate + 12 * (size_t)b0, tS, sizeof(double) * 12 * nb);
    memcpy(T.tn + 2 * (size_t)v0, tnS, sizeof(double) * 2 * nvt);
#else
    gcs_fence_async_smem();
    GCS_CTA_SYNC();
    if (threadIdx.x == GCS_COPY_THREAD) {
        if (nb) gcs_bulk_s2g(T.tstate + 12 * (size_t)b0, tS, (unsigned)(sizeof(double) * 12 * nb));
        gcs_bulk_s2g(T.tn + 2 * (size_t)v0, tnS, (unsigned)(sizeof(double) * 2 * nvt));
        gcs_bulk_commit();
    }
#endif
#undef bhe
#undef binfo
#undef bedge
#undef RHO
#undef MSC
#undef ACT
#undef ACT_W
}
