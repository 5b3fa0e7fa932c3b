/*
 * gcsadmm.h — C-ABI of libgcsadmm.so: the full-vertex-split ADMM iteration for shortest paths in
 * graphs of convex sets, as hand-written CUDA for sm_100a (B200).
 *
 * Drop-in scope.  The reference (Michaelszeng/GCS-ADMM) has no function API or FFI: its hot path is
 * the module-level loop of admm_solver_v3.py.  Each entry point below names the reference code it
 * replaces (file:line relative to the reference repository):
 *
 *   gcsadmm_create        ConsensusManager.__init__ + build_A_B_c_consensus_matrices   admm_solver_v3.py:68-198, :340-349
 *                         (variable/consensus bookkeeping; here: upload of the half-edge CSR layout)
 *   gcsadmm_vertex_update parallel_vertex_update / vertex_update / SolveInParallel     admm_solver_v3.py:352-540
 *   gcsadmm_edge_update   parallel_edge_update, dual_update, evaluate_*_residual,      admm_solver_v3.py:543-614, :690-713
 *                         eps_pri, eps_dual, rho adaptation, stop test (fused)
 *   gcsadmm_step / _run   the `while it <= MAX_IT` loop                                 admm_solver_v3.py:655-733
 *   gcsadmm_get_history   rho_seq / pri_res_seq / dual_res_seq                          admm_solver_v3.py:637-639, :771-773
 *   gcsadmm_get_solution  x_v_sol / y_v_sol / y_e_e_sol / z_v_sol slicing               admm_solver_v3.py:745-748
 *   gcsadmm_solve_host    the whole loop from host buffers to host buffers (what solve() calls)
 *
 * Conventions: plain C types; the caller owns every host buffer; the library owns device memory.
 * Every call returns 0 on success and a negative GCS_E_* code on failure (never throws, never
 * aborts); gcsadmm_last_error() returns the message of the last failure on the calling thread.
 * A handle is bound to one CUDA device and one stream and is not thread-safe; independent handles
 * may be used from different threads.  All floating point data is IEEE fp64; n (the ambient
 * dimension) must be 2.
 *
 * Data layout (see DESIGN.md).  Vertices in the order of the reference's vertex list V; directed
 * edges in the order of its edge list E; the half-edges of vertex v are he_off[v]..he_off[v+1] in
 * the reference's per-vertex order I_v_in[v] + I_v_out[v] (admm_solver_v3.py:105-116).  Each
 * half-edge h owns 5 consensus scalars, stored in edge-canonical order
 * xc[h] = (copy of z_u^e[:2], copy of z_w^e[:2], copy of y_e) for e = (u, w); z[e] has the same order.
 */
#ifndef GCSADMM_H
#define GCSADMM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GCS_OK 0
#define GCS_E_INVALID (-1)    /* bad argument / unsupported problem (n != 2, degree too large, ...) */
#define GCS_E_CUDA (-2)       /* CUDA runtime error (message has the CUDA error string) */
#define GCS_E_NOMEM (-3)
#define GCS_E_DIVERGED (-4)   /* non-finite residuals (reference: "BREAKING FOR Divergence") */

#define GCS_HE_FLAG_OUT 1     /* he_flags bit0: the owner is the edge's tail (outgoing half-edge) */
#define GCS_HE_FLAG_ZERO 2    /* he_flags bit1: flow forced to zero by the presolve */

typedef struct GcsHandle GcsHandle;

typedef struct GcsGraph {
    int32_t nV;                  /* local vertices */
    int32_t nE;                  /* local directed edges (incident to a local vertex) */
    int32_t n;                   /* ambient dimension, must be 2 */
    int32_t nH_own;              /* half-edges owned by local vertices (== he_off[nV]) */
    int32_t nH_ghost;            /* half-edge slots mirrored from another rank (0 on a single GPU) */
    const int32_t *poly_off;     /* [nV+1] rows of polytope v are poly_off[v]..poly_off[v+1] */
    const double *polyA;         /* [sum m][2] */
    const double *polyb;         /* [sum m] */
    const int32_t *he_off;       /* [nV+1] */
    const int32_t *he_edge;      /* [nH_own] local edge id of each half-edge */
    const uint8_t *he_flags;     /* [nH_own] GCS_HE_FLAG_* */
    const int32_t *edge_he_tail; /* [nE] half-edge slot (own or ghost) of the edge at its tail */
    const int32_t *edge_he_head; /* [nE] ... at its head */
    const uint8_t *edge_counted; /* [nE] or NULL: 1 if this rank accounts the edge in the z-norms (all 1 when NULL) */
    const uint8_t *vtype;        /* [nV] 0 generic, 1 source, 2 target, 3 no flow possible */
    const double *cent;          /* [nV][2] a strictly interior point of each polytope */
    int64_t n_x_global;          /* len(x_global) = 9|V| + 18|E| of the WHOLE graph (0: derive from nV, nE) */
    int64_t n_mu_global;         /* len(mu_global) = 10|E| of the whole graph (0: derive) */
    /* independent problems packed block-diagonally (batched queries): vertices / edges of problem p are the
     * contiguous ranges prob_voff[p]..prob_voff[p+1], prob_eoff[p]..prob_eoff[p+1]; each problem keeps its own
     * residuals, rho and stop decision.  nP <= 1: a single graph (pointers may be NULL). */
    int32_t nP;
    const int32_t *prob_voff;    /* [nP+1] */
    const int32_t *prob_eoff;    /* [nP+1] */
} GcsGraph;

typedef struct GcsParams {       /* literals of admm_solver_v3.py:621-651 */
    double rho0;                 /* 1 */
    double tau_incr, tau_decr;   /* 2, 2 */
    double nu;                   /* 10 */
    double frac;                 /* 0.1: rho adapts only while it < frac * max_it */
    double eps_abs, eps_rel;     /* 1e-4, 1e-3 */
    int32_t max_it;              /* 1000 */
    double inner_tol;            /* interior-point tolerance of the vertex programs (1e-8: gap and 10x that on the dual residual; MOSEK's default is 1e-8) */
    int32_t inner_max_iter;      /* 60 */
    int32_t check_every;         /* host polls the stop flag every this many iterations (8) */
    int32_t abs_stop;            /* 0: reference stop rule; 1: stop when max(pri, dual) < abs_tol */
    double abs_tol;              /* 1e-4 (metric "time to residual 1e-4") */
    double warm_theta;           /* interior-point warm start: previous optimum pulled this fraction towards the
                                    analytic centre (1e-3); 0 = cold start every iteration */
    double zero_tol;             /* a vertex whose consensus targets are all <= zero_tol in magnitude gets the zero
                                    solution without a solve (prox maps are non-expansive); 1e-12, 0 = exact zeros only */
    double outer_alpha;          /* over-relaxation of the consensus step (1 = the reference's plain ADMM; 1.5-1.8 is the usual
                                    accelerated choice, Boyd et al. 3.4.3) — perf-mode runs only, the parity mode keeps 1 */
    int32_t use_graph;           /* 1: gcsadmm_run replays one CUDA graph per chunk of check_every iterations (own stream only) */
    int32_t adapt_every;         /* 1 = the reference's per-iteration rho test (:703-709); N > 1: tested on every N-th iteration only */
    int32_t stop_ref;            /* abs_stop in perf mode with local frames: 0 (default) = the test uses the residuals of the local-frame
                                    formulation (translation-invariant); 1 = it uses the reference's definitions, i.e. the residuals in global
                                    coordinates (GcsStatus.pri_res_ref / dual_res_ref) — an absolute threshold on those depends on where the
                                    map's origin is: a flow mismatch eps at position c counts as eps * |c| */
} GcsParams;

typedef struct GcsStatus {
    int32_t iterations;          /* `it` of the last executed pass */
    int32_t converged;           /* reference `opt` */
    int32_t diverged;
    int32_t inner_fail;          /* vertex programs that ended above the noise-floor acceptance */
    int64_t inner_iters;         /* interior-point iterations summed over all vertex programs */
    int64_t skipped;             /* vertex programs answered by the zero-target shortcut */
    double rho, pri_res, dual_res, eps_pri, eps_dual;
    double inner_res;            /* perf mode: residual of the vertex programs' own cone constraints, |(M u + m0) - c| over all pairs
                                    (0 in the exact mode); part of the abs_stop test */
    double pri_res_ref, dual_res_ref;   /* the residuals by the reference's definitions (:598, :602), i.e. in global coordinates.  Equal to
                                    pri_res / dual_res except in perf mode with local frames near convergence, where the check variant
                                    of the edge kernel evaluates them (a flow mismatch far from the origin is a large position mismatch);
                                    the abs_stop test uses these */
} GcsStatus;

const char *gcsadmm_version(void);
const char *gcsadmm_last_error(void);
int gcsadmm_device_count(void);
void gcsadmm_default_params(GcsParams *p);

int gcsadmm_create(const GcsGraph *g, const GcsParams *p, int device, GcsHandle **out);
int gcsadmm_destroy(GcsHandle *h);
/* external != 0: enqueue on the caller's CUDA stream (e.g. torch's current stream; NULL = the legacy default
 * stream); external == 0: back to the handle's own stream */
int gcsadmm_set_stream(GcsHandle *h, void *cuda_stream, int external);

/* whole iterations */
int gcsadmm_run(GcsHandle *h, int max_iters, GcsStatus *st);   /* until the stop rule fires or max_iters passes */
int gcsadmm_step(GcsHandle *h, int k);                         /* exactly k passes, stop rule evaluated but ignored */
int gcsadmm_get_status(GcsHandle *h, GcsStatus *st);            /* batched handle: worst residuals, max iterations, all-converged */
int gcsadmm_get_problem_status(GcsHandle *h, int problem, GcsStatus *st);

/* the individual kernels (per-kernel parity tests, multi-GPU driver) */
int gcsadmm_vertex_update(GcsHandle *h);                       /* K1 */
int gcsadmm_edge_update(GcsHandle *h);                         /* K2-K4: z, mu, partial sums -> sums[8] on the device */
int gcsadmm_control(GcsHandle *h);                             /* K5: consumes sums[8]: residuals, rho, stop, history */
int gcsadmm_sums_device_ptr(GcsHandle *h, void **dev_ptr);     /* 8 doubles; all-reduce them between edge_update and control */
int gcsadmm_xc_device_ptr(GcsHandle *h, void **dev_ptr);       /* [(nH_own + nH_ghost)][5] doubles (halo pack / unpack) */

/* results */
int gcsadmm_get_history(GcsHandle *h, double *rho_seq, double *pri_seq, double *dual_seq, int cap); /* returns count or <0 */
int gcsadmm_get_problem_history(GcsHandle *h, int problem, double *rho_seq, double *pri_seq, double *dual_seq, int cap);
int gcsadmm_get_solution(GcsHandle *h, double *x_v, double *z_v, double *y_v, double *z_e);         /* any may be NULL */
int gcsadmm_get_state(GcsHandle *h, double *xc, double *mu, double *z, double *rho, int *it);
int gcsadmm_set_state(GcsHandle *h, const double *xc, const double *mu, const double *z, double rho, int it);

/* timing: k passes bracketed by CUDA events on the handle's stream; ms_k1 / ms_edge may be NULL */
int gcsadmm_time_steps(GcsHandle *h, int k, float *ms_total, float *ms_k1, float *ms_edge);

/* timing window (bench protocol): k iterations enqueued back to back, each preceded by an in-stream L2 eviction of flush_bytes
   (0: none) outside its own event pair; no host round trip between iterations.  ms_iter[k]; ms_k1[k] may be NULL */
int gcsadmm_time_window(GcsHandle *h, int k, long long flush_bytes, float *ms_iter, float *ms_k1);

/* evicts L2 between timed iterations (bench hygiene): overwrites a scratch buffer of `bytes` (0: 256 MiB) */
int gcsadmm_flush_l2(GcsHandle *h, long long bytes);

/* one call from host buffers to host buffers: create, run, copy back, destroy */
int gcsadmm_solve_host(const GcsGraph *g, const GcsParams *p, int device, int max_iters, GcsStatus *st,
                       double *x_v, double *z_v, double *y_v, double *z_e,
                       double *rho_seq, double *pri_seq, double *dual_seq, int hist_cap);

/* `perf` mode of the x-update (K1): K warm-started closed-form splitting iterations per ADMM iteration instead of
 * an exact interior-point solve (gcs-admm_b200/csrc/vertex_perf.cuh; north_star: "fixed-iteration inner projection /
 * primal-dual scheme").  Same fixed point, different trajectory: validated at convergence against the classic relaxation
 * optimum, not iteration by iteration.  All tables are built by the host (gcs-admm_b200/perf.py perf_tables). */
typedef struct GcsPerfConfig {
    int32_t inner_iters;         /* K */
    double alpha;                /* over-relaxation of the inner splitting (1.6) */
    double kappa;                /* sigma = kappa * rho */
    int32_t n_classes;           /* vertex classes (type, #live in-edges, #live out-edges) */
    const int32_t *vclass;       /* [nV] class of each vertex (-1 for vtype 3) */
    const double *cls_tab;       /* [n_classes][392]: the class's v-step in structured form: G TRANSPOSED (19 x 19: [19 j + k] = G[k, j]) | g0 (19) | dinv (2 x 5) | pad */
    const int32_t *cone_off;     /* [nV+1] polygon vertices of each region, counter-clockwise */
    const double *cone;          /* 12 doubles per polygon vertex: Vx, Vy, unit outward normal (3) of the cone face to the
                                    next vertex's ray, 1 / (Vx^2 + Vy^2 + 1), the face's two in-plane sector normals (3 + 3) */
    int32_t n_blocks;            /* blocks = live half-edges + one (z_v, y_v) block per live vertex */
    const int32_t *blk_off;      /* [nV+1]; a vertex's blocks are its in-blocks, then its out-blocks, then its z-block
                                    (any other order is refused with GCS_E_INVALID) */
    const int32_t *blk_he;       /* [n_blocks] half-edge of the block, -1 for the (z_v, y_v) block */
    const int32_t *blk_info;     /* [n_blocks] bits 0-7 vertex index inside its tile | 8-9 group (0 in, 1 out, 2 z-block) | 10 terminal */
    int32_t n_tiles;             /* a tile = the consecutive vertices one thread block works on */
    const int32_t *tile_voff;    /* [n_tiles+1] */
    int32_t cap_blocks, cap_verts, cap_cone;   /* largest tile: blocks, vertices, cone records (sizes the shared memory) */
    int32_t threads;             /* threads per tile's thread block (0 = 256; a multiple of 32 up to 256 — pairs of the tile's blocks) */
    double theta;                /* penalty of the flow scalars = theta * rho (0 or 1: the reference's single rho) */
    const double *edge_delta;    /* NULL: global coordinates.  [nE][2] = cent[tail] - cent[head]: LOCAL FRAMES — every vertex program runs in
                                    coordinates centred on its own region (the cone records must be built from the shifted polygons), the two
                                    copies of an edge agree through x_head = z_e, x_tail = B_e z_e.  Same optimisation problem, a differently
                                    conditioned ADMM: the perspective variables y * (p - cent) stay O(region size) instead of O(|p|), which is
                                    what lets large maps converge (DESIGN.md section 5b).  x_v / z_v come back in global coordinates; xc, mu, z
                                    (get_state) are in the local frames */
    const double *edge_cent;     /* local frames: [nE][2] = cent[tail] (NULL: the residuals of the abs_stop test stay in local coordinates).
                                    With it the check variant of the edge kernel evaluates the residuals in GLOBAL coordinates, i.e. by the
                                    reference's own definitions (GcsStatus.pri_res_ref / dual_res_ref) */
} GcsPerfConfig;
int gcsadmm_enable_perf(GcsHandle *h, const GcsPerfConfig *cfg);
/* the warm-start state of the perf mode (t = c + lam of every pair, 12 doubles per block, and 2 doubles per vertex for the
 * path-length item): with gcsadmm_get_state / _set_state a run can be checkpointed and resumed from host buffers */
int gcsadmm_get_perf_state(GcsHandle *h, double *tstate, double *tn);
int gcsadmm_set_perf_state(GcsHandle *h, const double *tstate, const double *tn);

/* Multi-GPU over NVLink peer memory (one process per GPU of one box; the graph vertex-partitioned by the host layer, ghost
 * slots as in GcsGraph.nH_ghost).  After connecting, gcsadmm_step / gcsadmm_run execute the partitioned iteration with no
 * collective library call inside it: cut half-edges are stored straight into the neighbours' ghost slots, the 6 residual
 * sums straight into every rank's inbox, flags in peer memory order the steps (gcsadmm.cu "peer mode").  Every rank must run
 * the same number of iterations.
 *   gcsadmm_peer_export: writes 128 bytes (two CUDA IPC handles: the xc buffer, the flag / inbox block) for the caller to
 *                        all-gather over its own channel;
 *   gcsadmm_peer_connect: all_handles = the gathered [world][128] table; peer_nHown / peer_nHghost = every rank's sizes;
 *                        send_he[j] = own half-edge j-th item of the halo, send_rank[j] = destination rank, send_slot[j] = index
 *                        of its ghost slot at the destination (0-based inside the destination's ghost range). */
int gcsadmm_peer_export(GcsHandle *h, void *handles128);
int gcsadmm_peer_connect(GcsHandle *h, int rank, int world, const void *all_handles, const int32_t *peer_nHown, const int32_t *peer_nHghost,
                         int nsend, const int32_t *send_he, const int32_t *send_rank, const int32_t *send_slot);
int gcsadmm_peer_error(GcsHandle *h);                           /* 1 if a peer wait timed out (a rank fell out of step) */

/* bytes of shared memory one vertex program needs (diagnostics) */
int gcsadmm_scratch_bytes(int max_live_degree, int max_rows);

#ifdef __cplusplus
}
#endif
#endif
