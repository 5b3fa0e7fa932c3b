// libgcsadmm.so — kernels and C-ABI (include/gcsadmm.h).  sm_100a only; no CPU path.
//
//   K1  vertex_kernel        one warp per vertex, interior-point prox solve in shared memory   (vertex_update.cuh)
//       vertex_perf_kernel   perf mode: persistent thread blocks walking tiles of vertices with two bulk-copy stage buffers,
//                            closed-form splitting iterations (vertex_perf.cuh)
//   K2-5 edge_coop_kernel    single-GPU throughput path: a warp per 32 consecutive edges, records moved HBM <-> shared memory in
//                            coalesced passes; z-update, dual update of both half-edges, the squared norms; block partials (no
//                            atomics on the data), and the LAST block to finish reduces them in a fixed order and applies the
//                            control step: residuals, rho adaptation, stop rule, history (reference admm_solver_v3.py:697-713)
//       edge_frames_kernel   the same with one thread per edge: partitions with ghost slots (multi-GPU), the check variant that
//                            also evaluates the residuals in global coordinates
//       batched_edge_kernel  packed independent problems: one block per problem, its own control step
//   control_kernel           the same control step as a separate launch (NCCL multi-GPU: the sums are all-reduced in between);
//   peer_control_kernel      peer-memory multi-GPU: waits for every rank's sums, then the control step
// Every kernel returns immediately once the stop flag is set, so the host can enqueue iterations in
// chunks (one CUDA graph per chunk) and poll the control block once per chunk while keeping the reference's exact
// stop iteration.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <new>
#include <nvtx3/nvToolsExt.h>     // header-only NVTX v3: ranges are no-ops unless a profiler injects itself

// NVTX range of a C-ABI call (nsys / ncu --nvtx timelines): create, enable_perf, every chunk of iterations, the downloads
struct NvtxRange {
    explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

#include "../../include/gcsadmm.h"
#include "gcs_ctrl.h"
#include "vertex_update.cuh"
#include "vertex_perf.cuh"

#define GCS_VERSION "gcsadmm 0.1.0 (sm_100a)"
#define K1_MAX_WARPS 12  // __launch_bounds__(384): <= 168 registers/thread, 12 warps (18.8 KB of shared memory each) fill one SM
#define EDGE_THREADS 256

static thread_local char g_err[512] = "";
static int set_err(int code, const char *fmt, const char *a = "", const char *b = "") {
    snprintf(g_err, sizeof g_err, fmt, a, b);
    return code;
}
#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) return set_err(GCS_E_CUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

// ------------------------------------------------------------------------------------------ peer mode (types)
// Vertex-partitioned graph, one process per GPU of one NVSwitch box.  Per ADMM iteration k a rank
//   K1, then the halo push: the 5 consensus scalars of every cut half-edge are stored straight into the neighbour's ghost slot
//         (peer pointer over NVLink), system fence, then halo_flag[me] = k is raised in the neighbour's block.  Perf mode: the
//         LAST block of K1 to finish does it (ticket); exact mode: peer_push_kernel
//   edge kernel (fuse = 2): every block first spins until each neighbour's flag has reached k; the last block to finish stores
//         this rank's 6 partial sums into EVERY rank's block and raises sums_flag[me] = k
//   peer_control_kernel: waits for all ranks' sums, adds them in rank order (identical on every rank) and applies the control step
// No NCCL call and no host round trip inside the iteration; the three (exact mode: four) launches are replayed from one CUDA graph.
// Ghost slots and the sums inbox are double-buffered by the parity of k, so a fast neighbour's iteration k + 1 never
// overwrites what iteration k still reads (it cannot reach k + 2 before this rank has raised its k + 1 flags).
#define GCS_MAX_PEERS 8
#define GCS_PEER_TIMEOUT_NS 20000000000ull
struct PeerComm {
    int halo_flag[GCS_MAX_PEERS];             // written by peer p: its halo of iteration k has landed here
    int sums_flag[GCS_MAX_PEERS];
    double sums_in[2][GCS_MAX_PEERS][NSUMS];  // [parity][source rank]
    int k;                                    // peer iterations completed by this rank
    int error;                                // a wait timed out
};
struct PeerView {
    int rank, world;
    unsigned neighbours;                      // bit p: ranks exchanging halos with this one
    double *xc[GCS_MAX_PEERS];                // every rank's xc buffer (own included)
    PeerComm *comm[GCS_MAX_PEERS];            // every rank's block
    int nHown[GCS_MAX_PEERS], nHghost[GCS_MAX_PEERS];
};

// what a kernel needs to push this rank's cut half-edges to its neighbours (PV == nullptr: nothing to push)
struct PeerPush { const int *send_he, *send_rank, *send_slot; int nsend; const PeerView *PV; unsigned int *ticket; };

struct GcsHandle {
    int device;
    cudaStream_t stream, own_stream;
    GcsParams p;
    int nV, nE, nHown, nHghost;
    int nP;             // independent problems packed block-diagonally (1 = a single graph)
    long long n_x, n_mu;
    int dcap, mcap;
    GcsScratchLayout L;
    int k1_smem, k1_blocks, k1_warps, edge_blocks, edge_coop, coop_blocks;
    // device
    int *poly_off, *he_off, *he_edge, *edge_he_tail, *edge_he_head;
    double *polyA, *polyb, *cent;
    unsigned char *he_flags, *vtype, *edge_counted;
    int *vprob, *prob_eoff; long long *prob_nx, *prob_nmu;   // batched mode (nP > 1)
    int *he_prob_host;  // host: problem of each half-edge (batched mode)
    unsigned int *ticket;   // edge kernels: blocks finished in the current launch (the last one reduces + controls)
    unsigned int *push_ticket;   // perf K1 in peer mode: blocks finished (the last one pushes the halo)
    double *xc, *mu, *z, *x_v, *z_v, *y_v;
    double *ws;         // [nV][gcs_ws_stride] interior-point warm-start records (null when warm_theta == 0)
    double *partials;   // [edge_blocks][NSUMS]
    double *hist;       // [3][hist_cap]
    int hist_cap;
    Ctrl *ctrl;         // device
    Ctrl *ctrl_host;    // pinned
    cudaEvent_t ev[4];
    void *flush_buf; size_t flush_bytes;
    // perf mode (inexact x-update by K closed-form splitting iterations)
    int perf_on, perf_smem, perf_threads, perf_grid;
    int inner_on;       // perf mode: the K1 variant that also produces the inner residual is in use (switched on by gcsadmm_run near convergence)
    GcsPerfLayout PL;
    GcsPerfTables PT;
    long long perf_nblocks;
    int *p_vclass, *p_cone_off, *p_blk_off, *p_blk_rec, *p_vrec, *p_tile_rec; double *p_cls_tab, *p_cone, *p_tstate, *p_tn, *p_edge_delta, *p_edge_cent, *p_tile_res;
    // one CUDA graph per chunk of `check_every` iterations (own stream only)
    cudaGraphExec_t graph_exec; int graph_iters;
    // peer mode (multi-GPU over NVLink peer memory, one process per GPU): see the "peer mode" section
    int peer_on, rank, world, nsend;
    PeerView PV; PeerView *PV_dev;        // host copy / device copy (the kernels index it at run time)
    PeerComm *comm;                       // own block (peers write their flags / partial sums into it)
    void *ipc_opened[2 * GCS_MAX_PEERS];  // mappings of the other ranks' xc / comm blocks
    int *send_he, *send_rank, *send_slot;
};

// ------------------------------------------------------------------------------------------ K1
__global__ void __launch_bounds__(K1_MAX_WARPS * 32)
vertex_kernel(GcsGraphView G, GcsStateView St, Ctrl *ctrl_all, const int *__restrict__ vprob, GcsScratchLayout L, double tol, int max_iter) {
    extern __shared__ double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int v = blockIdx.x * (blockDim.x >> 5) + warp;
    if (v >= G.nV) return;
    Ctrl *ctrl = ctrl_all + (vprob ? vprob[v] : 0);
    if (ctrl->stop && !ctrl->ignore_stop) return;
    double *S = smem + (size_t)warp * L.total;
    int status = 0;
    const int iters = gcs_vertex_update(G, St, v, ctrl->rho, ctrl->mu_scale, tol, max_iter, L, S, lane, &status);
    if (lane == 0) {
        if (iters) atomicAdd(&ctrl->inner_iters, (unsigned long long)iters);
        if (status > 0 && status != 5) atomicAdd(&ctrl->inner_fail, 1);
        if (status < 0) atomicAdd(&ctrl->skipped, 1ull);
    }
}

// ------------------------------------------------------------------------------------------ peer mode (device functions)
__device__ __forceinline__ unsigned long long gcs_globaltimer() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }

// one thread block: cut half-edges -> the neighbours' ghost slots of this iteration's parity, then the flags (NVLink peer stores)
__device__ __forceinline__ void peer_push(const double *xc, const int *__restrict__ send_he, const int *__restrict__ send_rank,
                                          const int *__restrict__ send_slot, int nsend, const PeerView &PV) {
    const int k = PV.comm[PV.rank]->k + 1, par = k & 1;
    for (int i = threadIdx.x; i < 5 * nsend; i += blockDim.x) {
        const int j = i / 5, c = i - 5 * j, q = send_rank[j];
        PV.xc[q][5 * ((size_t)PV.nHown[q] + (size_t)par * PV.nHghost[q] + send_slot[j]) + c] = __ldcg(xc + 5 * (size_t)send_he[j] + c);
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x < PV.world && ((PV.neighbours >> threadIdx.x) & 1u)) *(volatile int *)&PV.comm[threadIdx.x]->halo_flag[PV.rank] = k;
}
// start of the edge kernels in peer mode: wait until every neighbour's halo of this iteration has arrived
__device__ __forceinline__ void peer_wait_halo(const PeerView &PV) {
    PeerComm *me = PV.comm[PV.rank];
    const int k = me->k + 1, p = threadIdx.x;
    if (p < PV.world && ((PV.neighbours >> p) & 1u)) {
        const unsigned long long t0 = gcs_globaltimer();
        while (*(volatile int *)&me->halo_flag[p] < k)
            if (gcs_globaltimer() - t0 > GCS_PEER_TIMEOUT_NS) { me->error = 1; break; }
        __threadfence_system();
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------ K1 (perf mode)
// PERSISTENT thread blocks (4 per SM), each walking tiles blockIdx.x, blockIdx.x + gridDim.x, ... of consecutive vertices
// (<= 256 (point, flow) pairs per tile).  Two stage buffers: while a block computes tile i from one, the bulk copies (TMA unit,
// mbarrier-signalled) of tile i + gridDim.x fill the other, and the bulk stores of tile i - gridDim.x drain — the DRAM latency of
// the per-tile state, cone records and descriptors never sits on the critical path.  ~43 KB of shared memory per block.
// BATCH: several problems packed block-diagonally (vprob != null); the single-problem variant carries none of their bookkeeping.
template <bool INNER, bool BATCH>
__global__ void __launch_bounds__(GCS_PERF_THREADS, 4)
vertex_perf_kernel(GcsGraphView G, GcsStateView St, GcsPerfTables T, Ctrl *ctrl_all, GcsPerfLayout L, PeerPush P) {
    extern __shared__ __align__(16) double smem[];
    __shared__ __align__(8) unsigned long long bar[2];
    if (!BATCH) {
        if (ctrl_all->stop && !ctrl_all->ignore_stop) return;
        if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&ctrl_all->inner_iters, (unsigned long long)T.inner_iters * (unsigned long long)G.nV);   // K passes over every vertex
    }
    int tile = blockIdx.x;
    if (tile >= T.ntiles) return;
    double *const stage0 = smem + L.work;
#define STAGE(b) (stage0 + (b) * L.stage)
    if (threadIdx.x == 0) {
        gcs_mbar_init(&bar[0], 1);
        gcs_mbar_init(&bar[1], 1);
        gcs_perf_stage(T, L, STAGE(0), tile, &bar[0]);
    }
    __syncthreads();                   // the barrier objects are initialised before anybody polls them
    double rin = 0.0;                  // INNER: this thread's share of the block's squared inner residual
    for (unsigned n = 0; tile < T.ntiles; tile += gridDim.x, ++n) {
        const int buf = n & 1;         // the n-th tile of the block is the (n / 2)-th completion of bar[buf]: its parity is (n / 2) & 1
        gcs_mbar_wait(&bar[buf], (n >> 1) & 1u);
        // stages tile + gridDim.x into the other buffer once the tile's first barrier is passed
        gcs_perf_tile<INNER, BATCH>(G, St, T, L, smem, STAGE(buf), tile, ctrl_all, rin, STAGE(buf ^ 1), tile + gridDim.x, &bar[buf ^ 1]);
    }
    if (threadIdx.x == GCS_COPY_THREAD) gcs_bulk_wait_read();   // shared memory stays valid until the last stores have read it
#undef STAGE
    if (INNER) {     // one partial per thread block, summed in a fixed order (static tile assignment: reproducible run to run)
#pragma unroll
        for (int o = 16; o; o >>= 1) rin += __shfl_xor_sync(0xffffffffu, rin, o);
        __syncthreads();                                  // the work arrays are free
        if ((threadIdx.x & 31) == 0) smem[L.rin + (threadIdx.x >> 5)] = rin;
        __syncthreads();
        if (threadIdx.x == 0) {
            double s = 0.0;
            for (int w2 = 0; w2 < (int)(blockDim.x >> 5); ++w2) s += smem[L.rin + w2];
            T.tile_res[blockIdx.x] = s;
        }
    }
    if (P.PV) {      // peer mode: the LAST block to finish pushes the cut half-edges to the neighbours (no separate launch)
        __shared__ int is_last;
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) is_last = (atomicAdd(P.ticket, 1u) == gridDim.x - 1);
        __syncthreads();
        if (is_last) {
            __threadfence();
            peer_push(St.xc, P.send_he, P.send_rank, P.send_slot, P.nsend, *P.PV);
            if (threadIdx.x == 0) *P.ticket = 0u;
        }
    }
}
// x_v / z_v / y_v of vertices no flow can pass are constants: written once when the mode is enabled
__global__ void perf_init_dead_kernel(GcsGraphView G, GcsStateView St) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= G.nV || G.vtype[v] != GCS_VT_DEAD) return;
    for (int k = 0; k < 4; ++k) { St.z_v[4 * (size_t)v + k] = 0.0; St.x_v[4 * (size_t)v + k] = G.cent[2 * (size_t)v + (k & 1)]; }
    St.y_v[v] = 0.0;
}

// ------------------------------------------------------------------------------------------ K5 (device function)
// reference admm_solver_v3.py:697-713 and :733, on the reduced sums
__device__ void control_apply(Ctrl *ctrl, const GcsParams &p, long long n_x, long long n_mu, double *hist, int hist_cap) {
    const int it = ctrl->it + 1;
    const double *s = ctrl->sums;
    const double rho = ctrl->rho;
    const double pri = sqrt(s[0]);                       // :598  ||A x + B z - c||
    const double dual = rho * sqrt(2.0 * s[1]);          // :602  rho ||A'B dz|| = rho sqrt2 ||dz||
    double rho_new = rho, scale = 1.0;
    // adapt_every > 1 (perf-mode option): the balancing test is applied on every adapt_every-th iteration only — per-iteration
    // balancing over a long window reacts to the noise of nearly converged residuals and can keep rho oscillating
    const bool may = it < p.frac * p.max_it && (p.adapt_every <= 1 || it % p.adapt_every == 0);
    if (pri >= p.nu * dual && may) { rho_new = rho * p.tau_incr; scale = 1.0 / p.tau_incr; }        // :703-705
    else if (dual >= p.nu * pri && may) { rho_new = rho * (1.0 / p.tau_decr); scale = p.tau_incr; } // :706-708
    const double nAx = sqrt(s[2]), nBz = sqrt(2.0 * s[3]), nmu = scale * sqrt(s[4]);
    const double eps_pri = sqrt((double)n_x) * p.eps_abs + p.eps_rel * fmax(nAx, nBz);   // :605-610
    const double eps_dual = sqrt((double)n_mu) * p.eps_abs + p.eps_rel * nmu;            // :613-614
    const double inner = s[6] < 0.0 ? -1.0 : sqrt(s[6]);   // perf mode: residual of the vertex programs' own cone constraints (-1: not computed
                                                           // in this iteration, 0 in the exact mode)
    // local frames: the same two residuals evaluated in GLOBAL coordinates — what the reference's definitions (:598, :602) give for
    // this iterate.  A flow mismatch eps between the two copies of an edge at position c is a position mismatch eps * |c| there.
    const double pri_g = s[7] < 0.0 ? -1.0 : sqrt(s[7]), dual_g = s[8] < 0.0 ? -1.0 : rho * sqrt(2.0 * s[8]);
    ctrl->pri_g = pri_g; ctrl->dual_g = dual_g;
    ctrl->it = it; ctrl->pri = pri; ctrl->dual = dual; ctrl->eps_pri = eps_pri; ctrl->eps_dual = eps_dual; ctrl->inner = inner;
    ctrl->rho = rho_new; ctrl->mu_scale = scale;
    if (it < hist_cap) { hist[it] = rho_new; hist[hist_cap + it] = pri; hist[2 * hist_cap + it] = dual; }
    if (s[5] != 0.0 || !isfinite(pri) || !isfinite(dual)) { ctrl->diverged = 1; ctrl->stop = 1; return; }  // :662-664
    // abs_stop (the "residual < tol" metric): the inexact x-update's own residual counts too — an iterate whose consensus
    // residuals are small while its vertex programs still violate their cone constraints is not a solution
    const bool ref = p.stop_ref && pri_g >= 0.0 && dual_g >= 0.0;
    const bool opt = p.abs_stop ? (inner >= 0.0 && fmax(fmax(ref ? pri_g : pri, ref ? dual_g : dual), inner) < p.abs_tol)
                                : (pri < eps_pri && dual < eps_dual);        // :712
    if (opt) { ctrl->opt = 1; ctrl->stop = 1; }
}

// Block reduction of the six partial sums, then the LAST block to finish (ticket) adds all blocks' partials in a fixed order and
// applies the control step (fuse = 1), publishes this rank's sums to every peer (fuse = 2) or just leaves them in ctrl->sums (fuse = 0)
__device__ __forceinline__ void edge_finish(double r2, double dz2, double x2, double z2, double m2, double r2g, double dz2g, Ctrl *ctrl, double *__restrict__ partials,
                                            unsigned int *ticket, int fuse, const GcsParams &p, long long n_x, long long n_mu, double *hist,
                                            int hist_cap, const PeerView *PVp, const double *__restrict__ tile_res, int ntiles) {
    double bad = 0;
    if (!isfinite(r2) || !isfinite(dz2) || !isfinite(x2) || !isfinite(z2)) bad = 1.0;
    // block reduction (fixed order: shuffles, then warp partials in shared memory)
    // columns: 0-5 the six sums | 6 inner residual^2 (filled by the last block from K1's partials) | 7, 8 r2 / dz2 in global coordinates
    __shared__ double sh[EDGE_THREADS][9];
    __shared__ int is_last;
    double vals[8] = {r2, dz2, x2, z2, m2, bad, r2g, dz2g};
#pragma unroll
    for (int q = 0; q < 8; ++q)
#pragma unroll
        for (int o = 16; o; o >>= 1) vals[q] += __shfl_xor_sync(0xffffffffu, vals[q], o);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0)
#pragma unroll
        for (int q = 0; q < 8; ++q) sh[warp][q] = vals[q];
    __syncthreads();
    if (threadIdx.x < 8) {
        double s = 0.0;
        for (int w2 = 0; w2 < EDGE_THREADS / 32; ++w2) s += sh[w2][threadIdx.x];
        partials[(size_t)blockIdx.x * NSUMS + (threadIdx.x < 6 ? threadIdx.x : threadIdx.x + 1)] = s;      // (slot 6 belongs to the inner residual)
        __threadfence();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int t = atomicAdd(ticket, 1u);
        is_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    // last block: every block's partials are visible; sum them in an order that does not depend on which block is last
    // (seventh sum, perf mode: the tiles' squared inner residuals written by K1 of this iteration)
    double acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x)
#pragma unroll
        for (int q = 0; q < 9; ++q) if (q != 6) acc[q] += __ldcg(partials + (size_t)b * NSUMS + q);
    if (tile_res) { for (int b = threadIdx.x; b < ntiles; b += blockDim.x) acc[6] += __ldcg(tile_res + b); }
    else if (ntiles < 0 && threadIdx.x == 0) acc[6] = -1.0;           // perf mode, inner residual not computed in this iteration
#pragma unroll
    for (int q = 0; q < 9; ++q) sh[threadIdx.x][q] = acc[q];
    __syncthreads();
    for (int st = EDGE_THREADS / 2; st > 0; st >>= 1) {
        if (threadIdx.x < st)
#pragma unroll
            for (int q = 0; q < 9; ++q) sh[threadIdx.x][q] += sh[threadIdx.x + st][q];
        __syncthreads();
    }
    if (threadIdx.x < 9) ctrl->sums[threadIdx.x] = sh[0][threadIdx.x];
    __syncthreads();
    if (fuse == 2) {       // peer mode: this rank's sums into every rank's inbox, then the flag
        const int me = PVp->rank, world = PVp->world, k = PVp->comm[me]->k + 1, par = k & 1;
        if (threadIdx.x < 9)
            for (int q = 0; q < world; ++q) PVp->comm[q]->sums_in[par][me][threadIdx.x] = sh[0][threadIdx.x];
        __threadfence_system();
        __syncthreads();
        if (threadIdx.x < world) { *(volatile int *)&PVp->comm[threadIdx.x]->sums_flag[me] = k; }
        if (threadIdx.x == 0) *ticket = 0u;
        return;
    }
    if (threadIdx.x == 0) {
        *ticket = 0u;
        if (fuse) control_apply(ctrl, p, n_x, n_mu, hist, hist_cap);
    }
}

// ------------------------------------------------------------------------------------------ K2-K5
// z_e = 1/2 (xc_tail + xc_head)            reference admm_solver_v3.py:543-562 (live scalars only)
// mu_h <- mu_scale * mu_h + (z_e - xc_h)    :590-594  (mu_scale carries the rho-adaptation rescale :705/:708)
// partial sums of |z - xc|^2, |dz|^2, |xc|^2, |z|^2, |mu|^2     :597-614
// local frames (perf-mode option, vertex_perf.cuh GcsPerfTables.edge_delta): the consensus constraint of edge e is
//   x_head = z,  x_tail = B z,  B (p1, p2, y) = (p1, p2 - y delta, y)
// so the z-update is the least-squares solve  (I + B'B) z = x_head + B' x_tail  (the duals drop out: B' mu_tail + mu_head = 0 is an
// invariant of the iteration), closed form per edge; mu_head += z - x_head, mu_tail += B z - x_tail; the dual residual is
// rho sqrt(|dz|^2 + |B dz|^2).  Global frames are delta = 0.  The three coupled scalars (p2, y) are needed together, so a thread
// works on whole edges.
// oalpha != 1 (perf mode only) over-relaxes the consensus step (Boyd et al. 3.4.3): x is replaced by oalpha x + (1 - oalpha) (B) z_old
// in the z- and mu-updates; the primal residual keeps the true x.  B' mu_tail + mu_head = 0 stays invariant.
// fuse != 0: the last block to finish reduces the block partials in a fixed order and applies the control step.
// The two kernels below share the per-edge arithmetic through these helpers, so their z and mu agree bit for bit.

// z-update of one edge: the relaxed copies at / ah of the tail's and head's points, the new z and its tail-side image B z
template <bool OA>
__device__ __forceinline__ void edge_z_update(const double (&xt)[5], const double (&xh)[5], const double (&zo)[5], double d0, double d1,
                                              double oa, double ob, double (&at)[5], double (&ah)[5], double (&zn)[5], double (&bz)[5]) {
#pragma unroll
    for (int c = 0; c < 5; ++c) { at[c] = xt[c]; ah[c] = xh[c]; }
    if (OA) {          // (compile-time: without over-relaxation at / ah are xt / xh and cost no registers)
        const double bo[5] = {zo[0], zo[1], zo[2] - d0 * zo[4], zo[3] - d1 * zo[4], zo[4]};
#pragma unroll
        for (int c = 0; c < 5; ++c) { at[c] = oa * xt[c] + ob * bo[c]; ah[c] = oa * xh[c] + ob * zo[c]; }
    }
    zn[0] = 0.5 * (ah[0] + at[0]); zn[1] = 0.5 * (ah[1] + at[1]);
    const double q0 = ah[2] + at[2], q1 = ah[3] + at[3], q2 = ah[4] + at[4] - (d0 * at[2] + d1 * at[3]);
    zn[4] = (q2 + 0.5 * (d0 * q0 + d1 * q1)) / (2.0 + 0.5 * (d0 * d0 + d1 * d1));
    zn[2] = 0.5 * (q0 + d0 * zn[4]); zn[3] = 0.5 * (q1 + d1 * zn[4]);
    bz[0] = zn[0]; bz[1] = zn[1]; bz[2] = zn[2] - d0 * zn[4]; bz[3] = zn[3] - d1 * zn[4]; bz[4] = zn[4];
}

// |v|^2 + |B v|^2 of an edge vector v, its squared norm over both half-edge copies (the callers halve it); b2, b3: the two
// scalars of B v that differ from v
__device__ __forceinline__ double copies_sq(const double (&v)[5], double b2, double b3) {
    return 2.0 * (v[0] * v[0] + v[1] * v[1] + v[4] * v[4]) + v[2] * v[2] + v[3] * v[3] + b2 * b2 + b3 * b3;
}

// dual update of one half-edge with copy p of the edge's point (B z on the tail side, z on the head side), primal copy x and relaxed
// copy a: out[off + c] <- ms * mu + (p - a); with acc, adds |p - x|^2, |x|^2, |mu_new|^2, scalar by scalar.  (A base and an offset,
// not one pointer: with a pointer the warp-cooperative kernel's shared-memory addressing takes more instructions.)
__device__ __forceinline__ void half_edge_dual(const double (&p)[5], const double (&x)[5], const double (&a)[5], const double (&mu)[5], double ms,
                                               double *out, size_t off, bool acc, double &r2, double &x2, double &m2) {
#pragma unroll
    for (int c = 0; c < 5; ++c) {
        const double r = p[c] - x[c], mn = ms * mu[c] + (p[c] - a[c]);
        out[off + c] = mn;
        if (acc) { r2 += r * r; x2 += x[c] * x[c]; m2 += mn * mn; }
    }
}

// One thread per edge: partitions with ghost slots (multi-GPU), edge_counted weights, the check variant.
// GRES (check variant, local frames only): also the primal / dual residual sums in GLOBAL coordinates.  The copies of an edge
// (u, w) live in the frame of u (both points of the tail's copy, the first point of the head's copy) or of w (the head's own first
// point); adding  flow * centre-of-frame  to a point gives its global value, so  r_global = r_local + r_flow * centre.
// 128 registers (2 resident blocks per SM): all 25 loads of an edge are in flight together.
template <bool OA, bool GRES>
__global__ void __launch_bounds__(EDGE_THREADS, 2)
edge_frames_kernel(int nE, int nHown, const int *__restrict__ edge_he_tail, const int *__restrict__ edge_he_head,
                   const unsigned char *__restrict__ edge_counted, const double *__restrict__ edge_delta, const double *__restrict__ edge_cent, const double *__restrict__ xc,
                   double *__restrict__ mu, double *__restrict__ z, Ctrl *ctrl, double *__restrict__ partials, unsigned int *ticket, int fuse,
                   GcsParams p, long long n_x, long long n_mu, double *hist, int hist_cap, int nHghost, const PeerView *PVp, const double *__restrict__ tile_res, int ntiles) {
    if (ctrl->stop && !ctrl->ignore_stop) return;
    if (fuse == 2) peer_wait_halo(*PVp);
    const double ms = ctrl->mu_scale, oa = p.outer_alpha, ob = 1.0 - p.outer_alpha;
    // peer mode: the ghost slots of this iteration's parity (PVp lives in device memory: indexed at run time)
    const int gpar = fuse == 2 ? ((PVp->comm[PVp->rank]->k + 1) & 1) * nHghost : 0;
    double r2 = 0, dz2 = 0, x2 = 0, z2 = 0, m2 = 0, r2g = 0, dz2g = 0;
    if (!GRES && blockIdx.x == 0 && threadIdx.x == 0) r2g = dz2g = -1.0;      // "not computed in this iteration"
    // the half-edge indices of a thread's NEXT edge are loaded while the current one is processed: the dependent
    // index -> record load chain of a grid-stride step then starts with the indices already in registers
    const int estride = gridDim.x * blockDim.x;
    int e = blockIdx.x * blockDim.x + threadIdx.x, ht = 0, hh = 0;
    if (e < nE) { ht = edge_he_tail[e]; hh = edge_he_head[e]; }
    for (; e < nE; e += estride) {
        const int en = e + estride, ht_ = ht, hh_ = hh;       // this edge's half-edges; ht / hh now receive the next edge's
        if (en < nE) { ht = edge_he_tail[en]; hh = edge_he_head[en]; }
        const bool ot = ht_ < nHown, oh = hh_ < nHown;
        const double *pt = xc + 5 * (size_t)(ot ? ht_ : ht_ + gpar), *ph = xc + 5 * (size_t)(oh ? hh_ : hh_ + gpar);
        double xt[5], xh[5], zo[5], mt[5], mh[5];
#pragma unroll
        for (int c = 0; c < 5; ++c) { xt[c] = pt[c]; xh[c] = ph[c]; zo[c] = z[5 * (size_t)e + c]; }
#pragma unroll
        for (int c = 0; c < 5; ++c) { mt[c] = ot ? mu[5 * (size_t)ht_ + c] : 0.0; mh[c] = oh ? mu[5 * (size_t)hh_ + c] : 0.0; }
        const double d0 = edge_delta ? edge_delta[2 * (size_t)e] : 0.0, d1 = edge_delta ? edge_delta[2 * (size_t)e + 1] : 0.0;
        const double w = edge_counted ? (double)edge_counted[e] : 1.0;
        double at[5], ah[5], zn[5], bz[5], dd[5];
        edge_z_update<OA>(xt, xh, zo, d0, d1, oa, ob, at, ah, zn, bz);
#pragma unroll
        for (int c = 0; c < 5; ++c) { dd[c] = zn[c] - zo[c]; z[5 * (size_t)e + c] = zn[c]; }
        const double db2 = dd[2] - d0 * dd[4], db3 = dd[3] - d1 * dd[4];
        dz2 += 0.5 * w * copies_sq(dd, db2, db3);
        z2 += 0.5 * w * copies_sq(zn, bz[2], bz[3]);
        double cu0 = 0.0, cu1 = 0.0, cw0 = 0.0, cw1 = 0.0;
        if (GRES) {
            cu0 = edge_cent[2 * (size_t)e]; cu1 = edge_cent[2 * (size_t)e + 1]; cw0 = cu0 - d0; cw1 = cu1 - d1;
            const double g0 = dd[0] + dd[4] * cu0, g1 = dd[1] + dd[4] * cu1, g2 = dd[2] + dd[4] * cw0, g3 = dd[3] + dd[4] * cw1;
            dz2g += w * (g0 * g0 + g1 * g1 + g2 * g2 + g3 * g3 + dd[4] * dd[4]);
        }
        if (ot) {
            half_edge_dual(bz, xt, at, mt, ms, mu, 5 * (size_t)ht_, true, r2, x2, m2);
            if (GRES) {      // every slot of the tail's copy lives in the tail's frame
                const double ry = bz[4] - xt[4], a0 = bz[0] - xt[0] + ry * cu0, a1 = bz[1] - xt[1] + ry * cu1, a2 = bz[2] - xt[2] + ry * cu0, a3 = bz[3] - xt[3] + ry * cu1;
                r2g += a0 * a0 + a1 * a1 + a2 * a2 + a3 * a3 + ry * ry;
            }
        }
        if (oh) {
            half_edge_dual(zn, xh, ah, mh, ms, mu, 5 * (size_t)hh_, true, r2, x2, m2);
            if (GRES) {      // the tail's first point in the tail's frame, the head's own first point in the head's frame
                const double ry = zn[4] - xh[4], a0 = zn[0] - xh[0] + ry * cu0, a1 = zn[1] - xh[1] + ry * cu1, a2 = zn[2] - xh[2] + ry * cw0, a3 = zn[3] - xh[3] + ry * cw1;
                r2g += a0 * a0 + a1 * a1 + a2 * a2 + a3 * a3 + ry * ry;
            }
        }
    }
    edge_finish(r2, dz2, x2, z2, m2, r2g, dz2g, ctrl, partials, ticket, fuse, p, n_x, n_mu, hist, hist_cap, PVp, tile_res, ntiles);
}

// Warp-cooperative variant of the edge kernel for the single-GPU throughput path (every half-edge owned, no ghost slots, no
// check variant): a warp takes 32 consecutive edges.  The 5-double records of its 32 tail half-edges, 32 head half-edges and 32
// edges are moved between HBM and shared memory as five passes of 32 CONSECUTIVE doubles of the concatenated records (lane l of
// pass k handles double l + 32 k, i.e. scalar (l + 32 k) % 5 of record (l + 32 k) / 5, the record's index coming from the lane that
// owns the edge by a shuffle) — a request then touches ~7 records instead of 32, a third of the L1 wavefronts of the
// one-thread-per-record pattern; each lane then reads / writes its own edge's records in shared memory with stride 5 (conflict-free).
#define COOP_WARPS (EDGE_THREADS / 32)
#define COOP_SMEM_DOUBLES (COOP_WARPS * 5 * 160)
template <bool OA>
__global__ void __launch_bounds__(EDGE_THREADS, 2)
edge_coop_kernel(int nE, const int *__restrict__ edge_he_tail, const int *__restrict__ edge_he_head, const double *__restrict__ edge_delta,
                 const double *__restrict__ xc, double *__restrict__ mu, double *__restrict__ z, Ctrl *ctrl, double *__restrict__ partials,
                 unsigned int *ticket, int fuse, GcsParams p, long long n_x, long long n_mu, double *hist, int hist_cap,
                 const double *__restrict__ tile_res, int ntiles) {
    extern __shared__ __align__(16) double coop_sm[];
    if (ctrl->stop && !ctrl->ignore_stop) return;
    const double ms = ctrl->mu_scale, oa = p.outer_alpha, ob = 1.0 - p.outer_alpha;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double *xtS = coop_sm + (size_t)warp * 800, *xhS = xtS + 160, *zoS = xtS + 320, *mtS = xtS + 480, *mhS = xtS + 640;
    double r2 = 0, dz2 = 0, x2 = 0, z2 = 0, m2 = 0, r2g = 0, dz2g = 0;
    if (blockIdx.x == 0 && threadIdx.x == 0) r2g = dz2g = -1.0;      // global-coordinate residuals: not computed by this variant
    const int nchunks = (nE + 31) >> 5;
    for (int chunk = blockIdx.x * COOP_WARPS + warp; chunk < nchunks; chunk += gridDim.x * COOP_WARPS) {
        const int e = (chunk << 5) + lane;
        const bool valid = e < nE;
        const int ht = valid ? edge_he_tail[e] : 0, hh = valid ? edge_he_head[e] : 0;     // (lanes past the end read record 0 and store nothing)
        const double d0 = valid && edge_delta ? edge_delta[2 * (size_t)e] : 0.0, d1 = valid && edge_delta ? edge_delta[2 * (size_t)e + 1] : 0.0;
        const size_t zbase = (size_t)chunk * 160;
        // ---- HBM -> shared memory: 5 passes x 5 arrays, all 25 loads of a lane in flight before the first is used
        double vx[5], vh[5], vz[5], vm[5], vn[5];
        int tj[5], hj[5];
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            const int i = lane + 32 * k, j = i / 5, c = i - 5 * j;
            tj[k] = 5 * __shfl_sync(0xffffffffu, ht, j) + c;
            hj[k] = 5 * __shfl_sync(0xffffffffu, hh, j) + c;
        }
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            const int i = lane + 32 * k;
            vx[k] = xc[tj[k]]; vh[k] = xc[hj[k]]; vm[k] = mu[tj[k]]; vn[k] = mu[hj[k]];
            vz[k] = zbase + i < 5 * (size_t)nE ? z[zbase + i] : 0.0;
        }
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            const int i = lane + 32 * k;
            xtS[i] = vx[k]; xhS[i] = vh[k]; mtS[i] = vm[k]; mhS[i] = vn[k]; zoS[i] = vz[k];
        }
        __syncwarp();
        // ---- the lane's own edge
        double xt[5], xh[5], zo[5], mt[5], mh[5];
#pragma unroll
        for (int c = 0; c < 5; ++c) { xt[c] = xtS[5 * lane + c]; xh[c] = xhS[5 * lane + c]; zo[c] = zoS[5 * lane + c]; mt[c] = mtS[5 * lane + c]; mh[c] = mhS[5 * lane + c]; }
        __syncwarp();                    // every lane has read its records: the buffers can take the results
        double at[5], ah[5], zn[5], bz[5], dd[5];
        edge_z_update<OA>(xt, xh, zo, d0, d1, oa, ob, at, ah, zn, bz);
#pragma unroll
        for (int c = 0; c < 5; ++c) { dd[c] = zn[c] - zo[c]; zoS[5 * lane + c] = zn[c]; }
        // (db2 / db3 stay outside the branch: ptxas fuses a multiply and an add into one FMA only inside one block, so where they
        // are computed decides the last bits of dz2)
        const double db2 = dd[2] - d0 * dd[4], db3 = dd[3] - d1 * dd[4];
        if (valid) {
            dz2 += 0.5 * copies_sq(dd, db2, db3);
            z2 += 0.5 * copies_sq(zn, bz[2], bz[3]);
        }
        half_edge_dual(bz, xt, at, mt, ms, mtS, 5 * lane, valid, r2, x2, m2);
        half_edge_dual(zn, xh, ah, mh, ms, mhS, 5 * lane, valid, r2, x2, m2);
        __syncwarp();
        // ---- shared memory -> HBM, the same five passes
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            const int i = lane + 32 * k, j = i / 5;
            if ((chunk << 5) + j < nE) { z[zbase + i] = zoS[i]; mu[tj[k]] = mtS[i]; mu[hj[k]] = mhS[i]; }
        }
        __syncwarp();                    // the buffers are free for the warp's next chunk
    }
    edge_finish(r2, dz2, x2, z2, m2, r2g, dz2g, ctrl, partials, ticket, fuse, p, n_x, n_mu, hist, hist_cap, nullptr, tile_res, ntiles);
}

// ------------------------------------------------------------------------------------------ peer mode (kernels)
// exact mode: the push is a launch of its own after K1 (the perf kernel's last block does it itself)
__global__ void __launch_bounds__(1024)
peer_push_kernel(const double *__restrict__ xc, const int *__restrict__ send_he, const int *__restrict__ send_rank,
                 const int *__restrict__ send_slot, int nsend, Ctrl *ctrl, const PeerView *PVp) {
    if (ctrl->stop && !ctrl->ignore_stop) return;
    peer_push(xc, send_he, send_rank, send_slot, nsend, *PVp);
}
// one warp: waits for every rank's sums, adds them in rank order, control step, advances the peer iteration counter
__global__ void peer_control_kernel(Ctrl *ctrl, GcsParams p, long long n_x, long long n_mu, double *hist, int hist_cap, const PeerView *PVp) {
    if (ctrl->stop && !ctrl->ignore_stop) return;
    const PeerView &PV = *PVp;
    PeerComm *me = PV.comm[PV.rank];
    const int k = me->k + 1, par = k & 1, q = threadIdx.x;
    if (q < PV.world) {
        const unsigned long long t0 = gcs_globaltimer();
        while (*(volatile int *)&me->sums_flag[q] < k)
            if (gcs_globaltimer() - t0 > GCS_PEER_TIMEOUT_NS) { me->error = 1; break; }
    }
    __threadfence_system();
    __syncwarp();
    if (threadIdx.x == 0) {
        for (int j = 0; j < 9; ++j) {
            double s = 0.0;
            for (int r = 0; r < PV.world; ++r) s += *(volatile double *)&me->sums_in[par][r][j];
            ctrl->sums[j] = s;
        }
        if (me->error) { ctrl->diverged = 1; ctrl->stop = 1; }
        else control_apply(ctrl, p, n_x, n_mu, hist, hist_cap);
        me->k = k;
    }
}

__global__ void control_kernel(Ctrl *ctrl, GcsParams p, long long n_x, long long n_mu, double *hist, int hist_cap) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    if (ctrl->stop && !ctrl->ignore_stop) return;
    control_apply(ctrl, p, n_x, n_mu, hist, hist_cap);
}

// ------------------------------------------------------------------------------------------ batched K2-K5
// Independent problems packed block-diagonally (BASELINE config "batch of 4096 queries"): one block per problem
// does that problem's edges, its own residual sums and its own rho / stop decision — no communication, and a
// problem that has converged stops costing anything.
#define BATCH_THREADS 128
__global__ void __launch_bounds__(BATCH_THREADS)
batched_edge_kernel(int nP, const int *__restrict__ prob_eoff, int nHown, const int *__restrict__ edge_he_tail,
                    const int *__restrict__ edge_he_head, const double *__restrict__ xc, double *__restrict__ mu,
                    double *__restrict__ z, Ctrl *ctrl_all, GcsParams p, const long long *__restrict__ prob_nx,
                    const long long *__restrict__ prob_nmu, double *hist, int hist_cap) {
    __shared__ double sh[BATCH_THREADS / 32][6];
    for (int q = blockIdx.x; q < nP; q += gridDim.x) {
        Ctrl *ctrl = ctrl_all + q;
        if (ctrl->stop && !ctrl->ignore_stop) continue;
        const double ms = ctrl->mu_scale;
        double r2 = 0, dz2 = 0, x2 = 0, z2 = 0, m2 = 0, bad = 0;
        for (int e = prob_eoff[q] + threadIdx.x; e < prob_eoff[q + 1]; e += blockDim.x) {
            const int ht = edge_he_tail[e], hh = edge_he_head[e];
            double xt[5], xh[5], zn[5];
#pragma unroll
            for (int c = 0; c < 5; ++c) { xt[c] = xc[5 * (size_t)ht + c]; xh[c] = xc[5 * (size_t)hh + c]; }
#pragma unroll
            for (int c = 0; c < 5; ++c) {
                const double zo = z[5 * (size_t)e + c];
                zn[c] = 0.5 * (xt[c] + xh[c]);
                const double dd = zn[c] - zo;
                dz2 += dd * dd; z2 += zn[c] * zn[c];
                z[5 * (size_t)e + c] = zn[c];
            }
#pragma unroll
            for (int c = 0; c < 5; ++c) {
                const double rt = zn[c] - xt[c], mt = ms * mu[5 * (size_t)ht + c] + rt;
                mu[5 * (size_t)ht + c] = mt; r2 += rt * rt; x2 += xt[c] * xt[c]; m2 += mt * mt;
                const double rh = zn[c] - xh[c], mh = ms * mu[5 * (size_t)hh + c] + rh;
                mu[5 * (size_t)hh + c] = mh; r2 += rh * rh; x2 += xh[c] * xh[c]; m2 += mh * mh;
            }
        }
        if (!isfinite(r2) || !isfinite(dz2) || !isfinite(x2) || !isfinite(z2)) bad = 1.0;
        double vals[6] = {r2, dz2, x2, z2, m2, bad};
#pragma unroll
        for (int k = 0; k < 6; ++k)
#pragma unroll
            for (int o = 16; o; o >>= 1) vals[k] += __shfl_xor_sync(0xffffffffu, vals[k], o);
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        if (lane == 0)
            for (int k = 0; k < 6; ++k) sh[warp][k] = vals[k];
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int k = 0; k < 6; ++k) {
                double sum = 0.0;
                for (int w2 = 0; w2 < BATCH_THREADS / 32; ++w2) sum += sh[w2][k];
                ctrl->sums[k] = sum;
            }
            control_apply(ctrl, p, prob_nx[q], prob_nmu[q], hist + (size_t)q * 3 * hist_cap, hist_cap);
        }
        __syncthreads();
    }
}
__global__ void set_ignore_kernel(Ctrl *ctrl, int nP, int v) {
    for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < nP; q += gridDim.x * blockDim.x) ctrl[q].ignore_stop = v;
}

// ------------------------------------------------------------------------------------------ host side
extern "C" const char *gcsadmm_version(void) { return GCS_VERSION; }
extern "C" const char *gcsadmm_last_error(void) { return g_err; }
extern "C" int gcsadmm_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}
extern "C" void gcsadmm_default_params(GcsParams *p) {
    p->rho0 = 1.0; p->tau_incr = 2.0; p->tau_decr = 2.0; p->nu = 10.0; p->frac = 0.1;
    p->eps_abs = 1e-4; p->eps_rel = 1e-3; p->max_it = 1000; p->inner_tol = 1e-8; p->inner_max_iter = 60;
    p->check_every = 8; p->abs_stop = 0; p->abs_tol = 1e-4; p->warm_theta = 1e-3; p->zero_tol = 1e-12;
    p->outer_alpha = 1.0; p->use_graph = 1; p->adapt_every = 1; p->stop_ref = 0;
}
extern "C" int gcsadmm_scratch_bytes(int max_live_degree, int max_rows) {
    return (int)(gcs_scratch_layout(max_live_degree, max_rows).total * sizeof(double));
}

template <typename T>
static int upload(T **dst, const T *src, size_t n) {
    if (n == 0) n = 1, src = nullptr;
    cudaError_t e = cudaMalloc((void **)dst, n * sizeof(T));
    if (e != cudaSuccess) { char nb[32]; snprintf(nb, sizeof nb, "%zu", n * sizeof(T)); return set_err(GCS_E_NOMEM, "cudaMalloc(%s bytes): %s", nb, cudaGetErrorString(e)); }
    if (src) { e = cudaMemcpy(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice); if (e != cudaSuccess) return set_err(GCS_E_CUDA, "cudaMemcpy H2D: %s", cudaGetErrorString(e)); }
    else cudaMemset(*dst, 0, n * sizeof(T));
    return 0;
}

static int reset_ctrl(GcsHandle *h) {
    Ctrl c; memset(&c, 0, sizeof c);
    c.rho = h->p.rho0; c.mu_scale = 1.0;
    double first[3] = {h->p.rho0, 0.0, 0.0};   // admm_solver_v3.py:637-639: seeds of the three sequences
    for (int q = 0; q < h->nP; ++q) {
        h->ctrl_host[q] = c;
        for (int k = 0; k < 3; ++k)
            CK(cudaMemcpyAsync(h->hist + ((size_t)q * 3 + k) * h->hist_cap, &first[k], sizeof(double), cudaMemcpyHostToDevice, h->stream));
    }
    CK(cudaMemcpyAsync(h->ctrl, h->ctrl_host, sizeof(Ctrl) * h->nP, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

static void free_perf(GcsHandle *h) {
    void *pp[] = {h->p_vclass, h->p_cone_off, h->p_blk_off, h->p_blk_rec, h->p_vrec, h->p_tile_rec, h->p_cls_tab, h->p_cone, h->p_tstate, h->p_tn, h->p_edge_delta, h->p_edge_cent, h->p_tile_res};
    for (void *q : pp) if (q) cudaFree(q);
    h->p_vclass = h->p_cone_off = h->p_blk_off = h->p_blk_rec = h->p_vrec = h->p_tile_rec = nullptr;
    h->p_cls_tab = h->p_cone = h->p_tstate = h->p_tn = h->p_edge_delta = h->p_edge_cent = h->p_tile_res = nullptr;
    h->perf_on = 0;
}
static void drop_graph(GcsHandle *h) {
    if (h->graph_exec) { cudaGraphExecDestroy(h->graph_exec); h->graph_exec = nullptr; }
    h->graph_iters = 0;
}

extern "C" int gcsadmm_destroy(GcsHandle *h) {
    if (!h) return 0;
    cudaSetDevice(h->device);
    void *ptrs[] = {h->poly_off, h->he_off, h->he_edge, h->edge_he_tail, h->edge_he_head, h->polyA, h->polyb, h->cent,
                    h->he_flags, h->vtype, h->edge_counted, h->xc, h->mu, h->z, h->x_v, h->z_v, h->y_v, h->ws, h->partials, h->hist, h->ctrl,
                    h->vprob, h->prob_eoff, h->prob_nx, h->prob_nmu};
    for (void *p : ptrs) if (p) cudaFree(p);
    if (h->ctrl_host) cudaFreeHost(h->ctrl_host);
    free(h->he_prob_host);
    if (h->flush_buf) cudaFree(h->flush_buf);
    if (h->graph_exec) cudaGraphExecDestroy(h->graph_exec);
    for (void *m : h->ipc_opened) if (m) cudaIpcCloseMemHandle(m);
    { void *pp[] = {h->comm, h->send_he, h->send_rank, h->send_slot, h->PV_dev}; for (void *q : pp) if (q) cudaFree(q); }
    if (h->ticket) cudaFree(h->ticket);
    if (h->push_ticket) cudaFree(h->push_ticket);
    free_perf(h);
    for (int i = 0; i < 4; ++i) if (h->ev[i]) cudaEventDestroy(h->ev[i]);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    delete h;
    return 0;
}

// index ranges of the caller's arrays (a bad index would otherwise be an out-of-bounds access on the device)
static int validate_graph(const GcsGraph *g) {
    if (!g->poly_off || !g->polyA || !g->polyb || !g->he_off || !g->vtype || !g->cent) return set_err(GCS_E_INVALID, "null graph array%s", "");
    if (g->nH_own < 0 || g->nH_ghost < 0 || g->he_off[0] != 0 || g->he_off[g->nV] != g->nH_own) return set_err(GCS_E_INVALID, "he_off does not span nH_own%s", "");
    if (g->nH_own && (!g->he_edge || !g->he_flags)) return set_err(GCS_E_INVALID, "null half-edge array%s", "");
    if (g->nE && (!g->edge_he_tail || !g->edge_he_head)) return set_err(GCS_E_INVALID, "null edge array%s", "");
    if (g->poly_off[0] != 0) return set_err(GCS_E_INVALID, "poly_off[0] != 0%s", "");
    for (int v = 0; v < g->nV; ++v) {
        if (g->he_off[v + 1] < g->he_off[v] || g->poly_off[v + 1] < g->poly_off[v]) return set_err(GCS_E_INVALID, "offsets not monotone%s", "");
        if (g->vtype[v] > 3) return set_err(GCS_E_INVALID, "bad vertex type%s", "");
    }
    for (int hh = 0; hh < g->nH_own; ++hh) if (g->he_edge[hh] < 0 || g->he_edge[hh] >= g->nE) return set_err(GCS_E_INVALID, "he_edge out of range%s", "");
    const int nHall = g->nH_own + g->nH_ghost;
    for (int e = 0; e < g->nE; ++e)
        if (g->edge_he_tail[e] < 0 || g->edge_he_tail[e] >= nHall || g->edge_he_head[e] < 0 || g->edge_he_head[e] >= nHall)
            return set_err(GCS_E_INVALID, "edge_he_tail / edge_he_head out of range%s", "");
    return 0;
}

// everything of gcsadmm_create that can fail after the handle exists; the caller destroys the handle on failure
static int create_impl(GcsHandle *h, const GcsGraph *g) {
    // capacity of a vertex program: live degree and polytope rows
    int dcap = 1, mcap = 1;
    for (int v = 0; v < g->nV; ++v) {
        int d = 0;
        for (int hh = g->he_off[v]; hh < g->he_off[v + 1]; ++hh) if (!(g->he_flags[hh] & GCS_HE_FLAG_ZERO)) d++;
        if (d > dcap) dcap = d;
        int m = g->poly_off[v + 1] - g->poly_off[v];
        if (m > mcap) mcap = m;
        if (g->vtype[v] == GCS_VT_GENERIC && d < 2) return set_err(GCS_E_INVALID, "inconsistent presolve flags (generic vertex with < 2 live half-edges)%s", "");
    }
    h->dcap = dcap; h->mcap = mcap;
    h->L = gcs_scratch_layout(dcap, mcap);
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, h->device));
    {   // as many warps per block as shared memory allows (one block per SM when the programs are large)
        const size_t per_warp = (size_t)h->L.total * sizeof(double);
        const size_t budget = prop.sharedMemPerBlockOptin;
        int w = (int)(budget / per_warp);
        if (w < 1) return set_err(GCS_E_INVALID, "vertex program too large for shared memory (max live degree / polytope rows too high)%s", "");
        if (w > K1_MAX_WARPS) w = K1_MAX_WARPS;
        h->k1_warps = w;
        h->k1_smem = (int)(w * per_warp);
    }
    CK(cudaFuncSetAttribute(vertex_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, h->k1_smem));
    CK(cudaFuncSetAttribute(vertex_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    h->k1_blocks = (g->nV + h->k1_warps - 1) / h->k1_warps;
    {   // edge kernels.  Measured on the 100k-vertex grid: warp-cooperative 38 us (2 blocks per SM; 44 us with 3), one thread per
        // edge 54 us (2 blocks per SM).  The warp-cooperative kernel runs wherever it applies (single GPU, no ghost slots,
        // throughput path).  GCS_EDGE_KERNEL=per_edge runs the one-thread-per-edge kernel there too: this is how a test runs both
        // kernels on one state, which must agree bit for bit.
        const char *ek = getenv("GCS_EDGE_KERNEL");
        h->edge_coop = !(ek && !strcmp(ek, "per_edge"));
        h->coop_blocks = 2 * prop.multiProcessorCount;
        if (h->edge_coop) {
            const int smb = (int)(sizeof(double) * COOP_SMEM_DOUBLES);
            CK(cudaFuncSetAttribute(edge_coop_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smb));
            CK(cudaFuncSetAttribute(edge_coop_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smb));
        }
        // one thread per edge, at most 4 blocks per SM; at least as many blocks as the warp-cooperative launch (partials rows)
        const long long need = (g->nE + EDGE_THREADS - 1) / EDGE_THREADS, cap = 4ll * prop.multiProcessorCount;
        h->edge_blocks = (int)(need < 1 ? 1 : (need > cap ? cap : need));
    }
    CK(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    h->stream = h->own_stream;
    const size_t M = (size_t)g->poly_off[g->nV], Hall = (size_t)g->nH_own + g->nH_ghost;
    int rc = 0;
#define UP(field, src, n) if (!rc) rc = upload(&h->field, src, (size_t)(n))
    UP(poly_off, g->poly_off, g->nV + 1); UP(polyA, g->polyA, 2 * M); UP(polyb, g->polyb, M);
    UP(he_off, g->he_off, g->nV + 1); UP(he_edge, g->he_edge, g->nH_own); UP(he_flags, g->he_flags, g->nH_own);
    UP(edge_he_tail, g->edge_he_tail, g->nE); UP(edge_he_head, g->edge_he_head, g->nE);
    UP(vtype, g->vtype, g->nV); UP(cent, g->cent, 2 * (size_t)g->nV);
    if (g->edge_counted) UP(edge_counted, g->edge_counted, g->nE);
    UP(xc, (const double *)nullptr, 5 * (Hall + (size_t)g->nH_ghost));      // ghost slots twice: double-buffered in peer mode
    UP(mu, (const double *)nullptr, 5 * (size_t)g->nH_own); UP(z, (const double *)nullptr, 5 * (size_t)g->nE);
    UP(x_v, (const double *)nullptr, 4 * (size_t)g->nV); UP(z_v, (const double *)nullptr, 4 * (size_t)g->nV); UP(y_v, (const double *)nullptr, g->nV);
    if (h->p.warm_theta > 0.0) UP(ws, (const double *)nullptr, (size_t)g->nV * gcs_ws_stride(h->L));
    UP(partials, (const double *)nullptr, (size_t)h->edge_blocks * NSUMS);
    UP(ticket, (const unsigned int *)nullptr, 1);
    UP(push_ticket, (const unsigned int *)nullptr, 1);
    h->hist_cap = h->p.max_it + 2;
    UP(hist, (const double *)nullptr, 3 * (size_t)h->hist_cap * h->nP);
#undef UP
    if (rc) return rc;
    CK(cudaMalloc((void **)&h->ctrl, sizeof(Ctrl) * h->nP));
    CK(cudaMallocHost((void **)&h->ctrl_host, sizeof(Ctrl) * h->nP));
    if (h->nP > 1) {   // per-problem maps: vertex -> problem, edge ranges, len(x_global) / len(mu_global) of each problem
        int *vp = (int *)malloc(sizeof(int) * g->nV);
        long long *nx = (long long *)malloc(sizeof(long long) * h->nP), *nm = (long long *)malloc(sizeof(long long) * h->nP);
        h->he_prob_host = (int *)malloc(sizeof(int) * (size_t)(g->nH_own > 0 ? g->nH_own : 1));
        if (!vp || !nx || !nm || !h->he_prob_host) { free(vp); free(nx); free(nm); return set_err(GCS_E_NOMEM, "out of host memory%s", ""); }
        for (int q = 0; q < h->nP; ++q) {
            for (int v = g->prob_voff[q]; v < g->prob_voff[q + 1]; ++v) {
                vp[v] = q;
                for (int hh = g->he_off[v]; hh < g->he_off[v + 1]; ++hh) h->he_prob_host[hh] = q;
            }
            const long long nv = g->prob_voff[q + 1] - g->prob_voff[q], ne = g->prob_eoff[q + 1] - g->prob_eoff[q];
            nx[q] = 9 * nv + 18 * ne; nm[q] = 10 * ne;
        }
        rc = upload(&h->vprob, vp, (size_t)g->nV);
        if (!rc) rc = upload(&h->prob_eoff, g->prob_eoff, (size_t)h->nP + 1);
        if (!rc) rc = upload(&h->prob_nx, nx, (size_t)h->nP);
        if (!rc) rc = upload(&h->prob_nmu, nm, (size_t)h->nP);
        free(vp); free(nx); free(nm);
        if (rc) return rc;
    }
    for (int i = 0; i < 4; ++i) CK(cudaEventCreate(&h->ev[i]));
    return reset_ctrl(h);
}

extern "C" int gcsadmm_create(const GcsGraph *g, const GcsParams *p, int device, GcsHandle **out) {
    NvtxRange nvtx_("gcsadmm_create");
    if (!g || !out) return set_err(GCS_E_INVALID, "null argument%s", "");
    *out = nullptr;
    if (g->n != 2) return set_err(GCS_E_INVALID, "the CUDA path is specialised to n = 2 (2-D GCS)%s", "");
    if (g->nV <= 0 || g->nE < 0) return set_err(GCS_E_INVALID, "empty graph%s", "");
    int rc = validate_graph(g);
    if (rc) return rc;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return set_err(GCS_E_CUDA, "no CUDA device: libgcsadmm has no CPU path%s", ""); }
    if (device < 0 || device >= ndev) return set_err(GCS_E_INVALID, "bad device index%s", "");
    const int nP = g->nP > 1 ? g->nP : 1;
    if (nP > 1 && (g->nH_ghost > 0 || !g->prob_voff || !g->prob_eoff)) return set_err(GCS_E_INVALID, "batched problems need prob_voff / prob_eoff and cannot be vertex-partitioned%s", "");
    CK(cudaSetDevice(device));
    GcsHandle *h = new (std::nothrow) GcsHandle();
    if (!h) return set_err(GCS_E_NOMEM, "out of host memory%s", "");
    memset(h, 0, sizeof *h);
    h->device = device;
    if (p) h->p = *p; else gcsadmm_default_params(&h->p);
    if (h->p.check_every < 1) h->p.check_every = 1;
    if (!(h->p.outer_alpha > 0.0 && h->p.outer_alpha < 2.0)) h->p.outer_alpha = 1.0;
    h->nV = g->nV; h->nE = g->nE; h->nHown = g->nH_own; h->nHghost = g->nH_ghost;
    h->nP = nP;
    h->n_x = g->n_x_global ? g->n_x_global : 9LL * g->nV + 18LL * g->nE;
    h->n_mu = g->n_mu_global ? g->n_mu_global : 10LL * g->nE;
    rc = create_impl(h, g);
    if (rc) { gcsadmm_destroy(h); return rc; }      // single cleanup path: frees whatever was allocated so far
    *out = h;
    return 0;
}

extern "C" int gcsadmm_set_stream(GcsHandle *h, void *s, int external) {
    if (!h) return set_err(GCS_E_INVALID, "null handle%s", "");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    h->stream = external ? (cudaStream_t)s : h->own_stream;   // a NULL external stream is the legacy default stream
    drop_graph(h);
    return 0;
}

static GcsGraphView graph_view(const GcsHandle *h) {
    GcsGraphView G; G.nV = h->nV; G.nE = h->nE; G.poly_off = h->poly_off; G.polyA = h->polyA; G.polyb = h->polyb;
    G.he_off = h->he_off; G.he_edge = h->he_edge; G.he_flags = h->he_flags; G.vtype = h->vtype; G.cent = h->cent;
    return G;
}
static GcsStateView state_view(const GcsHandle *h) {
    GcsStateView S; S.xc = h->xc; S.mu = h->mu; S.z = h->z; S.x_v = h->x_v; S.z_v = h->z_v; S.y_v = h->y_v;
    S.ws = h->ws; S.theta = h->p.warm_theta; S.zero_tol = h->p.zero_tol;
    return S;
}
static int launch_k1(GcsHandle *h) {
    if (h->perf_on) {
        PeerPush P = {h->send_he, h->send_rank, h->send_slot, h->nsend, h->peer_on ? h->PV_dev : nullptr, h->push_ticket};
        auto *k = h->vprob ? (h->inner_on ? vertex_perf_kernel<true, true> : vertex_perf_kernel<false, true>)
                           : (h->inner_on ? vertex_perf_kernel<true, false> : vertex_perf_kernel<false, false>);
        k<<<h->perf_grid, h->perf_threads, h->perf_smem, h->stream>>>(graph_view(h), state_view(h), h->PT, h->ctrl, h->PL, P);
        return 0;
    }
    vertex_kernel<<<h->k1_blocks, h->k1_warps * 32, h->k1_smem, h->stream>>>(graph_view(h), state_view(h), h->ctrl, h->vprob, h->L, h->p.inner_tol, h->p.inner_max_iter);
    return 0;
}
// (tile_res, n) of the edge kernels: perf mode with the inner residual on -> the K1 blocks' partials; perf mode without -> (null, -1):
// "not computed this iteration" (sums[6] = -1, the absolute stop test cannot pass); exact mode -> (null, 0): sums[6] = 0
#define INNER_ARGS(h) ((h)->perf_on && (h)->inner_on ? (h)->p_tile_res : nullptr), ((h)->perf_on && (h)->nP == 1 ? ((h)->inner_on ? (h)->perf_grid : -1) : 0)
// K2-K5.  fuse: the control step runs inside the edge kernel's last block (single GPU); otherwise only sums[] is produced
static int launch_edge(GcsHandle *h, int fuse) {
    if (h->nP > 1) {   // edges, sums and control of every problem in one launch
        const int blocks = h->nP < 148 * 16 ? h->nP : 148 * 16;
        batched_edge_kernel<<<blocks, BATCH_THREADS, 0, h->stream>>>(h->nP, h->prob_eoff, h->nHown, h->edge_he_tail, h->edge_he_head, h->xc, h->mu, h->z,
                                                                     h->ctrl, h->p, h->prob_nx, h->prob_nmu, h->hist, h->hist_cap);
        return 0;
    }
    const bool oa = h->p.outer_alpha != 1.0;
    if (h->edge_coop && h->nHghost == 0 && !h->edge_counted && !(h->perf_on && h->inner_on)) {     // single-GPU throughput path
        const int nchunks = (h->nE + 31) / 32;
        int blocks = (nchunks + COOP_WARPS - 1) / COOP_WARPS;
        if (blocks > h->coop_blocks) blocks = h->coop_blocks;
        if (blocks < 1) blocks = 1;
        auto *k = oa ? edge_coop_kernel<true> : edge_coop_kernel<false>;
        k<<<blocks, EDGE_THREADS, sizeof(double) * COOP_SMEM_DOUBLES, h->stream>>>(h->nE, h->edge_he_tail, h->edge_he_head, h->perf_on ? h->p_edge_delta : nullptr,
            h->xc, h->mu, h->z, h->ctrl, h->partials, h->ticket, fuse, h->p, h->n_x, h->n_mu, h->hist, h->hist_cap, INNER_ARGS(h));
        return 0;
    }
    const bool gres = h->perf_on && h->inner_on && h->p_edge_delta && h->p_edge_cent;      // check variant in local frames
    auto *k = gres ? (oa ? edge_frames_kernel<true, true> : edge_frames_kernel<false, true>)
                   : (oa ? edge_frames_kernel<true, false> : edge_frames_kernel<false, false>);
    k<<<h->edge_blocks, EDGE_THREADS, 0, h->stream>>>(h->nE, h->nHown, h->edge_he_tail, h->edge_he_head, h->edge_counted,
        h->perf_on ? h->p_edge_delta : nullptr, h->perf_on ? h->p_edge_cent : nullptr, h->xc, h->mu, h->z, h->ctrl, h->partials, h->ticket, fuse, h->p,
        h->n_x, h->n_mu, h->hist, h->hist_cap, h->nHghost, h->PV_dev, INNER_ARGS(h));
    return 0;
}
static int launch_ctrl(GcsHandle *h) {
    if (h->nP > 1) return 0;   // fused into batched_edge_kernel
    control_kernel<<<1, 32, 0, h->stream>>>(h->ctrl, h->p, h->n_x, h->n_mu, h->hist, h->hist_cap);
    return 0;
}
// everything of an iteration after K1
static void launch_rest(GcsHandle *h) {
    if (!h->peer_on) { launch_edge(h, 1); return; }          // single GPU: 2 launches per ADMM iteration
    // perf mode: 3 launches per iteration (K1 + push by its last block | halo wait + edges + sums publish | sums wait + control)
    if (!h->perf_on) peer_push_kernel<<<1, 1024, 0, h->stream>>>(h->xc, h->send_he, h->send_rank, h->send_slot, h->nsend, h->ctrl, h->PV_dev);
    launch_edge(h, 2);
    peer_control_kernel<<<1, 32, 0, h->stream>>>(h->ctrl, h->p, h->n_x, h->n_mu, h->hist, h->hist_cap, h->PV_dev);
}
static void launch_iteration(GcsHandle *h) { launch_k1(h); launch_rest(h); }
// `iters` iterations as one CUDA graph launch (captured once per chunk length; the kernels read rho / stop from the control block)
static int launch_chunk(GcsHandle *h, int iters) {
    NvtxRange nvtx_("gcsadmm: chunk of ADMM iterations");
    // only whole chunks of check_every iterations are replayed (a remainder would force a re-instantiation every time)
    if (!h->p.use_graph || h->stream != h->own_stream || iters < 2 || iters != h->p.check_every) { for (int i = 0; i < iters; ++i) launch_iteration(h); return 0; }
    if (!h->graph_exec || h->graph_iters != iters) {
        drop_graph(h);
        cudaGraph_t graph = nullptr;
        CK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
        for (int i = 0; i < iters; ++i) launch_iteration(h);
        CK(cudaStreamEndCapture(h->stream, &graph));
        cudaError_t e = cudaGraphInstantiate(&h->graph_exec, graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) { h->graph_exec = nullptr; return set_err(GCS_E_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(e)); }
        h->graph_iters = iters;
    }
    CK(cudaGraphLaunch(h->graph_exec, h->stream));
    return 0;
}
static int set_ignore_stop(GcsHandle *h, int v) {
    if (h->nP > 1) { set_ignore_kernel<<<(h->nP + 255) / 256, 256, 0, h->stream>>>(h->ctrl, h->nP, v); return 0; }
    CK(cudaMemcpyAsync((char *)h->ctrl + offsetof(Ctrl, ignore_stop), &v, sizeof(int), cudaMemcpyHostToDevice, h->stream));
    return 0;
}
static int fetch_ctrl(GcsHandle *h) {
    CK(cudaMemcpyAsync(h->ctrl_host, h->ctrl, sizeof(Ctrl) * h->nP, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    return 0;
}
static void fill_status_one(const Ctrl *c, GcsStatus *st) {
    st->iterations = c->it; st->converged = c->opt; st->diverged = c->diverged; st->inner_fail = c->inner_fail;
    st->inner_iters = (int64_t)c->inner_iters; st->skipped = (int64_t)c->skipped; st->rho = c->rho; st->pri_res = c->pri; st->dual_res = c->dual;
    st->eps_pri = c->eps_pri; st->eps_dual = c->eps_dual; st->inner_res = c->inner; st->pri_res_ref = c->pri_g >= 0.0 ? c->pri_g : c->pri; st->dual_res_ref = c->dual_g >= 0.0 ? c->dual_g : c->dual;
}
// batched handles: iterations = max, converged = all, residuals = worst problem, counters summed
static void fill_status(const GcsHandle *h, GcsStatus *st) {
    fill_status_one(h->ctrl_host, st);
    for (int q = 1; q < h->nP; ++q) {
        GcsStatus t; fill_status_one(h->ctrl_host + q, &t);
        if (t.iterations > st->iterations) st->iterations = t.iterations;
        st->converged = st->converged && t.converged; st->diverged = st->diverged || t.diverged;
        st->inner_fail += t.inner_fail; st->inner_iters += t.inner_iters; st->skipped += t.skipped;
        if (t.pri_res > st->pri_res) { st->pri_res = t.pri_res; st->eps_pri = t.eps_pri; }
        if (t.dual_res > st->dual_res) { st->dual_res = t.dual_res; st->eps_dual = t.eps_dual; }
        if (t.inner_res > st->inner_res) st->inner_res = t.inner_res;
        if (t.pri_res_ref > st->pri_res_ref) st->pri_res_ref = t.pri_res_ref;
        if (t.dual_res_ref > st->dual_res_ref) st->dual_res_ref = t.dual_res_ref;
    }
}
static bool all_stopped(const GcsHandle *h) {
    for (int q = 0; q < h->nP; ++q) if (!h->ctrl_host[q].stop) return false;
    return true;
}
static bool any_diverged(const GcsHandle *h) {
    for (int q = 0; q < h->nP; ++q) if (h->ctrl_host[q].diverged) return true;
    return false;
}

extern "C" int gcsadmm_vertex_update(GcsHandle *h) { if (!h) return set_err(GCS_E_INVALID, "null handle%s", ""); CK(cudaSetDevice(h->device)); launch_k1(h); CK(cudaGetLastError()); return 0; }
extern "C" int gcsadmm_edge_update(GcsHandle *h) { if (!h) return set_err(GCS_E_INVALID, "null handle%s", ""); CK(cudaSetDevice(h->device)); launch_edge(h, 0); CK(cudaGetLastError()); return 0; }
extern "C" int gcsadmm_control(GcsHandle *h) { if (!h) return set_err(GCS_E_INVALID, "null handle%s", ""); CK(cudaSetDevice(h->device)); launch_ctrl(h); CK(cudaGetLastError()); return 0; }
extern "C" int gcsadmm_sums_device_ptr(GcsHandle *h, void **p) { if (!h || !p) return set_err(GCS_E_INVALID, "null argument%s", ""); *p = (char *)h->ctrl + offsetof(Ctrl, sums); return 0; }
extern "C" int gcsadmm_xc_device_ptr(GcsHandle *h, void **p) { if (!h || !p) return set_err(GCS_E_INVALID, "null argument%s", ""); *p = h->xc; return 0; }

extern "C" int gcsadmm_step(GcsHandle *h, int k) {
    if (!h) return set_err(GCS_E_INVALID, "null handle%s", "");
    CK(cudaSetDevice(h->device));
    int rc = set_ignore_stop(h, 1); if (rc) return rc;
    while (k > 0) {
        const int chunk = k < h->p.check_every ? k : h->p.check_every;
        rc = launch_chunk(h, chunk); if (rc) return rc;
        k -= chunk;
    }
    rc = set_ignore_stop(h, 0); if (rc) return rc;
    CK(cudaGetLastError());
    return fetch_ctrl(h);
}

extern "C" int gcsadmm_run(GcsHandle *h, int max_iters, GcsStatus *st) {
    NvtxRange nvtx_("gcsadmm_run");
    if (!h) return set_err(GCS_E_INVALID, "null handle%s", "");
    CK(cudaSetDevice(h->device));
    int rc = fetch_ctrl(h); if (rc) return rc;
    int done = 0;
    while (done < max_iters && !all_stopped(h)) {
        int chunk = h->p.check_every;
        if (chunk > max_iters - done) chunk = max_iters - done;
        rc = launch_chunk(h, chunk); if (rc) return rc;
        CK(cudaGetLastError());
        rc = fetch_ctrl(h); if (rc) return rc;
        done += chunk;
        if (h->perf_on && h->nP == 1 && h->p.abs_stop) {
            // near the absolute target the K1 variant that also measures the inner residual takes over (the stop test needs it);
            // far from it the throughput variant runs.  Every rank of a partitioned run sees the same control block, so all switch together.
            const int want = fmax(h->ctrl_host->pri, h->ctrl_host->dual) < 4.0 * h->p.abs_tol;
            if (want != h->inner_on) { h->inner_on = want; drop_graph(h); }
        }
    }
    if (st) fill_status(h, st);
    if (any_diverged(h)) return set_err(GCS_E_DIVERGED, "non-finite residuals (divergence)%s", "");
    return 0;
}

extern "C" int gcsadmm_get_status(GcsHandle *h, GcsStatus *st) {
    if (!h || !st) return set_err(GCS_E_INVALID, "null argument%s", "");
    CK(cudaSetDevice(h->device));
    int rc = fetch_ctrl(h); if (rc) return rc;
    fill_status(h, st);
    return 0;
}

extern "C" int gcsadmm_get_problem_status(GcsHandle *h, int problem, GcsStatus *st) {
    if (!h || !st || problem < 0 || problem >= h->nP) return set_err(GCS_E_INVALID, "bad argument%s", "");
    CK(cudaSetDevice(h->device));
    int rc = fetch_ctrl(h); if (rc) return rc;
    fill_status_one(h->ctrl_host + problem, st);
    return 0;
}
extern "C" int gcsadmm_get_problem_history(GcsHandle *h, int problem, double *rho, double *pri, double *dual, int cap) {
    if (!h || problem < 0 || problem >= h->nP) return set_err(GCS_E_INVALID, "bad argument%s", "");
    CK(cudaSetDevice(h->device));
    int rc = fetch_ctrl(h); if (rc) return rc;
    int n = h->ctrl_host[problem].it + 1;
    if (n > h->hist_cap) n = h->hist_cap;
    if (n > cap) n = cap;
    double *dst[3] = {rho, pri, dual};
    for (int k = 0; k < 3; ++k) if (dst[k]) CK(cudaMemcpy(dst[k], h->hist + ((size_t)problem * 3 + k) * h->hist_cap, sizeof(double) * n, cudaMemcpyDeviceToHost));
    return n;
}
extern "C" int gcsadmm_get_history(GcsHandle *h, double *rho, double *pri, double *dual, int cap) {
    if (!h) return set_err(GCS_E_INVALID, "null handle%s", "");
    CK(cudaSetDevice(h->device));
    int rc = fetch_ctrl(h); if (rc) return rc;
    int n = h->ctrl_host->it + 1;
    if (n > h->hist_cap) n = h->hist_cap;
    if (n > cap) n = cap;
    double *dst[3] = {rho, pri, dual};
    for (int q = 0; q < 3; ++q) if (dst[q]) CK(cudaMemcpy(dst[q], h->hist + (size_t)q * h->hist_cap, sizeof(double) * n, cudaMemcpyDeviceToHost));
    return n;
}

extern "C" int gcsadmm_get_solution(GcsHandle *h, double *x_v, double *z_v, double *y_v, double *z_e) {
    NvtxRange nvtx_("gcsadmm_get_solution");
    if (!h) return set_err(GCS_E_INVALID, "null handle%s", "");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    if (x_v) CK(cudaMemcpy(x_v, h->x_v, sizeof(double) * 4 * h->nV, cudaMemcpyDeviceToHost));
    if (z_v) CK(cudaMemcpy(z_v, h->z_v, sizeof(double) * 4 * h->nV, cudaMemcpyDeviceToHost));
    if (y_v) CK(cudaMemcpy(y_v, h->y_v, sizeof(double) * h->nV, cudaMemcpyDeviceToHost));
    if (z_e) CK(cudaMemcpy(z_e, h->z, sizeof(double) * 5 * h->nE, cudaMemcpyDeviceToHost));
    return 0;
}

extern "C" int gcsadmm_get_state(GcsHandle *h, double *xc, double *mu, double *z, double *rho, int *it) {
    if (!h) return set_err(GCS_E_INVALID, "null handle%s", "");
    CK(cudaSetDevice(h->device));
    int rc = fetch_ctrl(h); if (rc) return rc;
    if (xc) CK(cudaMemcpy(xc, h->xc, sizeof(double) * 5 * ((size_t)h->nHown + h->nHghost), cudaMemcpyDeviceToHost));
    if (mu) {   // stored duals carry a pending rho-adaptation rescale: return the effective values
        CK(cudaMemcpy(mu, h->mu, sizeof(double) * 5 * (size_t)h->nHown, cudaMemcpyDeviceToHost));
        if (h->nP > 1) { for (size_t hh = 0; hh < (size_t)h->nHown; ++hh) { const double s = h->ctrl_host[h->he_prob_host[hh]].mu_scale; if (s != 1.0) for (int c = 0; c < 5; ++c) mu[5 * hh + c] *= s; } }
        else { const double s = h->ctrl_host->mu_scale; if (s != 1.0) for (size_t i = 0; i < 5 * (size_t)h->nHown; ++i) mu[i] *= s; }
    }
    if (z) CK(cudaMemcpy(z, h->z, sizeof(double) * 5 * (size_t)h->nE, cudaMemcpyDeviceToHost));
    if (rho) *rho = h->ctrl_host->rho;
    if (it) *it = h->ctrl_host->it;
    return 0;
}

extern "C" int gcsadmm_set_state(GcsHandle *h, const double *xc, const double *mu, const double *z, double rho, int it) {
    if (!h) return set_err(GCS_E_INVALID, "null handle%s", "");
    CK(cudaSetDevice(h->device));
    int rc = fetch_ctrl(h); if (rc) return rc;
    if (xc) CK(cudaMemcpy(h->xc, xc, sizeof(double) * 5 * ((size_t)h->nHown + h->nHghost), cudaMemcpyHostToDevice));
    if (mu) CK(cudaMemcpy(h->mu, mu, sizeof(double) * 5 * (size_t)h->nHown, cudaMemcpyHostToDevice));
    if (z) CK(cudaMemcpy(h->z, z, sizeof(double) * 5 * (size_t)h->nE, cudaMemcpyHostToDevice));
    for (int q = 0; q < h->nP; ++q) { Ctrl &c = h->ctrl_host[q]; c.rho = rho; c.it = it; c.mu_scale = 1.0; c.stop = 0; c.opt = 0; c.diverged = 0; }
    CK(cudaMemcpy(h->ctrl, h->ctrl_host, sizeof(Ctrl) * h->nP, cudaMemcpyHostToDevice));
    return 0;
}

extern "C" int gcsadmm_time_steps(GcsHandle *h, int k, float *ms_total, float *ms_k1, float *ms_edge) {
    if (!h || !ms_total) return set_err(GCS_E_INVALID, "null argument%s", "");
    CK(cudaSetDevice(h->device));
    int rc = set_ignore_stop(h, 1); if (rc) return rc;
    CK(cudaStreamSynchronize(h->stream));
    float k1 = 0.f, ed = 0.f;
    const bool split = ms_k1 || ms_edge;
    CK(cudaEventRecord(h->ev[0], h->stream));
    for (int i = 0; i < k; ++i) {
        if (split) CK(cudaEventRecord(h->ev[1], h->stream));
        if (h->peer_on) launch_iteration(h); else launch_k1(h);
        if (split) CK(cudaEventRecord(h->ev[2], h->stream));
        if (!h->peer_on) launch_edge(h, 1);
        if (split) {
            CK(cudaEventRecord(h->ev[3], h->stream));
            CK(cudaEventSynchronize(h->ev[3]));
            float a = 0.f, b = 0.f;
            CK(cudaEventElapsedTime(&a, h->ev[1], h->ev[2])); CK(cudaEventElapsedTime(&b, h->ev[2], h->ev[3]));
            k1 += a; ed += b;
        }
    }
    CK(cudaEventRecord(h->ev[3], h->stream));
    CK(cudaEventSynchronize(h->ev[3]));
    CK(cudaEventElapsedTime(ms_total, h->ev[0], h->ev[3]));
    if (ms_k1) *ms_k1 = k1;
    if (ms_edge) *ms_edge = ed;
    rc = set_ignore_stop(h, 0); if (rc) return rc;
    CK(cudaGetLastError());
    return fetch_ctrl(h);
}

// k iterations enqueued back to back, each preceded by an L2 eviction (memset of flush_bytes on the same stream, outside the
// event pair) and bracketed by its own CUDA events: the host never waits between iterations, so launch latency and the skew
// between ranks of a multi-GPU run are not part of what is measured.  ms_iter[k], ms_k1[k] (optional): per-iteration times.
extern "C" int gcsadmm_time_window(GcsHandle *h, int k, long long flush_bytes, float *ms_iter, float *ms_k1) {
    NvtxRange nvtx_("gcsadmm_time_window");
    if (!h || !ms_iter || k < 1) return set_err(GCS_E_INVALID, "bad argument%s", "");
    CK(cudaSetDevice(h->device));
    if (flush_bytes > 0 && (!h->flush_buf || h->flush_bytes < (size_t)flush_bytes)) {
        if (h->flush_buf) cudaFree(h->flush_buf);
        h->flush_buf = nullptr;
        CK(cudaMalloc(&h->flush_buf, (size_t)flush_bytes));
        h->flush_bytes = (size_t)flush_bytes;
    }
    int rc = set_ignore_stop(h, 1); if (rc) return rc;
    cudaEvent_t *ev = (cudaEvent_t *)calloc(3 * (size_t)k, sizeof(cudaEvent_t));
    if (!ev) return set_err(GCS_E_NOMEM, "out of host memory%s", "");
    cudaError_t e = cudaSuccess;
    for (int i = 0; i < 3 * k && e == cudaSuccess; ++i) e = cudaEventCreate(&ev[i]);
    for (int i = 0; i < k && e == cudaSuccess; ++i) {
        if (flush_bytes > 0) cudaMemsetAsync(h->flush_buf, 0, (size_t)flush_bytes, h->stream);
        cudaEventRecord(ev[3 * i], h->stream);
        launch_k1(h);
        if (ms_k1) cudaEventRecord(ev[3 * i + 1], h->stream);
        launch_rest(h);
        e = cudaEventRecord(ev[3 * i + 2], h->stream);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    for (int i = 0; i < k && e == cudaSuccess; ++i) {
        e = cudaEventElapsedTime(&ms_iter[i], ev[3 * i], ev[3 * i + 2]);
        if (ms_k1 && e == cudaSuccess) e = cudaEventElapsedTime(&ms_k1[i], ev[3 * i], ev[3 * i + 1]);
    }
    for (int i = 0; i < 3 * k; ++i) if (ev[i]) cudaEventDestroy(ev[i]);
    free(ev);
    if (e != cudaSuccess) return set_err(GCS_E_CUDA, "time_window: %s", cudaGetErrorString(e));
    rc = set_ignore_stop(h, 0); if (rc) return rc;
    CK(cudaGetLastError());
    return fetch_ctrl(h);
}

extern "C" int gcsadmm_solve_host(const GcsGraph *g, const GcsParams *p, int device, int max_iters, GcsStatus *st,
                                  double *x_v, double *z_v, double *y_v, double *z_e,
                                  double *rho_seq, double *pri_seq, double *dual_seq, int hist_cap) {
    GcsHandle *h = nullptr;
    int rc = gcsadmm_create(g, p, device, &h);
    if (rc) return rc;
    GcsStatus local;
    rc = gcsadmm_run(h, max_iters, st ? st : &local);
    if (rc == 0 || rc == GCS_E_DIVERGED) {
        int rc2 = gcsadmm_get_solution(h, x_v, z_v, y_v, z_e);
        if (rc2 == 0 && (rho_seq || pri_seq || dual_seq)) { int n = gcsadmm_get_history(h, rho_seq, pri_seq, dual_seq, hist_cap); if (n < 0) rc2 = n; }
        if (rc == 0) rc = rc2;
    }
    gcsadmm_destroy(h);
    return rc;
}

// ------------------------------------------------------------------------------------------ peer mode (host)
// Every rank exports two CUDA IPC handles (its xc buffer and its PeerComm block); the host layer gathers them over its own
// channel (torch.distributed in gcs-admm_b200/dist.py) and hands every rank the full table.
extern "C" int gcsadmm_peer_export(GcsHandle *h, void *handles128) {
    if (!h || !handles128) return set_err(GCS_E_INVALID, "null argument%s", "");
    CK(cudaSetDevice(h->device));
    if (!h->comm) {
        CK(cudaMalloc((void **)&h->comm, sizeof(PeerComm)));
        CK(cudaMemset(h->comm, 0, sizeof(PeerComm)));
    }
    cudaIpcMemHandle_t a, b;
    CK(cudaIpcGetMemHandle(&a, h->xc));
    CK(cudaIpcGetMemHandle(&b, h->comm));
    memcpy(handles128, &a, 64); memcpy((char *)handles128 + 64, &b, 64);
    return 0;
}
extern "C" int gcsadmm_peer_connect(GcsHandle *h, int rank, int world, const void *all_handles, const int *peer_nHown, const int *peer_nHghost,
                                    int nsend, const int *send_he, const int *send_rank, const int *send_slot) {
    if (!h || !all_handles || !peer_nHown || !peer_nHghost || (nsend && (!send_he || !send_rank || !send_slot))) return set_err(GCS_E_INVALID, "null argument%s", "");
    if (world < 1 || world > GCS_MAX_PEERS || rank < 0 || rank >= world) return set_err(GCS_E_INVALID, "peer mode supports 1..8 ranks%s", "");
    if (h->nP > 1) return set_err(GCS_E_INVALID, "batched problems are not vertex-partitioned%s", "");
    if (!h->comm) return set_err(GCS_E_INVALID, "call gcsadmm_peer_export first%s", "");
    if (peer_nHown[rank] != h->nHown || peer_nHghost[rank] != h->nHghost) return set_err(GCS_E_INVALID, "peer table disagrees with this rank's sizes%s", "");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    drop_graph(h);
    PeerView V;
    memset(&V, 0, sizeof V);
    V.rank = rank; V.world = world;
    for (int j = 0; j < nsend; ++j) {
        const int q = send_rank[j];
        if (q < 0 || q >= world || q == rank || send_he[j] < 0 || send_he[j] >= h->nHown || send_slot[j] < 0 || send_slot[j] >= peer_nHghost[q])
            return set_err(GCS_E_INVALID, "bad halo send table%s", "");
        V.neighbours |= 1u << q;
    }
    for (int q = 0; q < world; ++q) {
        V.nHown[q] = peer_nHown[q]; V.nHghost[q] = peer_nHghost[q];
        if (q == rank) { V.xc[q] = h->xc; V.comm[q] = h->comm; continue; }
        cudaIpcMemHandle_t a, b;
        memcpy(&a, (const char *)all_handles + 128 * q, 64); memcpy(&b, (const char *)all_handles + 128 * q + 64, 64);
        void *px = nullptr, *pc = nullptr;
        CK(cudaIpcOpenMemHandle(&px, a, cudaIpcMemLazyEnablePeerAccess));
        h->ipc_opened[2 * q] = px;
        CK(cudaIpcOpenMemHandle(&pc, b, cudaIpcMemLazyEnablePeerAccess));
        h->ipc_opened[2 * q + 1] = pc;
        V.xc[q] = (double *)px; V.comm[q] = (PeerComm *)pc;
    }
    int rc = 0;
    if (!rc) rc = upload(&h->send_he, send_he, (size_t)nsend);
    if (!rc) rc = upload(&h->send_rank, send_rank, (size_t)nsend);
    if (!rc) rc = upload(&h->send_slot, send_slot, (size_t)nsend);
    if (rc) return rc;
    if (!h->PV_dev) CK(cudaMalloc((void **)&h->PV_dev, sizeof(PeerView)));
    CK(cudaMemcpy(h->PV_dev, &V, sizeof(PeerView), cudaMemcpyHostToDevice));
    h->nsend = nsend; h->rank = rank; h->world = world; h->PV = V; h->peer_on = 1;
    return 0;
}
extern "C" int gcsadmm_peer_error(GcsHandle *h) {
    if (!h || !h->comm) return 0;
    int e = 0;
    cudaSetDevice(h->device);
    cudaMemcpy(&e, (char *)h->comm + offsetof(PeerComm, error), sizeof(int), cudaMemcpyDeviceToHost);
    return e;
}

// Evicts the L2 (126 MB on B200) by overwriting a scratch buffer larger than it, on the handle's stream.
extern "C" int gcsadmm_flush_l2(GcsHandle *h, long long bytes) {
    if (!h) return set_err(GCS_E_INVALID, "null handle%s", "");
    CK(cudaSetDevice(h->device));
    if (bytes <= 0) bytes = 256ll << 20;
    if (!h->flush_buf || h->flush_bytes < (size_t)bytes) {
        if (h->flush_buf) cudaFree(h->flush_buf);
        h->flush_buf = nullptr;
        CK(cudaMalloc(&h->flush_buf, (size_t)bytes));
        h->flush_bytes = (size_t)bytes;
    }
    CK(cudaMemsetAsync(h->flush_buf, 0, (size_t)bytes, h->stream));
    return 0;
}

// Switches the x-update to the inexact `perf` mode (vertex_perf.cuh).  Tables are built by the host
// (gcs-admm_b200/perf.py): the structured v-step of every vertex class, the polygon cones, the block list and the tiling.
extern "C" int gcsadmm_enable_perf(GcsHandle *h, const GcsPerfConfig *c) {
    NvtxRange nvtx_("gcsadmm_enable_perf");
    if (!h || !c) return set_err(GCS_E_INVALID, "null argument%s", "");
    if (c->inner_iters < 1 || c->n_classes < 1 || c->n_tiles < 1 || c->n_blocks < 0 || !c->vclass || !c->cls_tab || !c->cone_off || !c->cone ||
        !c->blk_off || !c->tile_voff || (c->n_blocks && (!c->blk_he || !c->blk_info)))
        return set_err(GCS_E_INVALID, "incomplete perf-mode tables%s", "");
    if (!(c->alpha > 0.0 && c->alpha < 2.0) || !(c->kappa > 0.0)) return set_err(GCS_E_INVALID, "perf mode needs 0 < alpha < 2 and kappa > 0%s", "");
    // consistency of the tables with the graph (bad offsets would be out-of-bounds accesses in the kernel)
    if (c->tile_voff[0] != 0 || c->tile_voff[c->n_tiles] != h->nV || c->blk_off[0] != 0 || c->blk_off[h->nV] != c->n_blocks || c->cone_off[0] != 0)
        return set_err(GCS_E_INVALID, "perf-mode offsets do not span the graph%s", "");
    for (int t = 0; t < c->n_tiles; ++t) {
        const int a = c->tile_voff[t], b = c->tile_voff[t + 1];
        if (b <= a || b > h->nV || b - a > 255 || b - a > c->cap_verts || c->blk_off[b] - c->blk_off[a] > c->cap_blocks ||
            c->cone_off[b] - c->cone_off[a] > c->cap_cone || c->blk_off[b] < c->blk_off[a] || c->cone_off[b] < c->cone_off[a])
            return set_err(GCS_E_INVALID, "perf-mode tile exceeds the declared capacities%s", "");
    }
    for (int v = 0; v < h->nV; ++v) if (c->vclass[v] >= c->n_classes) return set_err(GCS_E_INVALID, "vclass out of range%s", "");
    for (int b = 0; b < c->n_blocks; ++b) if (c->blk_he[b] >= h->nHown) return set_err(GCS_E_INVALID, "blk_he out of range%s", "");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    drop_graph(h);
    free_perf(h);                 // a second call replaces the tables of the first
    int rc = 0;
    const size_t ncone = (size_t)c->cone_off[h->nV];
    if (!rc) rc = upload(&h->p_vclass, c->vclass, (size_t)h->nV);
    if (!rc) rc = upload(&h->p_cls_tab, c->cls_tab, (size_t)c->n_classes * GCS_CLS_STRIDE);
    if (!rc) rc = upload(&h->p_cone_off, c->cone_off, (size_t)h->nV + 1);
    if (!rc) rc = upload(&h->p_cone, c->cone, GCS_CONE_REC * ncone);
    if (!rc) rc = upload(&h->p_blk_off, c->blk_off, (size_t)h->nV + 1);
    if (!rc) {
        // packed descriptors the kernel stages with bulk copies: 4 ints per block, GCS_VI_N ints per vertex, 8 ints per tile
        const size_t nB = (size_t)c->n_blocks, nVt = (size_t)h->nV, nT = (size_t)c->n_tiles;
        int *brec = (int *)calloc(4 * (nB ? nB : 1), sizeof(int)), *vrec = (int *)calloc(GCS_VI_N * nVt, sizeof(int)), *trec = (int *)calloc(8 * nT, sizeof(int));
        int *he_edge = (int *)malloc(sizeof(int) * (size_t)(h->nHown > 0 ? h->nHown : 1)), *he_off = (int *)malloc(sizeof(int) * (nVt + 1));
        unsigned char *vtype = (unsigned char *)malloc(nVt), *he_flags = (unsigned char *)malloc((size_t)(h->nHown > 0 ? h->nHown : 1));
        int *vprob = (int *)calloc(nVt, sizeof(int));
        if (!brec || !vrec || !trec || !he_edge || !he_off || !vtype || !he_flags || !vprob) rc = set_err(GCS_E_NOMEM, "out of host memory%s", "");
        if (!rc) {
            cudaMemcpy(he_edge, h->he_edge, sizeof(int) * (size_t)h->nHown, cudaMemcpyDeviceToHost);
            cudaMemcpy(he_off, h->he_off, sizeof(int) * (nVt + 1), cudaMemcpyDeviceToHost);
            cudaMemcpy(vtype, h->vtype, nVt, cudaMemcpyDeviceToHost);
            cudaMemcpy(he_flags, h->he_flags, (size_t)h->nHown, cudaMemcpyDeviceToHost);
            if (h->vprob) cudaMemcpy(vprob, h->vprob, sizeof(int) * nVt, cudaMemcpyDeviceToHost);
            for (size_t b = 0; b < nB; ++b) {
                brec[4 * b] = c->blk_he[b]; brec[4 * b + 1] = c->blk_info[b]; brec[4 * b + 2] = c->blk_he[b] >= 0 ? he_edge[c->blk_he[b]] : -1;
            }
            for (int t = 0; t < c->n_tiles && !rc; ++t) {
                const int a = c->tile_voff[t], b = c->tile_voff[t + 1];
                int *r = trec + 8 * (size_t)t;
                r[0] = a; r[1] = b - a; r[2] = c->blk_off[a]; r[3] = c->blk_off[b] - c->blk_off[a];
                r[4] = c->cone_off[a]; r[5] = c->cone_off[b] - c->cone_off[a]; r[6] = he_off[a]; r[7] = he_off[b] - he_off[a];
                bool zero = false;
                for (int hh = he_off[a]; hh < he_off[b]; ++hh) zero = zero || (he_flags[hh] & GCS_HE_FLAG_ZERO);
                if (zero) r[7] |= 1 << 30;
                for (int v = a; v < b && !rc; ++v) {
                    // the kernel sums the in- and the out-blocks of a vertex as two ranges: in-blocks first, then out-blocks, then its z-block
                    int nin = 0, g = 0;
                    for (int bb = c->blk_off[v]; bb < c->blk_off[v + 1]; ++bb) {
                        const int gb = (c->blk_info[bb] >> 8) & 3;
                        if (gb < g || (gb == 2) != (bb == c->blk_off[v + 1] - 1)) rc = set_err(GCS_E_INVALID, "perf-mode blocks of a vertex are not in-, out-, z-block order%s", "");
                        g = gb; nin += gb == 0;
                    }
                    int *w = vrec + GCS_VI_N * (size_t)v;
                    w[GCS_VI_CONE] = c->cone_off[v] - c->cone_off[a]; w[GCS_VI_NV] = c->cone_off[v + 1] - c->cone_off[v];
                    w[GCS_VI_CLS] = c->vclass[v]; w[GCS_VI_TERM] = (vtype[v] != GCS_VT_GENERIC) | (nin << 1);
                    w[GCS_VI_BLK] = c->blk_off[v] - c->blk_off[a]; w[GCS_VI_NB] = c->blk_off[v + 1] - c->blk_off[v];
                    w[GCS_VI_ACTIVE] = vprob[v]; w[GCS_VI_HE] = he_off[v] - he_off[a];
                }
            }
            if (!rc) rc = upload(&h->p_blk_rec, brec, 4 * nB);
            if (!rc) rc = upload(&h->p_vrec, vrec, GCS_VI_N * nVt);
            if (!rc) rc = upload(&h->p_tile_rec, trec, 8 * nT);
        }
        free(brec); free(vrec); free(trec); free(he_edge); free(he_off); free(vtype); free(he_flags); free(vprob);
    }
    if (!rc) rc = upload(&h->p_tstate, (const double *)nullptr, 12 * (size_t)c->n_blocks);
    if (!rc) rc = upload(&h->p_tn, (const double *)nullptr, 2 * (size_t)h->nV);
    if (!rc) rc = upload(&h->p_tile_res, (const double *)nullptr, (size_t)c->n_tiles);
    if (!rc && c->edge_delta) rc = upload(&h->p_edge_delta, c->edge_delta, 2 * (size_t)h->nE);
    if (!rc && c->edge_delta && c->edge_cent) rc = upload(&h->p_edge_cent, c->edge_cent, 2 * (size_t)h->nE);
    if (rc) { free_perf(h); return rc; }
    h->perf_nblocks = c->n_blocks;
    h->PL = gcs_perf_layout(c->cap_blocks, c->cap_verts, c->cap_cone);
    h->PT.vclass = h->p_vclass; h->PT.cls_tab = h->p_cls_tab; h->PT.cone_off = h->p_cone_off; h->PT.cone = h->p_cone;
    h->PT.blk_off = h->p_blk_off; h->PT.blk_rec = h->p_blk_rec; h->PT.vrec = h->p_vrec; h->PT.tile_rec = h->p_tile_rec;
    h->PT.ntiles = c->n_tiles; h->PT.tstate = h->p_tstate; h->PT.tn = h->p_tn; h->PT.inner_iters = c->inner_iters;
    h->PT.alpha = c->alpha; h->PT.kappa = c->kappa; h->PT.theta = c->theta > 0.0 ? c->theta : 1.0; h->PT.edge_delta = h->p_edge_delta; h->PT.tile_res = h->p_tile_res;
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, h->device));
    const size_t bytes = (size_t)(h->PL.work + 2 * h->PL.stage) * sizeof(double);      // work arrays + two stage buffers
    if (bytes > prop.sharedMemPerBlockOptin) { free_perf(h); return set_err(GCS_E_INVALID, "perf-mode tile too large for shared memory (a vertex of very high degree)%s", ""); }
    h->perf_smem = (int)bytes;
    h->perf_threads = c->threads >= 32 && c->threads <= GCS_PERF_THREADS ? (c->threads / 32) * 32 : GCS_PERF_THREADS;
    {   // persistent grid: as many blocks as are resident at once (GCS_PERF_BLOCKS_PER_SM: tuning knob), never more than tiles
        const char *bps = getenv("GCS_PERF_BLOCKS_PER_SM");
        int per_sm = bps && atoi(bps) > 0 ? atoi(bps) : 4;
        const int by_smem = (int)(prop.sharedMemPerMultiprocessor / (bytes + 1024));
        if (per_sm > by_smem) per_sm = by_smem > 0 ? by_smem : 1;
        const long long cap = (long long)prop.multiProcessorCount * per_sm;
        h->perf_grid = (int)(c->n_tiles < cap ? c->n_tiles : cap);
    }
    for (auto *k : {vertex_perf_kernel<false, false>, vertex_perf_kernel<true, false>, vertex_perf_kernel<false, true>, vertex_perf_kernel<true, true>}) {
        CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, h->perf_smem));
        CK(cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    }
    perf_init_dead_kernel<<<(h->nV + 255) / 256, 256, 0, h->stream>>>(graph_view(h), state_view(h));
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(h->stream));
    h->perf_on = 1;
    return 0;
}

extern "C" int gcsadmm_get_perf_state(GcsHandle *h, double *tstate, double *tn) {
    if (!h || !h->perf_on) return set_err(GCS_E_INVALID, "perf mode is not enabled%s", "");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    if (tstate && h->perf_nblocks) CK(cudaMemcpy(tstate, h->p_tstate, sizeof(double) * 12 * (size_t)h->perf_nblocks, cudaMemcpyDeviceToHost));
    if (tn) CK(cudaMemcpy(tn, h->p_tn, sizeof(double) * 2 * (size_t)h->nV, cudaMemcpyDeviceToHost));
    return 0;
}
extern "C" int gcsadmm_set_perf_state(GcsHandle *h, const double *tstate, const double *tn) {
    if (!h || !h->perf_on) return set_err(GCS_E_INVALID, "perf mode is not enabled%s", "");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    if (tstate && h->perf_nblocks) CK(cudaMemcpy(h->p_tstate, tstate, sizeof(double) * 12 * (size_t)h->perf_nblocks, cudaMemcpyHostToDevice));
    if (tn) CK(cudaMemcpy(h->p_tn, tn, sizeof(double) * 2 * (size_t)h->nV, cudaMemcpyHostToDevice));
    return 0;
}
