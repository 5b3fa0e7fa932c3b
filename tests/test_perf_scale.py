"""GPU: perf mode at the scale of the benchmark, against the host build of the same kernel source (test_perf_mode.EmuPerfADMM),
iterate by iterate.  What only runs at scale: persistent K1 blocks that walk several tiles (second stage buffer, mbarrier phase
flip, refill while the previous tile's bulk stores drain), the grid-stride loop of the warp-cooperative edge kernel, the
mid-run switch to the INNER K1 and the edge kernel with global-coordinate residuals under CUDA graph replay, and tiles larger
than one pass of the block's threads."""
import functools

import numpy as np
import pytest

from conftest import load_golden
from gcs_admm_b200 import perf, warmstart
from gcs_admm_b200.generator import generate_test_2D, grid_packed_graph
from gcs_admm_b200.graph import pack_graph
import test_perf_mode as TPM

pytestmark = pytest.mark.gpu

# the accelerated configuration of bench.py's time-to-residual run (bench.TTR): local frames, rho0 = 3, over-relaxed consensus
# step, duals started from the portal-graph cost-to-go field, the reference rho rule during the first frac * max_it iterations
RHO0, OA, MAX_IT, FRAC = 3.0, 1.7, 1000, 0.1


@pytest.fixture(scope="module")
def lib():
    return TPM.load_emu()


@functools.lru_cache(maxsize=None)
def grid(G):
    return grid_packed_graph(G)


def box(x0, y0, x1, y1):
    return np.array([[1.0, 0.0], [-1.0, 0.0], [0.0, 1.0], [0.0, -1.0]]), np.array([x1, -x0, y1, -y0])


def hub(n):
    """a corridor box under a row of n unit boxes, each overlapping its neighbours: the corridor's live degree is 2 n"""
    As, bs = {}, {}
    As["s"], bs["s"] = box(0.2, 0.6, 0.4, 0.8)                   # inside the first box only
    As["t"], bs["t"] = box(n - 0.6, 0.6, n - 0.4, 0.8)           # inside the last box only
    As[0], bs[0] = box(-0.5, -0.25, n + 0.5, 0.25)
    for i in range(n):
        As[i + 1], bs[i + 1] = box(i - 0.1, 0.0, i + 1.1, 1.0)
    return As, bs


def problem(name):
    if name == "gen5":
        return pack_graph(*generate_test_2D(None, -20, 20, 1, 0.9, 40, seed=5)[:2])
    if name == "hub":
        return pack_graph(*hub(21))
    if name.startswith("grid"):
        return grid(int(name[4:]))
    return pack_graph(*load_golden(name)[:2])


class EmuBench(TPM.EmuPerfADMM):
    """the emulator with the device's adaptation window: the reference rho rule on iterations it < frac * max_it only"""

    def __init__(self, *args, frac=FRAC, max_it=MAX_IT, **kw):
        super().__init__(*args, adapt=True, **kw)
        self.window, self.rhos = frac * max_it, []

    def _adapt(self):
        self.adapt = len(self.pri) - 1 < self.window
        super()._adapt()
        self.rhos.append(self.rho)


def bench_pair(lib, g, check_every, rho0=RHO0, **params):
    """(device handle, emulator) in the bench's time-to-residual configuration, from the same warm start"""
    from gcs_admm_b200.lib import Solver
    T = perf.perf_tables(g, frames="local")
    s = Solver(g, max_it=MAX_IT, check_every=check_every, frac=FRAC, rho0=rho0, outer_alpha=OA, use_graph=1, **params)
    s.enable_perf(inner_iters=1, tables=T).warm_start("dijkstra", rho=rho0)
    a = EmuBench(lib, g, K=1, frames="local", outer_alpha=OA)
    a.rho, a.mu = rho0, warmstart.dual_start(g, T["edge_delta"], rho0)
    return s, a


def compare(s, a, tag):
    """every iterate of the device within 1e-9 of the emulator's (scaled by max(1, max |ref|)), rho exactly, residuals to 1e-9"""
    xc, mu, z, rho, it = s.state()
    t, tn = s.perf_state()
    x_v, z_v, y_v, z_e = s.solution()
    worst = {}
    for k, got, ref in (("xc", xc, a.xc), ("z", z, a.z), ("mu", mu, a.ms * a.mu), ("tstate", t, a.tstate), ("tn", tn, a.tn),
                        ("z_v", z_v, a.z_v), ("y_v", y_v, a.y_v)):
        worst[k] = float(np.max(np.abs(got - ref))) / max(1.0, float(np.max(np.abs(ref))))
    rh, pri, dual = s.history()
    worst["pri"] = float(np.max(np.abs(pri - a.pri) / np.maximum(np.abs(a.pri), 1e-3)))
    worst["dual"] = float(np.max(np.abs(dual - a.dual) / np.maximum(np.abs(a.dual), 1e-3)))
    print(f"{tag} it {it}: " + ", ".join(f"{k} {v:.1e}" for k, v in worst.items()))
    assert it == len(a.pri) - 1 and rho == a.rho and np.array_equal(rh[1:], a.rhos), tag
    assert all(worst[k] <= 1e-9 for k in ("xc", "z", "mu", "tstate", "tn", "z_v", "y_v")), (tag, worst)
    assert np.allclose(pri, a.pri, rtol=1e-9, atol=1e-12) and np.allclose(dual, a.dual, rtol=1e-9, atol=1e-12), tag
    return worst


@pytest.mark.parametrize("G,iters,check_every,blocks_per_sm,rho0", [(100, 150, 64, None, RHO0), (100, 150, 8, None, 30.0),
                                                                     (316, 40, 8, None, RHO0), (64, 60, 8, "1", 30.0)])
def test_bench_configuration_equals_emulation(lib, monkeypatch, G, iters, check_every, blocks_per_sm, rho0):
    """100 x 100: 1 423 tiles = 3 rounds of the 592 persistent K1 blocks, graph replays of 64 and of 8 iterations;
    316 x 316: 14 246 tiles (25 rounds) and 12 443 edge chunks (6 grid-stride passes per warp);
    64 x 64 with one K1 block per SM: 148 blocks walk 582 tiles (4 rounds).
    With rho0 = 3 the bench's residuals stay balanced and rho never moves; rho0 = 30 makes the reference rule lower it inside the
    adaptation window, so the deferred rescale of mu and lam runs inside a graph replay"""
    if blocks_per_sm:
        monkeypatch.setenv("GCS_PERF_BLOCKS_PER_SM", blocks_per_sm)      # read by gcsadmm_enable_perf
    g = grid(G)
    s, a = bench_pair(lib, g, check_every, rho0)
    print(f"grid {G}: {s.perf['n_tiles']} tiles, {(g.nE + 31) // 32} edge chunks")
    done = 0
    while done < iters:
        k = min(check_every, iters - done)
        for _ in range(k):
            a.step()
        s.step(k)                  # k == check_every: one CUDA graph launch of k iterations
        done += k
        compare(s, a, f"grid{G} check_every {check_every}")
    if rho0 != RHO0:
        assert len(set(a.rhos)) > 1
    s.close()


def test_inner_switch_at_scale(lib):
    """abs_stop with a huge tolerance: the first chunk runs the throughput kernels, then gcsadmm_run switches to the INNER K1 and the
    edge kernel with global-coordinate residuals (a new graph), and the run stops at iteration check_every + 1"""
    g = grid(316)
    s, a = bench_pair(lib, g, 8, abs_stop=1, abs_tol=1e9)
    st = s.run(8)
    assert st["iterations"] == 8 and not st["converged"] and st["inner_res"] == -1.0
    for _ in range(8):
        a.step()
    compare(s, a, "316 before the switch")
    xc8, mu8, z8, rho8, _ = s.state()
    st = s.run(56)
    assert st["converged"] == 1 and st["iterations"] == 9
    a.inner = True
    a.step()
    compare(s, a, "316 INNER")
    got, ref = st["inner_res"], float(np.sqrt(a.inner_sq))
    print(f"inner_res {got:.15e} emulator {ref:.15e} rel {abs(got - ref) / ref:.1e}")
    assert abs(got - ref) <= 1e-10 * ref
    xc, mu, z, rho, it = s.state()
    s.close()
    T = a.T
    d, cu = T["edge_delta"], T["edge_cent"]
    cw = cu - d
    xt, xh = xc[g.edge_he_tail], xc[g.edge_he_head]
    bz = z.copy()
    bz[:, 2:4] -= d * z[:, 4:5]
    rt, rh = bz - xt, z - xh
    gt = rt.copy(); gt[:, 0:2] += rt[:, 4:5] * cu; gt[:, 2:4] += rt[:, 4:5] * cu
    gh = rh.copy(); gh[:, 0:2] += rh[:, 4:5] * cu; gh[:, 2:4] += rh[:, 4:5] * cw
    pri_ref = np.sqrt(np.sum(gt ** 2) + np.sum(gh ** 2))
    dz = z - z8
    gz = dz.copy(); gz[:, 0:2] += dz[:, 4:5] * cu; gz[:, 2:4] += dz[:, 4:5] * cw
    dual_ref = rho8 * np.sqrt(2.0 * np.sum(gz ** 2))
    print(f"pri_res_ref {st['pri_res_ref']:.15e} numpy {pri_ref:.15e}; dual_res_ref {st['dual_res_ref']:.15e} numpy {dual_ref:.15e}")
    assert abs(st["pri_res_ref"] - pri_ref) <= 1e-10 * pri_ref
    assert abs(st["dual_res_ref"] - dual_ref) <= 1e-10 * dual_ref


@pytest.mark.parametrize("oa", [1.0, 1.7])
@pytest.mark.parametrize("name", ["grid316", "test1", "benchmark4"])
def test_edge_kernels_agree_bit_for_bit(monkeypatch, name, oa):
    """the warp-cooperative edge kernel (throughput path) and the one-thread-per-edge kernel (check variant, multi-GPU) on the
    same state: identical z and mu.  316 x 316: many chunks per warp; test1: 4 edges, one partial chunk."""
    from gcs_admm_b200.lib import Solver
    g = problem(name)
    T = perf.perf_tables(g, frames="local")
    rng = np.random.default_rng(7)
    xc, mu, z = rng.normal(size=(g.H, 5)), rng.normal(size=(g.H, 5)) * 0.3, rng.normal(size=(g.nE, 5))
    xc[:, 4] = rng.uniform(0, 1, g.H); z[:, 4] = rng.uniform(0, 1, g.nE)
    out = []
    for kernel in ("coop", "per_edge"):
        if kernel == "per_edge":
            monkeypatch.setenv("GCS_EDGE_KERNEL", "per_edge")     # read by gcsadmm_create
        s = Solver(g, max_it=100, outer_alpha=oa).enable_perf(inner_iters=1, tables=T)
        s.set_state(xc, mu, z, 2.0, 5)
        s.edge_update()
        out.append(s.state())
        s.close()
    (_, mu1, z1, _, _), (_, mu2, z2, _, _) = out
    print(f"{name} oa {oa}: max |dz| {np.max(np.abs(z1 - z2)):.1e}, max |dmu| {np.max(np.abs(mu1 - mu2)):.1e}")
    assert np.array_equal(z1, z2) and np.array_equal(mu1, mu2)


@pytest.mark.parametrize("threads", [64, 128, 256])
@pytest.mark.parametrize("name", ["benchmark3", "benchmark4", "gen5", "hub"])
def test_large_tiles_equal_emulation(lib, monkeypatch, name, threads):
    """tiles of up to 256 blocks: more consensus targets than the register prefetch covers (GCS_PF x threads) and more pairs than
    threads, so the strided target loop and the multi-pass P2 / P7 loops of the device build run"""
    from gcs_admm_b200.lib import Solver
    monkeypatch.setattr(perf, "TILE_BLOCKS", 256)
    monkeypatch.setattr(perf, "TILE_HE", 256)
    monkeypatch.setattr(perf, "TILE_THREADS", threads)
    g = problem(name)
    if name == "hub":
        assert g.max_live_degree == 42
    T = perf.perf_tables(g)
    nb = np.diff(T["blk_off"][T["tile_voff"]])
    print(f"{name}, {threads} threads: blocks per tile {nb.tolist()}, targets {(5 * nb).tolist()} "
          f"(prefetch {3 * threads}), pairs {(4 * nb).tolist()}")
    if threads == 64:
        assert np.any((5 * nb > 3 * threads) & (4 * nb > threads))
    a = TPM.EmuPerfADMM(lib, g, K=2, adapt=True)
    assert np.array_equal(a.T["tile_voff"], T["tile_voff"])
    s = Solver(g, frac=1.0, max_it=MAX_IT, use_graph=0).enable_perf(inner_iters=2, tables=T)
    a.rhos = []
    for it in range(60):
        a.step()
        a.rhos.append(a.rho)
        s.step(1)
        if it % 10 == 9:
            compare(s, a, f"{name} {threads} threads")
    s.close()


def test_hub_of_degree_64_is_refused():
    """gcsadmm_create sizes the exact-mode vertex program for the largest live degree: at 64 its scratch (481 KB per warp) does
    not fit in shared memory and the handle is refused, even when the caller means to run perf mode only"""
    from gcs_admm_b200.lib import GcsError, Solver
    g = pack_graph(*hub(32))
    assert g.max_live_degree == 64
    with pytest.raises(GcsError) as e:
        Solver(g)
    assert e.value.code == -1 and "vertex program too large" in str(e.value)
