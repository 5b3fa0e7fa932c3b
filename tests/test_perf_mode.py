"""`perf` mode of K1 (K closed-form splitting iterations per x-update) on the CPU: the kernel source compiled with
GCS_EMULATE against the numpy prototype of the same iteration written in the LITERAL variables of the reference
program (tools/prototypes/inner_first_order.py), and the convergence of the resulting inexact ADMM to the
classic relaxation optimum."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, load_golden
from gcs_admm_b200 import perf
from gcs_admm_b200.graph import pack_graph

sys.path.insert(0, os.path.join(ROOT, "tools", "prototypes"))
CSRC = os.path.join(ROOT, "gcs-admm_b200", "csrc")
_dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_ip = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_bp = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")


def load_emu():
    from conftest import build_emu
    lib = C.CDLL(build_emu())
    perf_args = [C.c_int, C.c_int, _ip, _dp, _dp, _ip, _ip, _bp, _bp, _dp, _dp, _dp, _dp, _dp, _dp, _dp,
                 C.c_double, C.c_double, _ip, _dp, _ip, _dp, _ip, _ip, _ip, _ip, _ip, C.c_int,
                 C.c_int, C.c_int, C.c_int, _dp, _dp, C.c_int, C.c_double, C.c_double, C.c_double, C.c_void_p]
    lib.gcsemu_vertex_update_perf_all.restype = C.c_int
    lib.gcsemu_vertex_update_perf_all.argtypes = perf_args
    lib.gcsemu_vertex_update_perf_inner.restype = C.c_int
    lib.gcsemu_vertex_update_perf_inner.argtypes = perf_args + [C.POINTER(C.c_double)]
    lib.gcsemu_cone_project.restype = None
    lib.gcsemu_cone_project.argtypes = [_dp, C.c_int, _dp, C.c_int, _dp]
    return lib


@pytest.fixture(scope="module")
def emu():
    return load_emu()


class EmuPerfADMM:
    """Outer ADMM (numpy edge / dual / residual / rho arithmetic of the kernels) around the emulated perf K1."""

    def __init__(self, lib, g, K, kappa=1.0, alpha=1.6, outer_alpha=1.0, adapt=False, nu=10.0, tau=2.0, theta=1.0, frames="global"):
        self.lib, self.g, self.K, self.alpha, self.oa, self.adapt, self.nu, self.tau = lib, g, K, alpha, outer_alpha, adapt, nu, tau
        self.T = perf.perf_tables(g, kappa, theta=theta, frames=frames)
        self.theta, self.delta = theta, self.T["edge_delta"]
        self.tstate, self.tn = np.zeros((self.T["blk_he"].shape[0], 12)), np.zeros((g.nV, 2))
        self.blk_edge = np.where(self.T["blk_he"] >= 0, g.he_edge[np.maximum(self.T["blk_he"], 0)], -1).astype(np.int32)
        self.xc, self.mu, self.z = np.zeros((g.H, 5)), np.zeros((g.H, 5)), np.zeros((g.nE, 5))
        self.x_v, self.z_v, self.y_v = np.zeros((g.nV, 4)), np.zeros((g.nV, 4)), np.zeros(g.nV)
        self.cent = np.ascontiguousarray(g.interior_points())
        self.rho, self.ms, self.pri, self.dual = 1.0, 1.0, [0.0], [0.0]
        self.inner = False                   # True: vertex_update runs the INNER variant of K1 and sets inner_sq
        self.inner_sq = None

    def vertex_update(self):
        """inner = True: the INNER variant of K1, which also leaves the squared inner residual of this update in inner_sq"""
        g, T = self.g, self.T
        args = (g.nV, g.nE, g.poly_off, g.polyA.reshape(-1), g.polyb, g.he_off, g.he_edge, g.he_flags,
                g.vtype, self.cent.reshape(-1), self.xc.reshape(-1), self.mu.reshape(-1), self.z.reshape(-1),
                self.x_v.reshape(-1), self.z_v.reshape(-1), self.y_v, self.rho, self.ms,
                T["vclass"], T["cls_tab"], T["cone_off"], T["cone"].reshape(-1), T["blk_off"], T["blk_he"],
                self.blk_edge, T["blk_info"], T["tile_voff"], T["tile_voff"].shape[0] - 1, T["caps"]["nb"], T["caps"]["nvt"],
                T["caps"]["cone"], self.tstate.reshape(-1), self.tn.reshape(-1), self.K, self.alpha, T["kappa"], self.theta,
                None if self.delta is None else self.delta.ctypes.data_as(C.c_void_p))
        if self.inner:
            sq = C.c_double()
            self.lib.gcsemu_vertex_update_perf_inner(*args, C.byref(sq))
            self.inner_sq = sq.value
        else:
            self.lib.gcsemu_vertex_update_perf_all(*args)

    def step_frames(self):
        """local frames: z = argmin |x_head - z|^2 + |x_tail - B z|^2,  B (p1, p2, y) = (p1, p2 - y delta, y)  (gcsadmm.cu edge_frames_kernel)"""
        g, d = self.g, self.delta
        self.vertex_update()
        xt, xh = self.xc[g.edge_he_tail], self.xc[g.edge_he_head]
        at, ah = xt, xh
        if self.oa != 1.0:                   # over-relaxed consensus step: x -> oa x + (1 - oa) (B) z_old in the z- and mu-updates
            bo = self.z.copy()
            bo[:, 2:4] -= d * self.z[:, 4:5]
            at, ah = self.oa * xt + (1 - self.oa) * bo, self.oa * xh + (1 - self.oa) * self.z
        xt_true, xh_true = xt, xh
        xt, xh = at, ah
        zn = np.empty_like(self.z)
        zn[:, 0:2] = 0.5 * (xh[:, 0:2] + xt[:, 0:2])
        q = xh[:, 2:4] + xt[:, 2:4]
        q2 = xh[:, 4] + xt[:, 4] - np.sum(d * xt[:, 2:4], axis=1)
        zn[:, 4] = (q2 + 0.5 * np.sum(d * q, axis=1)) / (2.0 + 0.5 * np.sum(d * d, axis=1))
        zn[:, 2:4] = 0.5 * (q + d * zn[:, 4:5])
        dz = zn - self.z
        self.z = zn
        bz, dbz = zn.copy(), dz.copy()
        bz[:, 2:4] -= d * zn[:, 4:5]; dbz[:, 2:4] -= d * dz[:, 4:5]
        r, rh = np.zeros_like(self.xc), np.zeros_like(self.xc)
        r[g.edge_he_head] = zn - xh_true
        r[g.edge_he_tail] = bz - xt_true
        rh[g.edge_he_head] = zn - xh
        rh[g.edge_he_tail] = bz - xt
        self.mu = self.ms * self.mu + rh
        self.pri.append(float(np.sqrt(np.sum(r * r)))); self.dual.append(self.rho * float(np.sqrt(np.sum(dz * dz) + np.sum(dbz * dbz))))
        self._adapt()

    def _adapt(self):
        pri, dual = self.pri[-1], self.dual[-1]
        self.ms = 1.0
        if self.adapt:                       # reference rho rule (:703-709) over the whole run; the rescale of mu is deferred like on the device
            if pri >= self.nu * dual:
                self.rho *= self.tau; self.ms = 1.0 / self.tau
            elif dual >= self.nu * pri:
                self.rho /= self.tau; self.ms = self.tau

    def step(self):
        if self.delta is not None:
            return self.step_frames()
        g = self.g
        self.vertex_update()
        xt, xh = self.xc[g.edge_he_tail], self.xc[g.edge_he_head]
        at, ah = (xt, xh) if self.oa == 1.0 else (self.oa * xt + (1 - self.oa) * self.z, self.oa * xh + (1 - self.oa) * self.z)
        zn = 0.5 * (at + ah)
        dz = zn - self.z
        self.z = zn
        r = zn[g.he_edge] - self.xc
        hat = self.xc if self.oa == 1.0 else None
        if hat is None:
            hat = np.empty_like(self.xc)
            hat[g.edge_he_tail] = at; hat[g.edge_he_head] = ah
        self.mu = self.ms * self.mu + (zn[g.he_edge] - hat)
        wz = np.array([1.0, 1.0, 1.0, 1.0, self.theta])          # the dual residual carries the penalty of every scalar
        pri, dual = float(np.sqrt(np.sum(r * r))), self.rho * float(np.sqrt(2 * np.sum((dz * wz) ** 2)))
        self.pri.append(pri); self.dual.append(dual)
        self._adapt()

    def cost(self):
        return float(np.sum(np.linalg.norm(self.z_v[:, :2] - self.z_v[:, 2:], axis=1)) + 1e-4 * np.sum(self.z[:, 4]))


def test_cone_projection_table_is_consistent():
    g = pack_graph(*load_golden("benchmark3")[:2])
    off, cone = perf.cone_table(g)
    cent = g.interior_points()
    for v in range(g.nV):
        ck = cone[off[v]:off[v + 1]]
        A, b = g.polyA[g.poly_off[v]:g.poly_off[v + 1]], g.polyb[g.poly_off[v]:g.poly_off[v + 1]]
        assert ck.shape[0] >= 3
        assert np.all(ck[:, :2] @ A.T <= b[None, :] + 1e-7)                               # polygon vertices are feasible
        assert np.all(ck[:, 2:5] @ np.r_[cent[v], 1.0] < 0)                                 # normals point outwards
        R = np.hstack([ck[:, :2], np.ones((ck.shape[0], 1))])
        assert np.allclose(np.sum(ck[:, 2:5] * R, axis=1), 0, atol=1e-7)                    # each face contains its two rays
        assert np.allclose(np.sum(ck[:, 2:5] * np.roll(R, -1, axis=0), axis=1), 0, atol=1e-7)


@pytest.mark.parametrize("name", ["benchmark1", "test3"])
def test_emulated_perf_kernel_equals_literal_prototype(emu, name):
    """Null-space kernel vs the literal-variable numpy prototype: the same inner iteration, iterate by iterate."""
    import inner_first_order as proto
    K = 3
    g = pack_graph(*load_golden(name)[:2])
    a = EmuPerfADMM(emu, g, K)
    o = proto.OracleADMM(g)
    splits = {v: proto.SplitVertex(g, v, p, 1.0) for v, p in enumerate(o.progs) if not (p.d == 0 or p.dead)}

    def inexact():
        for v, p in enumerate(o.progs):
            hs = p.hs
            if v not in splits:
                o.z_v[v] = 0.0; o.y_v[v] = 0.0
                for h in hs:
                    tgt = o.z[g.he_edge[h]] + o.mu[h]
                    o.xc[h] = 0.0
                    if not g.he_out[h]:
                        o.xc[h, 0:2] = tgt[0:2]
                continue
            u = splits[v].iterate(o.rho, o.z[g.he_edge[hs]] + o.mu[hs], K)
            o.x_v[v] = u[0:4]; o.z_v[v] = u[4:8]; o.y_v[v] = u[8]
            o.xc[hs] = u[p.sel].reshape(-1, 5)
    o.vertex_update = inexact
    for it in range(25):
        a.step(); o.step()
        assert np.max(np.abs(a.xc - o.xc)) < 1e-8, it
        assert np.max(np.abs(a.z_v - o.z_v)) < 1e-8 and np.max(np.abs(a.y_v - o.y_v)) < 1e-8


def test_inexact_admm_converges_to_classic_optimum(emu):
    As, bs, n, d, keys = load_golden("benchmark1")
    a = EmuPerfADMM(emu, pack_graph(As, bs), K=3)
    for _ in range(400):
        a.step()
    assert a.pri[-1] < 1e-6 and a.dual[-1] < 1e-6
    assert abs(a.cost() - float(d["classic_cost"])) < 1e-5


def test_local_tables_slice_the_global_ones():
    """multi-GPU perf mode: a rank's tables = its own vertices' cone records (sliced from the global table), and blocks /
    tiles / classes rebuilt for the local half-edge layout with the same class tables as the global graph"""
    from gcs_admm_b200.generator import grid_packed_graph
    from gcs_admm_b200.partition import partition_vertices, split_graph
    g = grid_packed_graph(10)
    T = perf.perf_tables(g)
    inv = {c: k for k, c in T["classes"].items()}
    seen = 0
    for lp in split_graph(g, partition_vertices(g, 3), 3):
        L = perf.local_tables(T, lp)
        linv = {c: k for k, c in L["classes"].items()}
        assert L["cone_off"][-1] == L["cone"].shape[0] and L["cone_off"].shape[0] == lp.nV + 1
        assert L["tile_voff"][0] == 0 and L["tile_voff"][-1] == lp.nV and L["blk_off"][-1] == L["blk_he"].shape[0]
        for i, v in enumerate(lp.global_vertices):
            assert (L["vclass"][i] < 0) == (T["vclass"][v] < 0)
            if L["vclass"][i] >= 0:
                assert linv[L["vclass"][i]] == inv[T["vclass"][v]]
                a, b = L["vclass"][i] * perf.CLS_STRIDE, T["vclass"][v] * perf.CLS_STRIDE
                assert np.array_equal(L["cls_tab"][a:a + perf.CLS_STRIDE], T["cls_tab"][b:b + perf.CLS_STRIDE])
            assert np.array_equal(L["cone"][L["cone_off"][i]:L["cone_off"][i + 1]], T["cone"][T["cone_off"][v]:T["cone_off"][v + 1]])
            assert L["blk_off"][i + 1] - L["blk_off"][i] == T["blk_off"][v + 1] - T["blk_off"][v]
        seen += lp.nV
    assert seen == g.nV


@pytest.mark.parametrize("key", [(0, 4, 4), (0, 1, 1), (0, 2, 1), (0, 1, 3), (1, 0, 3), (1, 0, 1), (2, 2, 0), (2, 1, 0), (0, 5, 7)])
@pytest.mark.parametrize("kappa", [1.0, 0.3])
def test_structured_vstep_equals_dense_solution_operator(key, kappa):
    """the class tables (G, g0, dinv) the kernel uses reproduce the dense solution operator of the v-step"""
    T = perf.class_tables(*key, kappa)
    rng = np.random.default_rng(1)
    for _ in range(4):
        r = rng.normal(size=perf.NCORE + 5 * T["d"]); r[perf.UT] = 0.0
        assert np.max(np.abs(T["Phi"] @ r + T["g0u"] - perf.structured_vstep(T, r))) < 1e-12


def test_tiles_respect_their_limits():
    from gcs_admm_b200.generator import generate_test_2D
    As, bs, s_pt, t_pt = generate_test_2D(None, -20, 20, 1, 0.9, 60, seed=3)
    g = pack_graph(As, bs)
    T = perf.perf_tables(g)
    tv = T["tile_voff"].astype(np.int64)
    assert np.all(np.diff(tv) >= 1) and tv[0] == 0 and tv[-1] == g.nV
    nb = T["blk_off"].astype(np.int64)[tv[1:]] - T["blk_off"].astype(np.int64)[tv[:-1]]
    single = np.diff(tv) == 1
    assert np.all((nb <= perf.TILE_BLOCKS) | single) and np.all(np.diff(tv) <= perf.TILE_VERTS)
    # block list: live half-edges of a vertex in half-edge order, then its (z_v, y_v) block
    for v in range(g.nV):
        bl = list(T["blk_he"][T["blk_off"][v]:T["blk_off"][v + 1]])
        live = [h for h in range(g.he_off[v], g.he_off[v + 1]) if not (g.he_flags[h] & 2)]
        assert bl == ((live + [-1]) if g.vtype[v] != 3 else [])


def test_emulated_perf_mode_reaches_our_classic_optimum_on_a_generated_problem(emu):
    """Irregular polygons (up to 10 rows), live degrees up to 14, no stored reference run: the perf-mode fixed point is
    compared with the Drake-free classic solver (north_star: "compare against classic_solver" where v3 has no run)."""
    from gcs_admm_b200.classic import solve_classic
    from gcs_admm_b200.generator import generate_test_2D
    As, bs, s_pt, t_pt = generate_test_2D(None, -20, 20, 1, 0.9, 40, seed=7)
    g = pack_graph(As, bs)
    assert g.max_live_degree > 8 and g.max_rows > 8
    ref = solve_classic(As, bs, 2, round_solution=False)
    assert ref["status"] == "optimal"
    a = EmuPerfADMM(emu, g, K=1)
    for _ in range(8000):
        a.step()
    assert a.pri[-1] < 1e-3 and a.dual[-1] < 1e-3
    assert abs(a.cost() - ref["cost"]) <= 5e-4 * ref["cost"]
