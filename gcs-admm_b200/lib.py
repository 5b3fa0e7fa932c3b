"""ctypes binding of ``libgcsadmm.so`` (``include/gcsadmm.h``).

There is no CPU fallback: if the shared library is missing it is built with nvcc; if that
fails, or no CUDA device is present when a handle is created, the call raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

_dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")

EXPORTS = [
    "gcsadmm_version", "gcsadmm_last_error", "gcsadmm_device_count", "gcsadmm_default_params",
    "gcsadmm_create", "gcsadmm_destroy", "gcsadmm_set_stream", "gcsadmm_run", "gcsadmm_step",
    "gcsadmm_get_status", "gcsadmm_vertex_update", "gcsadmm_edge_update", "gcsadmm_control",
    "gcsadmm_sums_device_ptr", "gcsadmm_xc_device_ptr", "gcsadmm_get_history", "gcsadmm_get_solution",
    "gcsadmm_get_state", "gcsadmm_set_state", "gcsadmm_time_steps", "gcsadmm_time_window", "gcsadmm_solve_host",
    "gcsadmm_scratch_bytes", "gcsadmm_flush_l2", "gcsadmm_get_problem_status", "gcsadmm_get_problem_history", "gcsadmm_enable_perf",
    "gcsadmm_get_perf_state", "gcsadmm_set_perf_state", "gcsadmm_peer_export", "gcsadmm_peer_connect", "gcsadmm_peer_error",
    "gcsadmm_set_problem_tolerance",
]


class GcsGraph(C.Structure):
    _fields_ = [("nV", C.c_int32), ("nE", C.c_int32), ("n", C.c_int32), ("nH_own", C.c_int32), ("nH_ghost", C.c_int32),
                ("poly_off", C.c_void_p), ("polyA", C.c_void_p), ("polyb", C.c_void_p),
                ("he_off", C.c_void_p), ("he_edge", C.c_void_p), ("he_flags", C.c_void_p),
                ("edge_he_tail", C.c_void_p), ("edge_he_head", C.c_void_p), ("edge_counted", C.c_void_p),
                ("vtype", C.c_void_p), ("cent", C.c_void_p),
                ("n_x_global", C.c_int64), ("n_mu_global", C.c_int64),
                ("nP", C.c_int32), ("prob_voff", C.c_void_p), ("prob_eoff", C.c_void_p)]


class GcsParams(C.Structure):
    _fields_ = [("rho0", C.c_double), ("tau_incr", C.c_double), ("tau_decr", C.c_double), ("nu", C.c_double),
                ("frac", C.c_double), ("eps_abs", C.c_double), ("eps_rel", C.c_double), ("max_it", C.c_int32),
                ("inner_tol", C.c_double), ("inner_max_iter", C.c_int32), ("check_every", C.c_int32),
                ("abs_stop", C.c_int32), ("abs_tol", C.c_double), ("warm_theta", C.c_double), ("zero_tol", C.c_double),
                ("outer_alpha", C.c_double), ("use_graph", C.c_int32), ("adapt_every", C.c_int32), ("stop_ref", C.c_int32)]


class GcsPerfConfig(C.Structure):
    _fields_ = [("inner_iters", C.c_int32), ("alpha", C.c_double), ("kappa", C.c_double), ("n_classes", C.c_int32),
                ("vclass", C.c_void_p), ("cls_tab", C.c_void_p), ("cone_off", C.c_void_p), ("cone", C.c_void_p),
                ("n_blocks", C.c_int32), ("blk_off", C.c_void_p), ("blk_he", C.c_void_p), ("blk_info", C.c_void_p),
                ("n_tiles", C.c_int32), ("tile_voff", C.c_void_p),
                ("cap_blocks", C.c_int32), ("cap_verts", C.c_int32), ("cap_cone", C.c_int32), ("threads", C.c_int32),
                ("theta", C.c_double), ("edge_delta", C.c_void_p), ("edge_cent", C.c_void_p)]


class GcsStatus(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("converged", C.c_int32), ("diverged", C.c_int32),
                ("inner_fail", C.c_int32), ("inner_iters", C.c_int64), ("skipped", C.c_int64), ("rho", C.c_double), ("pri_res", C.c_double),
                ("dual_res", C.c_double), ("eps_pri", C.c_double), ("eps_dual", C.c_double), ("inner_res", C.c_double),
                ("pri_res_ref", C.c_double), ("dual_res_ref", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


_LIB = None


def library_path():
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), "libgcsadmm.so")


def load():
    """Load (building if needed) libgcsadmm.so.  Raises if it cannot be had."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = _build.build()          # no-op when libgcsadmm.so is newer than its sources; raises if nvcc is missing
    L = C.CDLL(path)
    L.gcsadmm_version.restype = C.c_char_p
    L.gcsadmm_last_error.restype = C.c_char_p
    L.gcsadmm_default_params.argtypes = [C.POINTER(GcsParams)]
    L.gcsadmm_default_params.restype = None
    L.gcsadmm_create.argtypes = [C.POINTER(GcsGraph), C.POINTER(GcsParams), C.c_int, C.POINTER(C.c_void_p)]
    L.gcsadmm_destroy.argtypes = [C.c_void_p]
    L.gcsadmm_set_stream.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    L.gcsadmm_run.argtypes = [C.c_void_p, C.c_int, C.POINTER(GcsStatus)]
    L.gcsadmm_step.argtypes = [C.c_void_p, C.c_int]
    L.gcsadmm_get_status.argtypes = [C.c_void_p, C.POINTER(GcsStatus)]
    L.gcsadmm_get_problem_status.argtypes = [C.c_void_p, C.c_int, C.POINTER(GcsStatus)]
    L.gcsadmm_set_problem_tolerance.argtypes = [C.c_void_p, C.c_void_p]
    L.gcsadmm_get_problem_history.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    for f in ("gcsadmm_vertex_update", "gcsadmm_edge_update", "gcsadmm_control"):
        getattr(L, f).argtypes = [C.c_void_p]
    L.gcsadmm_sums_device_ptr.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    L.gcsadmm_xc_device_ptr.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    L.gcsadmm_get_history.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    L.gcsadmm_get_solution.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.gcsadmm_get_state.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int)]
    L.gcsadmm_set_state.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_int]
    L.gcsadmm_time_steps.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float)]
    L.gcsadmm_time_window.argtypes = [C.c_void_p, C.c_int, C.c_longlong, C.c_void_p, C.c_void_p]
    L.gcsadmm_solve_host.argtypes = [C.POINTER(GcsGraph), C.POINTER(GcsParams), C.c_int, C.c_int, C.POINTER(GcsStatus),
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    L.gcsadmm_enable_perf.argtypes = [C.c_void_p, C.POINTER(GcsPerfConfig)]
    L.gcsadmm_get_perf_state.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.gcsadmm_set_perf_state.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.gcsadmm_peer_export.argtypes = [C.c_void_p, C.c_void_p]
    L.gcsadmm_peer_connect.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    L.gcsadmm_peer_error.argtypes = [C.c_void_p]
    L.gcsadmm_scratch_bytes.argtypes = [C.c_int, C.c_int]
    L.gcsadmm_flush_l2.argtypes = [C.c_void_p, C.c_longlong]
    _LIB = L
    return L


class GcsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libgcsadmm error {code}: {msg}")
        self.code = code


GCS_E_DIVERGED = -4


def _check(rc, allow_diverged=False):
    """Negative codes raise, except GCS_E_DIVERGED where the caller asked for it: the reference breaks out of its loop on
    non-finite iterates (``admm_solver_v3.py:662-664, :679-681``) and still reports / rounds / pickles the last iterates, so
    ``run`` and ``solve_host`` return normally with ``status['diverged'] = 1`` (the library has copied everything back)."""
    if rc < 0 and not (allow_diverged and rc == GCS_E_DIVERGED):
        raise GcsError(rc, load().gcsadmm_last_error().decode())
    return rc


def default_params(**overrides):
    p = GcsParams()
    load().gcsadmm_default_params(C.byref(p))
    for k, v in overrides.items():
        if not hasattr(p, k):
            raise TypeError(f"unknown ADMM parameter {k!r}")
        setattr(p, k, v)
    return p


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def graph_struct(g):
    """``PackedGraph`` (or a partition's local view with the same attributes) -> (GcsGraph, keepalive)."""
    keep = dict(
        poly_off=np.ascontiguousarray(g.poly_off, np.int32), polyA=np.ascontiguousarray(g.polyA, np.float64),
        polyb=np.ascontiguousarray(g.polyb, np.float64), he_off=np.ascontiguousarray(g.he_off, np.int32),
        he_edge=np.ascontiguousarray(g.he_edge, np.int32), he_flags=np.ascontiguousarray(g.he_flags, np.uint8),
        edge_he_tail=np.ascontiguousarray(g.edge_he_tail, np.int32),
        edge_he_head=np.ascontiguousarray(g.edge_he_head, np.int32),
        vtype=np.ascontiguousarray(g.vtype, np.uint8),
        cent=np.ascontiguousarray(getattr(g, "cent", None) if getattr(g, "cent", None) is not None else g.interior_points(), np.float64),
    )
    ec = getattr(g, "edge_counted", None)
    if ec is not None:
        keep["edge_counted"] = np.ascontiguousarray(ec, np.uint8)
    s = GcsGraph()
    s.nV, s.nE, s.n = g.nV, g.nE, 2
    s.nH_own = int(keep["he_off"][-1])
    s.nH_ghost = int(getattr(g, "nH_ghost", 0))
    for k in ("poly_off", "polyA", "polyb", "he_off", "he_edge", "he_flags", "edge_he_tail", "edge_he_head", "vtype", "cent"):
        setattr(s, k, _ptr(keep[k]))
    s.edge_counted = _ptr(keep.get("edge_counted"))
    pv = getattr(g, "prob_voff", None)
    if pv is not None and len(pv) > 2:
        keep["prob_voff"] = np.ascontiguousarray(pv, np.int32)
        keep["prob_eoff"] = np.ascontiguousarray(g.prob_eoff, np.int32)
        s.nP = len(pv) - 1
        s.prob_voff, s.prob_eoff = _ptr(keep["prob_voff"]), _ptr(keep["prob_eoff"])
    else:
        s.nP = 1
    s.n_x_global = int(getattr(g, "n_x_global", 0))
    s.n_mu_global = int(getattr(g, "n_mu_global", 0))
    return s, keep


class Solver:
    """One device-resident problem (handle of ``gcsadmm_create``)."""

    def __init__(self, g, device=0, **params):
        L = load()
        self.g = g
        self.params = default_params(**params)
        self._gs, self._keep = graph_struct(g)
        h = C.c_void_p()
        _check(L.gcsadmm_create(C.byref(self._gs), C.byref(self.params), int(device), C.byref(h)))
        self._h = h
        self.nHall = self._gs.nH_own + self._gs.nH_ghost

    def enable_perf(self, inner_iters=1, alpha=1.6, kappa=1.0, tables=None, frames="global"):
        """Switch the x-update to the inexact `perf` mode (K closed-form splitting iterations per ADMM iteration)."""
        from . import perf
        T = tables if tables is not None else perf.perf_tables(self.g, kappa, frames=frames)
        i32, f64 = np.int32, np.float64
        keep = dict(vclass=np.ascontiguousarray(T["vclass"], i32), cls_tab=np.ascontiguousarray(T["cls_tab"], f64),
                    cone_off=np.ascontiguousarray(T["cone_off"], i32), cone=np.ascontiguousarray(T["cone"], f64),
                    blk_off=np.ascontiguousarray(T["blk_off"], i32), blk_he=np.ascontiguousarray(T["blk_he"], i32),
                    blk_info=np.ascontiguousarray(T["blk_info"], i32), tile_voff=np.ascontiguousarray(T["tile_voff"], i32))
        c = GcsPerfConfig()
        c.inner_iters, c.alpha, c.kappa, c.n_classes = int(inner_iters), float(alpha), float(T["kappa"]), len(T["classes"])
        for k in ("vclass", "cls_tab", "cone_off", "cone", "blk_off", "blk_he", "blk_info", "tile_voff"):
            setattr(c, k, _ptr(keep[k]))
        c.n_blocks, c.n_tiles = int(keep["blk_he"].shape[0]), int(keep["tile_voff"].shape[0] - 1)
        c.cap_blocks, c.cap_verts, c.cap_cone = int(T["caps"]["nb"]), int(T["caps"]["nvt"]), int(T["caps"]["cone"])
        c.theta = float(T.get("theta", 1.0))
        c.threads = int(T.get("threads", 0))
        if T.get("edge_delta") is not None:
            keep["edge_delta"] = np.ascontiguousarray(T["edge_delta"], f64)
            c.edge_delta = _ptr(keep["edge_delta"])
            if T.get("edge_cent") is not None:
                keep["edge_cent"] = np.ascontiguousarray(T["edge_cent"], f64)
                c.edge_cent = _ptr(keep["edge_cent"])
        _check(load().gcsadmm_enable_perf(self._h, C.byref(c)))
        self._frames = T.get("edge_delta") is not None
        self._edge_delta = keep.get("edge_delta")
        self.perf = dict(inner_iters=int(inner_iters), alpha=float(alpha), kappa=float(T["kappa"]), classes=len(T["classes"]),
                         n_blocks=c.n_blocks, n_tiles=c.n_tiles, frames="local" if self._frames else "global")
        return self

    def warm_start(self, field="dijkstra", rho=None):
        """perf mode, before the first iteration: duals from a cost-to-go field over the portal graph (``warmstart.dual_start``);
        primal variables stay zero.  Same fixed point, far fewer iterations on large maps."""
        from . import warmstart
        if not getattr(self, "perf", None):
            raise GcsError(-1, "warm_start is an option of the perf mode (enable_perf first)")
        rho = float(self.status()["rho"] if rho is None else rho)
        mu = warmstart.dual_start(self.g, self._edge_delta, rho, field=field)
        self.set_state(None, mu, None, rho, 0)
        return self

    def perf_state(self):
        t, tn = np.zeros((self.perf["n_blocks"], 12)), np.zeros((self.g.nV, 2))
        _check(load().gcsadmm_get_perf_state(self._h, _ptr(t), _ptr(tn)))
        return t, tn

    def set_perf_state(self, tstate, tn):
        a, b = np.ascontiguousarray(tstate, np.float64), np.ascontiguousarray(tn, np.float64)
        _check(load().gcsadmm_set_perf_state(self._h, _ptr(a), _ptr(b)))

    def close(self):
        if getattr(self, "_h", None):
            load().gcsadmm_destroy(self._h)
            self._h = None

    __del__ = close

    def set_stream(self, stream_ptr, external=True):
        _check(load().gcsadmm_set_stream(self._h, C.c_void_p(stream_ptr), int(external)))

    def run(self, max_iters=None):
        st = GcsStatus()
        _check(load().gcsadmm_run(self._h, int(max_iters or self.params.max_it), C.byref(st)), allow_diverged=True)
        return st.as_dict()

    def step(self, k=1):
        _check(load().gcsadmm_step(self._h, int(k)))

    def status(self):
        st = GcsStatus()
        _check(load().gcsadmm_get_status(self._h, C.byref(st)))
        return st.as_dict()

    def problem_status(self, p):
        st = GcsStatus()
        _check(load().gcsadmm_get_problem_status(self._h, int(p), C.byref(st)))
        return st.as_dict()

    def set_problem_tolerance(self, tols):
        """each problem's own ``abs_tol`` of the absolute stop rule (one value per packed problem; 0: the handle's ``abs_tol``)"""
        t = np.ascontiguousarray(tols, np.float64).reshape(-1)
        if t.shape[0] != self._gs.nP:
            raise ValueError(f"{self._gs.nP} tolerances expected, got {t.shape[0]}")
        _check(load().gcsadmm_set_problem_tolerance(self._h, _ptr(t)))

    def problem_history(self, p):
        cap = self.params.max_it + 2
        rho, pri, dual = np.zeros(cap), np.zeros(cap), np.zeros(cap)
        n = _check(load().gcsadmm_get_problem_history(self._h, int(p), _ptr(rho), _ptr(pri), _ptr(dual), cap))
        return rho[:n].copy(), pri[:n].copy(), dual[:n].copy()

    def vertex_update(self):
        _check(load().gcsadmm_vertex_update(self._h))

    def edge_update(self):
        _check(load().gcsadmm_edge_update(self._h))

    def control(self):
        _check(load().gcsadmm_control(self._h))

    def sums_ptr(self):
        p = C.c_void_p()
        _check(load().gcsadmm_sums_device_ptr(self._h, C.byref(p)))
        return p.value

    def xc_ptr(self):
        p = C.c_void_p()
        _check(load().gcsadmm_xc_device_ptr(self._h, C.byref(p)))
        return p.value

    def history(self):
        cap = self.params.max_it + 2
        rho, pri, dual = np.zeros(cap), np.zeros(cap), np.zeros(cap)
        n = _check(load().gcsadmm_get_history(self._h, _ptr(rho), _ptr(pri), _ptr(dual), cap))
        return rho[:n].copy(), pri[:n].copy(), dual[:n].copy()

    def solution(self):
        nV, nE = self.g.nV, self.g.nE
        x_v, z_v, y_v, z_e = np.zeros((nV, 4)), np.zeros((nV, 4)), np.zeros(nV), np.zeros((nE, 5))
        _check(load().gcsadmm_get_solution(self._h, _ptr(x_v), _ptr(z_v), _ptr(y_v), _ptr(z_e)))
        if getattr(self, "_frames", False) and hasattr(self.g, "edge_tail"):
            # local frames: the edge variables (p1 in the tail's frame, p2 in the head's, y) back to global coordinates
            c = np.asarray(self.g.interior_points())
            z_e[:, 0:2] += z_e[:, 4:5] * c[self.g.edge_tail]
            z_e[:, 2:4] += z_e[:, 4:5] * c[self.g.edge_head]
        return x_v, z_v, y_v, z_e

    def state(self):
        xc, mu, z = np.zeros((self.nHall, 5)), np.zeros((self._gs.nH_own, 5)), np.zeros((self.g.nE, 5))
        rho, it = C.c_double(), C.c_int()
        _check(load().gcsadmm_get_state(self._h, _ptr(xc), _ptr(mu), _ptr(z), C.byref(rho), C.byref(it)))
        return xc, mu, z, rho.value, it.value

    def set_state(self, xc=None, mu=None, z=None, rho=1.0, it=0):
        a = [None if x is None else np.ascontiguousarray(x, np.float64) for x in (xc, mu, z)]
        _check(load().gcsadmm_set_state(self._h, _ptr(a[0]), _ptr(a[1]), _ptr(a[2]), float(rho), int(it)))

    def peer_export(self):
        """128 bytes: the CUDA IPC handles of this rank's xc buffer and flag / inbox block (to be all-gathered by the caller)"""
        buf = np.zeros(128, dtype=np.uint8)
        _check(load().gcsadmm_peer_export(self._h, _ptr(buf)))
        return buf

    def peer_connect(self, rank, world, all_handles, nHown, nHghost, send_he, send_rank, send_slot):
        a = np.ascontiguousarray(all_handles, np.uint8)
        i = [np.ascontiguousarray(x, np.int32) for x in (nHown, nHghost, send_he, send_rank, send_slot)]
        _check(load().gcsadmm_peer_connect(self._h, int(rank), int(world), _ptr(a), _ptr(i[0]), _ptr(i[1]), int(i[2].shape[0]), _ptr(i[2]), _ptr(i[3]), _ptr(i[4])))

    def peer_error(self):
        return int(load().gcsadmm_peer_error(self._h))

    def flush_l2(self, nbytes=0):
        _check(load().gcsadmm_flush_l2(self._h, int(nbytes)))

    def time_steps(self, k, split=False):
        tot, k1, ed = C.c_float(), C.c_float(), C.c_float()
        _check(load().gcsadmm_time_steps(self._h, int(k), C.byref(tot), C.byref(k1) if split else None,
                                         C.byref(ed) if split else None))
        return tot.value, k1.value, ed.value


    def time_window(self, k, flush_bytes=256 << 20, split=False):
        """k iterations enqueued back to back, L2 evicted in-stream before each (outside the event pairs) -> (ms per iteration [k], K1 ms [k] | None)"""
        it = np.zeros(int(k), dtype=np.float32)
        k1 = np.zeros(int(k), dtype=np.float32) if split else None
        _check(load().gcsadmm_time_window(self._h, int(k), int(flush_bytes), _ptr(it), _ptr(k1)))
        return it, k1


def solve_host(g, device=0, max_iters=None, **params):
    """create + run + copy back + destroy in one C call (host buffers in, host buffers out)."""
    L = load()
    p = default_params(**params)
    gs, keep = graph_struct(g)
    nV, nE = g.nV, g.nE
    cap = p.max_it + 2
    x_v, z_v, y_v, z_e = np.zeros((nV, 4)), np.zeros((nV, 4)), np.zeros(nV), np.zeros((nE, 5))
    rho, pri, dual = np.zeros(cap), np.zeros(cap), np.zeros(cap)
    st = GcsStatus()
    _check(L.gcsadmm_solve_host(C.byref(gs), C.byref(p), int(device), int(max_iters or p.max_it), C.byref(st),
                                _ptr(x_v), _ptr(z_v), _ptr(y_v), _ptr(z_e), _ptr(rho), _ptr(pri), _ptr(dual), cap), allow_diverged=True)
    n = st.iterations + 1
    return dict(status=st.as_dict(), x_v=x_v, z_v=z_v, y_v=y_v, z_e=z_e, rho_seq=rho[:n].copy(),
                pri_res_seq=pri[:n].copy(), dual_res_seq=dual[:n].copy())
