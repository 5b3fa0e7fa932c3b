"""The two-point form of the perf-mode cone projection (`gcs_cone_project2`, csrc/vertex_perf.cuh), which K1 uses for the
fam-0 and fam-1 pairs of one half-edge point, against two calls of the one-point form, on the CPU through the host build of
the kernel source.  Both evaluate each point with the same expressions, so they must agree bit for bit.  Also the block order
the kernel's per-vertex sums rely on (in-blocks, then out-blocks), which perf.perf_tables enforces."""
import ctypes as C

import numpy as np
import pytest

from test_cone_projection import generated_cones, grid_cones, project, sample_points, stored_cones
from test_perf_mode import load_emu

_dp = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")


@pytest.fixture(scope="module")
def emu():
    lib = load_emu()
    lib.gcsemu_cone_project2.restype = None
    lib.gcsemu_cone_project2.argtypes = [_dp, C.c_int, _dp, C.c_int, _dp]
    return lib


def project2(lib, rec, pts):
    pts = np.ascontiguousarray(pts, dtype=np.float64)
    out = np.zeros_like(pts)
    lib.gcsemu_cone_project2(np.ascontiguousarray(rec).reshape(-1), rec.shape[0], pts.reshape(-1), pts.shape[0], out.reshape(-1))
    return out


@pytest.mark.parametrize("cones", [stored_cones, generated_cones, grid_cones])
def test_two_point_projection_is_two_one_point_projections(emu, cones):
    rng = np.random.default_rng(11)
    for c in cones():
        t = sample_points(c, rng)
        t = t[: t.shape[0] // 2 * 2]
        # pairs of unrelated points and of a point with itself, in both orders
        for pts in (t, t[rng.permutation(t.shape[0])], np.repeat(t[: t.shape[0] // 2], 2, axis=0)):
            q1 = project(emu, c.rec, pts)
            q2 = project2(emu, c.rec, pts)
            assert np.array_equal(q1.view(np.uint64), q2.view(np.uint64)), c.tag


def test_perf_tables_refuse_an_out_half_edge_before_an_in_half_edge():
    """K1 sums a vertex's in-blocks and out-blocks as two contiguous ranges, so the tables must list in-half-edges first"""
    import copy

    from conftest import load_golden
    from gcs_admm_b200 import perf
    from gcs_admm_b200.graph import pack_graph
    g = pack_graph(*load_golden("benchmark4")[:2])
    perf.perf_tables(g)
    flags = np.asarray(g.he_flags)
    off = np.asarray(g.he_off)
    live = (flags & 2) == 0
    v = next(v for v in range(g.nV) if np.any(live[off[v]:off[v + 1]] & ((flags[off[v]:off[v + 1]] & 1) == 0))
             and np.any(live[off[v]:off[v + 1]] & ((flags[off[v]:off[v + 1]] & 1) == 1)))
    h = off[v] + int(np.nonzero(live[off[v]:off[v + 1]])[0][0])       # the vertex's first live half-edge (an in-half-edge)
    bad = copy.copy(g)
    bad.he_flags = flags.copy()
    bad.he_flags[h] |= 1                                                 # now an out-half-edge ahead of the in-half-edges
    with pytest.raises(ValueError, match="in-half-edges before"):
        perf.perf_tables(bad)
