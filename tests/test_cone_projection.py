"""The exact 3-D cone projection of perf-mode K1 (`gcs_cone_project`, csrc/vertex_perf.cuh) and the inner residual of the
INNER variant of K1, both on the CPU through the host build of the kernel source (csrc/emulate.cpp).

The projection is checked by its optimality conditions, which need no second implementation: by Moreau's decomposition q is
the projection of t onto the closed convex cone K = {(p, h): A p <= h b} exactly when q is in K, t - q is in the polar cone
K° = {w: w.(V_k, 1) <= 0 for every polygon vertex V_k} and <q, t - q> = 0.  It is also compared with scipy's NNLS on the ray
matrix R = [V_k, 1]': q* = R lam*.  q is feasible, so |q - q*|^2 <= |t - q|^2 - |t - q*|^2 and the comparison bounds the point
error, not only the distance error."""
import ctypes as C

import numpy as np
import pytest
from scipy.optimize import nnls

from conftest import ALL_PROBLEMS, load_golden
from gcs_admm_b200 import perf
from gcs_admm_b200.generator import generate_test_2D, grid_problem
from gcs_admm_b200.graph import _vertices_batch, pack_graph
from test_perf_mode import EmuPerfADMM, load_emu

EPS = np.finfo(np.float64).eps
# Errors are measured in units of  s = max(1, |t|) * max(1, max_k |V_k|)  (s^2 for the complementarity product and for the
# excess of squared distance over the NNLS point's): the kernel forms dot products of t with records whose entries are up to
# max |V_k| (rays) or 1 (unit normals), so a correct projection leaves a few ulps of s.
# Regular cones (every pair of adjacent rays at an angle whose sine is >= 1e-4): worst measured 7.8 EPS (distance to the NNLS
# point), 4.6 EPS (squared-distance excess), 2.0 EPS (complementarity), 1.3 EPS (polar cone); tolerance 64 EPS.  Membership
# (A p <= h b) also carries the error of the polygon vertices the records are built from (intersections of the rows): 149 EPS
# measured on the 316 x 316 grid in global frames, tolerance 1024 EPS.
TOL_REG, TOL_REG_MEMBER = 64 * EPS, 1024 * EPS
# Needle cones: the 's' / 't' regions of the stored and generated problems are boxes of side 2e-6, so adjacent rays are parallel
# to 1e-7 or better.  The kernel's inside test, sector tests and ray comparison are then decided at the rounding level and it may
# return a neighbouring candidate: a point of the cone (or within rounding of it) whose squared distance exceeds the optimum by
# up to 1.6e4 EPS s^2 (measured), i.e. |q - q*| up to 1.5e-9 s (6.9e6 EPS), membership 3.1e5 EPS, polar 4.4e4 EPS.  Tolerances:
# 8x those.  Well-posed cones never come near these numbers, and a projection that misses a candidate is off by O(1).
NEEDLE = 1e-4
TOL_NEEDLE = dict(member=2.5e6 * EPS, polar=3.5e5 * EPS, comp=64 * EPS, excess=1.3e5 * EPS, dist=5.5e7 * EPS)


@pytest.fixture(scope="module")
def emu():
    return load_emu()


def project(lib, rec, pts):
    pts = np.ascontiguousarray(pts, dtype=np.float64)
    out = np.zeros_like(pts)
    lib.gcsemu_cone_project(np.ascontiguousarray(rec).reshape(-1), rec.shape[0], pts.reshape(-1), pts.shape[0], out.reshape(-1))
    return out


class Cone:
    """One region's perspective cone: rows (A, b) and the kernel's records, in the same coordinates"""

    def __init__(self, A, b, rec, tag):
        self.A, self.b, self.rec, self.tag = A, b, rec, tag
        self.R = np.hstack([rec[:, :2], np.ones((rec.shape[0], 1))])        # rays (V_k, 1)
        self.vmax = max(1.0, float(np.max(np.linalg.norm(rec[:, :2], axis=1))))
        Ru = self.R / np.linalg.norm(self.R, axis=1, keepdims=True)
        self.sin_min = float(np.min(np.linalg.norm(np.cross(Ru, np.roll(Ru, -1, axis=0)), axis=1)))      # smallest angle between adjacent rays
        self.needle = self.sin_min < NEEDLE
        reg = dict(member=TOL_REG_MEMBER, polar=TOL_REG, comp=TOL_REG, excess=TOL_REG, dist=TOL_REG)
        self.tol = TOL_NEEDLE if self.needle else reg


def cones_of(off, A, b, frames, tag, only=None):
    """Cone records of every region (or of the regions `only`), global frames or centred on the region's vertex centroid"""
    off = np.asarray(off, np.int64)
    if only is not None:                  # repack the chosen regions
        rows = [np.arange(off[v], off[v + 1]) for v in only]
        off = np.concatenate([[0], np.cumsum([r.shape[0] for r in rows])])
        A, b = A[np.concatenate(rows)], b[np.concatenate(rows)]
    verts, cnt = _vertices_batch(off, A, b)
    cent = np.array([verts[v, :cnt[v]].mean(axis=0) for v in range(cnt.shape[0])])

    class G:
        pass
    G.poly_off, G.polyA, G.polyb, G.nV = off, A, b, cnt.shape[0]
    coff, rec = perf.cone_table(G, shift=cent if frames == "local" else None)
    out = []
    for v in range(cnt.shape[0]):
        Av, bv = A[off[v]:off[v + 1]], b[off[v]:off[v + 1]]
        if frames == "local":
            bv = bv - Av @ cent[v]
        out.append(Cone(Av, bv, rec[coff[v]:coff[v + 1]], f"{tag}/{frames}/{v}"))
    return out


def stored_cones():
    res = []
    for name in ALL_PROBLEMS:
        g = pack_graph(*load_golden(name)[:2])
        for fr in ("global", "local"):
            res += cones_of(g.poly_off, g.polyA, g.polyb, fr, name)
    return res


def generated_cones():
    res = []
    for seed in (3, 5, 7):
        g = pack_graph(*generate_test_2D(None, -20, 20, 1, 0.9, 40, seed=seed)[:2])
        assert g.max_rows >= 8
        for fr in ("global", "local"):
            res += cones_of(g.poly_off, g.polyA, g.polyb, fr, f"gen{seed}")
    return res


def grid_cones():
    """chamfered boxes of the 316 x 316 grid (the bench's headline map): the four corners, the rows and columns at the far
    edges and a seeded sample.  In global frames the far corner's polygon is ~447 from the origin: its rays are nearly parallel"""
    G = 316
    off, A, b, s_pt, t_pt = grid_problem(G)
    rng = np.random.default_rng(0)
    cells = [(0, 0), (0, G - 1), (G - 1, 0), (G - 1, G - 1)] + [(G - 1, int(j)) for j in rng.integers(0, G, 6)] + \
            [(int(i), G - 1) for i in rng.integers(0, G, 6)] + [tuple(int(x) for x in rng.integers(0, G, 2)) for _ in range(12)]
    only = [2 + i * G + j for i, j in cells]
    res = []
    for fr in ("global", "local"):
        res += cones_of(off, A, b, fr, "grid316", only)
    assert max(c.vmax for c in res) > 440
    return res


def sample_points(c, rng):
    """points where the choice between apex, ray, face and interior is decided"""
    R, rec = c.R, c.rec
    nv = R.shape[0]
    N, MA, MB = rec[:, 2:5], rec[:, 6:9], rec[:, 9:12]
    Rn = np.roll(R, -1, axis=0)
    pts = []
    for s in (1e-3, 1.0, 1e3):
        for k in range(nv):
            r = s * R[k]
            pts.append(r)
            for eps in (1e-14, 1e-11, 1e-8):                     # on the ray, nudged to either side
                u = rng.normal(size=3); u /= np.linalg.norm(u)
                pts += [r + eps * np.linalg.norm(r) * u, r - eps * np.linalg.norm(r) * u]
            a, bb = rng.uniform(0.1, 1.0, 2)
            f = s * (a * R[k] + bb * Rn[k])                       # on face k, and above it (projects onto the face)
            d = s * rng.uniform(0.01, 10.0)
            pts += [f, f + d * N[k], f + 1e-9 * s * N[k]]
            # exactly on the sector planes of face k: above the face's two bounding rays (t.ma = 0, t.mb = 0), and just outside
            pts += [s * Rn[k] + d * N[k], s * R[k] + d * N[k]]
            pts += [s * Rn[k] + d * N[k] - 1e-9 * s * MA[k] / np.linalg.norm(MA[k]), s * R[k] + d * N[k] - 1e-9 * s * MB[k] / np.linalg.norm(MB[k])]
        lam = rng.uniform(0.0, 1.0, (8, nv))
        pts += list(s * lam @ R)                                  # inside
        mu = rng.uniform(0.0, 1.0, (8, nv))
        pts += list(s * mu @ N)                                   # in the polar cone: the answer is the apex
        h = rng.normal(size=(8, 3)); h[:, 2] = -np.abs(h[:, 2]) - 1e-3
        pts += list(s * h * np.array([c.vmax, c.vmax, 1.0]))     # below the apex (h < 0)
    for s in (1e-6, 1.0, 1e6):
        pts += list(s * rng.normal(size=(12, 3)))
        axis = R.mean(axis=0)
        pts += list(s * (axis + rng.normal(size=(12, 3)) * np.array([c.vmax, c.vmax, 1.0]) * 0.05))      # around the cone's axis
    return np.array(pts)


def certificate(c, t, q):
    """worst membership, polar, complementarity, squared-distance excess over the NNLS point and distance to it, of the
    projections q of points t, in units of s (s^2)"""
    s = np.maximum(1.0, np.linalg.norm(t, axis=1)) * c.vmax
    An = c.A / np.linalg.norm(c.A, axis=1, keepdims=True)
    bn = c.b / np.linalg.norm(c.A, axis=1)
    Ru = c.R / np.linalg.norm(c.R, axis=1, keepdims=True)
    qs = np.array([c.R.T @ nnls(c.R.T, ti)[0] for ti in t])
    return dict(member=np.maximum(np.max(q[:, :2] @ An.T - q[:, 2:3] * bn[None, :], axis=1), -q[:, 2]) / s,
                polar=np.max((t - q) @ Ru.T, axis=1) / s,
                comp=np.abs(np.sum(q * (t - q), axis=1)) / s ** 2,
                excess=(np.sum((t - q) ** 2, axis=1) - np.sum((t - qs) ** 2, axis=1)) / s ** 2,
                dist=np.linalg.norm(q - qs, axis=1) / s)


def check_cones(lib, cones, seed):
    rng = np.random.default_rng(seed)
    worst = {k: {True: 0.0, False: 0.0} for k in TOL_NEEDLE}
    for c in cones:
        t = sample_points(c, rng)
        q = project(lib, c.rec, t)
        for k, v in certificate(c, t, q).items():
            i = int(np.argmax(v))
            worst[k][c.needle] = max(worst[k][c.needle], float(v[i]))
            assert v[i] <= c.tol[k], (c.tag, k, v[i] / EPS, t[i], q[i])
    n = sum(c.needle for c in cones)
    print(f"{len(cones)} cones ({n} needles), worst in units of eps, regular | needle: " +
          ", ".join(f"{k} {w[False] / EPS:.1f} | {w[True] / EPS:.1f}" for k, w in worst.items()))


def test_projection_certificate_stored_problems(emu):
    check_cones(emu, stored_cones(), 1)


def test_projection_certificate_generated_problems(emu):
    check_cones(emu, generated_cones(), 2)


def test_projection_certificate_grid316_far_from_the_origin(emu):
    check_cones(emu, grid_cones(), 3)


def test_projection_is_exact_at_the_apex_and_inside(emu):
    """cases with an exact answer: the apex is its own projection, points of the polar cone go to the apex, interior points stay"""
    for c in [c for c in generated_cones() if not c.needle][:40]:
        assert np.array_equal(project(emu, c.rec, np.zeros((1, 3))), np.zeros((1, 3)))
        q = project(emu, c.rec, 3.0 * (c.rec[:, 2:5] + c.rec[:, 2:5].sum(axis=0)))      # strictly inside the polar cone
        assert np.array_equal(q, np.zeros_like(q)), c.tag
        inside = 0.5 * (c.R + np.roll(c.R, -1, axis=0)) * 0.5 + 0.5 * c.R.mean(axis=0)
        assert np.array_equal(project(emu, c.rec, inside), inside), c.tag


# ------------------------------------------------------------------------------------------ inner residual (INNER K1)

def soft_threshold(a, thr):
    n = np.linalg.norm(a, axis=1, keepdims=True)
    return np.where(n > 0, np.maximum(0.0, 1.0 - thr / np.where(n > 0, n, 1.0)), 0.0) * a


def inner_residual_numpy(a, t_old, tn_old):
    """squared inner residual of one K = 1 step with mu_scale = 1, from the state t (per pair) and tn (per vertex) before it and
    after it (a.tstate, a.tn): c = Proj_K(t_old) by NNLS, lam = t_old - c, pv = (t_new - (1 - alpha) c - lam) / alpha, summed
    |pv - c|^2 over the live pairs and the path-length items (their c: block soft-threshold of tn_old at 1 / sigma, sigma = kappa rho)"""
    T, g, alpha = a.T, a.g, a.alpha
    blk_off, info = T["blk_off"].astype(np.int64), T["blk_info"]
    owner = np.repeat(np.arange(g.nV), np.diff(blk_off))
    total = 0.0
    npairs = 0
    for b in range(blk_off[-1]):
        v = owner[b]
        c0, c1 = T["cone_off"][v], T["cone_off"][v + 1]
        R = np.hstack([T["cone"][c0:c1, :2], np.ones((c1 - c0, 1))])
        term = (info[b] >> 10) & 1
        for p in range(4):
            if term and (p & 1):                   # 's' / 't' blocks have no fam-1 pairs
                continue
            to = t_old[b, 3 * p:3 * p + 3]
            c = R.T @ nnls(R.T, to)[0]
            pv = (a.tstate[b, 3 * p:3 * p + 3] - (1 - alpha) * c - (to - c)) / alpha
            total += float(np.sum((pv - c) ** 2))
            npairs += 1
    live = T["vclass"] >= 0
    c = soft_threshold(tn_old[live], 1.0 / (T["kappa"] * a.rho))
    pv = (a.tn[live] - (1 - alpha) * c - (tn_old[live] - c)) / alpha
    return total + float(np.sum((pv - c) ** 2)), npairs


@pytest.mark.parametrize("frames", ["global", "local"])
@pytest.mark.parametrize("name", ["benchmark2", "benchmark4", "gen5"])
def test_inner_residual_of_the_inner_variant_equals_numpy(emu, name, frames):
    if name == "gen5":
        g = pack_graph(*generate_test_2D(None, -20, 20, 1, 0.9, 40, seed=5)[:2])
    else:
        g = pack_graph(*load_golden(name)[:2])
    a = EmuPerfADMM(emu, g, K=1, frames=frames, outer_alpha=1.7 if frames == "local" else 1.0)
    for _ in range(6):
        a.step()
    assert a.ms == 1.0
    t_old, tn_old = a.tstate.copy(), a.tn.copy()
    a.inner = True
    a.vertex_update()
    ref, npairs = inner_residual_numpy(a, t_old, tn_old)
    print(f"{name} {frames}: {npairs} pairs, inner_sq {a.inner_sq:.6e} numpy {ref:.6e} rel {abs(a.inner_sq - ref) / ref:.2e}")
    assert ref > 0.0 and abs(a.inner_sq - ref) <= 1e-10 * ref
    # the INNER variant updates the state exactly like the throughput variant
    b = EmuPerfADMM(emu, g, K=1, frames=frames, outer_alpha=1.7 if frames == "local" else 1.0)
    for _ in range(6):
        b.step()
    b.vertex_update()
    for x, y in ((a.tstate, b.tstate), (a.tn, b.tn), (a.xc, b.xc), (a.z_v, b.z_v), (a.y_v, b.y_v)):
        assert np.array_equal(x, y)
