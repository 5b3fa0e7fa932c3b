"""Host-side tables of the `perf` mode of K1 (``csrc/vertex_perf.cuh``).

* ``class_inverse``: for a vertex class (type, #live in-edges, #live out-edges) the matrix
  ``K1 = N'(S'S + kappa M'M)N`` of the v-step and its inverse.  ``N`` is the null-space map of the equalities
  C6/C7 (reference ``admm_solver_v3.py:450-464``), ``S`` selects the consensus scalars that carry the rho-quadratic
  (``:390-413``), ``M`` maps the variables to the (point, flow) pairs of C1-C4 (``:416-440``) and to ``z_1 - z_2``.
  All three have 0/+-1 entries and depend on the class only — not on the polygon.
* ``cone_table``: the rays / face normals of every region's perspective cone for the exact 3-D projection.

The Python functions ``_forward`` / ``_pair_values`` restate ``gcs_forward`` / ``gcs_pair_values`` of the kernels.
"""
from __future__ import annotations

import numpy as np

from .graph import _vertices_batch

NCORE, UX, UT, UZ, UYV = 10, 0, 4, 5, 9


def _uw(j):
    return NCORE + 5 * j


def _forward(v, d, jstar, prim, term, affine):
    u = np.zeros(NCORE + 5 * d)
    u[UX:UX + 4] = v[0:4]
    u[UT] = v[4]
    zy = np.zeros(5)
    other = np.zeros(5)
    if term:
        zy[0:4] = v[0:4]
        zy[4] = 1.0 if affine else 0.0
    for jj in range(d - 1):
        j = jj if jj < jstar else jj + 1
        w = v[5 + 5 * jj: 10 + 5 * jj]
        u[_uw(j):_uw(j) + 5] = w
        if prim[j]:
            other += w
        else:
            zy += w
    u[UZ:UZ + 5] = zy
    u[_uw(jstar):_uw(jstar) + 5] = zy - other
    return u


def _pair_values(u, d, term):
    npair = 4 * (d + 1)
    pv = np.zeros(3 * npair + 2)
    for blk in range(d + 1):
        for i in range(2):
            po = (_uw(blk) if blk < d else UZ) + 2 * i
            yo = _uw(blk) + 4 if blk < d else UYV
            xo = UX + 2 * i
            for fam in range(1 if term else 2):
                o = 3 * ((blk * 2 + i) * 2 + fam)
                if fam:
                    pv[o:o + 3] = (u[xo] - u[po], u[xo + 1] - u[po + 1], 1.0 - u[yo])
                else:
                    pv[o:o + 3] = (u[po], u[po + 1], u[yo])
    pv[3 * npair] = u[UZ] - u[UZ + 2]
    pv[3 * npair + 1] = u[UZ + 1] - u[UZ + 3]
    return pv


def class_pattern(vtype, din, dout):
    """(d, out flags, prim flags, jstar, term) of a class, in the kernels' half-edge order (in-edges then out-edges)."""
    d = din + dout
    out = [0] * din + [1] * dout
    term = vtype != 0
    prim = [1] * d if vtype == 2 else list(out)
    jstar = max(j for j in range(d) if prim[j])
    return d, out, prim, jstar, term


def class_inverse(vtype, din, dout, kappa):
    d, out, prim, jstar, term = class_pattern(vtype, din, dout)
    n, nu = 5 * d, NCORE + 5 * d
    N = np.zeros((nu, n))
    for k in range(n):
        e = np.zeros(n); e[k] = 1.0
        N[:, k] = _forward(e, d, jstar, prim, term, False)
    pv0 = _pair_values(np.zeros(nu), d, term)
    M = np.zeros((pv0.shape[0], nu))
    for k in range(nu):
        e = np.zeros(nu); e[k] = 1.0
        M[:, k] = _pair_values(e, d, term) - pv0
    S = np.zeros(nu)
    for j in range(d):
        o = _uw(j)
        S[o:o + 2] = 1.0
        if out[j]:
            S[o + 2:o + 4] = 1.0
        S[o + 4] = 1.0
    K1 = N.T @ (np.diag(S) + kappa * M.T @ M) @ N
    K1[4, :] = 0.0; K1[:, 4] = 0.0; K1[4, 4] = 1.0          # the epigraph variable t is unused in this mode
    w = np.linalg.eigvalsh(K1)
    if w[0] <= 1e-12 * w[-1]:
        raise ValueError(f"singular v-step matrix for class {(vtype, din, dout)}")
    Kinv = np.linalg.inv(K1)
    Kinv[4, :] = 0.0; Kinv[:, 4] = 0.0
    return np.ascontiguousarray(Kinv)


def cone_table(g, shift=None):
    """Per region: polygon vertices (counter-clockwise) with the unit outward normal of the cone face spanned by the
    rays through vertex k and k+1, 1/|r_k|^2 (r_k = (V_k, 1)) and the two in-plane sector normals of that face
    (12 doubles per polygon vertex).  Vectorised over regions with the same vertex count."""
    verts, cnt = g.polygon_vertices_batch() if hasattr(g, "polygon_vertices_batch") else _vertices_batch(g.poly_off.astype(np.int64), g.polyA, g.polyb)
    if shift is not None:            # local frames: the polygon of region v translated by -shift[v]
        verts = verts - np.asarray(shift)[:, None, :]
    nV = g.nV
    # duplicates (redundant rows meeting in one vertex) are rare: handle those regions one by one
    per = [None] * nV
    for k in np.unique(cnt):
        idx = np.nonzero(cnt == k)[0]
        P = verts[idx, :k]                                            # (g, k, 2)
        c = P.mean(axis=1, keepdims=True)
        ang = np.arctan2(P[..., 1] - c[..., 1], P[..., 0] - c[..., 0])
        order = np.argsort(ang, axis=1)
        P = np.take_along_axis(P, order[..., None], axis=1)
        nxt = np.roll(P, -1, axis=1)
        dup = np.max(np.abs(P - nxt), axis=2) <= 1e-12 * np.maximum(1.0, np.abs(P).max(axis=2))
        clean = ~np.any(dup, axis=1)
        R = np.concatenate([P, np.ones(P.shape[:2] + (1,))], axis=2)
        Nn = np.cross(R, np.roll(R, -1, axis=1))
        nrm = np.linalg.norm(Nn, axis=2, keepdims=True)
        Nn = Nn / np.where(nrm > 0, nrm, 1.0)
        inner = np.concatenate([c, np.ones((c.shape[0], 1, 1))], axis=2)
        flip = np.sum(Nn * inner, axis=2) > 0
        Nn = np.where(flip[..., None], -Nn, Nn)
        Rn = np.roll(R, -1, axis=1)
        # in-plane sector tests of face k: p = a r + b s with a, b >= 0  <=>  p.ma >= 0 and p.mb >= 0, where
        # ma = n x s (zero on s, positive on r) and mb = r x n (zero on r, positive on s), n = outward unit normal
        ma = np.cross(Nn, Rn); mb = np.cross(R, Nn)
        ma *= np.sign(np.sum(ma * R, axis=2, keepdims=True)); mb *= np.sign(np.sum(mb * Rn, axis=2, keepdims=True))
        rec = np.concatenate([P, Nn, 1.0 / np.sum(R * R, axis=2, keepdims=True), ma, mb], axis=2)      # (g, k, 12)
        for gi, v in enumerate(idx):
            per[v] = rec[gi] if clean[gi] else None
    for v in range(nV):
        if per[v] is None:
            per[v] = _cone_one(verts[v, :cnt[v]])
    off = np.zeros(nV + 1, dtype=np.int64)
    np.cumsum([p.shape[0] for p in per], out=off[1:])
    return off.astype(np.int32), np.ascontiguousarray(np.vstack(per))


def _cone_one(P):
    keep = []
    for p in P:
        if not any(np.max(np.abs(p - q)) <= 1e-12 * max(1.0, np.abs(p).max()) for q in keep):
            keep.append(p)
    P = np.array(keep)
    c = P.mean(axis=0)
    P = P[np.argsort(np.arctan2(P[:, 1] - c[1], P[:, 0] - c[0]))]
    R = np.hstack([P, np.ones((P.shape[0], 1))])
    Nn = np.cross(R, np.roll(R, -1, axis=0))
    Nn /= np.linalg.norm(Nn, axis=1, keepdims=True)
    flip = (Nn @ np.array([c[0], c[1], 1.0])) > 0
    Nn[flip] *= -1.0
    Rn = np.roll(R, -1, axis=0)
    ma = np.cross(Nn, Rn); mb = np.cross(R, Nn)
    ma *= np.sign(np.sum(ma * R, axis=1, keepdims=True)); mb *= np.sign(np.sum(mb * Rn, axis=1, keepdims=True))
    return np.hstack([P, Nn, 1.0 / np.sum(R * R, axis=1, keepdims=True), ma, mb])


CORE_IDX = (0, 1, 2, 3, 5, 6, 7, 8, 9)      # x(4), z(4), y_v in the u-space layout (index 4 is the unused epigraph variable)
NCX = 19                                      # extended core: x(4) z(4) y_v | beta_in(5) | beta_out(5)
CLS_STRIDE = NCX * NCX + NCX + 10 + 2          # G transposed (19 x 19) | g0 (19) | dinv (2 x 5) | pad -> 392 doubles per class


def class_tables(vtype, din, dout, kappa, theta=1.0):
    """Structured form of the v-step of one vertex class (``csrc/vertex_perf.cuh``).

    The v-step minimises  1/2 u'D u - r'u  over the equalities C6/C7 (reference ``admm_solver_v3.py:450-464``), with
    ``D = S'S + kappa M'M``.  Its solution operator ``u = Phi r + g0`` has a block structure the kernel exploits:
    every variable (tau = a1x, a1y, a2x, a2y, y) of a half-edge block b in group g (in- / out-edges) is

        u[b, tau] = dinv[g, tau] * r[b, tau] + beta[g, tau]

    and the extended core  (x, z, y_v, beta_in, beta_out)  is a 19 x 19 linear map ``G`` of
    (r_x, r_z, r_yv, R_in, R_out) with ``R_g = sum of r over the blocks of group g``, plus a constant ``g0`` (the affine
    part: y_v = 1 at 's' / 't').  ``Phi`` is formed densely here (once per class) and the structure is read off it."""
    d, out, prim, jstar, term = class_pattern(vtype, din, dout)
    n, nu = 5 * d, NCORE + 5 * d
    N = np.zeros((nu, n))
    for k in range(n):
        e = np.zeros(n); e[k] = 1.0
        N[:, k] = _forward(e, d, jstar, prim, term, False)
    pv0 = _pair_values(np.zeros(nu), d, term)
    M = np.zeros((pv0.shape[0], nu))
    for k in range(nu):
        e = np.zeros(nu); e[k] = 1.0
        M[:, k] = _pair_values(e, d, term) - pv0
    S = np.zeros(nu)
    for j in range(d):
        o = _uw(j)
        S[o:o + 2] = 1.0
        if out[j]:
            S[o + 2:o + 4] = 1.0
        S[o + 4] = theta            # the flow scalar's penalty is theta * rho (theta = 1: the reference's single rho)
    D = np.diag(S) + kappa * M.T @ M
    K1 = N.T @ D @ N
    K1[4, :] = 0.0; K1[:, 4] = 0.0; K1[4, 4] = 1.0          # the epigraph variable t is unused in this mode
    w = np.linalg.eigvalsh(K1)
    if w[0] <= 1e-12 * w[-1]:
        raise ValueError(f"singular v-step matrix for class {(vtype, din, dout)}")
    Kinv = np.linalg.inv(K1)
    Kinv[4, :] = 0.0; Kinv[:, 4] = 0.0
    Phi = N @ Kinv @ N.T
    up = _forward(np.zeros(n), d, jstar, prim, term, True)
    g0u = up - Phi @ (D @ up)
    nfam = 1 if term else 2
    dinv = np.zeros((2, 5))
    for g in range(2):
        s = np.array([1.0, 1.0, float(g), float(g), 1.0])       # rho-quadratic: first point always, second point of out-edges, flow
        dinv[g, :4] = 1.0 / (s[:4] + nfam * kappa)
        dinv[g, 4] = 1.0 / (theta + 2 * nfam * kappa)
    members = [[j for j in range(d) if not out[j]], [j for j in range(d) if out[j]]]
    G = np.zeros((NCX, NCX)); g0 = np.zeros(NCX)

    def col(k):          # u-space column(s) an input of the extended core stands for (a representative block per group)
        if k < 9:
            return CORE_IDX[k]
        g, tau = divmod(k - 9, 5)
        return _uw(members[g][0]) + tau if members[g] else None
    for k in range(9):
        g0[k] = g0u[CORE_IDX[k]]
        for j in range(NCX):
            cj = col(j)
            if cj is not None:
                G[k, j] = Phi[CORE_IDX[k], cj]
    for g in range(2):
        if not members[g]:
            continue
        b0 = members[g][0]
        for tau in range(5):
            row = _uw(b0) + tau
            g0[9 + 5 * g + tau] = g0u[row]
            for j in range(NCX):
                if j < 9:
                    G[9 + 5 * g + tau, j] = Phi[row, CORE_IDX[j]]
                    continue
                g2, tau2 = divmod(j - 9, 5)
                if not members[g2]:
                    continue
                if g2 != g:
                    G[9 + 5 * g + tau, j] = Phi[row, _uw(members[g2][0]) + tau2]
                elif len(members[g]) >= 2:
                    G[9 + 5 * g + tau, j] = Phi[row, _uw(members[g][1]) + tau2]
                else:
                    G[9 + 5 * g + tau, j] = Phi[row, _uw(b0) + tau2] - (dinv[g, tau] if tau2 == tau else 0.0)
    return dict(G=G, g0=g0, dinv=dinv, Phi=Phi, g0u=g0u, members=members, term=term, d=d)


def structured_vstep(T, r):
    """Reference evaluation of the structured v-step (what the kernel does): ``r`` in the u-space layout -> u."""
    d, members = T["d"], T["members"]
    inp = np.zeros(NCX)
    inp[:9] = r[list(CORE_IDX)]
    for g in range(2):
        for j in members[g]:
            inp[9 + 5 * g:14 + 5 * g] += r[_uw(j):_uw(j) + 5]
    core = T["G"] @ inp + T["g0"]
    u = np.zeros(NCORE + 5 * d)
    u[list(CORE_IDX)] = core[:9]
    for g in range(2):
        for j in members[g]:
            u[_uw(j):_uw(j) + 5] = T["dinv"][g] * r[_uw(j):_uw(j) + 5] + core[9 + 5 * g:14 + 5 * g]
    return u


# limits of one tile (= one thread block of the perf kernel): consecutive vertices are packed greedily up to these.
# TILE_BLOCKS blocks = 4 * TILE_BLOCKS (point, flow) pairs = one pair per thread of a block of TILE_THREADS threads.
import os as _os
TILE_BLOCKS = int(_os.environ.get("GCS_TILE_BLOCKS", "64"))
TILE_THREADS = int(_os.environ.get("GCS_TILE_THREADS", str(min(256, 4 * TILE_BLOCKS))))
TILE_VERTS, TILE_CONE, TILE_HE = 32, 160, 128


def perf_tables(g, kappa=1.0, cone=None, theta=1.0, frames="global", edge_delta=None, edge_cent=None):
    """Everything ``gcsadmm_enable_perf`` uploads (``include/gcsadmm.h`` ``GcsPerfConfig``): class tables, cone records,
    the block list (one block per live half-edge plus one per vertex for (z_v, y_v)) and the tiling of the vertices.
    ``cone = (cone_off, cone)`` reuses records computed elsewhere (multi-GPU: sliced from the global graph).
    ``frames="local"``: every vertex program runs in coordinates centred on its own region (cone records of the shifted
    polygons + ``edge_delta``); same optimisation problem, translation-invariant and far better conditioned on large maps."""
    nV = g.nV
    owner = np.repeat(np.arange(nV, dtype=np.int64), np.diff(np.asarray(g.he_off, dtype=np.int64)))
    flags = np.asarray(g.he_flags)
    live = (flags & 2) == 0
    outm = (flags & 1) == 1
    vtype = np.asarray(g.vtype)
    din = np.bincount(owner[live & ~outm], minlength=nV)
    dout = np.bincount(owner[live & outm], minlength=nV)
    alive = vtype != 3
    keys = {}
    vclass = np.full(nV, -1, dtype=np.int32)
    code = vtype.astype(np.int64) * 1000000 + din * 1000 + dout
    tabs = []
    for cd in np.unique(code[alive]):
        key = (int(cd // 1000000), int((cd // 1000) % 1000), int(cd % 1000))
        keys[key] = len(keys)
        T = class_tables(*key, kappa, theta)
        tabs.append(np.concatenate([np.ascontiguousarray(T["G"].T).reshape(-1), T["g0"], T["dinv"].reshape(-1), np.zeros(2)]))      # G transposed (coalesced lanes)
        vclass[(code == cd) & alive] = keys[key]
    cls_tab = np.ascontiguousarray(np.concatenate(tabs)) if tabs else np.zeros(CLS_STRIDE)
    # frames = "local": every vertex program in coordinates centred on its own region (gcsadmm.h GcsPerfConfig.edge_delta)
    cent = np.asarray(g.interior_points()) if frames == "local" else None
    if cone is None:
        cone_off, cone_rec = cone_table(g, shift=cent)
    else:
        cone_off, cone_rec = cone
    if frames == "local" and edge_delta is None:
        if not hasattr(g, "edge_tail"):
            raise ValueError("local frames need edge_tail / edge_head (single-GPU graphs)")
        edge_delta = np.ascontiguousarray(cent[np.asarray(g.edge_tail, dtype=np.int64)] - cent[np.asarray(g.edge_head, dtype=np.int64)])
        edge_cent = np.ascontiguousarray(cent[np.asarray(g.edge_tail, dtype=np.int64)])       # residuals in global coordinates (check variant)
    # blocks: live half-edges of every live vertex in half-edge order, then its (z_v, y_v) block
    nlive = np.where(alive, din + dout, 0).astype(np.int64)
    nblk = np.where(alive, nlive + 1, 0).astype(np.int64)
    blk_off = np.zeros(nV + 1, dtype=np.int64)
    np.cumsum(nblk, out=blk_off[1:])
    Btot = int(blk_off[-1])
    blk_he = np.full(Btot, -1, dtype=np.int32)
    blk_v = np.repeat(np.arange(nV, dtype=np.int64), nblk)
    hl = np.nonzero(live & alive[owner])[0]                     # live half-edges, already grouped by owner in half-edge order
    rank_in_v = np.arange(hl.shape[0]) - np.repeat(np.cumsum(nlive) - nlive, nlive)
    blk_he[blk_off[owner[hl]] + rank_in_v] = hl
    grp = np.full(Btot, 2, dtype=np.int64)
    grp[blk_off[owner[hl]] + rank_in_v] = outm[hl].astype(np.int64)
    # the kernel sums a vertex's in-blocks and out-blocks as two contiguous ranges: in-blocks first, then out-blocks, then the z-block
    if Btot and not np.all((np.diff(grp) >= 0) | (np.diff(blk_v) != 0)):
        raise ValueError("perf tables need every vertex's in-half-edges before its out-half-edges")
    # tiles: greedy over consecutive vertices
    he_cnt = np.diff(np.asarray(g.he_off, dtype=np.int64))
    cone_cnt = np.diff(np.asarray(cone_off, dtype=np.int64))
    tile_voff = _greedy_tiles(nblk, he_cnt, cone_cnt)
    tile_of_v = np.repeat(np.arange(tile_voff.shape[0] - 1), np.diff(tile_voff))
    vloc = np.arange(nV, dtype=np.int64) - tile_voff[tile_of_v]
    term = (vtype != 0)
    blk_info = (vloc[blk_v] | (grp << 8) | (term[blk_v].astype(np.int64) << 10)).astype(np.int32)
    tv0, tv1 = tile_voff[:-1], tile_voff[1:]
    caps = dict(nb=int((blk_off[tv1] - blk_off[tv0]).max()) if nV else 1, nvt=int((tv1 - tv0).max()) if nV else 1,
                cone=int((np.asarray(cone_off, np.int64)[tv1] - np.asarray(cone_off, np.int64)[tv0]).max()) if nV else 1,
                he=int((np.asarray(g.he_off, np.int64)[tv1] - np.asarray(g.he_off, np.int64)[tv0]).max()) if nV else 1)
    return dict(vclass=vclass, cls_tab=cls_tab, cone_off=np.asarray(cone_off, dtype=np.int32), cone=np.ascontiguousarray(cone_rec),
                blk_off=blk_off.astype(np.int32), blk_he=blk_he, blk_info=blk_info, tile_voff=tile_voff.astype(np.int32),
                caps=caps, classes=keys, kappa=float(kappa), theta=float(theta), edge_delta=edge_delta, edge_cent=edge_cent if frames == "local" else None,
                frames=frames, threads=TILE_THREADS)


def _greedy_tiles(nblk, he_cnt, cone_cnt):
    """Tile boundaries: consecutive vertices while blocks <= TILE_BLOCKS, vertices <= TILE_VERTS, cone records <= TILE_CONE
    and half-edges <= TILE_HE (a single vertex above a limit gets a tile of its own)."""
    nV = nblk.shape[0]
    cb, ch, cc = np.concatenate([[0], np.cumsum(nblk)]), np.concatenate([[0], np.cumsum(he_cnt)]), np.concatenate([[0], np.cumsum(cone_cnt)])
    bounds = [0]
    v = 0
    while v < nV:
        # furthest end with every limit respected (binary search per limit on the cumulative sums)
        e = min(int(np.searchsorted(cb, cb[v] + TILE_BLOCKS, side="right")) - 1,
                int(np.searchsorted(ch, ch[v] + TILE_HE, side="right")) - 1,
                int(np.searchsorted(cc, cc[v] + TILE_CONE, side="right")) - 1, v + TILE_VERTS, nV)
        e = max(e, v + 1)
        bounds.append(e)
        v = e
    return np.array(bounds, dtype=np.int64)


def local_tables(T, lp):
    """Tables of one rank's share of the graph (``partition.LocalProblem``): the cone records are sliced from the global
    table in the rank's vertex order, blocks / tiles / classes are rebuilt for the local half-edge layout."""
    lv = np.asarray(lp.global_vertices, dtype=np.int64)
    off = T["cone_off"].astype(np.int64)
    cnt = off[lv + 1] - off[lv]
    loff = np.zeros(lv.shape[0] + 1, dtype=np.int64)
    np.cumsum(cnt, out=loff[1:])
    rec = T["cone"].reshape(-1, 12)
    idx = np.repeat(off[lv] - loff[:-1], cnt) + np.arange(int(loff[-1]))
    frames = T.get("frames", "global")
    delta = np.ascontiguousarray(T["edge_delta"][np.asarray(lp.global_edges, dtype=np.int64)]) if frames == "local" else None
    ecent = np.ascontiguousarray(T["edge_cent"][np.asarray(lp.global_edges, dtype=np.int64)]) if frames == "local" and T.get("edge_cent") is not None else None
    return perf_tables(lp, T["kappa"], cone=(loff.astype(np.int32), np.ascontiguousarray(rec[idx])), theta=T.get("theta", 1.0), frames=frames, edge_delta=delta,
                       edge_cent=ecent)
