"""Dual warm start of the perf mode from a cost-to-go field (an accelerator of the PERF mode only; the parity mode keeps the
reference's cold start ``admm_solver_v3.py:621-652``: all zeros).

Why: at a fixed point of the full-vertex-split ADMM the scaled dual of the head-side copy of edge e = (u, w) is the gradient of
the head's cost-to-go in the perspective variables,

    rho mu_head(e) = ( 0, 0,  grad J_w(p),  J_w(p) - grad J_w(p) . p )        slots: tail's first point | head's first point | flow

(J_w(p) = cheapest continuation from entering region w at p; the tail's first point is a free copy on the head side, so its
dual vanishes), and the tail side follows from the invariant B' mu_tail + mu_head = 0 of the consensus step
(``csrc/gcsadmm.cu`` ``edge_frames_kernel``).  J is a distance field with the range of the whole map: a cold start has to build
it one hop per iteration, which is what makes the iteration count grow with the square of the graph diameter.  A shortest-path
computation over the PORTALS (one point in the overlap of every edge's two regions) gives J and its gradient up to the
discretisation of the portal points in O(|E| log |E|) on the host; the ADMM then only has to correct local errors.

The primal variables and the inner (cone-splitting) state start from zero as before; any start gives the same fixed point (the
relaxation's optimum) because the iteration is a convergent ADMM from every initial dual.  (Also starting the primal variables
from the unit flow along the portal path was tried and dropped: the single path is not the relaxation's fractional optimum and
the inner duals of the cone constraints are unknown, so the first x-update moves away from it — same residuals after 50 iterations.)
"""
from __future__ import annotations

import numpy as np

__all__ = ["portal_points", "cost_to_go", "dual_start", "portal_path"]


def portal_points(g):
    """one point per edge in (or near) the overlap of its two regions: the midpoint of the regions' interior points, for edges
    of 's' / 't' (point regions) the terminal's own point"""
    c = np.asarray(g.interior_points())
    tail, head = np.asarray(g.edge_tail, np.int64), np.asarray(g.edge_head, np.int64)
    p = 0.5 * (c[tail] + c[head])
    vt = np.asarray(g.vtype)
    for term in (tail, head):
        m = (vt[term] == 1) | (vt[term] == 2)
        p[m] = c[term[m]]
    return p


def cost_to_go(g, field="dijkstra", return_next=False):
    """(J[nE], grad[nE, 2]): cost-to-go from the portal of every edge and its gradient (minus the unit direction of travel).
    ``field="euclid"``: straight-line distance to the target (exact on obstacle-free maps); ``"dijkstra"``: shortest path over
    the portal graph (portal of e = (u, w) -> portal of f = (w, x), weight = their distance), valid for any region graph.
    Edges that cannot reach the target get J = 0, grad = 0 (their flow is forced to zero by the presolve anyway).
    A block-diagonal batch (``graph.pack_batch``) has one target per problem (``g.dsts``): every edge is measured to its own
    problem's target, and since the problems are disconnected one search gives each of them its own field."""
    p = portal_points(g)
    c = np.asarray(g.interior_points())
    nE = g.nE
    dsts = np.atleast_1d(np.asarray(getattr(g, "dsts", [g.dst]), np.int64))
    eoff = getattr(g, "prob_eoff", None)
    prob = np.searchsorted(np.asarray(eoff), np.arange(nE), side="right") - 1 if eoff is not None else np.zeros(nE, np.int64)
    tgt = c[dsts[prob]]                                  # [nE, 2]: the target of every edge's problem
    tail, head = np.asarray(g.edge_tail, np.int64), np.asarray(g.edge_head, np.int64)
    if field == "euclid":
        d = tgt - p
        J = np.linalg.norm(d, axis=1)
        grad = -d / np.where(J > 0, J, 1.0)[:, None]
        if return_next:
            raise ValueError("the euclid field has no successor structure; use field='dijkstra'")
        return J, grad
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import dijkstra
    # arcs e -> f for head(e) == tail(f): all (in-edge, out-edge) pairs of every vertex, built without Python loops
    order_in = np.argsort(head, kind="stable")          # edges grouped by head
    order_out = np.argsort(tail, kind="stable")         # edges grouped by tail
    din = np.bincount(head, minlength=g.nV)
    dout = np.bincount(tail, minlength=g.nV)
    in_off = np.concatenate([[0], np.cumsum(din)])
    out_off = np.concatenate([[0], np.cumsum(dout)])
    npair = din * dout
    pv = np.repeat(np.arange(g.nV), npair)              # vertex of every pair
    k = np.arange(int(npair.sum())) - np.repeat(np.cumsum(npair) - npair, npair)
    ei = order_in[in_off[pv] + k // np.maximum(dout[pv], 1)]
    fo = order_out[out_off[pv] + k % np.maximum(dout[pv], 1)]
    keep = tail[ei] != head[fo]                          # no immediate U-turn
    ei, fo = ei[keep], fo[keep]
    w = np.linalg.norm(p[fo] - p[ei], axis=1) + 1e-12
    # node nE = the target(s): every edge into t connects to it at the remaining distance
    into_t = np.nonzero(np.isin(head, dsts[dsts >= 0]))[0]
    rows = np.concatenate([fo, np.full(into_t.shape[0], nE)])          # reversed arcs: search from the target
    cols = np.concatenate([ei, into_t])
    vals = np.concatenate([w, np.linalg.norm(tgt[into_t] - p[into_t], axis=1) + 1e-12])
    A = csr_matrix((vals, (rows, cols)), shape=(nE + 1, nE + 1))
    dist, pred = dijkstra(A, directed=True, indices=nE, return_predecessors=True)
    J = dist[:nE].copy()
    nxt = pred[:nE]                                      # next portal on the way to the target (nE = the target itself)
    ok = np.isfinite(J) & (nxt >= 0)
    J[~ok] = 0.0
    to = np.where(nxt[:, None] == nE, tgt, p[np.clip(nxt, 0, nE - 1)])
    d = to - p
    n = np.linalg.norm(d, axis=1)
    grad = np.where((ok & (n > 1e-9))[:, None], -d / np.where(n > 1e-9, n, 1.0)[:, None], 0.0)
    if return_next:
        return J, grad, np.where(ok, nxt, -1)
    return J, grad


def dual_start(g, edge_delta, rho, field="dijkstra"):
    """mu[H, 5] (scaled duals, the kernels' sign convention: the x-update's target is z + mu) for local frames
    (``edge_delta`` = cent[tail] - cent[head], ``perf.perf_tables(frames="local")``) or global frames (``edge_delta`` None)."""
    J, grad = cost_to_go(g, field)
    p = portal_points(g)
    c = np.asarray(g.interior_points())
    head = np.asarray(g.edge_head, np.int64)
    pl = p - c[head] if edge_delta is not None else p           # the portal in the head's coordinates
    mu = np.zeros((g.H if hasattr(g, "H") else 2 * g.nE, 5))
    mh = np.zeros((g.nE, 5))
    mh[:, 2:4] = grad
    mh[:, 4] = J - np.sum(grad * pl, axis=1)
    mt = -mh
    if edge_delta is not None:                                   # B' mu_tail + mu_head = 0 with B (p1, p2, y) = (p1, p2 - y delta, y)
        mt[:, 4] = -mh[:, 4] - np.sum(np.asarray(edge_delta) * mh[:, 2:4], axis=1)
    # an edge with a forced-zero half-edge keeps zero duals on BOTH sides: B' mu_tail + mu_head is conserved by the iteration,
    # so a start that violates it would shift the fixed point
    live = (np.asarray(g.he_flags) & 2) == 0
    hh, ht = np.asarray(g.edge_he_head, np.int64), np.asarray(g.edge_he_tail, np.int64)
    dead = ~(live[hh] & live[ht])
    mh[dead] = 0.0
    mt[dead] = 0.0
    mu[hh] = mh
    mu[ht] = mt
    return mu / float(rho)


def portal_path(g):
    """edges of the shortest s-t path over the portal graph (None if the target cannot be reached)"""
    J, _, nxt = cost_to_go(g, "dijkstra", return_next=True)
    tail = np.asarray(g.edge_tail, np.int64)
    p = portal_points(g)
    c = np.asarray(g.interior_points())
    start = np.nonzero((tail == g.src) & (nxt >= 0))[0]
    if start.shape[0] == 0:
        return None
    e = int(start[np.argmin(J[start] + np.linalg.norm(p[start] - c[g.src], axis=1))])
    path = [e]
    while nxt[e] != g.nE:
        e = int(nxt[e])
        if e < 0 or len(path) > g.nE:
            return None
        path.append(e)
    return path
