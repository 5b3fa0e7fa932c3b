"""``solve(As, bs, n)`` — host mirror of the reference's ``admm_solver_v3.py`` script.

The reference has no callable entry point (its loop runs at module level,
``admm_solver_v3.py:621-775``); this function packages the same sequence:
build graph (:53) -> ADMM loop on the GPU (:655-733) -> last iterates as dicts (:745-748)
-> cost (:750) -> rounding (:759).  The graph is converted once to the half-edge CSR layout and
every iteration runs in ``libgcsadmm.so``; there is no CPU path for the loop.
"""
from __future__ import annotations

import time

import numpy as np

from . import lib
from .graph import build_graph, pack_batch, pack_graph
from .rounding import compute_cost, rounding

__all__ = ["solve", "solve_batch", "MAX_IT"]

MAX_IT = 1000     # reference admm_solver_v3.py:651

# Contract of the perf mode (DESIGN.md section 5a).  Its trajectory is not the reference's, so it is not stopped by the
# reference's loose rule (eps_rel = 1e-3 halts at residuals ~1e-2, where the flows of different trajectories still round
# differently) but iterated to the fixed point all trajectories share: max(pri, dual) < PERF_ABS_TOL.  At that point
# (tests/test_gpu_perf.py, all nine problem files) the relaxed cost is within 1e-4 relative of the classic optimum and the
# rounded result equals the reference's stored one (same curve, same final cost).  rho adapts during the first
# PERF_ADAPT_WINDOW iterations only (the reference's window, :703-709, is 0.1 * MAX_IT = 100 iterations as well).
PERF_ABS_TOL = 3e-5          # for problems whose s-t distance is >= PERF_LENGTH_SCALE (all four benchmarks); scaled down below it
PERF_LENGTH_SCALE = 3.0
PERF_MAX_IT = 400000
PERF_ADAPT_WINDOW = 100


def perf_abs_tol(g):
    """Stop tolerance of the perf mode: residuals are absolute lengths, so for a problem smaller than the benchmarks (s-t
    distance below ``PERF_LENGTH_SCALE``) the tolerance shrinks with it — the contract is a RELATIVE cost error of 1e-4."""
    c = g.interior_points()
    if g.src < 0 or g.dst < 0:
        return PERF_ABS_TOL
    dist = float(np.linalg.norm(c[g.src] - c[g.dst]))
    return PERF_ABS_TOL * min(1.0, max(dist, 1e-3) / PERF_LENGTH_SCALE)


def solve(As, bs, n, *, device=0, max_it=MAX_IT, round_solution=True, seed=None, verbose=False,
          graph=None, one_call=True, mode="parity", inner_iters=1, rounding_kw=None, frames="global", warm_start=None, **params):
    """Solve the convex relaxation of the GCS shortest-path problem by full-vertex-split ADMM.

    Parameters mirror the reference's literals (``rho0, tau_incr, tau_decr, nu, frac, eps_abs,
    eps_rel`` — ``admm_solver_v3.py:621-651``) plus ``inner_tol``/``inner_max_iter`` for the vertex
    programs and ``abs_stop``/``abs_tol`` for the "residual < 1e-4" metric.

    ``mode="parity"`` (default) solves every vertex program exactly and reproduces the reference's trajectory;
    ``mode="perf"`` does ``inner_iters`` closed-form splitting iterations per x-update instead (same fixed point,
    far cheaper iterations, not the reference's trajectory) and, unless told otherwise, iterates to
    max(pri, dual) < ``PERF_ABS_TOL`` (at most ``PERF_MAX_IT`` iterations) — the stop rule its parity gate is defined for.

    Returns a dict: cost (pre-rounding, what the reference pickles), final_cost, x_v_sol, y_v_sol,
    z_v_sol, y_e_sol (also under the short names x_v, y_v, z_v, y_e), x_v_rounded, y_v_rounded, path, iterations,
    converged, diverged, rho_seq, pri_res_seq, dual_res_seq, solve_time, status, mode, V, E.
    ``rounding_kw``: overrides of the rounding literals ``N=5, M=20`` (reference ``GCS_utils.py:92``).
    ``frames="local"`` (perf mode): vertex programs in coordinates centred on their own regions — the same problem, a
    translation-invariant and much better conditioned ADMM on large maps (``perf.perf_tables``).
    ``warm_start="dijkstra"`` (perf mode): the duals start from a shortest-path cost-to-go field over the portal graph instead
    of zero (``warmstart.py``; the reference starts cold, ``admm_solver_v3.py:621-652``) — same fixed point, about half the
    iterations on large maps; ``outer_alpha`` (1 < a < 2, e.g. 1.7) over-relaxes the consensus step.
    """
    if int(n) != 2:
        raise ValueError("gcs-admm_b200 implements the 2-D case (n = 2), like all reference data")
    if graph is None:
        V, E, I_v_in, I_v_out = build_graph(As, bs)
        g = pack_graph(As, bs, V, E)
    else:
        V, E, I_v_in, I_v_out, g = graph
    t0 = time.perf_counter()
    max_it = _mode_defaults(mode, max_it, params)
    if mode == "perf":
        params.setdefault("abs_tol", perf_abs_tol(g))
    if one_call and mode == "parity":
        out = lib.solve_host(g, device=device, max_iters=max_it, max_it=max_it, **params)
    else:
        s = lib.Solver(g, device=device, max_it=max_it, **params)
        if mode == "perf":
            s.enable_perf(inner_iters=inner_iters, frames=frames)
            if warm_start:
                s.warm_start(field=warm_start)
        st = s.run(max_it)
        x_v, z_v, y_v, z_e = s.solution()
        rho, pri, dual = s.history()
        s.close()
        out = dict(status=st, x_v=x_v, z_v=z_v, y_v=y_v, z_e=z_e, rho_seq=rho, pri_res_seq=pri, dual_res_seq=dual)
    solve_time = time.perf_counter() - t0
    st = out["status"]
    if verbose:
        print(f"it = {st['iterations']}/{max_it}, pri_res_seq[-1]={st['pri_res']}, dual_res_seq[-1]={st['dual_res']}")
    return _result(out, V, E, I_v_out, As, bs, n, mode, solve_time, round_solution, seed, rounding_kw)


def solve_batch(queries, *, device=0, max_it=MAX_IT, round_solution=True, seed=None, mode="parity", inner_iters=1,
                rounding_kw=None, frames="global", warm_start=None, **params):
    """Solve many independent problems (start / goal queries) in one handle: ``queries`` is a list of ``(As, bs)`` in the
    reference's format (n = 2).  The problems are packed block-diagonally (``graph.pack_batch``); each keeps its own residuals,
    rho, stop decision and, in the perf mode, its own tolerance ``perf_abs_tol`` (unless ``abs_tol`` is given).  A query's
    iterates, iteration count and stop are those of ``solve()`` on it alone with the same options.

    Takes ``solve()``'s keyword arguments and returns a list with one ``solve()`` result dict per query; ``solve_time`` is the
    time of the whole batch.  Rounding runs per query on the host."""
    built = []
    for As, bs in queries:
        V, E, I_v_in, I_v_out = build_graph(As, bs)
        built.append((V, E, I_v_out, pack_graph(As, bs, V, E)))
    big = pack_batch([b[3] for b in built])
    t0 = time.perf_counter()
    max_it = _mode_defaults(mode, max_it, params)
    tols = [perf_abs_tol(b[3]) for b in built] if mode == "perf" and "abs_tol" not in params else None
    s = lib.Solver(big, device=device, max_it=max_it, **params)
    try:
        if mode == "perf":
            s.enable_perf(inner_iters=inner_iters, frames=frames)
            if tols is not None:
                s.set_problem_tolerance(tols)
            if warm_start:
                s.warm_start(field=warm_start)
        s.run(max_it)
        x_v, z_v, y_v, z_e = s.solution()
        per = [(s.problem_status(q), s.problem_history(q)) for q in range(len(built))]
    finally:
        s.close()
    solve_time = time.perf_counter() - t0
    out = []
    for q, ((V, E, I_v_out, g), (st, (rho, pri, dual))) in enumerate(zip(built, per)):
        v0, v1, e0, e1 = big.prob_voff[q], big.prob_voff[q + 1], big.prob_eoff[q], big.prob_eoff[q + 1]
        arrays = dict(status=st, x_v=x_v[v0:v1], z_v=z_v[v0:v1], y_v=y_v[v0:v1], z_e=z_e[e0:e1], rho_seq=rho, pri_res_seq=pri, dual_res_seq=dual)
        As, bs = queries[q]
        out.append(_result(arrays, V, E, I_v_out, As, bs, 2, mode, solve_time, round_solution, seed, rounding_kw))
    return out


def _mode_defaults(mode, max_it, params):
    """the perf mode's stop rule and adaptation window (DESIGN.md section 5a) unless the caller set them -> max_it"""
    if mode not in ("parity", "perf"):
        raise ValueError("mode must be 'parity' or 'perf'")
    if mode == "perf":
        if max_it == MAX_IT:
            max_it = PERF_MAX_IT
        params.setdefault("abs_stop", 1)
        params.setdefault("frac", PERF_ADAPT_WINDOW / max_it)
        params.setdefault("check_every", 64)
    return max_it


def _result(out, V, E, I_v_out, As, bs, n, mode, solve_time, round_solution, seed, rounding_kw):
    """one problem's arrays (status, x_v, z_v, y_v, z_e, rho / pri / dual sequences) -> the result dict of ``solve()``"""
    st = out["status"]
    x_v_sol = {v: out["x_v"][i].copy() for i, v in enumerate(V)}        # :745
    y_v_sol = {v: float(out["y_v"][i]) for i, v in enumerate(V)}        # :746
    y_e_sol = {e: float(out["z_e"][i, 4]) for i, e in enumerate(E)}     # :747
    z_v_sol = {v: out["z_v"][i].copy() for i, v in enumerate(V)}        # :748
    cost = compute_cost(z_v_sol, y_e_sol)                               # :750
    res = dict(cost=cost, x_v_sol=x_v_sol, y_v_sol=y_v_sol, z_v_sol=z_v_sol, y_e_sol=y_e_sol,
               iterations=int(st["iterations"]), converged=bool(st["converged"]), diverged=bool(st["diverged"]),
               rho_seq=out["rho_seq"], pri_res_seq=out["pri_res_seq"], dual_res_seq=out["dual_res_seq"],
               solve_time=solve_time, status=st, V=V, E=E, final_cost=None, x_v_rounded=None, y_v_rounded=None, path=None,
               mode=mode)
    res.update(x_v=x_v_sol, y_v=y_v_sol, z_v=z_v_sol, y_e=y_e_sol)      # short names of SURVEY.md section 8b (same objects)
    if round_solution:
        if res["diverged"]:      # the reference would round NaN flows (:662-664 then :759): no path can be sampled from them
            y_e_sol = {e: (y if np.isfinite(y) else 0.0) for e, y in y_e_sol.items()}
        fc, xr, yr, path = rounding(y_e_sol, V, E, I_v_out, As, bs, n, rng=seed, return_path=True, **(rounding_kw or {}))   # :759
        res.update(final_cost=fc, x_v_rounded=xr, y_v_rounded=yr, path=path)
    return res
