"""Batched start/goal queries under the perf-mode contract: a query packed into a batch (graph.pack_batch) does what its
stand-alone run does — local frames, over-relaxation, the dual warm start, its own tolerance and its own inner residual in the
stop test — and solver.solve_batch returns solve()'s result for every query."""
import numpy as np
import pytest

from conftest import load_golden
from gcs_admm_b200.graph import pack_batch, pack_graph

BENCH = ["benchmark1", "benchmark2", "benchmark3", "benchmark4"]


def _queries():
    """benchmark1, benchmark2, test3, benchmark4 and four seeded benchmark4 queries; the last one's s-t distance is below
    PERF_LENGTH_SCALE, so its tolerance is scaled down"""
    from gcs_admm_b200.queries import make_queries
    qs = make_queries(63, seed=1)
    return [load_golden(n)[:2] for n in ("benchmark1", "benchmark2", "test3", "benchmark4")] + [qs[i] for i in (0, 1, 2, 62)]


def _accelerated(g, **kw):
    """the accelerated perf configuration: local frames, rho0 = 3, over-relaxation 1.7, absolute stop every 64 iterations"""
    from gcs_admm_b200 import solver
    from gcs_admm_b200.lib import Solver
    p = dict(max_it=solver.PERF_MAX_IT, abs_stop=1, check_every=64, frac=solver.PERF_ADAPT_WINDOW / solver.PERF_MAX_IT,
             rho0=3.0, outer_alpha=1.7)
    p.update(kw)
    return Solver(g, **p).enable_perf(inner_iters=1, frames="local")


# ------------------------------------------------------------------------------------------------------------------ CPU

def _old_cost_to_go(g, field="dijkstra"):
    """warmstart.cost_to_go as it was for a single target (the reference of the single-graph check)"""
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import dijkstra
    from gcs_admm_b200.warmstart import portal_points
    p = portal_points(g)
    c = np.asarray(g.interior_points())
    tgt = c[g.dst]
    nE = g.nE
    tail, head = np.asarray(g.edge_tail, np.int64), np.asarray(g.edge_head, np.int64)
    if field == "euclid":
        d = tgt[None, :] - p
        J = np.linalg.norm(d, axis=1)
        return J, -d / np.where(J > 0, J, 1.0)[:, None]
    order_in = np.argsort(head, kind="stable")
    order_out = np.argsort(tail, kind="stable")
    din = np.bincount(head, minlength=g.nV)
    dout = np.bincount(tail, minlength=g.nV)
    in_off = np.concatenate([[0], np.cumsum(din)])
    out_off = np.concatenate([[0], np.cumsum(dout)])
    npair = din * dout
    pv = np.repeat(np.arange(g.nV), npair)
    k = np.arange(int(npair.sum())) - np.repeat(np.cumsum(npair) - npair, npair)
    ei = order_in[in_off[pv] + k // np.maximum(dout[pv], 1)]
    fo = order_out[out_off[pv] + k % np.maximum(dout[pv], 1)]
    keep = tail[ei] != head[fo]
    ei, fo = ei[keep], fo[keep]
    w = np.linalg.norm(p[fo] - p[ei], axis=1) + 1e-12
    into_t = np.nonzero(head == g.dst)[0]
    rows = np.concatenate([fo, np.full(into_t.shape[0], nE)])
    cols = np.concatenate([ei, into_t])
    vals = np.concatenate([w, np.linalg.norm(tgt[None, :] - p[into_t], axis=1) + 1e-12])
    A = csr_matrix((vals, (rows, cols)), shape=(nE + 1, nE + 1))
    dist, pred = dijkstra(A, directed=True, indices=nE, return_predecessors=True)
    J = dist[:nE].copy()
    nxt = pred[:nE]
    ok = np.isfinite(J) & (nxt >= 0)
    J[~ok] = 0.0
    to = np.where(nxt[:, None] == nE, tgt[None, :], p[np.clip(nxt, 0, nE - 1)])
    d = to - p
    n = np.linalg.norm(d, axis=1)
    return J, np.where((ok & (n > 1e-9))[:, None], -d / np.where(n > 1e-9, n, 1.0)[:, None], 0.0)


def _edge_delta(g):
    c = np.asarray(g.interior_points())
    return c[np.asarray(g.edge_tail)] - c[np.asarray(g.edge_head)]


@pytest.mark.parametrize("field", ["dijkstra", "euclid"])
def test_dual_start_of_a_batch_is_the_concatenation_of_its_queries(field):
    from gcs_admm_b200 import warmstart
    graphs = [pack_graph(A, b) for A, b in _queries()]
    big = pack_batch(graphs)
    for delta in (None, _edge_delta(big)):
        mu = warmstart.dual_start(big, delta, 3.0, field=field)
        parts = [warmstart.dual_start(g, None if delta is None else _edge_delta(g), 3.0, field=field) for g in graphs]
        assert np.array_equal(mu, np.concatenate(parts))


@pytest.mark.parametrize("field", ["dijkstra", "euclid"])
@pytest.mark.parametrize("name", ["benchmark1", "benchmark3", "test3"])
def test_cost_to_go_of_a_single_graph_is_unchanged(name, field):
    from gcs_admm_b200 import warmstart
    g = pack_graph(*load_golden(name)[:2])
    J, grad = warmstart.cost_to_go(g, field)
    J0, grad0 = _old_cost_to_go(g, field)
    assert np.array_equal(J, J0) and np.array_equal(grad, grad0)


# ------------------------------------------------------------------------------------------------------------------ GPU

@pytest.mark.gpu
def test_batch_equals_its_queries_in_the_accelerated_configuration():
    """every query of the batch stops at the iteration of its stand-alone run, below its own tolerance with its own inner
    residual, with the same iterates and the same rho history.  (On a B200, 1000 W: in this configuration benchmark4 and the
    benchmark4 queries stall at a dual residual of ~5e-5 and run to PERF_MAX_IT, stand-alone as in the batch; the others stop.)"""
    from gcs_admm_b200.solver import PERF_MAX_IT, perf_abs_tol
    graphs = [pack_graph(A, b) for A, b in _queries()]
    tols = [perf_abs_tol(g) for g in graphs]
    assert min(tols) < max(tols)
    big = pack_batch(graphs)
    sb = _accelerated(big)
    sb.set_problem_tolerance(tols)
    sb.warm_start("dijkstra")
    sb.run()
    x_v, z_v, y_v, z_e = sb.solution()
    stopped = 0
    for q, g in enumerate(graphs):
        s = _accelerated(g, abs_tol=tols[q]).warm_start("dijkstra")
        st = s.run()
        ps = sb.problem_status(q)
        assert ps["iterations"] == st["iterations"] and ps["converged"] == st["converged"], (q, ps, st)
        for k in ("pri_res", "dual_res", "inner_res"):      # only the order of the residual sums differs
            assert abs(ps[k] - st[k]) <= 1e-12 * abs(st[k]), (q, k, ps[k], st[k])
        assert ps["inner_res"] >= 0.0
        if ps["converged"]:
            stopped += 1
            assert 0.0 <= ps["inner_res"] < tols[q] and max(ps["pri_res"], ps["dual_res"]) < tols[q]
        else:
            assert ps["iterations"] == PERF_MAX_IT
        xs, zs, ys, es = s.solution()
        v0, v1, e0, e1 = big.prob_voff[q], big.prob_voff[q + 1], big.prob_eoff[q], big.prob_eoff[q + 1]
        assert np.max(np.abs(zs - z_v[v0:v1])) <= 1e-12 and np.max(np.abs(es - z_e[e0:e1])) <= 1e-12, q
        assert np.array_equal(s.history()[0], sb.problem_history(q)[0]), q
        s.close()
    assert stopped >= 3
    sb.close()


@pytest.mark.gpu
def test_batch_reports_unmeasured_residuals_before_the_switch():
    """far from the tolerance the inner residual is not measured (-1) and the reference-definition residuals fall back to the
    frame residuals"""
    graphs = [pack_graph(A, b) for A, b in _queries()]
    sb = _accelerated(pack_batch(graphs))
    sb.step(50)
    for q in range(len(graphs)):
        ps = sb.problem_status(q)
        assert ps["inner_res"] == -1.0 and ps["pri_res_ref"] == ps["pri_res"] and ps["dual_res_ref"] == ps["dual_res"], (q, ps)
    sb.close()


@pytest.mark.gpu
def test_batch_reference_definition_residuals_vs_numpy():
    """stop_ref in a batch: each query's primal residual in global coordinates, from its own slice of the state (the formula of
    test_gpu_perf.test_reference_definition_residuals_in_local_frames_vs_numpy)"""
    from gcs_admm_b200 import perf
    from gcs_admm_b200.lib import Solver
    graphs = [pack_graph(*load_golden(n)[:2]) for n in BENCH]
    big = pack_batch(graphs)
    T = perf.perf_tables(big, frames="local")
    s = Solver(big, abs_stop=1, abs_tol=1e9, stop_ref=1, check_every=8, frac=0.0, max_it=1000).enable_perf(inner_iters=1, tables=T)
    st = s.run(64)
    assert st["converged"] == 1 and st["iterations"] == 9
    xc, mu, z, rho, it = s.state()
    d, cu = T["edge_delta"], T["edge_cent"]
    cw = cu - d
    xt, xh = xc[big.edge_he_tail], xc[big.edge_he_head]
    bz = z.copy()
    bz[:, 2:4] -= d * z[:, 4:5]
    rt, rh = bz - xt, z - xh
    gt = rt.copy(); gt[:, 0:2] += rt[:, 4:5] * cu; gt[:, 2:4] += rt[:, 4:5] * cu
    gh = rh.copy(); gh[:, 0:2] += rh[:, 4:5] * cu; gh[:, 2:4] += rh[:, 4:5] * cw
    for q in range(len(graphs)):
        e = slice(big.prob_eoff[q], big.prob_eoff[q + 1])
        ps = s.problem_status(q)
        assert ps["iterations"] == 9 and ps["inner_res"] >= 0.0
        loc = np.sqrt(np.sum(rt[e] ** 2) + np.sum(rh[e] ** 2))
        ref = np.sqrt(np.sum(gt[e] ** 2) + np.sum(gh[e] ** 2))
        assert abs(loc - ps["pri_res"]) < 1e-10 * max(1.0, loc)
        assert abs(ref - ps["pri_res_ref"]) < 1e-10 * max(1.0, ref), (q, ref, ps)
    s.close()


@pytest.mark.gpu
def test_per_query_tolerance():
    """one query with a 100x tighter tolerance runs on past the iteration it stops at with the shared one and ends below its own
    tolerance; the other queries stop where they stop without it"""
    from gcs_admm_b200.lib import GcsError, _check, load
    from gcs_admm_b200.solver import perf_abs_tol
    graphs = [pack_graph(*load_golden(n)[:2]) for n in BENCH]
    loose = [perf_abs_tol(g) for g in graphs]
    tight = [loose[0] / 100.0] + loose[1:]
    runs = []
    for tols in (loose, tight):
        sb = _accelerated(pack_batch(graphs), rho0=1.0, outer_alpha=1.0)      # local frames and warm start: all four converge
        sb.warm_start("dijkstra")
        for bad in (-1.0, float("nan")):
            with pytest.raises(GcsError):
                sb.set_problem_tolerance([bad] + tols[1:])
        with pytest.raises(GcsError):
            _check(load().gcsadmm_set_problem_tolerance(sb._h, None))
        sb.set_problem_tolerance(tols)
        assert sb.run()["converged"] == 1
        ps = [sb.problem_status(q) for q in range(len(graphs))]
        for q, p in enumerate(ps):
            assert p["converged"] == 1 and 0.0 <= p["inner_res"] < tols[q] and max(p["pri_res"], p["dual_res"]) < tols[q], (q, p)
        runs.append([p["iterations"] for p in ps])
        sb.close()
    assert runs[1][0] > runs[0][0] and runs[1][1:] == runs[0][1:], runs


@pytest.mark.gpu
def test_global_frames_batch_iterates_are_bit_identical_to_stand_alone_runs():
    """global frames, no over-relaxation: z and mu of every query after 200 iterations equal its stand-alone run's bit for bit"""
    from gcs_admm_b200.lib import Solver
    graphs = [pack_graph(*load_golden(n)[:2]) for n in ("benchmark1", "benchmark2", "test3", "benchmark4")]
    big = pack_batch(graphs)
    sb = Solver(big, max_it=1000).enable_perf(inner_iters=2)
    sb.step(200)
    _, mub, zb, _, _ = sb.state()
    for q, g in enumerate(graphs):
        s = Solver(g, max_it=1000).enable_perf(inner_iters=2)
        s.step(200)
        _, mu, z, _, _ = s.state()
        h0, h1 = big.he_off[big.prob_voff[q]], big.he_off[big.prob_voff[q + 1]]
        assert np.array_equal(z, zb[big.prob_eoff[q]:big.prob_eoff[q + 1]]) and np.array_equal(mu, mub[h0:h1]), q
        s.close()
    sb.close()


def _same_result(a, b):
    assert a["iterations"] == b["iterations"] and a["converged"] == b["converged"]
    assert abs(a["cost"] - b["cost"]) <= 1e-12 * abs(b["cost"])
    assert a["path"] == b["path"] and a["final_cost"] == b["final_cost"]
    assert set(a) == set(b)


@pytest.mark.gpu
def test_solve_batch_equals_solve_in_perf_mode():
    from gcs_admm_b200.solver import solve, solve_batch
    probs = [load_golden(n) for n in BENCH]
    kw = dict(mode="perf", frames="local", warm_start="dijkstra", seed=0)
    res = solve_batch([(As, bs) for As, bs, *_ in probs], **kw)
    for (As, bs, n, d, keys), r in zip(probs, res):
        _same_result(r, solve(As, bs, n, **kw))
        assert abs(r["cost"] - float(d["classic_cost"])) <= 1e-4 * float(d["classic_cost"])


@pytest.mark.gpu
def test_solve_batch_equals_solve_in_parity_mode():
    from gcs_admm_b200.solver import solve, solve_batch
    probs = [load_golden(n) for n in ("benchmark1", "benchmark2")]
    res = solve_batch([(As, bs) for As, bs, *_ in probs], seed=0)
    for (As, bs, n, d, keys), r in zip(probs, res):
        _same_result(r, solve(As, bs, n, seed=0))
