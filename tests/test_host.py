"""Host-side logic that needs no GPU: the C-ABI library's exports, problem files, rounding, generators."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ALL_PROBLEMS, ROOT, load_golden
from gcs_admm_b200.graph import build_graph, pack_graph


def test_library_exports_every_declared_symbol():
    """include/gcsadmm.h is the contract: every function it declares must be exported (no compute call here)."""
    from gcs_admm_b200 import lib
    hdr = open(os.path.join(ROOT, "include", "gcsadmm.h")).read()
    declared = set(re.findall(r"\b(gcsadmm_\w+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    L = lib.load()
    for name in sorted(declared):
        assert hasattr(L, name), f"libgcsadmm.so does not export {name}"
    assert declared == set(lib.EXPORTS)
    assert L.gcsadmm_version().startswith(b"gcsadmm")
    p = lib.default_params()
    assert (p.rho0, p.tau_incr, p.tau_decr, p.nu, p.frac, p.eps_abs, p.eps_rel, p.max_it) == (1.0, 2.0, 2.0, 10.0, 0.1, 1e-4, 1e-3, 1000)
    assert L.gcsadmm_scratch_bytes(8, 8) < 32 * 1024


def test_no_gpu_is_a_loud_error():
    """The product path must fail loudly without CUDA (no CPU fallback)."""
    from gcs_admm_b200 import lib
    if lib.load().gcsadmm_device_count() > 0:
        pytest.skip("a GPU is present")
    As, bs, n, d, keys = load_golden("benchmark1")
    with pytest.raises(lib.GcsError, match="no CPU path"):
        lib.Solver(pack_graph(As, bs))


@pytest.mark.parametrize("name", ALL_PROBLEMS)
def test_problem_files_load_and_match_fixtures(name):
    from gcs_admm_b200.problem_io import load_test_file
    As, bs, n = load_test_file(name)
    Ag, bg, ng, d, keys = load_golden(name)
    assert n == ng == 2 and list(As.keys()) == keys
    for k in keys:
        assert np.array_equal(As[k], Ag[k]) and np.array_equal(bs[k], bg[k])


def test_write_then_load_roundtrip(tmp_path):
    from gcs_admm_b200.problem_io import load_test_file, write_test_file
    As, bs, n, d, keys = load_golden("benchmark2")
    write_test_file(str(tmp_path / "rt.py"), As, bs, s=d["s"], t=d["t"])
    A2, b2, n2 = load_test_file("rt", str(tmp_path))
    assert list(A2.keys()) == keys and all(np.array_equal(A2[k], As[k]) and np.array_equal(b2[k], bs[k]) for k in keys)
    with pytest.raises(ModuleNotFoundError):
        load_test_file("does_not_exist", str(tmp_path))


@pytest.mark.parametrize("name", ["benchmark1", "benchmark2", "benchmark3", "benchmark4"])
def test_rounding_reproduces_stored_path(name):
    """Flows from the (pinned) oracle -> randomized DFS + convex restriction = the reference's stored rounded
    solution: same curve (Hausdorff distance <= 1e-3, the north-star waypoint tolerance), same final cost, and the same
    vertex labels where the optimal curve has one labelling (benchmark1 through the tie policy, benchmark4)."""
    from c_oracle import COracle
    from gcs_admm_b200.rounding import rounding
    from path_utils import gold_path, hausdorff, polyline
    As, bs, n, d, keys = load_golden(name)
    V, E, I_in, I_out = build_graph(As, bs)
    g = pack_graph(As, bs, V, E)
    o = COracle(g)
    o.run()
    _, _, z = o.state()
    y_e = {e: float(z[i, 4]) for i, e in enumerate(E)}
    kw = dict(N=20, M=100) if name == "benchmark3" else {}      # loose relaxation: see tests/test_gpu_perf.py ROUND_KW
    cost, x_r, y_r, path = rounding(y_e, V, E, I_out, As, bs, n, rng=0, return_path=True, **kw)
    gpath, gold_x, gold_cost = gold_path(As, d, keys, "v3")
    assert path[0] == 's' and path[-1] == 't'
    assert abs(cost - gold_cost) < 1e-6 * max(1.0, gold_cost)
    assert hausdorff(polyline(x_r, path), polyline(gold_x, gpath)) <= 1e-3
    if name in ("benchmark1", "benchmark4"):
        assert path == gpath
    # waypoints: feasible, continuous, same length as the stored solution.  (Interior waypoints of collinear
    # stretches can slide along the line at equal cost, so they are compared through the length, and point-wise
    # only at the terminals.)
    for a, b in zip(path[:-1], path[1:]):
        assert np.max(np.abs(x_r[a][2:] - x_r[b][:2])) < 1e-7
    for v in path:
        for i in range(2):
            assert np.all(As[v] @ x_r[v][2 * i: 2 * i + 2] <= bs[v] + 1e-7)
    assert np.max(np.abs(x_r['s'] - gold_x['s'])) < 1e-3 and np.max(np.abs(x_r['t'] - gold_x['t'])) < 1e-3
    assert all(y_r[v] == (1 if v in path else 0) for v in V)


def test_compute_cost_and_pickle_schema(tmp_path):
    import pickle
    import utils
    from gcs_admm_b200.rounding import compute_cost
    z = {0: np.array([0.0, 0.0, 3.0, 4.0]), 1: np.array([1.0, 1.0, 1.0, 1.0])}
    assert abs(compute_cost(z, {(0, 1): 0.5, (1, 0): 1.0}) - (5.0 + 1.5e-4)) < 1e-15
    f = tmp_path / "sub" / "x.pkl"
    utils.save_data(str(f), {}, {}, 1.0, 2.0, {}, {}, {}, {}, True, 7, np.ones(8), np.zeros(8), np.zeros(8))
    dd = pickle.load(open(f, "rb"))
    assert list(dd) == ["As", "bs", "solve_time", "cost", "x_v_sol", "y_v_sol", "x_v_rounded", "y_v_rounded", "ADMM",
                        "iterations", "rho_seq", "pri_res_seq", "dual_res_seq"]


def test_grid_generator_and_random_generator():
    from gcs_admm_b200.generator import generate_test_2D, grid_packed_graph
    g = grid_packed_graph(7)
    assert g.nV == 51 and g.nE == 4 * 7 * 6 + 4 and g.max_rows == 8 and g.max_live_degree == 8
    assert list(np.bincount(g.vtype)) == [49, 1, 1]
    As, bs, s, t = generate_test_2D(None, -10, 10, 1, 0.9, 12, seed=3)
    V, E, _, _ = build_graph(As, bs)
    assert V[:2] == ["s", "t"] and len(V) == 14 and len(E) % 2 == 0
    for k in As:
        assert As[k].shape[1] == 2 and As[k].shape[0] == bs[k].shape[0] >= 3
    assert np.all(As["s"] @ s <= bs["s"])


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours): one JSON line with the contract's keys."""
    import json, subprocess, sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--grid", "24", "--steps", "2", "--warmup", "1", "--no-classic"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["metric"] == "admm_iterations_per_second" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # rank != 0 under torchrun: exits 0 without work and without output
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_cli_divergence_landmarks_and_pickle(tmp_path, monkeypatch, capsys):
    """reference :662-664 then :745-775: after "BREAKING FOR Divergence" the script still prints the cost, rounds and pickles.
    The GPU loop is replaced by a canned diverged result here (the device side is tests/test_gpu_solve.py)."""
    import importlib
    import pickle
    import gcs_admm_b200.solver as solver_mod
    cli = importlib.import_module("admm_solver_v3")

    def fake_solve(As, bs, n, **kw):
        V, E, I_in, I_out, g = kw["graph"]
        nan = float("nan")
        return dict(cost=nan, x_v_sol={v: np.zeros(4) for v in V}, y_v_sol={v: nan for v in V}, iterations=7, converged=False, diverged=True,
                    rho_seq=np.ones(8), pri_res_seq=np.r_[0.0, np.ones(6), nan], dual_res_seq=np.r_[0.0, np.ones(6), nan], solve_time=0.1,
                    x_v_rounded=None, y_v_rounded=None, final_cost=float("inf"), path=None)
    monkeypatch.setattr(solver_mod, "solve", fake_solve)
    cli.main(["--test_file=benchmark1", "--show_plot=False", f"--out_dir={tmp_path}"])
    out = capsys.readouterr().out
    assert "BREAKING FOR Divergence" in out and "BREAKING FOR OPT" not in out and "it = 7/1000" not in out
    assert "Cost before rounding" in out and "POST-ROUNDING" in out
    d = pickle.load(open(tmp_path / "admm_solver_v3_benchmark1.pkl", "rb"))
    assert d["iterations"] == 7 and d["ADMM"] is True and len(d["pri_res_seq"]) == 8


def test_cli_pickles_max_it_plus_one_when_exhausted(tmp_path, monkeypatch, capsys):
    """the reference leaves `while it <= MAX_IT` with it = MAX_IT + 1 and pickles that (:733, :775); progress lines every 100 (:716-718)"""
    import importlib
    import pickle
    import gcs_admm_b200.solver as solver_mod
    cli = importlib.import_module("admm_solver_v3")

    def fake_solve(As, bs, n, **kw):
        V, E, I_in, I_out, g = kw["graph"]
        return dict(cost=1.0, x_v_sol={v: np.zeros(4) for v in V}, y_v_sol={v: 0.0 for v in V}, iterations=1000, converged=False, diverged=False,
                    rho_seq=np.ones(1001), pri_res_seq=np.r_[0.0, np.full(1000, 0.5)], dual_res_seq=np.r_[0.0, np.full(1000, 0.25)], solve_time=0.1,
                    x_v_rounded={v: np.zeros(4) for v in V}, y_v_rounded={v: 0 for v in V}, final_cost=1.0, path=["s", "t"])
    monkeypatch.setattr(solver_mod, "solve", fake_solve)
    cli.main(["--test_file=benchmark1", "--show_plot=False", f"--out_dir={tmp_path}"])
    out = capsys.readouterr().out
    assert out.count("it = ") == 10 and "it = 100/1000, pri_res_seq[-1]=0.5, dual_res_seq[-1]=0.25" in out and "it = 1000/1000" in out
    d = pickle.load(open(tmp_path / "admm_solver_v3_benchmark1.pkl", "rb"))
    assert d["iterations"] == 1001
