"""BASELINE config 4: a batch of independent start/goal queries on the benchmark4 region set.

    python tools/batch_queries.py --queries 4096 [--gpus N via torchrun: each rank takes queries rank::world]

Every query is the 40 benchmark4 regions plus its own (s, t) drawn by rejection sampling inside two distinct
random regions (np.random.default_rng(1)); queries are packed block-diagonally (gcs_admm_b200.graph.pack_batch)
and solved in one handle per GPU with per-problem residuals / rho / stop — no communication.
Prints one JSON line: problems/s, aggregate ADMM iterations/s, iteration statistics, the largest per-query
max(pri, dual, inner) at the stop, and the card's name and power limit.

The perf mode's accelerated configuration (DESIGN.md section 5a) on the same batch:

    python tools/batch_queries.py --mode perf --abs-stop --frames local --outer-alpha 1.7 --warm-start dijkstra --rho0 3

--abs-stop stops every query at its own tolerance (solver.perf_abs_tol) with its inner residual in the test.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import utils  # noqa: E402,F401
from gcs_admm_b200.graph import pack_batch, pack_graph  # noqa: E402
from gcs_admm_b200.queries import make_queries  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=4096)
    ap.add_argument("--max-it", type=int, default=1000)
    ap.add_argument("--mode", default="parity", choices=["parity", "perf"])
    ap.add_argument("--inner", type=int, default=1, help="K of the perf mode")
    ap.add_argument("--eps-rel", type=float, default=1e-3, help="reference stop rule (1e-3); perf mode wants a tighter one")
    ap.add_argument("--eps-abs", type=float, default=1e-4)
    ap.add_argument("--frames", default="global", choices=["global", "local"], help="perf mode: coordinates of the vertex programs")
    ap.add_argument("--outer-alpha", type=float, default=1.0, help="perf mode: over-relaxation of the consensus step")
    ap.add_argument("--warm-start", default=None, choices=["dijkstra", "euclid"], help="perf mode: dual start from a cost-to-go field")
    ap.add_argument("--rho0", type=float, default=1.0)
    ap.add_argument("--abs-stop", action="store_true", help="perf mode: max(pri, dual, inner) < each query's perf_abs_tol")
    ap.add_argument("--all-pairs", action="store_true", help="draw (s, t) from any two regions (46 %% of the pairs then have no path); default: same component")
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    from gcs_admm_b200 import lib
    from gcs_admm_b200.solver import PERF_ADAPT_WINDOW, perf_abs_tol
    t0 = time.perf_counter()
    qs = make_queries(args.queries, feasible_only=not args.all_pairs)[rank::world]
    graphs = [pack_graph(A, b) for A, b in qs]
    big = pack_batch(graphs)
    t_build = time.perf_counter() - t0
    t0 = time.perf_counter()
    abs_stop = args.mode == "perf" and args.abs_stop
    extra = dict(abs_stop=1, check_every=64, frac=PERF_ADAPT_WINDOW / args.max_it) if abs_stop else dict(check_every=16)
    s = lib.Solver(big, device=local, max_it=args.max_it, eps_rel=args.eps_rel, eps_abs=args.eps_abs, rho0=args.rho0,
                   outer_alpha=args.outer_alpha, **extra)
    if args.mode == "perf":
        s.enable_perf(inner_iters=args.inner, frames=args.frames)
        if abs_stop:
            s.set_problem_tolerance([perf_abs_tol(g) for g in graphs])
        if args.warm_start:
            s.warm_start(field=args.warm_start)
    t1 = time.perf_counter()
    st = s.run(args.max_it)
    t_run = time.perf_counter() - t1
    x_v, z_v, y_v, z_e = s.solution()
    dt = time.perf_counter() - t0
    ps = [s.problem_status(p) for p in range(len(graphs))]
    its = np.array([p["iterations"] for p in ps])
    conv = np.array([p["converged"] for p in ps])
    worst = max(max(p["pri_res"], p["dual_res"], p["inner_res"]) for p in ps)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local)],
                          capture_output=True, text=True).stdout.strip()
    line = {"mode": args.mode + (f" K={args.inner}" if args.mode == "perf" else ""), "eps_rel": args.eps_rel, "eps_abs": args.eps_abs, "max_it": args.max_it,
            "frames": args.frames, "outer_alpha": args.outer_alpha, "warm_start": args.warm_start, "rho0": args.rho0,
            "abs_stop": "per-query perf_abs_tol" if abs_stop else None, "card": card,
            "rank": rank, "world": world, "queries": len(graphs), "vertices": int(big.nV), "edges": int(big.nE),
            "host_build_s": t_build, "solve_s": dt, "seconds_to_all_stopped": t_run, "problems_per_s": len(graphs) / dt,
            "aggregate_problem_iterations_per_s": float(its.sum()) / dt, "converged": int(conv.sum()),
            "iterations_min_median_max": [int(its.min()), int(np.median(its)), int(its.max())],
            "max_query_residual_at_stop": worst,
            "inner_fail": st["inner_fail"], "inner_iters": st["inner_iters"]}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
