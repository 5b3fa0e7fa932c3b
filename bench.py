"""bench.py — ADMM iterations/s of the full-vertex-split iteration (reference admm_solver_v3.py:655-733) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload grid316|grid100|grid1000|batch4096] [--impl reference]
                    [--dump-outputs DIR]

A "step" is one ADMM iteration (K1 vertex programs + the fused edge / dual / residual / control kernel) over the whole
workload.  `value` = iterations/s with everything resident in HBM (CUDA events on the library's stream, L2 flushed before
every timed iteration); `e2e` = the same K iterations through the host-buffer C-ABI calls: graph + warm state uploaded
from host memory, K iterations, solution downloaded — all inside the timed region.  One JSON line on stdout (rank 0).

Headline mode.  The perf mode (north_star kernel (1): fixed-iteration inner scheme) is the headline only if its parity
gate passes IN THIS RUN (benchmark1-4 solved by solve(mode="perf") to its stop rule: relaxed cost within 1e-4 of the
stored classic optimum, rounded result = the reference's stored one); otherwise the parity mode (exact vertex programs,
the reference's trajectory) is the headline and the perf numbers stay nested.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "admm_iterations_per_second"
UNIT = "it/s"
WORKLOADS = {"grid316": 316, "grid100": 100, "grid1000": 1000}     # BASELINE metric config, config 3, config 5 (+ batch4096 = config 4)
PERF_STATE_BYTES_PER_BLOCK = 96 * 2          # t state of one block, read + written by K1 every iteration (not algorithmic: warm-start state)


def algorithmic_bytes(g):
    """SURVEY.md section 8d: compulsory fp64 traffic of one ADMM iteration.
    K1: targets z (gather, H*5) + mu (H*5) read, xc (H*5) written, polytopes, CSR indices.
    K2-5: xc read (H*5), z read+written (2*E*5), mu read+written (2*H*5), edge->half-edge indices."""
    E, H, V = g.nE, 2 * g.nE, g.nV
    sum_m = int(g.poly_off[-1])
    k1 = 8 * (3 * 5 * H + 3 * sum_m) + 4 * (V + 1) + 4 * H + H + V + 16 * V
    k2 = 8 * (3 * 5 * H + 2 * 5 * E) + 8 * E
    return k1, k2


class ClockSampler(threading.Thread):
    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.samples, self._halt = index, [], threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._halt.wait(0.1)

    def finish(self):
        self._halt.set()
        self.join(timeout=6)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(s) > 2 + i and s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.samples[0][1]) if self.samples[0][1].isdigit() else None,
                "reasons": reasons}


def build_workload(name, rank=0, world=1):
    """-> (PackedGraph, description).  Grids: SURVEY 8d recipe (generator.grid_problem); batch4096: queries rank::world."""
    import utils  # noqa: F401
    if name in WORKLOADS:
        from gcs_admm_b200.generator import grid_packed_graph
        G = WORKLOADS[name]
        g = grid_packed_graph(G)
        return g, f"grid{G}x{G} 2-D GCS: {g.nV} vertices, {g.nE} directed edges, m=8 rows/region"
    if name.startswith("batch"):
        from gcs_admm_b200.graph import pack_batch, pack_graph
        from gcs_admm_b200.queries import make_queries
        nq = int(name[5:] or 4096)
        qs = make_queries(nq)[rank::world]
        g = pack_batch([pack_graph(A, b) for A, b in qs])
        return g, (f"batch of {nq} independent benchmark4-sized start/goal queries (s, t in one component of the region graph), "
                   f"{len(qs)} on this GPU: {g.nV} vertices, {g.nE} directed edges, block-diagonal, per-problem residuals / rho / stop")
    raise SystemExit(f"unknown workload {name!r}")


DUMP_BYTES = 60 * 10 ** 6        # payload cap of --dump-outputs: with the .npy headers the files stay under 64 MB


def dump_outputs(out_dir, outputs):
    """Writes every array of `outputs` (one row per vertex, edge or problem) as <out_dir>/<name>.npy in float64.  When
    together they exceed DUMP_BYTES (the million-vertex grid, long runs of a batch), each keeps the same fraction of its
    rows, at least one, drawn by default_rng(0) and kept in order: the sample depends only on the array's length, so two
    runs with the same arguments store the same rows."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in outputs.items()}
    one_row = sum(a[:1].nbytes for a in arrays.values())
    if one_row > DUMP_BYTES:
        raise SystemExit(f"--dump-outputs: one row of every output is {one_row} bytes, more than the {DUMP_BYTES} allowed; use fewer --steps")
    frac = min(1.0, (DUMP_BYTES - one_row) / sum(a.nbytes for a in arrays.values()))    # sum of max(1, n * frac) rows <= DUMP_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        if frac < 1.0:
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], max(1, int(a.shape[0] * frac)), replace=False))]
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


def steady_state(g, burn, mode="parity", tables=None, inner=1):
    """burn-in on the GPU -> host copies of (xc, mu, z, rho, it[, tstate, tn]): the state every arm's timed iterations start from"""
    from gcs_admm_b200 import lib
    s = lib.Solver(g, device=0, max_it=max(1000, burn + 8), eps_abs=0.0, eps_rel=0.0)
    if mode == "perf":
        s.enable_perf(inner_iters=inner, tables=tables)
    s.step(burn)
    st = list(s.state())
    if mode == "perf":
        st += list(s.perf_state())
    s.close()
    return st


def oracle_rate(g, state, iters, warmup=1):
    """the C oracle (port of the reference's algorithm: exact vertex programs, OpenMP over vertices) on the FULL workload,
    started from `state`; every timed step is one real ADMM iteration.  -> (it/s, seconds per step list, cores)"""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import c_oracle
    cores = c_oracle.use_all_cores()
    o = c_oracle.COracle(g, max_it=10 ** 6, eps_abs=0.0, eps_rel=0.0)
    if state is not None:
        o.set_state(state[0][:g.H], state[1], state[2], state[3], state[4])
    for _ in range(warmup):
        o.step(1)
    per = []
    for _ in range(iters):
        t0 = time.perf_counter()
        o.step(1)
        per.append(time.perf_counter() - t0)
    return iters / sum(per), per, cores


def run_reference(args):
    """--impl reference: the reference's own algorithm on the host cores.  The reference itself (pydrake + MOSEK) is not
    installable offline, so the oracle port stands in (kind='port').  Every step is one real ADMM iteration at the
    workload's full size; the start state is the steady state after the same burn-in as the GPU arm (produced by the GPU
    library when a device is present — untimed, only to skip ~20 minutes of CPU burn-in — else a cold start)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    g, desc = build_workload(args.workload if not args.workload.startswith("batch") else "batch256")
    G = WORKLOADS.get(args.workload, 0)
    burn = (G + 10) if args.burn_in < 0 else args.burn_in
    state, how = None, "cold start (no CUDA device for the burn-in): early iterations answer most vertex programs by the zero shortcut"
    try:
        from gcs_admm_b200 import lib
        if lib.load().gcsadmm_device_count() > 0 and burn > 0:
            state = steady_state(g, burn)
            how = f"state after {burn} burn-in iterations in parity mode, produced on the GPU (untimed) and injected with set_state"
    except Exception as e:       # the arm must still run without the CUDA library
        how += f" [{type(e).__name__}]"
    W = max(0, min(args.warmup, 2))
    val, per, cores = oracle_rate(g, state, args.steps, warmup=W)
    sample = f"{args.steps} real ADMM iterations of the C oracle at the workload's full size ({g.nV} vertices), {W} untimed before; start = {how}"
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sum(per) / len(per), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": desc, "sample": sample},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if not args.no_classic:
        # the reference's other CPU solver (classic_solver.py: one monolithic conic program), Drake-free restatement, bounded sample
        from gcs_admm_b200.classic import solve_classic
        from gcs_admm_b200.generator import grid_problem, packed_to_dicts
        off, A, b, _, _ = grid_problem(8)
        As, bs = packed_to_dicts(off, A, b)
        t0 = time.perf_counter()
        rc = solve_classic(As, bs, 2, round_solution=False)
        line["classic_solver"] = {"workload": f"grid8x8 ({len(As)} vertices)", "seconds": time.perf_counter() - t0, "status": rc["status"],
                                  "ip_iterations": rc["iterations"], "cost": rc["cost"], "kind": "port (gcs_admm_b200.classic, sparse interior point, 1 thread)",
                                  "note": "whole solve to optimality, not an iteration rate"}
    print(json.dumps(line))


MODE_TEXT = {"parity": "parity (every vertex program solved to 1e-8 by the interior-point kernel; the reference's trajectory)",
             "perf": "perf (inexact x-update: K warm-started closed-form splitting iterations per ADMM iteration, gcsadmm_enable_perf; "
                     "same fixed point, gated by the parity gate of this run)"}


def parity_gate(verbose=False):
    """The perf mode's contract, checked in this run on benchmark1-4 (the problems with stored reference runs):
    solve(mode="perf") to its stop rule -> relaxed cost within 1e-4 relative of the stored classic optimum, rounded
    final cost within 1e-4 relative of the stored v3 result, same curve (Hausdorff <= 1e-3), same vertex labels where
    the optimum has one labelling (benchmark1, benchmark4).  The full gate (9 problems) is tests/test_gpu_perf.py."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import utils  # noqa: F401
    from conftest import load_golden
    from path_utils import gold_path, hausdorff, polyline
    from gcs_admm_b200.solver import solve
    out, ok = {}, True
    for name in ("benchmark1", "benchmark2", "benchmark3", "benchmark4"):
        As, bs, n, d, keys = load_golden(name)
        t0 = time.perf_counter()
        res = solve(As, bs, n, mode="perf", seed=0, rounding_kw=dict(N=20, M=100) if name == "benchmark3" else None)
        gpath, gx, gcost = gold_path(As, d, keys, "v3")
        rel = abs(res["cost"] - float(d["classic_cost"])) / float(d["classic_cost"])
        frel = abs(res["final_cost"] - gcost) / gcost
        hd = hausdorff(polyline(res["x_v_rounded"], res["path"]), polyline(gx, gpath))
        same = res["path"] == gpath
        good = bool(res["converged"] and rel <= 1e-4 and frel <= 1e-4 and hd <= 1e-3 and (same or name in ("benchmark2", "benchmark3")))
        ok = ok and good
        out[name] = {"ok": good, "iterations": res["iterations"], "seconds": round(time.perf_counter() - t0, 3), "cost_rel_err_vs_classic": rel,
                     "final_cost_rel_err_vs_v3": frel, "curve_hausdorff": hd, "same_vertex_labels": same}
    return {"passed": ok, "stop_rule": "max(pri, dual) < 3e-5 (solver.PERF_ABS_TOL), K=1", "problems": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", type=str, default="grid316", help="grid316 (BASELINE metric config, 99 858 vertices) | grid100 (config 3) | "
                    "grid1000 (config 5) | batch4096 (config 4: independent queries, sharded rank::world)")
    ap.add_argument("--grid", type=int, default=0, help="shorthand: --grid G = --workload gridG")
    ap.add_argument("--impl", type=str, default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-classic", action="store_true", help="reference arm: skip the classic-solver sample")
    ap.add_argument("--burn-in", type=int, default=-1, help="untimed iterations before the timed window (default: grid side + 10, so that the\n                    cold-start wave has reached every vertex and no vertex program is the trivial all-zero one)")
    ap.add_argument("--mode", type=str, default="auto", choices=["auto", "parity", "perf"],
                    help="auto: perf if the parity gate passes in this run, else parity; parity: exact interior-point x-update (reference trajectory); "
                         "perf: K closed-form splitting iterations per x-update")
    ap.add_argument("--inner", type=int, default=1, help="K of the perf mode")
    ap.add_argument("--no-gate", action="store_true", help="skip the parity gate (then --mode auto means parity)")
    ap.add_argument("--no-other-mode", action="store_true", help="do not also time the non-headline mode as a nested report")
    ap.add_argument("--dist", type=str, default="peer", choices=["peer", "nccl"],
                    help="N > 1: peer = halos and residual sums as flag-ordered peer-memory stores over NVLink (no collective call in the iteration); "
                         "nccl = all_to_all_single + all_reduce per iteration")
    ap.add_argument("--dist-graph", action="store_true", help="N > 1, --dist nccl: replay one captured CUDA graph per ADMM iteration (kernels + NCCL collectives)")
    ap.add_argument("--residual-budget", type=float, default=-1.0,
                    help="seconds allowed for the time-to-residual-1e-4 run (perf mode); -1: 330 for the metric workload on 1 GPU, else 0; N > 1: any value > 0 enables the run (bounded by --residual-cap)")
    ap.add_argument("--residual-cap", type=int, default=1_200_000, help="N > 1: iteration cap of the time-to-residual run (ranks cannot agree on a wall-clock budget)")
    ap.add_argument("--outer-alpha", type=float, default=1.0, help="over-relaxation of the consensus step in the time-to-residual run")
    ap.add_argument("--dump-outputs", type=str, default=None, metavar="DIR",
                    help="1 GPU: write what the timed path returns after its last step (solution x_v, z_v, y_v, z_e; rho / pri_res / dual_res "
                         "of the timed steps, one row per problem of a batch) as DIR/<name>.npy, float64, at most 64 MB (a seeded row sample of larger outputs)")
    args = ap.parse_args()
    if args.grid:
        WORKLOADS.setdefault(f"grid{args.grid}", args.grid)
        args.workload = f"grid{args.grid}"
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (args.impl == "reference" or world > 1 or args.gpus > 1):
        ap.error("--dump-outputs is implemented for the single-GPU path only")
    if args.impl == "reference":
        return run_reference(args)
    if world > 1 or args.gpus > 1:
        from gcs_admm_b200 import dist_bench  # multi-GPU path (vertex-partitioned grids / sharded query batches)
        import gcs_admm_b200  # noqa: F401
        return dist_bench.main(args)

    from gcs_admm_b200 import lib, perf as perf_mod
    W = max(3, args.warmup)
    g, desc = build_workload(args.workload)
    batched = args.workload.startswith("batch")
    G = WORKLOADS.get(args.workload, 0)
    burn = max(W, (G + 10 if G else 100) if args.burn_in < 0 else args.burn_in)
    k1_bytes, k2_bytes = algorithmic_bytes(g)
    tables = perf_mod.perf_tables(g)
    gate = None
    if args.mode in ("auto", "perf") and not args.no_gate:
        gate = parity_gate()
    headline = "perf" if (args.mode == "perf" or (args.mode == "auto" and gate and gate["passed"])) else "parity"
    if args.mode == "perf" and gate and not gate["passed"]:
        headline = "parity"        # the gate decides, not the flag

    def timed(mode, steps, burn_it, keep_outputs=False):
        """burn-in, then `steps` iterations timed one by one with CUDA events on the solver's stream, L2 flushed before each;
        keep_outputs: also return what a caller of this path receives after the last timed iteration"""
        s = lib.Solver(g, device=0, max_it=max(1000, steps + burn_it + 8), eps_abs=0.0, eps_rel=0.0)
        if mode == "perf":
            s.enable_perf(inner_iters=args.inner, tables=tables)
        s.step(burn_it)
        st0 = s.status()
        sampler = ClockSampler(0)
        sampler.start()
        # the whole window is enqueued ahead (no host round trip between iterations); every iteration has its own CUDA event
        # pair on the solver's stream and an in-stream L2 eviction before it, outside the pair
        it_ms, k1_ms_ = s.time_window(steps, 256 << 20, split=True)
        tot, k1 = float(it_ms.sum()), float(k1_ms_.sum())
        ed = tot - k1
        clocks = sampler.finish()
        st = s.status()
        state = list(s.state()) + (list(s.perf_state()) if mode == "perf" else [])
        outputs = None
        if keep_outputs:
            outputs = dict(zip(("x_v", "z_v", "y_v", "z_e"), s.solution()))
            # rho / residuals of the timed iterations, one row per problem (a batch keeps them per problem); NaN after a
            # problem's own stop
            n_prob = len(g.prob_voff) - 1 if getattr(g, "prob_voff", None) is not None else 1
            hist = np.full((3, n_prob, steps), np.nan)
            for p in range(n_prob):
                for q, h in enumerate(s.problem_history(p)):
                    seg = h[st0["iterations"] + 1: st0["iterations"] + 1 + steps]
                    hist[q, p, :len(seg)] = seg
            outputs.update(zip(("rho", "pri_res", "dual_res"), hist))
        s.close()
        return dict(ms=tot / steps, k1_ms=k1 / steps, ed_ms=ed / steps, clocks=clocks, st0=st0, st=st, state=state, outputs=outputs)

    def end_to_end(mode, state, n):
        """host buffers -> host buffers through the C-ABI, wall clock: graph / tables / warm state upload + n iterations + download"""
        t0 = time.perf_counter()
        s = lib.Solver(g, device=0, max_it=max(1000, state[4] + n + 8), check_every=max(1, min(64, n)), eps_abs=0.0, eps_rel=0.0)
        if mode == "perf":
            s.enable_perf(inner_iters=args.inner, tables=tables)
        s.set_state(state[0], state[1], state[2], state[3], state[4])
        if mode == "perf":
            s.set_perf_state(state[5], state[6])
        s.run(n)
        s.solution(); s.history()
        dt = time.perf_counter() - t0             # results are in host memory; the handle's teardown (~50 ms of cudaFree) is not part of it
        it = s.status()["iterations"]
        s.close()
        assert it == state[4] + n, (it, state[4], n)
        return dt

    def state_bytes(mode, state):
        gs = sum(np.asarray(a).nbytes for a in (g.poly_off, g.polyA, g.polyb, g.he_off, g.he_edge, g.he_flags, g.edge_he_tail, g.edge_he_head, g.vtype)) + 16 * g.nV
        gs += sum(np.asarray(a).nbytes for a in state if isinstance(a, np.ndarray))
        if mode == "perf":
            gs += sum(np.asarray(tables[k]).nbytes for k in ("vclass", "cls_tab", "cone_off", "cone", "blk_off", "blk_he", "blk_info", "tile_voff"))
        return gs

    m = timed(headline, args.steps, burn, keep_outputs=bool(args.dump_outputs))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, m["outputs"])
    ms, k1_ms, ed_ms, clocks = m["ms"], m["k1_ms"], m["ed_ms"], m["clocks"]
    e2e_s = end_to_end(headline, m["state"], args.steps)
    n_long = 1000 if headline == "perf" else 50
    e2e_long = end_to_end(headline, m["state"], n_long)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    traffic = None          # dram__bytes_read.sum + dram__bytes_write.sum of one K1 launch, from the committed ncu capture of this round
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_k1perf_traffic.json" if headline == "perf" else "r01_k1_traffic.json")))
        if tj.get("workload") in (args.workload, f"grid{G}x{G}") and (headline == "parity" or tj.get("inner_iters") == args.inner):
            traffic = tj["traffic_bytes_per_launch"]
    except Exception:
        pass
    out_bytes = 8 * (9 * g.nV + 5 * g.nE) + 3 * 8 * (args.steps + 1)
    achieved = k1_bytes / (k1_ms * 1e-3) / 1e9
    nblk = int(tables["blk_he"].shape[0])
    line = {
        "metric": METRIC, "value": 1e3 / ms, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": W,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": desc + (" (BASELINE.json metric config: 100k-vertex 2-D GCS)" if args.workload == "grid316" else ""),
                   "mode": MODE_TEXT[headline] + (f", K={args.inner}" if headline == "perf" else ""),
                   "l2": "flushed (256 MiB memset in-stream before every timed iteration, outside its event pair)", "burn_in_iterations": burn,
                   "inner_iters_per_vertex": (m["st"]["inner_iters"] - m["st0"]["inner_iters"]) / max(1, args.steps * g.nV)},
        "clocks": clocks,
        "e2e": {"value": args.steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": state_bytes(headline, m["state"]) / args.steps,
                "d2h_bytes_per_step": out_bytes / args.steps, "seconds": e2e_s,
                "note": "the SAME steady-state work as `value`, from host buffers: gcsadmm_create (graph upload) [+ gcsadmm_enable_perf (tables)] + gcsadmm_set_state "
                        "[+ set_perf_state] (warm state of the timed window's start) + gcsadmm_run(K = steps) + get_solution / get_history (clock stops when the results are in host "
                        "memory, before gcsadmm_destroy); wall clock; pageable host memory",
                f"amortised_over_{n_long}_iterations": {"value": n_long / e2e_long, "seconds": e2e_long}},
        "gpu_launches": 2 * args.steps,
        "roofline": {"bound": "hbm", "kernel": "vertex_kernel (K1)" if headline == "parity" else "vertex_perf_kernel (K1, perf mode)",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "peak_source": "measured (MEASURED_PEAKS.json)" if peaks else "fallback",
                     "algorithmic_bytes_per_launch": k1_bytes, "kernel_ms": k1_ms,
                     "warm_state_bytes_per_launch": PERF_STATE_BYTES_PER_BLOCK * nblk if headline == "perf" else None,
                     "whole_iteration": {"bytes": k1_bytes + k2_bytes, "achieved": (k1_bytes + k2_bytes) / (ms * 1e-3) / 1e9,
                                         "frac": (k1_bytes + k2_bytes) / (ms * 1e-3) / 1e9 / peak},
                     "edge_kernel": {"bytes": k2_bytes, "ms": ed_ms, "achieved": k2_bytes / (ed_ms * 1e-3) / 1e9,
                                     "frac": k2_bytes / (ed_ms * 1e-3) / 1e9 / peak}},
    }
    if gate is not None:
        line["parity_gate"] = gate
    if not args.no_other_mode and not batched:
        other = "parity" if headline == "perf" else "perf"
        if other == "parity" or (gate is None or True):
            osteps = max(3, min(args.steps, 10)) if other == "parity" else args.steps
            om = timed(other, osteps, burn)
            line[other + "_mode"] = {"what": "the other mode on the same workload with the same timing protocol: " + MODE_TEXT[other],
                                     "value": 1e3 / om["ms"], "unit": UNIT, "ms_per_step": om["ms"], "kernel_ms": om["k1_ms"], "edge_ms": om["ed_ms"], "steps": osteps,
                                     "roofline_frac_k1": k1_bytes / (om["k1_ms"] * 1e-3) / 1e9 / peak,
                                     "roofline_frac_iteration": (k1_bytes + k2_bytes) / (om["ms"] * 1e-3) / 1e9 / peak, "clocks": om["clocks"]}
            if other == "parity":
                parity_state = om["state"]
    if not args.no_cpu_baseline and not batched:
        # the reference's algorithm on the host cores at the SAME size, from the parity-mode steady state (no |V| scaling)
        pst = locals().get("parity_state") or steady_state(g, burn)
        n_cpu = 3
        val, per, cores = oracle_rate(g, pst, n_cpu, warmup=1)
        line["cpu_baseline"] = {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"{n_cpu} real ADMM iterations of the C oracle (exact vertex programs, OpenMP) on the whole workload ({g.nV} vertices), "
                                          f"1 untimed before, started from the GPU's parity-mode state after {burn} iterations (set_state)",
                                "seconds_per_iteration": per}
    budget = args.residual_budget if args.residual_budget >= 0 else (330.0 if args.workload == "grid316" else 0.0)
    if budget > 0 and not batched:
        line["time_to_residual_1e-4"] = time_to_residual(g, tables, budget, args.outer_alpha, ms if headline == "perf" else None)
    print(json.dumps(line))


# the accelerated perf-mode configuration of the time-to-residual run (profiles/r02_convergence_sweep_grid100_local_frames_warm_alpha.log)
TTR = dict(rho0=3.0, outer_alpha=1.7, warm="dijkstra", frames="local", inner=1, window=100, cap=4_000_000)


def time_to_residual(g, tables, budget_s, outer_alpha=None, ms_hint=None, tol=1e-4, certify=True):
    """BASELINE metric, second half: wall time of a perf-mode run to max(pri, dual, inner) < 1e-4 with pri / dual by the reference's
    definitions (global coordinates: GcsStatus.pri_res_ref / dual_res_ref; device-side stop test every iteration, host polls every 256).  Local coordinate frames (perf.perf_tables frames="local": the same problem, vertex programs
    centred on their regions), rho0 = 3, over-relaxed consensus step (1.7) and duals started from the portal-graph cost-to-go
    field (gcs_admm_b200.warmstart; primal variables start at zero) — all three change the trajectory, not the fixed point.
    The clock covers the host-side table build and warm start too.  Bounded by `budget_s`; reports what was reached, plus the
    certificate of gcs_admm_b200.certify (straight-line lower bound, relaxed cost, Dijkstra-path upper bound)."""
    from gcs_admm_b200 import lib, perf as perf_mod
    oa = TTR["outer_alpha"] if outer_alpha in (None, 1.0) else outer_alpha
    cap = TTR["cap"]
    t_all = time.perf_counter()
    tables = perf_mod.perf_tables(g, frames=TTR["frames"])
    t_tab = time.perf_counter() - t_all
    s = lib.Solver(g, device=0, max_it=cap, abs_stop=1, abs_tol=tol, check_every=256, frac=TTR["window"] / cap, outer_alpha=oa, rho0=TTR["rho0"])
    s.enable_perf(inner_iters=TTR["inner"], tables=tables)
    t_w = time.perf_counter()
    s.warm_start(field=TTR["warm"], rho=TTR["rho0"])
    t_w = time.perf_counter() - t_w
    t0 = time.perf_counter()
    st = s.status()
    chunk = 20000
    while not st["converged"] and not st["diverged"] and st["iterations"] < cap - chunk and time.perf_counter() - t0 < budget_s:
        st = s.run(chunk)
    dt = time.perf_counter() - t0
    out = {"definition": "max(pri, dual, inner) < tolerance with the residuals of the local-frame formulation the run iterates on (translation-invariant); "
                         "inner = residual of the vertex programs' own cone constraints",
           "reached": bool(st["converged"]), "seconds": dt, "seconds_with_host_setup": time.perf_counter() - t_all, "iterations": st["iterations"],
           "pri_res": st["pri_res"], "dual_res": st["dual_res"], "inner_res": st["inner_res"], "pri_res_reference_definition": st["pri_res_ref"],
           "dual_res_reference_definition": st["dual_res_ref"], "rho": st["rho"], "tolerance": tol, "budget_seconds": budget_s, "outer_alpha": oa,
           "mode": f"perf K={TTR['inner']}, local coordinate frames, rho0 = {TTR['rho0']} (reference rho rule during the first {TTR['window']} iterations), "
                   f"over-relaxed consensus step, duals started from the portal-graph cost-to-go field ({TTR['warm']}), primal start 0",
           "host_table_seconds": t_tab, "host_warm_start_seconds": t_w,
           "reference_definition_note": "pri_res / dual_res by the reference's formulas (:598, :602) are in GLOBAL coordinates, where a flow mismatch eps at "
                                        "position c counts as eps * |c| (|c| up to 447 on this map) and an absolute threshold depends on the map's origin; "
                                        "the values of this iterate are reported above.  Stopping on them (GcsParams.stop_ref): 1e-4 reached at the 10k-vertex "
                                        "grid after 167 290 iterations / 7.8 s; at 100k vertices 1.9e-3 after 1.7 M iterations / 547 s, relaxed cost within "
                                        "1e-4 relative of its limit from ~1.5 M iterations on (profiles/r02_time_to_residual_grid316_ref_definition.jsonl)"}
    x_v, z_v, y_v, z_e = s.solution()
    out["relaxed_cost"] = float(np.sum(np.linalg.norm(z_v[:, :2] - z_v[:, 2:], axis=1)) + 1e-4 * np.sum(z_e[:, 4]))
    s.close()
    if certify:
        try:
            from gcs_admm_b200.certify import certificate
            out["certificate"] = certificate(g, z_v, z_e)
        except Exception as e:
            out["certificate"] = {"error": f"{type(e).__name__}: {e}"}
    return out


if __name__ == "__main__":
    main()
