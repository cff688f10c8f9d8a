"""Candidate-list 2-opt (Mode N) from the nearest-neighbour tour: phases, step times and results.

Uniform instances of the BASELINE generator (seed = n) at 10k, 100k and 10^6 cities, k in {5, 8, 10},
the f32 metric everywhere and also nint at 100k.  Per run: wall time of tl_problem_set_candidates,
tl_nn_tour and the search from host buffers (tl_local_search), the search's device time, moves /
scans / evals, us per step over a steady window (CUDA events of the session's own timing), final
length.  At 10k, full Mode B (nint matrix and f32 recompute) to its optimum in the same run; at
100k, tl_session_time_scans of one full Mode B scan next to one Mode N scan.  The card's name, power
limit and max SM clock are read in the same run.  Writes one JSON file under --out.

    python scripts/two_opt_neighbor_timing.py --out DIR [--sizes 10000,100000,1000000]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import oracle as O  # noqa: E402  (instance generator only)
import teeline_b200 as T  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def wall(f):
    t0 = time.perf_counter()
    r = f()
    return r, (time.perf_counter() - t0) * 1e3


def length(prob, t):
    return float(prob.tour_lengths(t)[0])


def step_us(prob, start, moves):
    """us per Mode N step over a steady window in the middle of the search (after the long early reversals)."""
    if moves < 40:
        return None
    a = moves // 2
    w = min(2000, moves // 4)
    s = prob.session(T.ALGO_TWO_OPT_NEIGHBOR, start)
    s.run(a)
    ms0 = s.stats().device_ms
    s.run(a + w)
    st = s.stats()
    s.close()
    return (st.device_ms - ms0) * 1e3 / w


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--sizes", default="10000,100000,1000000")
    ap.add_argument("--ks", default="5,8,10")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    sizes = [int(v) for v in args.sizes.split(",")]
    ks = [int(v) for v in args.ks.split(",")]
    ctx = T.Context(0)
    res = {"card": card(), "runs": [], "mode_b_10k": [], "scan_100k": None}
    print(res["card"], flush=True)
    for n in sizes:
        x, y = O.gen_uniform(n, n)
        for metric in (["f32", "nint"] if n == 100_000 else ["f32"]):
            prob = T.Problem.euc2d(ctx, x, y, T.DIST_NINT_I32 if metric == "nint" else T.DIST_F32_EXACT)
            prob.set_candidates(1)  # warm-up: modules loaded before anything is timed
            start, nn_ms = wall(lambda: prob.nn_tour(3))
            for k in ks:
                _, cand_ms = wall(lambda: prob.set_candidates(k))
                (t, st, _), search_ms = wall(lambda: prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR, start))
                r = {"n": n, "metric": metric, "k": k, "set_candidates_ms": cand_ms, "nn_tour_ms": nn_ms,
                     "search_wall_ms": search_ms, "search_device_ms": st.device_ms, "moves": int(st.moves),
                     "scans": int(st.passes), "evals": int(st.evals), "converged": int(st.converged),
                     "nn_length": length(prob, start), "length": length(prob, t),
                     "step_us": step_us(prob, start, int(st.moves))}
                if n == 100_000 and k == 8:
                    s = prob.session(T.ALGO_TWO_OPT_NEIGHBOR, start)
                    r["scan_ms_time_scans"] = s.time_scans(200)
                    s.close()
                res["runs"].append(r)
                print(json.dumps(r), flush=True)
            if n == 100_000 and metric == "f32":
                s = prob.session(T.ALGO_TWO_OPT_BEST, start)
                res["scan_100k"] = {"mode_b_full_scan_ms": s.time_scans(10)}
                s.close()
                print(json.dumps(res["scan_100k"]), flush=True)
            if n == 10_000:
                for mb_metric, path in (("nint", T.PATH_MATRIX), ("f32", T.PATH_RECOMPUTE)):
                    pb = prob if mb_metric == "f32" else T.Problem.euc2d(ctx, x, y, T.DIST_NINT_I32)
                    (t, st, _), ms = wall(lambda: pb.local_search(T.ALGO_TWO_OPT_BEST, start, path=path))
                    r = {"n": n, "metric": mb_metric, "path": "matrix" if path == T.PATH_MATRIX else "recompute",
                         "wall_ms": ms, "device_ms": st.device_ms, "moves": int(st.moves), "length": length(pb, t)}
                    res["mode_b_10k"].append(r)
                    print(json.dumps(r), flush=True)
            prob.close()
    if res["scan_100k"]:
        nl = [r for r in res["runs"] if r["n"] == 100_000 and r["metric"] == "f32" and r["k"] == 8]
        if nl:
            res["scan_100k"]["mode_n_k8_scan_ms"] = nl[0]["scan_ms_time_scans"]
            res["scan_100k"]["mode_n_k8_step_us"] = nl[0]["step_us"]
            res["scan_100k"]["ratio_full_scan_over_mode_n_step"] = \
                res["scan_100k"]["mode_b_full_scan_ms"] * 1e3 / nl[0]["step_us"]
    with open(os.path.join(args.out, "two_opt_neighbor_timing.json"), "w") as f:
        json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
