"""Multi-move candidate-list Or-opt (Or-opt NM) next to Or-opt N: steps, moves, time and length to the Or-opt optimum.

BASELINE instances (seed = n): uniform f32 at 10^5 and 10^6 cities, the integer grid (NINT_I32) at 10^5; k = 8.
Per instance, the starts are the Mode NM optima of the greedy-edge tour and of the NN tour.  From each, in one run:
Or-opt N to its optimum, and Or-opt NM to its optimum for each block size in --blocks (set through the
TL_MULTI_BLOCK environment variable, read when a session is created).  Each records scans (steps + 1), moves, wall
and device time, device time per scan and the final length.  The card's name, power limit and max SM clock are read
in the same run.  Writes one JSON file.

    python scripts/or_opt_neighbor_multi_timing.py --out FILE [--cases f32:100000,f32:1000000,nint:100000]
                                                              [--blocks 1024,4096,16384]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import oracle as O  # noqa: E402  (instance generator only)
import teeline_b200 as T  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def length(prob, t):
    return float(prob.tour_lengths(t)[0])


def search(prob, algo, start, block=None):
    if block:
        os.environ["TL_MULTI_BLOCK"] = str(block)
    try:
        t0 = time.perf_counter()
        t, st, _ = prob.local_search(algo, start)
        ms = (time.perf_counter() - t0) * 1e3
    finally:
        os.environ.pop("TL_MULTI_BLOCK", None)
    return t, {"scans": int(st.passes), "moves": int(st.moves), "wall_ms": ms, "device_ms": st.device_ms,
               "device_us_per_scan": st.device_ms * 1e3 / max(1, int(st.passes)), "length": length(prob, t),
               "converged": int(st.converged)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--cases", default="f32:100000,f32:1000000,nint:100000")
    ap.add_argument("--blocks", default="1024,4096,16384")
    args = ap.parse_args()
    blocks = [int(b) for b in args.blocks.split(",")]
    ctx = T.Context(0)
    res = {"card": card(), "k": 8, "built_block": T.OR_MULTI_BLOCK, "runs": []}
    print(res["card"], flush=True)
    # first launches load the modules: warm every kernel the timed calls use on a small instance
    for kind in (T.DIST_F32_EXACT, T.DIST_NINT_I32):
        x, y = O.gen_uniform(20000, 1)
        w = T.Problem.euc2d(ctx, x, y, kind)
        w.set_candidates(8)
        t, _ = w.greedy_tour()
        t = w.local_search(T.ALGO_TWO_OPT_NEIGHBOR_MULTI, t)[0]
        w.local_search(T.ALGO_OR_OPT_NEIGHBOR, t)
        w.local_search(T.ALGO_OR_OPT_NEIGHBOR_MULTI, t)
        w.nn_tour(3)
        w.close()
    for case in args.cases.split(","):
        metric, n = case.split(":")
        n = int(n)
        x, y = O.gen_grid(n, n) if metric == "nint" else O.gen_uniform(n, n)
        prob = T.Problem.euc2d(ctx, x, y, T.DIST_NINT_I32 if metric == "nint" else T.DIST_F32_EXACT)
        prob.set_candidates(8)
        g, _ = prob.greedy_tour()
        r = {"n": n, "metric": metric}
        for name, tour0 in (("from_greedy_mode_nm", g), ("from_nn_mode_nm", prob.nn_tour(3))):
            start, nm = search(prob, T.ALGO_TWO_OPT_NEIGHBOR_MULTI, tour0)
            s = {"mode_nm": nm, "start_length": length(prob, start)}
            _, s["or_opt_n"] = search(prob, T.ALGO_OR_OPT_NEIGHBOR, start)
            print(case, name, "or_opt_n", json.dumps(s["or_opt_n"]), flush=True)
            for b in blocks:
                _, s[f"or_opt_nm_b{b}"] = search(prob, T.ALGO_OR_OPT_NEIGHBOR_MULTI, start, b)
                o = s[f"or_opt_nm_b{b}"]
                o["scan_ratio_vs_or_opt_n"] = s["or_opt_n"]["scans"] / o["scans"]
                o["device_ratio_vs_or_opt_n"] = s["or_opt_n"]["device_ms"] / o["device_ms"]
                print(case, name, f"or_opt_nm_b{b}", json.dumps(o), flush=True)
            r[name] = s
        res["runs"].append(r)
        prob.close()
    d = os.path.dirname(os.path.abspath(args.out))
    os.makedirs(d, exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
