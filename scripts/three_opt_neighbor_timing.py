"""Candidate-list 3-opt (3-opt N) after Or-opt N: step and scan times, and the way to its optimum.

Uniform instances of the BASELINE generator (seed = n), f32 metric.  At 100k and 10^6 cities, from the
Or-opt N optimum of the nn -> Mode N -> Or-opt N pipeline (k = 8), for k in {5, 8}: us per 3-opt N step
over the first moves (CUDA events of the session's own timing), one scan alone (tl_session_time_scans),
and moves, scans, wall and device time and length before and after the search to the 3-opt N optimum.
A search that stops at --budget moves first says so ("converged": 0, "budget").  At 10k, one full K6
3-opt scan next to one 3-opt N scan (k = 8) on the same tour.  The card's name, power limit and max SM
clock are read in the same run.  Writes one JSON file.

    python scripts/three_opt_neighbor_timing.py --out FILE [--sizes 100000,1000000] [--ks 5,8]
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


def wall(f):
    t0 = time.perf_counter()
    r = f()
    return r, (time.perf_counter() - t0) * 1e3


def length(prob, t):
    return float(prob.tour_lengths(t)[0])


def first_steps_us(prob, start, steps):
    """us per step over the first `steps` 3-opt N steps (device time of the session's batches)."""
    s = prob.session(T.ALGO_THREE_OPT_NEIGHBOR, start)
    s.run(steps)
    st = s.stats()
    s.close()
    return st.device_ms * 1e3 / max(1, int(st.passes))


def pipeline(prob):
    """nn -> Mode N -> Or-opt N, k = 8: the start of 3-opt N."""
    prob.set_candidates(8)
    nn = prob.nn_tour(3)
    (t2, st2, _), ms2 = wall(lambda: prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR, nn))
    (t3, st3, _), ms3 = wall(lambda: prob.local_search(T.ALGO_OR_OPT_NEIGHBOR, t2))
    return t3, {"mode_n_k8_moves": int(st2.moves), "mode_n_k8_wall_ms": ms2, "or_opt_n_k8_moves": int(st3.moves),
                "or_opt_n_k8_wall_ms": ms3, "or_opt_n_length": length(prob, t3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--sizes", default="100000,1000000")
    ap.add_argument("--ks", default="5,8")
    ap.add_argument("--budget", type=int, default=10000, help="move budget of the 10^6-city searches")
    args = ap.parse_args()
    ks = [int(v) for v in args.ks.split(",")]
    ctx = T.Context(0)
    res = {"card": card(), "runs": [], "k6_vs_three_opt_n_10k": None}
    print(res["card"], flush=True)
    for n in [int(v) for v in args.sizes.split(",")]:
        x, y = O.gen_uniform(n, n)
        prob = T.Problem.euc2d(ctx, x, y)
        start, base = pipeline(prob)
        base = dict(n=n, **base)
        print(json.dumps(base), flush=True)
        budget = args.budget if n >= 1_000_000 else -1
        for k in ks:
            prob.set_candidates(k)
            s = prob.session(T.ALGO_THREE_OPT_NEIGHBOR, start)
            scan_ms = s.time_scans(20)
            s.close()
            step_us = first_steps_us(prob, start, 200)
            (t, st, _), search_ms = wall(lambda: prob.local_search(T.ALGO_THREE_OPT_NEIGHBOR, start, max_moves=budget))
            r = dict(base, k=k, scan_ms_time_scans=scan_ms, step_us_first_200=step_us, budget=budget,
                     search_wall_ms=search_ms, search_device_ms=st.device_ms, moves=int(st.moves),
                     scans=int(st.passes), evals=int(st.evals), converged=int(st.converged),
                     length_before=base["or_opt_n_length"], length_after=length(prob, t))
            res["runs"].append(r)
            print(json.dumps(r), flush=True)
        prob.close()
    n = 10_000
    x, y = O.gen_uniform(n, n)
    prob = T.Problem.euc2d(ctx, x, y)
    start, base = pipeline(prob)
    s = prob.session(T.ALGO_THREE_OPT_NEIGHBOR, start)
    nl_ms = s.time_scans(20)
    s.close()
    s = prob.session(T.ALGO_THREE_OPT, start)
    k6_ms = s.time_scans(1)
    s.close()
    res["k6_vs_three_opt_n_10k"] = {"n": n, "start": "or_opt_n_optimum", "k6_full_scan_ms": k6_ms,
                                     "three_opt_n_k8_scan_ms": nl_ms}
    print(json.dumps(res["k6_vs_three_opt_n_10k"]), flush=True)
    prob.close()
    d = os.path.dirname(os.path.abspath(args.out))
    os.makedirs(d, exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
