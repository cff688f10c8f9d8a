"""Candidate-list Or-opt (Or-opt N) after 2-opt: step and scan times, and the way to its optimum.

Uniform instances of the BASELINE generator (seed = n), f32 metric.  At 100k and 10^6 cities, from
the Mode N optimum of the nearest-neighbour tour (k = 8), for k in {5, 8, 10}: us per Or-opt N step
over the first moves (CUDA events of the session's own timing), one scan alone
(tl_session_time_scans), and moves, scans, wall and device time and final length of the search to the
Or-opt N optimum.  At 100k also one full K3 Or-opt scan.  At 10k, Or-opt N (k = 8) against K3 Or-opt
from the same Mode B optimum: time and final length.  The card's name, power limit and max SM clock are
read in the same run.  Writes one JSON file under --out.

    python scripts/or_opt_neighbor_timing.py --out DIR [--sizes 100000,1000000] [--ks 5,8,10]
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


def first_steps_us(prob, start, steps=2000):
    """us per step over the first `steps` Or-opt N steps (device time of the session's batches)."""
    s = prob.session(T.ALGO_OR_OPT_NEIGHBOR, start)
    s.run(steps)
    st = s.stats()
    s.close()
    return st.device_ms * 1e3 / max(1, int(st.passes))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--sizes", default="100000,1000000")
    ap.add_argument("--ks", default="5,8,10")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    ks = [int(v) for v in args.ks.split(",")]
    ctx = T.Context(0)
    res = {"card": card(), "runs": [], "or_opt_full_scan_100k_ms": None, "vs_k3_10k": []}
    print(res["card"], flush=True)
    for n in [int(v) for v in args.sizes.split(",")]:
        x, y = O.gen_uniform(n, n)
        prob = T.Problem.euc2d(ctx, x, y)
        prob.set_candidates(8)
        nn = prob.nn_tour(3)
        (start, st2, _), ms2 = wall(lambda: prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR, nn))
        base = {"n": n, "mode_n_k8_moves": int(st2.moves), "mode_n_k8_wall_ms": ms2, "mode_n_length": length(prob, start)}
        print(json.dumps(base), flush=True)
        for k in ks:
            prob.set_candidates(k)
            s = prob.session(T.ALGO_OR_OPT_NEIGHBOR, start)
            scan_ms = s.time_scans(200)
            s.close()
            step_us = first_steps_us(prob, start)
            (t, st, _), search_ms = wall(lambda: prob.local_search(T.ALGO_OR_OPT_NEIGHBOR, start))
            r = dict(base, k=k, scan_ms_time_scans=scan_ms, step_us_first_2000=step_us, search_wall_ms=search_ms,
                     search_device_ms=st.device_ms, moves=int(st.moves), scans=int(st.passes), evals=int(st.evals),
                     converged=int(st.converged), length=length(prob, t))
            res["runs"].append(r)
            print(json.dumps(r), flush=True)
        if n == 100_000:
            s = prob.session(T.ALGO_OR_OPT, start)
            res["or_opt_full_scan_100k_ms"] = s.time_scans(5)
            s.close()
            print(json.dumps({"or_opt_full_scan_100k_ms": res["or_opt_full_scan_100k_ms"]}), flush=True)
        prob.close()
    n = 10_000
    x, y = O.gen_uniform(n, n)
    prob = T.Problem.euc2d(ctx, x, y)
    prob.set_candidates(8)
    start, _, _ = prob.local_search(T.ALGO_TWO_OPT_BEST, prob.nn_tour(3))
    for name, algo in (("or_opt_n_k8", T.ALGO_OR_OPT_NEIGHBOR), ("k3_or_opt", T.ALGO_OR_OPT)):
        prob.local_search(algo, start, max_moves=1)  # warm-up
        (t, st, _), ms = wall(lambda: prob.local_search(algo, start))
        r = {"n": n, "start": "mode_b_optimum", "start_length": length(prob, start), "algo": name, "wall_ms": ms,
             "device_ms": st.device_ms, "moves": int(st.moves), "scans": int(st.passes), "length": length(prob, t)}
        res["vs_k3_10k"].append(r)
        print(json.dumps(r), flush=True)
    prob.close()
    with open(os.path.join(args.out, "or_opt_neighbor_timing.json"), "w") as f:
        json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
