"""The greedy-edge constructor (tl_greedy_tour) next to the NN tour, and what each start costs Mode N and Or-opt N.

BASELINE instances (seed = n): uniform f32 at 10^5 and 10^6 cities, the integer grid (NINT_I32) at 10^5.
Per instance, in one run: the k = 8 list build (tl_problem_set_candidates) alone; the greedy tour's wall and
device time, device rounds, list rebuilds and length; the NN tour's wall time and length; and from each start,
with k = 8, Mode N to its optimum and then Or-opt N to its optimum, with moves, wall and device time and
lengths.  The card's name, power limit and max SM clock are read in the same run.  Writes one JSON file.

    python scripts/greedy_timing.py --out FILE [--cases f32:100000,f32:1000000,nint:100000]
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


def searches(prob, start):
    (t2, st2, _), ms2 = wall(lambda: prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR, start))
    (t3, st3, _), ms3 = wall(lambda: prob.local_search(T.ALGO_OR_OPT_NEIGHBOR, t2))
    return {"start_length": length(prob, start),
            "mode_n_moves": int(st2.moves), "mode_n_wall_ms": ms2, "mode_n_device_ms": st2.device_ms,
            "mode_n_length": length(prob, t2),
            "or_opt_n_moves": int(st3.moves), "or_opt_n_wall_ms": ms3, "or_opt_n_device_ms": st3.device_ms,
            "or_opt_n_length": length(prob, t3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--cases", default="f32:100000,f32:1000000,nint:100000")
    args = ap.parse_args()
    ctx = T.Context(0)
    res = {"card": card(), "k": 8, "runs": []}
    print(res["card"], flush=True)
    # first launches load the modules: warm every kernel the timed calls use on a small instance
    for kind in (T.DIST_F32_EXACT, T.DIST_NINT_I32):
        x, y = O.gen_grid(2000, 1)
        w = T.Problem.euc2d(ctx, x, y, kind)
        w.set_candidates(8)
        t, _ = w.greedy_tour()
        w.local_search(T.ALGO_OR_OPT_NEIGHBOR, w.local_search(T.ALGO_TWO_OPT_NEIGHBOR, t)[0])
        w.nn_tour(3)
        w.close()
    for case in args.cases.split(","):
        metric, n = case.split(":")
        n = int(n)
        x, y = O.gen_grid(n, n) if metric == "nint" else O.gen_uniform(n, n)
        prob = T.Problem.euc2d(ctx, x, y, T.DIST_NINT_I32 if metric == "nint" else T.DIST_F32_EXACT)
        _, knn_ms = wall(lambda: prob.set_candidates(8))
        (g, gst), g_ms = wall(prob.greedy_tour)
        nn, nn_ms = wall(lambda: prob.nn_tour(3))
        r = {"n": n, "metric": metric, "knn_k8_wall_ms": knn_ms,
             "greedy": {"wall_ms": g_ms, "device_ms": gst.device_ms, "rounds": int(gst.passes),
                        "list_rebuilds": int(gst.repermutes), "launches": int(gst.launches), "length": length(prob, g)},
             "nn": {"wall_ms": nn_ms, "length": length(prob, nn)}}
        print(json.dumps(r), flush=True)
        r["from_nn"] = searches(prob, nn)
        print(json.dumps(r["from_nn"]), flush=True)
        r["from_greedy"] = searches(prob, g)
        print(json.dumps(r["from_greedy"]), flush=True)
        res["runs"].append(r)
        prob.close()
    d = os.path.dirname(os.path.abspath(args.out))
    os.makedirs(d, exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
