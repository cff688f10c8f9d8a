"""bench.py --steps / --dump-outputs: the run applies exactly --warmup + --steps moves to the NN start
tour, and the tour and last move it dumps are the CPU oracle's after that many best-improvement moves
on the same seeded instance (TSPLIB-nint matrix)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WARMUP, STEPS = 3, 5
WORKLOADS = {"n1k": (1_000, 1_000), "n10k": (10_000, 10_000)}  # bench.WORKLOADS: (n, seed)


def run_bench(out_dir, workload, *extra):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--steps", str(STEPS),
           "--warmup", str(WARMUP), "--dump-outputs", str(out_dir), *extra]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def check_dump(out_dir, workload):
    n, seed = WORKLOADS[workload]
    x, y = O.gen_grid(n, seed)
    P = O.Problem(tri=O.matrix_packed_nint(x, y), n=n)
    moves = WARMUP + STEPS
    want_tour, st, want_moves = O.two_opt_best(P, O.nn_tour(P, 3), max_moves=moves, nthreads=os.cpu_count() or 1,
                                               log_cap=moves)
    assert st.moves == moves
    tour = np.load(os.path.join(out_dir, "tour.npy"))
    last = np.load(os.path.join(out_dir, "last_move.npy"))
    assert tour.dtype == np.float64 and last.dtype == np.float64
    assert (tour == want_tour).all()
    assert last.tolist() == [float(v) for v in want_moves[-1][:3]]


def test_reference_arm_takes_exactly_the_requested_steps(tmp_path):
    line = run_bench(tmp_path, "n1k", "--impl", "reference")
    assert line["steps"] == STEPS and line["warmup"] == WARMUP
    check_dump(tmp_path, "n1k")


@pytest.mark.gpu
def test_timed_path_outputs_equal_the_oracle(tmp_path):
    line = run_bench(tmp_path, "n10k", "--no-partitioned", "--cpu-budget", "0.1", "--e2e-steps", "1")
    assert line["steps"] == STEPS and line["moves_applied"] == STEPS
    check_dump(tmp_path, "n10k")
