#!/usr/bin/env python
"""bench.py -- headline benchmark: 2-opt moves evaluated per second at n = 10 000.

`python bench.py --gpus N --steps K --warmup W` prints ONE JSON line on rank 0; exactly K steps
are timed, after W (at least 3) untimed warm-up steps.  `--dump-outputs DIR` also writes what the
timed path returned after its last step (the tour and the move that step applied) as DIR/*.npy, so
that two builds can be compared output for output: the inputs depend on the arguments only.

Workload (BASELINE.json configs[2], the config the metric is quoted on): 10 000 cities on the
DIMACS-style 10^6 integer grid (splitmix64, seed 10000), TSPLIB nint distances, the int32
distance matrix resident in HBM (n x ld x 4 B = 400 MB, larger than L2), nearest-neighbour
start tour, best-improvement 2-opt ("Mode B").  A STEP is one full scan of the
P(n) = (n-3)(n-2)/2 = 49 975 003 candidate moves plus the application of the best one.
`value` = moves evaluated per second with everything resident in HBM.
`e2e`   = the same metric through the C ABI with HOST buffers: one e2e step is the call a
          `teeline solve nn,2opt` user makes -- tl_problem_create_euc2d (coordinates up),
          tl_local_search to the 2-opt local optimum (matrix build + every scan+apply), tour
          read-back -- so it is also BASELINE's second figure, wall time to the local optimum.
`--path recompute --dist f32` benches the coordinate-recompute path instead; both alternatives
are always reported under `other_paths`.
With N > 1 every rank runs an independent instance (seed + rank; no data-path collective) ->
weak scaling.

`--impl reference` times the CPU oracle port of the same step on the same configuration (the
reference itself is Rust and cannot be built in this image) with all host threads.
"""
from __future__ import annotations

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

METRIC = "2-opt moves evaluated/sec at n=10k (best-improvement scan+apply)"
UNIT = "moves/s"

WORKLOADS = {
    # name: (n, seed)
    "n10k": (10_000, 10_000),
    "n1k": (1_000, 1_000),
    "n100k": (100_000, 100_000),
}


# ---- synthetic instance (same stream as oracle/teeline_oracle.c: tlo_gen_uniform) ----------------

def splitmix64_stream(seed: int, count: int) -> np.ndarray:
    with np.errstate(over="ignore"):
        idx = np.arange(1, count + 1, dtype=np.uint64)
        z = np.uint64(seed) + idx * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def gen_uniform(n: int, seed: int):
    u = (splitmix64_stream(seed, 2 * n) >> np.uint64(40)).astype(np.float32)
    scale = np.float32(1000.0) / np.float32(16777216.0)
    xy = (u * scale).astype(np.float32)
    return np.ascontiguousarray(xy[0::2]), np.ascontiguousarray(xy[1::2])


def gen_grid(n: int, seed: int):
    """Integer grid floor(u * 10^6) from the same stream (NINT_I32 workloads; oracle: tlo_gen_grid)."""
    u = (splitmix64_stream(seed, 2 * n) >> np.uint64(40)).astype(np.float64)
    g = np.floor(u / 16777216.0 * 1.0e6).astype(np.float32)
    return np.ascontiguousarray(g[0::2]), np.ascontiguousarray(g[1::2])


def shuffle_tour(n: int, seed: int) -> np.ndarray:
    """Fisher-Yates driven by splitmix64(seed) (oracle: tlo_shuffle_tour)."""
    r = splitmix64_stream(seed, n - 1)
    t = np.arange(n, dtype=np.uint32)
    k = 0
    for i in range(n - 1, 0, -1):
        j = int(r[k] % np.uint64(i + 1))
        k += 1
        t[i], t[j] = t[j], t[i]
    return t


def shuffle_tours(n: int, seeds) -> np.ndarray:
    """shuffle_tour for many seeds at once (vectorised over the tours; same permutations)."""
    seeds = np.asarray(list(seeds), dtype=np.uint64)
    with np.errstate(over="ignore"):
        idx = np.arange(1, n, dtype=np.uint64)
        z = seeds[:, None] + idx[None, :] * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        r = z ^ (z >> np.uint64(31))
    t = np.tile(np.arange(n, dtype=np.uint32), (len(seeds), 1))
    rows = np.arange(len(seeds))
    for k, i in enumerate(range(n - 1, 0, -1)):
        j = (r[:, k] % np.uint64(i + 1)).astype(np.int64)
        ti = t[rows, i].copy()
        t[rows, i] = t[rows, j]
        t[rows, j] = ti
    return t


def pairs_per_scan(n: int) -> int:
    return (n - 3) * (n - 2) // 2


def instance(n: int, seed: int, dist: str):
    return gen_grid(n, seed) if dist == "nint" else gen_uniform(n, seed)


def describe(workload: str, n: int, seed: int, path: str, dist: str) -> str:
    coords = "10^6 integer grid, TSPLIB nint int32 distances" if dist == "nint" else \
        "uniform [0,1000)^2 on a 2^-24 grid, f32 distances"
    src = f"{'int32' if dist == 'nint' else 'f32'} distance matrix in HBM" if path == "matrix" else \
        "distances recomputed from coordinates"
    return (f"{workload}: n={n} EUC_2D ({coords}; splitmix64 seed {seed}), {src}, NN start tour, "
            f"best-improvement 2-opt, one step = full scan of {pairs_per_scan(n)} moves + apply")


def bench_config(args, world: int) -> dict:
    """`config` of the JSON line: a function of the command line only, so that both arms (ours and
    --impl reference) print the SAME dictionary for the same invocation."""
    n, seed = WORKLOADS[args.workload]
    ld = (n + 31) // 32 * 32
    return {
        "workload": describe(args.workload, n, seed, args.path, args.dist),
        "path": args.path, "dist": args.dist,
        "l2": (f"inputs larger than L2 ({4 * n * ld / 1e6:.0f} MB matrix, {4 * pairs_per_scan(n) / 1e6:.0f} MB read per "
               "scan, L2 126 MB); no flush") if args.path == "matrix" else
              "compute-bound path: 16 B per city of tour-ordered points, L2 state irrelevant",
        "timed_region": f"{args.steps} steps after {args.warmup} untimed warm-up steps; ms_per_step is the timed "
                        f"time / {args.steps}",
        "parallelism": f"independent instances x{world} (seed + rank), no data-path collective; the partitioned "
                       "cases (configs 4 and 5) are under `partitioned`",
    }


# an NN tour converges after ~1500 (10k) / ~170 (1k) moves: start a fresh session before that
SESSION_CAPS = {"n10k": 1400, "n1k": 150, "n100k": 4000}
SCAN_REPS = 200  # scan-kernel launches averaged for the roofline, whatever --steps is


# ---- clocks sampling ------------------------------------------------------------------------------

class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML every ~2 ms from a
    thread (the timed region is tens of ms), nvidia-smi -lms as the fallback."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.rows, self.proc = device, [], None
        self.sm, self.reasons, self.mx, self.th, self.stop_flag = [], set(), None, None, False
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[device]) if vis and vis.split(",")[device].isdigit() else device
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _poll(self):
        nv = self.nvml
        names = {nv.nvmlClocksEventReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksEventReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksEventReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksEventReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nvml is not None:
            self.stop_flag = False
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._pump, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def pause(self):
        """Stop sampling between timed chunks (NVML mode only)."""
        if self.nvml is not None and self.th is not None:
            self.stop_flag = True
            self.th.join()
            self.th = None

    def stop(self):
        if self.nvml is not None:
            self.pause()
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.mx,
                    "samples": len(self.sm), "reasons": sorted(self.reasons), "source": "nvml, 2 ms period, "
                    "sampled only while the timed steps were running"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [c.strip() for c in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi -lms 20"}


# ---- CPU baseline (the oracle; never on the product path) ----------------------------------------------

def oracle_problem(n: int, seed: int, path: str, dist: str):
    """The CPU twin of the benched configuration: packed int32/f32 triangle for the matrix-backed
    paths (what DistanceMatrix holds, distance_matrix.rs:122-153), coordinates for recompute."""
    import oracle as O
    x, y = instance(n, seed, dist)
    if dist == "nint":
        P = O.Problem(tri=O.matrix_packed_nint(x, y), n=n)
    elif path == "matrix":
        P = O.Problem(tri=O.matrix_packed_f32(x, y), n=n)
    else:
        P = O.Problem(x, y)
    return O, P


def cpu_scan_rate(n: int, seed: int, path: str, dist: str, threads: int, budget_s: float):
    """Times full Mode B scans of the oracle on the host cores; returns (moves/s, scans, seconds)."""
    O, P = oracle_problem(n, seed, path, dist)
    tour = O.nn_tour(P, 3)
    O.two_opt_best_scan(P, tour, nthreads=threads)  # warm
    t0 = time.perf_counter()
    scans = 0
    while True:
        O.two_opt_best_scan(P, tour, nthreads=threads)
        scans += 1
        if time.perf_counter() - t0 >= budget_s:
            break
    dt = time.perf_counter() - t0
    return scans * pairs_per_scan(n) / dt, scans, dt


def dump_outputs(out_dir: str, tour, move) -> None:
    """What a caller of the timed path receives after its last step, as float64 .npy files: the tour
    (city indices in tour order) and the move that step applied, (delta, i, j); empty when the tour
    had no improving move left."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "tour.npy"), np.asarray(tour, dtype=np.float64))
    np.save(os.path.join(out_dir, "last_move.npy"), np.array(move[:3] if move else [], dtype=np.float64))


def run_reference(args, rank: int, world: int):
    """--impl reference: the CPU port of the same step (scan + apply), all host threads."""
    if rank != 0:
        return
    n, seed = WORKLOADS[args.workload]
    threads = os.cpu_count() or 1
    O, P = oracle_problem(n, seed, args.path, args.dist)
    tour = O.nn_tour(P, 3).copy()
    t_all = 0.0
    for k in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        mv = O.two_opt_best_scan(P, tour, nthreads=threads)
        if mv is not None:
            tour = O.swap_2opt(tour, mv[1] + 1, mv[2])
        if k >= args.warmup:
            t_all += time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, tour, mv)
    value = args.steps * pairs_per_scan(n) / t_all
    sample = f"{args.steps} full scan+apply steps of the n={n} workload"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_all / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int32" if args.dist == "nint" else "f32",
        "data": "synthetic",
        "config": bench_config(args, world),
        "note": "CPU oracle port of the reference semantics over the packed lower-triangle matrix, "
                "row-parallel over all host threads (the Rust reference is single-threaded and cannot "
                "be built here: no cargo)",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---- product arm -------------------------------------------------------------------------------------

def run_partitioned(args, T, ctx, torch, dist, rank: int, world: int, hbm_peak: float) -> dict:
    """The two cases of BASELINE.json that split ONE job over the GPUs (SURVEY.md section 8(e)).

    config 4: n = 100 000, coordinate recompute, the (i,j) triangle sharded over the ranks; every step
              the per-rank minima are exchanged inside the scan kernel over NVLink peer memory
              (csrc/shard_exchange.cuh) and every rank applies the same move to its replica.
    config 5: 1024 start tours on the 1k instance, tours sharded by index, no data-path collective.
    Every figure is measured in this run: the unsharded single-GPU baseline first (same process, same
    instance), then the sharded run; times are CUDA-event / wall times, max over ranks."""
    from teeline_b200 import multi

    def rmax(v):
        if dist is None:
            return float(v)
        t = torch.tensor([float(v)], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def rmin_flag(ok):
        if dist is None:
            return bool(ok)
        t = torch.tensor([1 if ok else 0], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    def sync():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    out = {"n_gpus": world}
    if world > 1:
        multi.attach_nccl(ctx, dist)

    # ---- config 4 ------------------------------------------------------------------------------------
    n, seed = WORKLOADS["n100k"]
    P4 = pairs_per_scan(n)
    x, y = gen_uniform(n, seed)
    prob = T.Problem.euc2d(ctx, x, y)
    start = prob.nn_tour(3)
    W4, K4 = 5, max(50, min(args.partitioned_steps, 400))

    def timed_steps(sess):
        sess.enqueue(W4)
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        sess.enqueue(K4)
        e1.record()
        sync()
        return rmax(e0.elapsed_time(e1)) / K4

    base = prob.session(T.ALGO_TWO_OPT_BEST, start, T.PATH_RECOMPUTE)
    base_step = timed_steps(base)
    base_log, base_tour = base.log(W4 + K4), base.tour()
    base_scan = rmax(base.time_scans(20))
    base.close()
    ffma, _ = ctx.microbench_fp32()
    c4 = {"workload": f"n={n} uniform f32 (seed {seed}), coordinate recompute, NN start, Mode B, {K4} timed steps "
                      f"after {W4} warm-up", "pairs_per_scan": P4,
          "single_gpu": {"step_ms": base_step, "scan_ms": base_scan, "moves_per_s": P4 / (base_step * 1e-3),
                         "roofline_frac_fp32_issue": 15.0 * P4 / (base_scan * 1e-3) / ffma}}
    if world > 1:
        sh = prob.session(T.ALGO_TWO_OPT_BEST, start, T.PATH_RECOMPUTE)
        sh.set_shard(rank, world)
        first = sh.scan()  # (all-gather + host reduction path) the global best move from the start tour
        step = timed_steps(sh)
        log, tour = sh.log(W4 + K4), sh.tour()
        scan = rmax(sh.time_scans(20))
        sh.close()
        same = log == base_log and bool((tour == base_tour).all()) and first is not None and \
            first[1:3] == base_log[0][1:3]
        c4["sharded"] = {
            "step_ms": step, "scan_ms_slowest_rank": scan, "exchange_plus_apply_ms": step - scan,
            "moves_per_s": P4 / (step * 1e-3), "speedup_vs_single_gpu_step": base_step / step,
            "scan_speedup": base_scan / scan,
            "roofline_frac_fp32_issue_aggregate": 15.0 * P4 / (scan * 1e-3) / (ffma * world),
            "identical_to_unsharded": rmin_flag(same),
            "transport": os.environ.get("TL_SHARD_TRANSPORT", "peer mailboxes over NVLink inside the scan kernel "
                                                                 "(ncclAllGather only if peers cannot be mapped)")}
    if rank == 0 and args.partitioned_oracle_check:
        # one oracle-checked scan (the checker, outside every timed region): the first logged move of
        # the (sharded) search must be the CPU oracle's best move from the same start tour
        import oracle as O
        t0 = time.perf_counter()
        want = O.two_opt_best_scan(O.Problem(x, y), start, nthreads=os.cpu_count() or 1)
        got = base_log[0]
        c4["oracle_checked_first_move"] = {
            "ok": bool(want is not None and (want[1], want[2]) == (got[1], got[2]) and
                       np.float32(want[0]) == np.float32(got[0])),
            "oracle_scan_s": time.perf_counter() - t0, "move": [float(got[0]), int(got[1]), int(got[2])]}
    prob.close()
    out["config4_100k_sharded_triangle"] = c4

    # ---- config 5 ------------------------------------------------------------------------------------
    n, seed = WORKLOADS["n1k"]
    B = 1024
    x, y = gen_uniform(n, seed)
    prob = T.Problem.euc2d(ctx, x, y)
    tours = np.concatenate([prob.nn_tour(3)[None, :], shuffle_tours(n, range(1, B))])
    prob.two_opt_batch(tours[:8], max_moves=2)  # warm
    sync()
    t0 = time.perf_counter()
    got, st, lengths = prob.two_opt_batch(tours)
    torch.cuda.synchronize()
    single_wall = rmax(time.perf_counter() - t0)
    evals = int(st.evals)
    c5 = {"workload": f"{B} start tours (NN + {B - 1} splitmix64 shuffles) on the n={n} instance, every tour to its "
                      "2-opt local optimum, host buffers in and out",
          "evals": evals, "moves_applied": int(st.moves),
          "single_gpu": {"wall_s": single_wall, "device_ms": float(st.device_ms), "moves_per_s": evals / single_wall,
                         "best_length": float(lengths.min())}}
    if world > 1:
        # untimed warm-up of the whole sharded call on a tiny batch: the first all_gather / broadcast of a
        # process group connects NCCL's channels for those collectives (milliseconds, once per job)
        multi.sharded_population(tours[:2 * world], lambda t: prob.two_opt_batch(t, max_moves=2)[::2], dist)
        dev_ms = []

        def solve_shard(t):
            got_t, st_t, len_t = prob.two_opt_batch(t)
            dev_ms.append(float(st_t.device_ms))
            return got_t, len_t

        sync()
        t0 = time.perf_counter()
        (lo, hi), mine, all_len, best, best_tour = multi.sharded_population(tours, solve_shard, dist)
        torch.cuda.synchronize()
        wall = rmax(time.perf_counter() - t0)
        same = bool((np.float32(all_len) == lengths).all()) and best == int(np.argmin(lengths)) and \
            bool((best_tour == got[best]).all()) and bool((mine == got[lo:hi]).all())
        c5["sharded"] = {"wall_s": wall, "device_ms_slowest_rank": rmax(dev_ms[0] if dev_ms else 0.0),
                         "moves_per_s": evals / wall, "speedup_vs_single_gpu": single_wall / wall,
                         "identical_lengths_and_best_tour": rmin_flag(same), "tours_per_gpu": B // world}
    prob.close()
    out["config5_1024_tours"] = c5
    return out


def run_ours(args, rank: int, world: int, local_rank: int):
    import torch
    import teeline_b200 as T

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    n, seed0 = WORKLOADS[args.workload]
    seed = seed0 + rank  # one independent instance per rank
    P = pairs_per_scan(n)
    kinds = {"nint": T.DIST_NINT_I32, "f32": T.DIST_F32_EXACT}
    paths = {"recompute": T.PATH_RECOMPUTE, "matrix": T.PATH_MATRIX, "auto": T.PATH_AUTO}
    x, y = instance(n, seed, args.dist)
    stream = torch.cuda.current_stream().cuda_stream
    ctx = T.Context(local_rank, stream=stream)
    prob = T.Problem.euc2d(ctx, x, y, kinds[args.dist])
    start = prob.nn_tour(3)  # the reference's `nn,2opt` pipeline
    path = paths[args.path]

    # --- device-resident timing: exactly K = --steps timed steps, each stretch of them after W untimed
    #     warm-up steps, bracketed by barrier + synchronize on both sides and timed with CUDA events on
    #     the library's stream.  A tour runs out of improving moves after about SESSION_CAPS steps, so
    #     a K larger than that is timed in pieces, each on a fresh session from the same start tour.
    #     The reported step time is the timed device time (max over ranks) / K.
    cap = SESSION_CAPS[args.workload]
    sampler = ClockSampler(local_rank)
    ms, launches, left, sess = 0.0, 0, args.steps, None
    while left > 0:
        k = min(left, max(1, cap - args.warmup))
        if sess is not None:
            sess.close()
        sess = prob.session(T.ALGO_TWO_OPT_BEST, start, path)
        sess.enqueue(args.warmup)
        barrier()
        if rank == 0:
            sampler.start()
        l0 = ctx.launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        sess.enqueue(k)
        e1.record()
        barrier()
        if rank == 0:
            sampler.pause()
        ms += e0.elapsed_time(e1)
        launches += ctx.launches - l0
        left -= k
    real = int(sess.stats().moves)
    if real < args.warmup + k:
        raise SystemExit(f"bench invalid: the tour converged after {real} moves, fewer than the {args.warmup + k} "
                         f"steps enqueued on it; lower SESSION_CAPS[{args.workload!r}]")
    if dist is not None:
        t_ms = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        ms = float(t_ms.item())
    clocks = sampler.stop() if rank == 0 else None
    value = world * args.steps * P / (ms * 1e-3)
    moves_applied = args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sess.tour(), sess.log()[-1])

    # --- dominant kernel: average launch duration of the scan kernel (CUDA events, same stream)
    scan_ms = sess.time_scans(SCAN_REPS)
    stats_path = int(sess.stats().path_used)
    sess.close()

    # --- the alternatives on the same workload size, always reported
    def probe(label, p_path, p_dist):
        gx, gy = instance(n, seed, p_dist)
        p2 = T.Problem.euc2d(ctx, gx, gy, kinds[p_dist])
        s2 = p2.session(T.ALGO_TWO_OPT_BEST, p2.nn_tour(3), paths[p_path])
        s2.enqueue(args.warmup)
        torch.cuda.synchronize()
        k = 200
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        s2.enqueue(k)
        a1.record()
        torch.cuda.synchronize()
        step_ms2 = a0.elapsed_time(a1) / k
        scan_ms2 = s2.time_scans(SCAN_REPS)
        s2.close()
        p2.close()
        kern = "two_opt_scan_matrix_kernel" if p_path == "matrix" else "two_opt_scan_recompute_kernel"
        return {"path": p_path, "dist": p_dist, "ms_per_step": step_ms2, "value": P / (step_ms2 * 1e-3),
                "kernel_ms": scan_ms2, "kernel": kern, "scan_moves_per_s": P / (scan_ms2 * 1e-3)}

    other_paths = {}
    if rank == 0 and args.workload != "n100k":
        for label, p_path, p_dist in (("matrix_nint_i32", "matrix", "nint"), ("matrix_f32", "matrix", "f32"),
                                      ("recompute_f32", "recompute", "f32")):
            if (p_path, p_dist) != (args.path, args.dist):
                other_paths[label] = probe(label, p_path, p_dist)

    # --- the metric's second half, "wall time to 2-opt local optimum", per mode (SURVEY.md section 8(d)):
    #     host buffers in, NN start tour, the whole search through the C ABI, tour back; median of 3 calls.
    #     Mode R is the reference's own first-improvement loop (the local optimum the Rust two_opt::solve
    #     reaches, bit for bit); Mode B is the best-improvement scan the headline counts.
    def to_optimum(algo, p_dist, p_path):
        gx, gy = instance(n, seed, p_dist)
        walls, st3 = [], None
        for _ in range(4):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            p3 = T.Problem.euc2d(ctx, gx, gy, kinds[p_dist])
            t3, st3, _ = p3.local_search(algo, p3.nn_tour(3), path=paths[p_path])
            p3.close()
            walls.append(time.perf_counter() - t0)
        return {"dist": p_dist, "path": "matrix" if st3.path_used == T.PATH_MATRIX else "recompute",
                "wall_ms": 1e3 * float(np.median(walls[1:])), "wall_ms_all": [1e3 * w for w in walls],
                "device_ms": float(st3.device_ms),
                "moves": int(st3.moves), "passes_or_scans": int(st3.passes), "evals": int(st3.evals),
                "launches": int(st3.launches)}

    def or_opt_after_two_opt(p_dist, p_path):
        """BASELINE config 3's second stage: Or-opt (the reference's or_opt::solve, bit-exact) from the
        Mode B local optimum, to its own local optimum."""
        gx, gy = instance(n, seed, p_dist)
        p3 = T.Problem.euc2d(ctx, gx, gy, kinds[p_dist])
        t2, _, _ = p3.local_search(T.ALGO_TWO_OPT_BEST, p3.nn_tour(3), path=paths[p_path])
        walls, st3 = [], None
        for _ in range(4):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            _t, st3, _ = p3.local_search(T.ALGO_OR_OPT, t2, path=paths[p_path])
            walls.append(time.perf_counter() - t0)
        p3.close()
        return {"dist": p_dist, "path": "matrix" if st3.path_used == T.PATH_MATRIX else "recompute",
                "wall_ms": 1e3 * float(np.median(walls[1:])), "device_ms": float(st3.device_ms), "moves": int(st3.moves),
                "scans": int(st3.passes), "evals": int(st3.evals),
                "candidates_per_s": int(st3.evals) / (1e-3 * float(st3.device_ms))}

    wall_to_optimum = None
    if rank == 0 and args.workload != "n100k":
        wall_to_optimum = {
            "note": f"n={n}: tl_problem_create_euc2d + tl_nn_tour + tl_local_search to the local optimum + tour read-back, "
                    "wall clock, median of 3 calls after one warm-up",
            "mode_r_reference_exact_f32": to_optimum(T.ALGO_TWO_OPT_REF, "f32", "auto"),
            "mode_r_reference_exact_nint": to_optimum(T.ALGO_TWO_OPT_REF, "nint", "auto"),
            "mode_b_best_improvement_nint_matrix": to_optimum(T.ALGO_TWO_OPT_BEST, "nint", "matrix"),
            "mode_b_best_improvement_f32_recompute": to_optimum(T.ALGO_TWO_OPT_BEST, "f32", "recompute"),
            # the same moves and the same tour as Mode B, from cached row minima: a step re-evaluates only the
            # pairs the previous move changed (`evals` = pair deltas actually computed)
            "mode_b_cached_nint_matrix": to_optimum(T.ALGO_TWO_OPT_BEST_CACHED, "nint", "matrix"),
            "mode_b_cached_f32_recompute": to_optimum(T.ALGO_TWO_OPT_BEST_CACHED, "f32", "recompute"),
            "or_opt_from_the_mode_b_optimum_nint_matrix": or_opt_after_two_opt("nint", "matrix"),
        }

    # --- the partitioned cases (configs 4 and 5): sharded across the ranks, measured against this
    #     run's own single-GPU baseline
    partitioned = None
    if not args.no_partitioned:
        peaks0 = {}
        try:
            peaks0 = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        partitioned = run_partitioned(args, T, ctx, torch, dist, rank, world, float(peaks0.get("hbm_gbs", 6650.0)))

    # --- end to end through the C ABI with host buffers (pinned), copies inside the timed region:
    #     coordinates up, the whole local search to the 2-opt optimum, tour back
    e2e_steps = max(1, args.e2e_steps)
    hx = torch.from_numpy(x).pin_memory().numpy()
    hy = torch.from_numpy(y).pin_memory().numpy()

    def e2e_step():
        """What `teeline solve 2opt` does with a problem file already parsed (2opt auto-expands to the
        nn,2opt pipeline, src/tsp/mod.rs:129-139): coordinates up, NN start tour (device, read back as the
        stage's Solution), 2-opt to the local optimum from that seed, tour back."""
        ta = time.perf_counter()
        p2 = T.Problem.euc2d(ctx, hx, hy, kinds[args.dist])
        tb = time.perf_counter()
        seed_tour = p2.nn_tour(3)
        tn = time.perf_counter()
        t2, st2, _ = p2.local_search(T.ALGO_TWO_OPT_BEST, seed_tour, path=path, max_moves=args.e2e_moves)
        tc = time.perf_counter()
        p2.close()
        if os.environ.get("TL_DEBUG_TIMING"):
            print(f"[bench] e2e call: create {1e3 * (tb - ta):.2f} ms, nn_tour {1e3 * (tn - tb):.2f} ms, "
                  f"local_search {1e3 * (tc - tn):.2f} ms, close {1e3 * (time.perf_counter() - tc):.2f} ms",
                  file=sys.stderr)
        return int(st2.evals), int(st2.moves), t2, tn - tb

    e2e_step()
    barrier()
    evals = e2e_applied = 0
    nn_s = 0.0
    call_s = []
    t_all0 = time.perf_counter()
    for _ in range(e2e_steps):
        t0 = time.perf_counter()
        ev, mv, _t, nn_dt = e2e_step()
        torch.cuda.synchronize()
        call_s.append(time.perf_counter() - t0)
        evals += ev
        e2e_applied += mv
        nn_s += nn_dt
    dt_total = time.perf_counter() - t_all0
    # one e2e step = one call; the reported rate is evaluations per call / the MEDIAN call time, max
    # over ranks (every call does identical work; a single slow call -- first touch of a pool block, a
    # host hiccup -- would otherwise decide the headline).  The total over all calls is kept beside it.
    dt = float(np.median(call_s))
    evals_per_call = evals / e2e_steps
    evals_all_ranks = evals_per_call
    if dist is not None:
        # every rank solves its own instance (seed + rank), which takes its own number of moves: the
        # job's rate is the evaluations of ALL ranks over the slowest rank's time
        tdt = torch.tensor([dt, dt_total], device="cuda", dtype=torch.float64)
        dist.all_reduce(tdt, op=dist.ReduceOp.MAX)
        dt, dt_total = float(tdt[0].item()), float(tdt[1].item())
        tev = torch.tensor([evals_per_call], device="cuda", dtype=torch.float64)
        dist.all_reduce(tev, op=dist.ReduceOp.SUM)
        evals_all_ranks = float(tev.item())
    e2e_value = evals_all_ranks / dt
    h2d = 2 * 4 * n + 4 * n  # x, y; the NN tour goes back up as the 2-opt stage's seed
    d2h = 4 * n + 4 * n + 64  # NN tour, final tour, stats

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # --- roofline for the dominant kernel
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    traffic = {}
    try:  # dram__bytes_read.sum + dram__bytes_write.sum per launch, from the committed `ncu --set full` captures
        traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except Exception:
        pass

    def hbm_roofline(kernel_ms, key):
        achieved = 4.0 * P / (kernel_ms * 1e-3) / 1e9  # 4 algorithmic bytes per move (DESIGN.md section 4)
        t = traffic.get(key, {}) if args.workload == "n10k" else {}
        return {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                "traffic": t.get("bytes_per_launch"), "traffic_source": t.get("source"), "peak_source": peak_src,
                "kernel": "two_opt_scan_matrix_kernel", "kernel_ms": kernel_ms, "algorithmic_bytes_per_move": 4,
                "algorithmic_bytes_per_launch": 4 * P}

    def fp32_roofline(kernel_ms):
        ffma, mufu = ctx.microbench_fp32()
        flops = 15.0 * P / (kernel_ms * 1e-3)  # 13 FP32 ops + 2 sqrt per move (SURVEY.md section 8(d))
        t = traffic.get("recompute", {}) if args.workload == "n10k" else {}
        return {"bound": "fp32_issue", "achieved": flops / 1e12, "peak": ffma / 1e12, "unit": "TFLOP/s",
                "frac": flops / ffma,
                "peak_source": "measured here: dependent-free FFMA stream, lane-instructions/s "
                               "(tl_microbench_fp32); MEASURED_PEAKS.json has no FP32 figure",
                "kernel": "two_opt_scan_recompute_kernel", "kernel_ms": kernel_ms,
                "algorithmic_flop_per_move": 15, "mufu_peak_per_s": mufu,
                "traffic": t.get("bytes_per_launch"), "traffic_source": t.get("source"),
                "note": "coordinate-recompute path: ~0 bytes/move, bound by FP32 issue, not HBM or tensor"}

    for label, o in other_paths.items():
        o["roofline"] = hbm_roofline(o["kernel_ms"], label) if o["path"] == "matrix" else fp32_roofline(o["kernel_ms"])
    if stats_path == T.PATH_MATRIX:
        roofline = hbm_roofline(scan_ms, "matrix_nint_i32" if args.dist == "nint" else "matrix_f32")
    else:
        roofline = fp32_roofline(scan_ms)
    roofline["kernel_share_of_step"] = scan_ms / (ms / args.steps)
    roofline["kernel_reps_timed"] = SCAN_REPS

    # --- CPU baseline: the oracle port on the host cores (bounded sample)
    threads = os.cpu_count() or 1
    cpu_v, cpu_scans, cpu_dt = cpu_scan_rate(n, seed, args.path, args.dist, threads, args.cpu_budget)
    cpu_v1, cpu_scans1, cpu_dt1 = cpu_scan_rate(n, seed, args.path, args.dist, 1, min(args.cpu_budget, 4.0))
    cpu_baseline = {
        "value": cpu_v, "unit": UNIT, "cores": threads, "kind": "port",
        "sample": f"{cpu_scans} full Mode B scans of the same n={n} tour in {cpu_dt:.1f} s, {threads} threads "
                  f"(row-parallel oracle scan over the same {'packed matrix' if args.path == 'matrix' or args.dist == 'nint' else 'coordinates'})",
        "single_thread_value": cpu_v1,
        "note": "C oracle with flat arrays; the Rust reference is single-threaded and pays 2 SipHash "
                "lookups per distance, so this over-states the reference's speed",
    }

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "timed_ms_total": ms,
        "vs_baseline": None, "dtype": "int32" if args.dist == "nint" else "f32", "data": "synthetic",
        "config": bench_config(args, world),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "step": "tl_problem_create_euc2d + tl_nn_tour + tl_local_search(" +
                        ("to the 2-opt local optimum" if args.e2e_moves < 0 else f"max_moves={args.e2e_moves}") +
                        f") + tour read-back, pinned host buffers; median of {e2e_steps} calls",
                "seconds": dt_total, "wall_ms_per_call": 1e3 * dt, "wall_ms_per_call_all": [1e3 * c for c in call_s],
                "value_from_total_time": evals_all_ranks * e2e_steps / dt_total,
                "moves_applied_per_call": e2e_applied / e2e_steps,
                "nn_tour_ms_per_call": 1e3 * nn_s / e2e_steps,
                "metric_note": "moves evaluated by the 2-opt stage / wall time of the WHOLE call (NN start tour "
                               "construction and all copies included)"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "cpu_baseline": cpu_baseline,
        "other_paths": other_paths,
        "wall_to_local_optimum": wall_to_optimum,
        "moves_applied": moves_applied,
        "partitioned": partitioned,
    }
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="n10k", choices=sorted(WORKLOADS))
    ap.add_argument("--path", default="matrix", choices=["recompute", "matrix"])
    ap.add_argument("--dist", default="nint", choices=["nint", "f32"])
    ap.add_argument("--no-partitioned", action="store_true", help="skip the configs 4/5 block")
    ap.add_argument("--partitioned-steps", type=int, default=60, help="timed steps of the 100k sharded case")
    ap.add_argument("--partitioned-oracle-check", type=int, default=1,
                    help="rank 0 checks the first 100k move against one CPU oracle scan (5-15 s)")
    ap.add_argument("--e2e-moves", type=int, default=-1, help="-1: to the local optimum")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-budget", type=float, default=10.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the timed path's outputs after its last step "
                    "as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.path == "recompute" and args.dist == "nint":
        args.dist = "f32"  # the recompute kernels evaluate the f32 metric
    if args.workload == "n100k":
        args.path, args.dist = "recompute", "f32"
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
