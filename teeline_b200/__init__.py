"""teeline_b200 -- B200-native local-search hot path of teeline behind a C ABI.

The product is `libteeline_cuda.so` (hand-written sm_100a CUDA, built by
`teeline_b200/build.py`) and the C++ host mirror under `teeline_b200/host/`.  This
Python package only wraps the C ABI with ctypes so that tests and bench.py can call
it with numpy arrays; it never computes anything itself and never falls back to a
CPU path.
"""
from __future__ import annotations

import ctypes as C
import weakref

import numpy as np

from . import _capi as capi
from ._capi import (ALGO_OR_OPT, ALGO_OR_OPT_NEIGHBOR, ALGO_OR_OPT_NEIGHBOR_MULTI, ALGO_THREE_OPT, ALGO_TWO_OPT_BEST, ALGO_TWO_OPT_BEST_CACHED, ALGO_TWO_OPT_BEST_CYCLIC,
                    ALGO_THREE_OPT_NEIGHBOR, ALGO_TWO_OPT_NEIGHBOR, ALGO_TWO_OPT_NEIGHBOR_MULTI, ALGO_TWO_OPT_REF,
                    CANDIDATES_DEFAULT, MULTI_BLOCK, OR_MULTI_BLOCK,
                    DIST_F32_EXACT, DIST_NINT_I32, LEN_EXACT, LEN_FAST, PATH_AUTO, PATH_MATRIX,
                    PATH_RECOMPUTE, Move, Stats, TeelineError)

__all__ = ["Context", "Problem", "Session", "TeelineError", "capi"]


def _u32(a):
    return np.ascontiguousarray(a, dtype=np.uint32)


class Context:
    """tl_ctx: one device + one stream."""

    def __init__(self, device: int = 0, stream: int | None = None):
        self._lib = capi.load()
        h = C.c_void_p()
        if stream is None:
            capi.check(self._lib.tl_ctx_create(device, C.byref(h)))
        else:
            capi.check(self._lib.tl_ctx_create_on_stream(device, C.c_void_p(stream), C.byref(h)))
        self.h = h
        self.device = device
        # handles created from this context; close() destroys them first (the C handles point back
        # at the tl_ctx, so a Problem collected after its Context would touch freed memory)
        self._children = weakref.WeakSet()

    def sync(self):
        capi.check(self._lib.tl_ctx_sync(self.h))

    @property
    def launches(self) -> int:
        return int(self._lib.tl_ctx_launch_count(self.h))

    def attach_nccl(self, unique_id: bytes, rank: int, world: int):
        buf = (C.c_uint8 * capi.NCCL_ID_BYTES).from_buffer_copy(unique_id)
        capi.check(self._lib.tl_ctx_attach_nccl(self.h, buf, rank, world))

    @staticmethod
    def nccl_unique_id() -> bytes:
        buf = (C.c_uint8 * capi.NCCL_ID_BYTES)()
        capi.check(capi.load().tl_nccl_unique_id(buf))
        return bytes(buf)

    def selftest_sqrt(self, lo_bits: int, hi_bits: int) -> int:
        out = C.c_uint64()
        capi.check(self._lib.tl_selftest_sqrt(self.h, lo_bits, hi_bits, C.byref(out)))
        return int(out.value)

    def microbench_fp32(self):
        a, b = C.c_double(), C.c_double()
        capi.check(self._lib.tl_microbench_fp32(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def close(self):
        if getattr(self, "h", None):
            for child in list(self._children):
                child.close()
            self._lib.tl_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Problem:
    """tl_problem: coordinates (EUC_2D) or an explicit packed triangle, resident on the device."""

    def __init__(self, ctx: Context, h, n: int, kind: str):
        self.ctx, self.h, self.n, self.kind = ctx, h, n, kind
        self._lib = ctx._lib
        self._children = weakref.WeakSet()  # sessions: destroyed before the problem they point at
        ctx._children.add(self)

    @classmethod
    def euc2d(cls, ctx: Context, x, y, dist_kind: int = DIST_F32_EXACT) -> "Problem":
        x = np.ascontiguousarray(x, dtype=np.float32)
        y = np.ascontiguousarray(y, dtype=np.float32)
        if x.shape != y.shape or x.ndim != 1:
            raise ValueError("x and y must be 1-D arrays of equal length")
        h = C.c_void_p()
        capi.check(ctx._lib.tl_problem_create_euc2d(ctx.h, len(x), capi.ptr(x), capi.ptr(y), dist_kind,
                                                    C.byref(h)))
        return cls(ctx, h, len(x), "nint" if dist_kind == DIST_NINT_I32 else "f32")

    @classmethod
    def explicit(cls, ctx: Context, packed_tri, n: int) -> "Problem":
        t = np.ascontiguousarray(packed_tri, dtype=np.float32)
        if t.size != n * (n - 1) // 2:
            raise ValueError("packed triangle must hold n(n-1)/2 values")
        h = C.c_void_p()
        capi.check(ctx._lib.tl_problem_create_explicit(ctx.h, n, capi.ptr(t), C.byref(h)))
        return cls(ctx, h, n, "explicit")

    def matrix_packed(self) -> np.ndarray:
        cnt = self.n * (self.n - 1) // 2
        if self.kind == "nint":
            out = np.empty(cnt, dtype=np.int32)
            capi.check(self._lib.tl_dist_matrix_packed_i32(self.h, capi.ptr(out)))
        else:
            out = np.empty(cnt, dtype=np.float32)
            capi.check(self._lib.tl_dist_matrix_packed(self.h, capi.ptr(out)))
        return out

    def knn(self, k: int) -> np.ndarray:
        out = np.empty((self.n, k), dtype=np.uint32)
        capi.check(self._lib.tl_knn(self.h, k, capi.ptr(out)))
        return out

    def set_candidates(self, k: int = CANDIDATES_DEFAULT):
        """tl_problem_set_candidates: the k-nearest candidate lists that later ALGO_TWO_OPT_NEIGHBOR[_MULTI],
        ALGO_OR_OPT_NEIGHBOR[_MULTI] and ALGO_THREE_OPT_NEIGHBOR sessions of this problem search (1 <= k <= 32)."""
        capi.check(self._lib.tl_problem_set_candidates(self.h, k))

    def nn_tour(self, k: int = 3) -> np.ndarray:
        out = np.empty(self.n, dtype=np.uint32)
        capi.check(self._lib.tl_nn_tour(self.h, k, capi.ptr(out)))
        return out

    def greedy_tour(self):
        """tl_greedy_tour: the greedy-edge tour, built on the device from the candidate lists (default lists
        are built and kept when there are none).  Returns (tour, Stats)."""
        out = np.empty(self.n, dtype=np.uint32)
        st = Stats()
        capi.check(self._lib.tl_greedy_tour(self.h, capi.ptr(out), C.byref(st)))
        return out, st

    def tour_lengths(self, tours, mode: int = LEN_EXACT) -> np.ndarray:
        t = _u32(tours)
        if t.ndim == 1:
            t = t[None, :]
        if t.shape[1] != self.n:
            raise ValueError("tours must be batch x n")
        if self.kind == "nint":
            out = np.empty(t.shape[0], dtype=np.int64)
            capi.check(self._lib.tl_tour_lengths_i64(self.h, capi.ptr(t), t.shape[0], capi.ptr(out)))
        else:
            out = np.empty(t.shape[0], dtype=np.float32)
            capi.check(self._lib.tl_tour_lengths(self.h, capi.ptr(t), t.shape[0], mode, capi.ptr(out)))
        return out

    def local_search(self, algo: int, tour, path: int = PATH_AUTO, max_moves: int = -1,
                     log_cap: int = 0):
        """tl_local_search: returns (tour, Stats, [moves])."""
        t = _u32(tour).copy()
        if t.shape != (self.n,):
            raise ValueError("tour must have n entries")
        st = Stats()
        log = (Move * max(log_cap, 1))()
        capi.check(self._lib.tl_local_search(self.h, algo, path, capi.ptr(t), max_moves, C.byref(st),
                                             log if log_cap else None, log_cap))
        three = algo in (ALGO_THREE_OPT, ALGO_THREE_OPT_NEIGHBOR)
        moves = [log[k].astuple3() if three else log[k].astuple() for k in range(min(int(st.moves), log_cap))]
        return t, st, moves

    def two_opt_batch(self, tours, algo: int = ALGO_TWO_OPT_BEST, max_moves: int = -1):
        t = _u32(tours).copy()
        if t.ndim != 2 or t.shape[1] != self.n:
            raise ValueError("tours must be batch x n")
        st = Stats()
        lengths = np.empty(t.shape[0], dtype=np.float32)
        capi.check(self._lib.tl_two_opt_batch(self.h, algo, capi.ptr(t), t.shape[0], max_moves,
                                              C.byref(st), capi.ptr(lengths)))
        return t, st, lengths

    def aco(self, seed: int, init_tour=None, alpha: float = 1.0, beta: float = 2.0, evaporation_rate: float = 0.5,
            num_ants: int = 25, epochs: int = 150):
        """tl_aco with the reference's AcoOptions defaults: returns (best_tour, best_cost, Stats)."""
        o = capi.AcoOptions(alpha, beta, evaporation_rate, num_ants, epochs, 0, seed)
        best = np.empty(self.n, dtype=np.uint32)
        cost, st = C.c_float(), Stats()
        it = _u32(init_tour) if init_tour is not None else None
        capi.check(self._lib.tl_aco(self.h, C.byref(o), capi.ptr(it) if it is not None else None, capi.ptr(best),
                                    C.byref(cost), C.byref(st)))
        return best, float(cost.value), st

    def ga(self, seed: int, init_tour=None, mutation_probability: float = 0.001, n_elite: int = 3, epochs: int = 10000):
        """tl_ga with the reference's GAOptions defaults: returns (best_tour, best_length, Stats)."""
        o = capi.GaOptions(mutation_probability, n_elite, epochs, 0, seed)
        best = np.empty(self.n, dtype=np.uint32)
        cost, st = C.c_float(), Stats()
        it = _u32(init_tour) if init_tour is not None else None
        capi.check(self._lib.tl_ga(self.h, C.byref(o), capi.ptr(it) if it is not None else None, capi.ptr(best),
                                   C.byref(cost), C.byref(st)))
        return best, float(cost.value), st

    def session(self, algo: int, tour, path: int = PATH_AUTO) -> "Session":
        return Session(self, algo, path, tour)

    def close(self):
        if getattr(self, "h", None):
            for child in list(self._children):
                child.close()
            self._lib.tl_problem_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Session:
    """tl_session: a device-resident local search that can be stepped."""

    def __init__(self, problem: Problem, algo: int, path: int, tour):
        self.problem = problem
        self.algo = algo
        self._lib = problem._lib
        t = _u32(tour)
        h = C.c_void_p()
        capi.check(self._lib.tl_session_create(problem.h, algo, path, capi.ptr(t), C.byref(h)))
        self.h = h
        problem._children.add(self)

    def set_shard(self, index: int, count: int):
        capi.check(self._lib.tl_session_set_shard(self.h, index, count))

    def scan(self):
        mv, found = Move(), C.c_int32()
        capi.check(self._lib.tl_session_scan(self.h, C.byref(mv), C.byref(found)))
        if not found.value:
            return None
        return mv.astuple3() if self.algo in (ALGO_THREE_OPT, ALGO_THREE_OPT_NEIGHBOR) else mv.astuple()

    def time_scans(self, reps: int) -> float:
        """Average scan-kernel launch duration in ms (CUDA events on the context's stream)."""
        out = C.c_double()
        capi.check(self._lib.tl_session_time_scans(self.h, reps, C.byref(out)))
        return out.value

    def enqueue(self, steps: int):
        capi.check(self._lib.tl_session_enqueue(self.h, steps))

    def run(self, max_moves: int = -1):
        capi.check(self._lib.tl_session_run(self.h, max_moves))

    def tour(self) -> np.ndarray:
        out = np.empty(self.problem.n, dtype=np.uint32)
        capi.check(self._lib.tl_session_tour(self.h, capi.ptr(out)))
        return out

    def stats(self) -> Stats:
        st = Stats()
        capi.check(self._lib.tl_session_stats(self.h, C.byref(st)))
        return st

    def log(self, cap: int = 1 << 16):
        log = (Move * max(cap, 1))()
        got = C.c_size_t()
        capi.check(self._lib.tl_session_log(self.h, log, cap, C.byref(got)))
        three = self.algo in (ALGO_THREE_OPT, ALGO_THREE_OPT_NEIGHBOR)
        return [log[k].astuple3() if three else log[k].astuple() for k in range(got.value)]

    def close(self):
        if getattr(self, "h", None):
            self._lib.tl_session_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
