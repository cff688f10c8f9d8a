"""ctypes binding of libteeline_cuda.so (include/teeline_cuda.h), one-to-one.

This is the thinnest possible layer: it exists so that the parity tests and
bench.py can drive the C ABI exactly as the reference-side Rust shim would
(INTEGRATION.md).  There is no CPU fallback: if the shared library is missing or
no CUDA device is present the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TL_LIB") or os.path.join(_HERE, "libteeline_cuda.so")  # TL_LIB: tuning builds only

# enums (teeline_cuda.h)
TL_OK = 0
DIST_F32_EXACT, DIST_NINT_I32 = 0, 1
ALGO_TWO_OPT_REF, ALGO_TWO_OPT_BEST, ALGO_TWO_OPT_BEST_CYCLIC, ALGO_OR_OPT, ALGO_THREE_OPT = 0, 1, 2, 3, 4
ALGO_TWO_OPT_BEST_CACHED = 5
ALGO_TWO_OPT_NEIGHBOR = 6
ALGO_OR_OPT_NEIGHBOR = 7
ALGO_THREE_OPT_NEIGHBOR = 8
ALGO_TWO_OPT_NEIGHBOR_MULTI = 9
ALGO_OR_OPT_NEIGHBOR_MULTI = 10
MULTI_BLOCK = 4096
OR_MULTI_BLOCK = 16384
CANDIDATES_DEFAULT = 8
PATH_AUTO, PATH_MATRIX, PATH_RECOMPUTE = 0, 1, 2
LEN_EXACT, LEN_FAST = 0, 1
NCCL_ID_BYTES = 128

EXPORTS = [
    "tl_ctx_create", "tl_ctx_create_on_stream", "tl_ctx_destroy", "tl_ctx_sync", "tl_last_error",
    "tl_version", "tl_ctx_launch_count", "tl_nccl_unique_id", "tl_ctx_attach_nccl",
    "tl_problem_create_euc2d", "tl_problem_create_explicit", "tl_problem_destroy",
    "tl_dist_matrix_packed", "tl_dist_matrix_packed_i32", "tl_knn", "tl_problem_set_candidates", "tl_nn_tour", "tl_greedy_tour", "tl_tour_lengths",
    "tl_tour_lengths_i64", "tl_local_search", "tl_two_opt_batch", "tl_session_create",
    "tl_session_destroy", "tl_session_set_shard", "tl_session_scan", "tl_session_time_scans",
    "tl_session_enqueue",
    "tl_session_run", "tl_session_tour", "tl_session_stats", "tl_session_log", "tl_selftest_sqrt",
    "tl_microbench_fp32", "tl_aco", "tl_ga",
]


class Move(C.Structure):
    _fields_ = [("delta", C.c_float), ("i", C.c_uint32), ("j", C.c_uint32), ("seg_len", C.c_uint8),
                ("reversed", C.c_uint8), ("pad", C.c_uint16), ("k", C.c_uint32)]

    def astuple(self):
        return (float(self.delta), int(self.i), int(self.j), int(self.seg_len), int(self.reversed))

    def astuple3(self):
        """3-opt view: (delta, i, j, k, case)."""
        return (float(self.delta), int(self.i), int(self.j), int(self.k), int(self.seg_len))


class Stats(C.Structure):
    _fields_ = [("passes", C.c_uint64), ("moves", C.c_uint64), ("evals", C.c_uint64),
                ("launches", C.c_uint64), ("repermutes", C.c_uint64), ("device_ms", C.c_double),
                ("converged", C.c_int32), ("path_used", C.c_int32)]

    def asdict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class AcoOptions(C.Structure):
    _fields_ = [("alpha", C.c_float), ("beta", C.c_float), ("evaporation_rate", C.c_float),
                ("num_ants", C.c_uint32), ("epochs", C.c_uint32), ("pad", C.c_uint32), ("seed", C.c_uint64)]


class GaOptions(C.Structure):
    _fields_ = [("mutation_probability", C.c_float), ("n_elite", C.c_uint32), ("epochs", C.c_uint32),
                ("pad", C.c_uint32), ("seed", C.c_uint64)]


class TeelineError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__(f"tl_status={status}: {msg}")
        self.status = status


_lib = None


def load():
    """dlopen the in-tree library.  Raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(teeline_b200 has no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    L.tl_last_error.restype = C.c_char_p
    L.tl_version.restype = C.c_char_p
    L.tl_ctx_launch_count.restype = C.c_uint64
    L.tl_ctx_launch_count.argtypes = [C.c_void_p]
    L.tl_ctx_create.argtypes = [C.c_int32, C.POINTER(C.c_void_p)]
    L.tl_ctx_create_on_stream.argtypes = [C.c_int32, C.c_void_p, C.POINTER(C.c_void_p)]
    L.tl_ctx_destroy.argtypes = [C.c_void_p]
    L.tl_ctx_destroy.restype = None
    L.tl_ctx_sync.argtypes = [C.c_void_p]
    L.tl_nccl_unique_id.argtypes = [C.c_void_p]
    L.tl_ctx_attach_nccl.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]
    L.tl_problem_create_euc2d.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_int32,
                                          C.POINTER(C.c_void_p)]
    L.tl_problem_create_explicit.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.POINTER(C.c_void_p)]
    L.tl_problem_destroy.argtypes = [C.c_void_p]
    L.tl_problem_destroy.restype = None
    L.tl_dist_matrix_packed.argtypes = [C.c_void_p, C.c_void_p]
    L.tl_dist_matrix_packed_i32.argtypes = [C.c_void_p, C.c_void_p]
    L.tl_knn.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
    L.tl_problem_set_candidates.argtypes = [C.c_void_p, C.c_uint32]
    L.tl_nn_tour.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
    L.tl_greedy_tour.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Stats)]
    L.tl_tour_lengths.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int32, C.c_void_p]
    L.tl_tour_lengths_i64.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    L.tl_local_search.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int64,
                                  C.POINTER(Stats), C.c_void_p, C.c_size_t]
    L.tl_two_opt_batch.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_size_t, C.c_int64,
                                   C.POINTER(Stats), C.c_void_p]
    L.tl_session_create.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.POINTER(C.c_void_p)]
    L.tl_session_destroy.argtypes = [C.c_void_p]
    L.tl_session_destroy.restype = None
    L.tl_session_set_shard.argtypes = [C.c_void_p, C.c_int32, C.c_int32]
    L.tl_session_scan.argtypes = [C.c_void_p, C.POINTER(Move), C.POINTER(C.c_int32)]
    L.tl_session_enqueue.argtypes = [C.c_void_p, C.c_uint32]
    L.tl_session_time_scans.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_double)]
    L.tl_session_run.argtypes = [C.c_void_p, C.c_int64]
    L.tl_session_tour.argtypes = [C.c_void_p, C.c_void_p]
    L.tl_session_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
    L.tl_session_log.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
    L.tl_selftest_sqrt.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint64)]
    L.tl_microbench_fp32.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.tl_aco.argtypes = [C.c_void_p, C.POINTER(AcoOptions), C.c_void_p, C.c_void_p, C.POINTER(C.c_float),
                         C.POINTER(Stats)]
    L.tl_ga.argtypes = [C.c_void_p, C.POINTER(GaOptions), C.c_void_p, C.c_void_p, C.POINTER(C.c_float),
                        C.POINTER(Stats)]
    _lib = L
    return L


def check(status: int):
    if status != TL_OK:
        raise TeelineError(status, load().tl_last_error().decode(errors="replace"))


def ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)
