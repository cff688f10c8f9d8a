"""ctypes loader for the CPU ORACLES of candidate-list 2-opt, Or-opt and 3-opt and of the greedy-edge constructor
(oracle_nl/libteeline_oracle_nl.so).

TEST INFRASTRUCTURE ONLY, like `oracle`: tests and measurement scripts load it, the product package
(teeline_b200/) never does.  Problems are `oracle.Problem` instances; the definitions are in
two_opt_nl.h, or_opt_nl.h, three_opt_nl.h, greedy_nl.h and include/teeline_cuda.h (tl_problem_set_candidates,
tl_greedy_tour).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

import oracle as O

_DIR = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_DIR, "libteeline_oracle_nl.so")
_ORACLE_DIR = os.path.dirname(os.path.abspath(O.__file__))


def build(force: bool = False) -> str:
    """Compile with gcc (oracle_nl/Makefile)."""
    srcs = [os.path.join(_DIR, f) for f in ("two_opt_nl.c", "two_opt_nl.h", "or_opt_nl.c", "or_opt_nl.h", "three_opt_nl.c",
                                         "three_opt_nl.h", "greedy_nl.c", "greedy_nl.h", "Makefile")] + \
        [os.path.join(_ORACLE_DIR, f) for f in ("teeline_oracle.c", "algos.inc", "teeline_oracle.h")]
    stale = not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs)
    if force or stale:
        subprocess.run(["make", "-C", _DIR, "-s"], check=True)
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_SO)
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _cand(cand):
    """n x k candidate positions as int32 (the GPU's UINT32_MAX padding becomes -1)."""
    c = np.ascontiguousarray(cand)
    if c.dtype == np.uint32:
        c = c.view(np.int32)
    c = np.ascontiguousarray(c, dtype=np.int32)
    assert c.ndim == 2
    return c


def two_opt_nl_scan(p: O.Problem, tour, cand, nthreads: int = 1):
    """One scan.  Returns (move or None, evals); move = (delta, i, j, 0, 0) as O.two_opt_best_scan."""
    t = np.ascontiguousarray(tour, dtype=np.int32)
    c = _cand(cand)
    mv, ev = O.Move(), C.c_int64()
    found = lib().tlo_two_opt_nl_scan(p.ref, _p(t), _p(c), C.c_int32(c.shape[1]), C.c_int(nthreads), C.byref(mv),
                                      C.byref(ev))
    return (mv.astuple() if found else None), ev.value


def two_opt_nl(p: O.Problem, tour, cand, max_moves: int = -1, nthreads: int = 1, log_cap: int = 0):
    """Mode N to its local optimum (or max_moves).  Returns (tour, stats, moves) as O.two_opt_best."""
    t = np.ascontiguousarray(tour, dtype=np.int32).copy()
    c = _cand(cand)
    st, log = O.Stats(), (O.Move * max(log_cap, 1))()
    lib().tlo_two_opt_nl(p.ref, _p(t), _p(c), C.c_int32(c.shape[1]), C.c_int64(max_moves), C.c_int(nthreads),
                         C.byref(st), log, C.c_int64(log_cap))
    return t, st, [log[m].astuple() for m in range(min(st.moves, log_cap))]


def two_opt_nl_multi(p: O.Problem, tour, cand, block: int, step0: int = 0, max_moves: int = -1, nthreads: int = 1,
                     log_cap: int = 0):
    """Mode NM (multi-move Mode N) with blocks of `block` positions, first step numbered step0, to its local
    optimum (or max_moves).  Returns (tour, stats, moves, converged); moves as two_opt_nl's."""
    assert block >= 2 and block & (block - 1) == 0, "block must be a power of two >= 2"
    t = np.ascontiguousarray(tour, dtype=np.int32).copy()
    c = _cand(cand)
    st, log = O.Stats(), (O.Move * max(log_cap, 1))()
    conv = lib().tlo_two_opt_nl_multi(p.ref, _p(t), _p(c), C.c_int32(c.shape[1]), C.c_int32(block), C.c_int64(step0),
                                      C.c_int64(max_moves), C.c_int(nthreads), C.byref(st), log, C.c_int64(log_cap))
    return t, st, [log[m].astuple() for m in range(min(st.moves, log_cap))], int(conv)


def or_opt_nl_scan(p: O.Problem, tour, cand, nthreads: int = 1):
    """One Or-opt N scan.  Returns (move or None, evals); move = (delta, i, j, seg_len, reversed)."""
    t = np.ascontiguousarray(tour, dtype=np.int32)
    c = _cand(cand)
    mv, ev = O.Move(), C.c_int64()
    found = lib().tlo_or_opt_nl_scan(p.ref, _p(t), _p(c), C.c_int32(c.shape[1]), C.c_int(nthreads), C.byref(mv),
                                     C.byref(ev))
    return (mv.astuple() if found else None), ev.value


def or_opt_nl(p: O.Problem, tour, cand, max_moves: int = -1, nthreads: int = 1, log_cap: int = 0):
    """Or-opt N to its local optimum (or max_moves).  Returns (tour, stats, moves) as O.or_opt."""
    t = np.ascontiguousarray(tour, dtype=np.int32).copy()
    c = _cand(cand)
    st, log = O.Stats(), (O.Move * max(log_cap, 1))()
    lib().tlo_or_opt_nl(p.ref, _p(t), _p(c), C.c_int32(c.shape[1]), C.c_int64(max_moves), C.c_int(nthreads),
                        C.byref(st), log, C.c_int64(log_cap))
    return t, st, [log[m].astuple() for m in range(min(st.moves, log_cap))]


def or_opt_nl_multi(p: O.Problem, tour, cand, block: int, step0: int = 0, max_moves: int = -1, nthreads: int = 1,
                    log_cap: int = 0):
    """Or-opt NM (multi-move Or-opt N) with blocks of `block` positions, first step numbered step0, to its local
    optimum (or max_moves).  Returns (tour, stats, moves, converged); moves as or_opt_nl's."""
    assert block >= 2 and block & (block - 1) == 0, "block must be a power of two >= 2"
    t = np.ascontiguousarray(tour, dtype=np.int32).copy()
    c = _cand(cand)
    st, log = O.Stats(), (O.Move * max(log_cap, 1))()
    conv = lib().tlo_or_opt_nl_multi(p.ref, _p(t), _p(c), C.c_int32(c.shape[1]), C.c_int32(block), C.c_int64(step0),
                                     C.c_int64(max_moves), C.c_int(nthreads), C.byref(st), log, C.c_int64(log_cap))
    return t, st, [log[m].astuple() for m in range(min(st.moves, log_cap))], int(conv)


def three_opt_nl_eval(p: O.Problem, tour, i: int, j: int, k: int):
    """The evaluation of the triple i < j < k on tour: (delta = -savings, case), or None when no case improves."""
    t = np.ascontiguousarray(tour, dtype=np.int32)
    s, kase = C.c_double(), C.c_int32()
    ok = lib().tlo_three_opt_nl_eval(p.ref, _p(t), C.c_int32(i), C.c_int32(j), C.c_int32(k), C.byref(s),
                                     C.byref(kase))
    return (-s.value, kase.value) if ok else None


def three_opt_nl_scan(p: O.Problem, tour, cand, nthreads: int = 1):
    """One 3-opt N scan.  Returns (move or None, evals); move = (delta = -savings, i, j, k, case) as
    O.three_opt_find_best."""
    t = np.ascontiguousarray(tour, dtype=np.int32)
    c = _cand(cand)
    mv, k, ev = O.Move(), C.c_int32(), C.c_int64()
    found = lib().tlo_three_opt_nl_scan(p.ref, _p(t), _p(c), C.c_int32(c.shape[1]), C.c_int(nthreads), C.byref(mv),
                                        C.byref(k), C.byref(ev))
    return ((mv.delta, mv.i, mv.j, k.value, mv.seg_len) if found else None), ev.value


def three_opt_nl(p: O.Problem, tour, cand, max_moves: int = -1, nthreads: int = 1, log_cap: int = 0):
    """3-opt N to its local optimum (or max_moves).  Returns (tour, stats, moves) as O.three_opt, with
    moves = (delta, i, j, k, case)."""
    t = np.ascontiguousarray(tour, dtype=np.int32).copy()
    c = _cand(cand)
    st, log = O.Stats(), (O.Move * max(log_cap, 1))()
    ks = np.zeros(max(log_cap, 1), dtype=np.int32)
    lib().tlo_three_opt_nl(p.ref, _p(t), _p(c), C.c_int32(c.shape[1]), C.c_int64(max_moves), C.c_int(nthreads),
                           C.byref(st), log, _p(ks), C.c_int64(log_cap))
    mv = [(log[m].delta, log[m].i, log[m].j, int(ks[m]), log[m].seg_len) for m in range(min(st.moves, log_cap))]
    return t, st, mv


def _greedy(fn, x, y, metric):
    x = np.ascontiguousarray(x, dtype=np.float32)
    y = np.ascontiguousarray(y, dtype=np.float32)
    out = np.empty(len(x), dtype=np.int32)
    getattr(lib(), fn)(C.c_int32(len(x)), _p(x), _p(y), C.c_int(metric == "nint"), _p(out))
    return out


def greedy_brute(x, y, metric: str = "f32"):
    """The greedy-edge tour by sorting all n(n-1)/2 edges (metric "f32" or "nint"); a few thousand cities."""
    return _greedy("tlo_greedy_brute", x, y, metric)


def greedy_lazy(x, y, metric: str = "f32"):
    """The greedy-edge tour by Bentley's lazy greedy on a uniform grid; fast enough for 10^6 cities."""
    return _greedy("tlo_greedy_lazy", x, y, metric)
