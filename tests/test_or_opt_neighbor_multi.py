"""Multi-move candidate-list Or-opt ("Or-opt NM", TL_ALGO_OR_OPT_NEIGHBOR_MULTI).

CPU: the Or-opt NM oracle (oracle_nl) against Or-opt N's when one block covers the tour, against an independent
numpy restatement of a step, and on its own properties (hulls, exact length change, Or-opt N local optimum,
budgets, thread count); the ABI and the CLI without a device.  GPU: the library bit for bit against the oracle
(move log, tour, moves / scans / evals) with the built block size and with small blocks, a long G applied together
with block moves, Or-opt N on the GPU for n <= TL_OR_MULTI_BLOCK/2, budgets and resumed sessions, 10^6 cities from the
Mode NM optimum of the greedy tour, and the CLI.  The nint oracle needs the packed triangle, so nint runs stop at
10^4 cities against it."""
import os
import subprocess

import numpy as np
import pytest

import oracle as O
import oracle_nl as NL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
SPAN = 4096  # kOrNlCtaSpan: longer relocations of G go through the apply grids


def f32_bits(v):
    return np.float32(v).view(np.uint32)


def key(m):
    return (int(f32_bits(m[0])), int(m[1]), int(m[2]), int(m[3]), int(m[4]))


def same_moves(got, want):
    """GPU log (f32 delta) against the oracle's (widened delta): (delta bits, i, j, s, rev) per move."""
    return [key(m) for m in got] == [key(m) for m in want]


def replay(start, moves):
    cur = np.asarray(start).copy()
    for _, i, j, s, r in moves:
        cur = O.or_opt_apply(cur, i, s, j, r)
    return cur


def wraps(m, n):
    _, i, j, s, _ = m
    return i == 0 or i + s == n or j == n - 1


def hull(m):
    _, i, j, s, _ = m
    return min(i - 1, j), max(i + s, j + 1)


def span(m):
    a0, a1 = hull(m)
    return a1 - a0 - 1


def oracle_problem(x, y, metric):
    return O.Problem(tri=O.matrix_packed_nint(x, y), n=len(x)) if metric == "nint" else O.Problem(x, y)


def step_ref(x, y, tour, K, block, t):
    """One Or-opt NM step restated with numpy (f32 metric): the moves it applies, in log order, as 5-tuples."""
    n = len(tour)
    tour = np.asarray(tour, dtype=np.int64)
    pos = np.empty(n, dtype=np.int64)
    pos[tour] = np.arange(n)
    q = np.repeat(np.arange(n), K.shape[1])
    b = K[tour].reshape(-1).astype(np.int64)
    keep = b >= 0
    q, r = q[keep], pos[b[keep]]
    rm = (r - 1) % n
    parts = []  # the ten roles: (i, j, s, rev)
    for s in (1, 2, 3):
        parts.append((q, r, s, 0))              # (f, x) forward
        parts.append((q - s + 1, rm, s, 0))     # (l, y) forward
        if s > 1:
            parts.append((q - s + 1, r, s, 1))  # (l, x) reversed
            parts.append((q, rm, s, 1))         # (f, y) reversed
    I = np.concatenate([p[0] for p in parts])
    J = np.concatenate([p[1] for p in parts])
    S = np.concatenate([np.full(len(p[0]), p[2]) for p in parts])
    R = np.concatenate([np.full(len(p[0]), p[3]) for p in parts])
    prev = np.where(I == 0, n - 1, I - 1)
    legal = (n > S + 1) & (I >= 0) & (I + S <= n) & (J != prev) & ~((J >= I) & (J < I + S))
    I, J, S, R = I[legal], J[legal], S[legal], R[legal]

    def d(u, v):
        dx = (x[tour[u]] - x[tour[v]]).astype(np.float32)
        dy = (y[tour[u]] - y[tour[v]]).astype(np.float32)
        return np.sqrt(dx * dx + dy * dy, dtype=np.float32)

    a, f, l, dd = np.where(I == 0, n - 1, I - 1), I, I + S - 1, (I + S) % n
    xx, yy = J, (J + 1) % n
    rg = (d(a, f) + d(l, dd)) - d(a, dd)
    fwd = ((-rg + d(xx, f)) + d(l, yy)) - d(xx, yy)
    rev = ((-rg + d(xx, l)) + d(f, yy)) - d(xx, yy)
    delta = np.where(R == 1, rev, fwd).astype(np.float32)
    below = delta < np.float32(-1e-3)
    delta, I, J, S, R = delta[below], I[below], J[below], S[below], R[below]
    if len(delta) == 0:
        return []
    order = np.lexsort((R, J, I, S, delta))
    delta, I, J, S, R = delta[order], I[order], J[order], S[order], R[order]
    G = (float(delta[0]), int(I[0]), int(J[0]), int(S[0]), int(R[0]))
    if wraps(G, n):
        return [G]
    g0, g1 = hull(G)
    a0, a1 = np.minimum(I - 1, J), np.maximum(I + S, J + 1)
    off = (t % 2) * (block // 2)
    blk = (a0 + off) // block
    inb = (I != 0) & (I + S != n) & (J != n - 1) & (blk == (a1 + off) // block)
    ub, first = np.unique(blk[inb], return_index=True)  # sorted by Or-opt's order: first per block is its best
    sel = np.flatnonzero(inb)[first]
    acc = (a1[sel] <= g0) | (a0[sel] >= g1)
    rest = [(float(delta[k]), int(I[k]), int(J[k]), int(S[k]), int(R[k])) for k in sel[acc]]  # increasing block
    return [G] + rest


def next_pow2(v):
    return 1 << max(1, (v - 1).bit_length())


# ---- CPU: the oracle ------------------------------------------------------------------------------------

@pytest.mark.parametrize("metric", ["f32", "nint"])
def test_oracle_one_block_is_or_opt_n(metric):
    wrapping = 0
    for n in list(range(4, 34)) + [1000]:
        x, y = O.gen_uniform(n, 500 + n)
        P = oracle_problem(x, y, metric)
        K = O.knn(O.Problem(x, y) if metric == "f32" else P, min(8, n - 1))
        start = O.shuffle_tour(n, 9 + n)
        tn, sn, mn = NL.or_opt_nl(P, start, K, log_cap=1 << 14)
        wrapping += sum(wraps(m, n) for m in mn)
        for block in (next_pow2(2 * n), 4 * next_pow2(2 * n)):
            tm, sm, mm, conv = NL.or_opt_nl_multi(P, start, K, block, log_cap=1 << 14)
            assert mm == mn and (tm == tn).all() and conv == 1, (n, block)
            assert (sm.moves, sm.passes, sm.evals) == (sn.moves, sn.passes, sn.evals)
    assert wrapping > 0  # G that wraps (applied alone) is covered


@pytest.fixture(scope="module")
def inst20k():
    n = 20000
    x, y = O.gen_uniform(n, n)
    P = O.Problem(x, y)
    K = O.knn(P, 8)
    start, _, _ = NL.two_opt_nl(P, NL.greedy_lazy(x, y), K, nthreads=8)  # Mode N optimum of the greedy tour
    return x, y, P, K, start


@pytest.mark.parametrize("block", [256, 1024])
def test_oracle_properties_20k(inst20k, block):
    x, y, P, K, start = inst20k
    n = len(x)
    t, st, moves, conv = NL.or_opt_nl_multi(P, start, K, block, nthreads=8, log_cap=1 << 16)
    assert conv == 1 and st.moves == len(moves) and sorted(t.tolist()) == list(range(n))
    # step by step against the numpy restatement: G first, then the accepted block bests in block order
    cur, at, steps, multi = start.copy(), 0, 0, 0
    while True:
        want = step_ref(x, y, cur, K, block, steps)
        if not want:
            break
        got = moves[at:at + len(want)]
        assert [key(m) for m in got] == [key(m) for m in want], steps
        hulls = sorted(hull(m) for m in want)
        assert all(a[1] <= b[0] for a, b in zip(hulls, hulls[1:]))  # at most an end position in common
        multi += len(want) > 1
        cur = replay(cur, got)
        at += len(want)
        steps += 1
    assert at == len(moves) and st.passes == steps + 1 and (cur == t).all() and multi > 0
    assert NL.or_opt_nl_scan(P, t, K, nthreads=8)[0] is None
    assert steps < NL.or_opt_nl(P, start, K, nthreads=8)[1].passes
    # f32: the length falls by the logged deltas up to the rounding of each edge sum
    drop = O.tour_length(P, start) - O.tour_length(P, t)
    assert drop > 0 and abs(drop + sum(m[0] for m in moves)) < 1e-3 * drop
    # budgets: the first m moves of the unbudgeted log, and the tour they give
    for m in (1, 2, 3, len(step_ref(x, y, start, K, block, 0)) - 1, st.moves // 2, st.moves - 1):
        tb, sb, mb, cb = NL.or_opt_nl_multi(P, start, K, block, max_moves=m, nthreads=8, log_cap=1 << 16)
        assert mb == moves[:m] and sb.moves == m and cb == 0 and (tb == replay(start, moves[:m])).all()
    # thread count
    t1, s1, m1, _ = NL.or_opt_nl_multi(P, start, K, block, nthreads=1, log_cap=1 << 16)
    assert m1 == moves and (t1 == t).all() and (s1.passes, s1.evals) == (st.passes, st.evals)


def test_oracle_nint_length_exact_and_resume():
    n = 10000
    x, y = O.gen_uniform(n, 3 * n)
    P = oracle_problem(x, y, "nint")
    K = O.knn(P, 8)
    start = O.nn_tour(P, 3)
    t, st, moves, conv = NL.or_opt_nl_multi(P, start, K, 256, nthreads=8, log_cap=1 << 20)
    assert conv == 1 and all(m[0] < 0 and m[0] == int(m[0]) for m in moves)
    assert int(O.tour_length(P, start)) + int(sum(m[0] for m in moves)) == int(O.tour_length(P, t))
    assert NL.or_opt_nl_scan(P, t, K, nthreads=8)[0] is None
    # budget a at the end of a step, then b more from that tour with the step count carried over: the
    # unbudgeted log (a resumed search starts a new step, so a cut inside a step would not give it)
    a = next(a for a in range(st.moves // 3, st.moves)
             if NL.or_opt_nl_multi(P, start, K, 256, max_moves=a + 1, nthreads=8)[1].passes >
             NL.or_opt_nl_multi(P, start, K, 256, max_moves=a, nthreads=8)[1].passes)
    b = st.moves // 3
    ta, sa, ma, _ = NL.or_opt_nl_multi(P, start, K, 256, max_moves=a, nthreads=8, log_cap=1 << 20)
    tb, sb, mb, _ = NL.or_opt_nl_multi(P, ta, K, 256, step0=sa.passes, max_moves=b, nthreads=8, log_cap=1 << 20)
    assert ma + mb == moves[:a + b] and (tb == replay(start, moves[:a + b])).all()


# ---- CPU: ABI and CLI without a device --------------------------------------------------------------------

@pytest.fixture(scope="module")
def cli():
    from teeline_b200 import build as tb, build_host
    tb.build()
    return build_host.build()


def run(cmd):
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    return p.returncode, p.stdout, p.stderr


def test_abi_constants():
    import teeline_b200 as T
    assert T.ALGO_OR_OPT_NEIGHBOR_MULTI == 10 and T.OR_MULTI_BLOCK == 16384 and T.MULTI_BLOCK == 4096
    hdr = open(os.path.join(ROOT, "include", "teeline_cuda.h")).read()
    assert "TL_ALGO_OR_OPT_NEIGHBOR_MULTI = 10" in hdr and "#define TL_OR_MULTI_BLOCK 16384" in hdr


def test_cli_without_device(cli, tmp_path):
    import torch
    rc, out, _ = run([cli, "solvers"])
    assert rc == 0 and "or_opt --mode neighbor_multi" in out
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    inp = os.path.join(GOLDEN, "berlin52.tsp")
    rc, out, err = run([cli, "solve", "or_opt", "--mode", "neighbor_multi", "--candidates", "8", "-i", inp])
    assert rc == 101 and out == "" and "no CPU fallback" in err
    cfg = tmp_path / "onm.toml"
    cfg.write_text("[[stage]]\nsolver = \"greedy_edge\"\n[[stage]]\nsolver = \"or_opt\"\n[stage.cuda]\n"
                   "mode = \"neighbor_multi\"\ncandidates = 8\n")
    rc, out, err = run([cli, "pipeline", "--config", str(cfg), "-i", inp])
    assert rc == 101 and out == "" and "no CPU fallback" in err


# ---- GPU ----------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def ctx():
    import teeline_b200 as T
    c = T.Context(0)
    yield c
    c.close()


def instance(name):
    if name in ("berlin52", "att532"):
        _, x, y = O.read_tsplib_coords(os.path.join(GOLDEN, name + ".tsp"))
    else:
        x, y = O.gen_uniform(int(name), 7000 + int(name))
    return x, y


def make_problem(ctx, x, y, metric, k):
    import teeline_b200 as T
    prob = T.Problem.euc2d(ctx, x, y, T.DIST_NINT_I32 if metric == "nint" else T.DIST_F32_EXACT)
    prob.set_candidates(k)
    return prob


def starts(prob, x, y):
    """The Mode N optimum of the greedy tour (computed on the GPU: it is only an input here) and the NN tour."""
    import teeline_b200 as T
    g, _ = prob.greedy_tour()
    return prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR, g)[0], O.nn_tour(O.Problem(x, y), 3)


def gpu_vs_oracle(prob, P, K, start, block=None, max_moves=-1):
    import teeline_b200 as T
    cap = 1 << 20
    got_t, st, got_m = prob.local_search(T.ALGO_OR_OPT_NEIGHBOR_MULTI, start, max_moves=max_moves, log_cap=cap)
    want_t, wst, want_m, conv = NL.or_opt_nl_multi(P, start, K, block or T.OR_MULTI_BLOCK, max_moves=max_moves,
                                                   nthreads=16, log_cap=cap)
    assert same_moves(got_m, want_m)
    assert (got_t.astype(np.int64) == want_t).all()
    assert (int(st.moves), int(st.passes), int(st.evals)) == (wst.moves, wst.passes, wst.evals)
    assert st.converged == conv and st.path_used == T.PATH_RECOMPUTE
    return got_t, want_m


def check_instance(ctx, x, y, metric, k, block=None):
    prob = make_problem(ctx, x, y, metric, k)
    P = O.Problem(x, y) if metric == "f32" else oracle_problem(x, y, metric)
    K = prob.knn(k)
    for start in starts(prob, x, y):
        gpu_vs_oracle(prob, P, K, start, block)
    prob.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["4", "5", "6", "7", "13", "20", "33", "257", "1000", "berlin52", "att532"])
@pytest.mark.parametrize("metric", ["f32", "nint"])
def test_gpu_equals_oracle(ctx, name, metric):
    x, y = instance(name)
    for k in (5, 8, 10):
        check_instance(ctx, x, y, metric, k)


@pytest.mark.gpu
@pytest.mark.parametrize("block", ["8", "64", "256"])
@pytest.mark.parametrize("n", [1000, 5000])
def test_gpu_equals_oracle_small_blocks(ctx, monkeypatch, block, n):
    """Many blocks: boundaries, both offsets and moves that straddle a boundary."""
    monkeypatch.setenv("TL_MULTI_BLOCK", block)
    x, y = O.gen_uniform(n, 3 * n)
    for metric in ("f32", "nint"):
        check_instance(ctx, x, y, metric, 8, block=int(block))


@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["f32", "nint"])
def test_gpu_equals_oracle_10k(ctx, metric):
    x, y = O.gen_uniform(10000, 10000)
    check_instance(ctx, x, y, metric, 8)


@pytest.mark.gpu
def test_gpu_equals_oracle_100k(ctx):
    import teeline_b200 as T
    x, y = O.gen_uniform(100_000, 100_000)
    prob = make_problem(ctx, x, y, "f32", 8)
    g, _ = prob.greedy_tour()
    gpu_vs_oracle(prob, O.Problem(x, y), prob.knn(8), prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR, g)[0])


@pytest.mark.gpu
def test_gpu_ties_on_a_lattice(ctx):
    side = 24
    q = np.arange(side * side)
    lattice = ((q % side).astype(np.float32), (q // side).astype(np.float32))
    for x, y in (lattice, O.gen_grid(900, 900)):
        for metric in ("f32", "nint"):
            for k in (3, 8):
                prob = make_problem(ctx, x, y, metric, k)
                P = O.Problem(x, y) if metric == "f32" else oracle_problem(x, y, metric)
                gpu_vs_oracle(prob, P, prob.knn(k), O.shuffle_tour(len(x), 3))


@pytest.mark.gpu
def test_gpu_long_g_with_block_moves(ctx, monkeypatch):
    """Steps whose G spans more than one CTA relocates (the apply grids) together with block moves."""
    monkeypatch.setenv("TL_MULTI_BLOCK", "4096")
    n = 20000
    x, y = O.gen_uniform(n, 2 * n)
    prob = make_problem(ctx, x, y, "f32", 8)
    P, K = O.Problem(x, y), prob.knn(8)
    start = O.shuffle_tour(n, 17)
    _, moves = gpu_vs_oracle(prob, P, K, start, block=4096, max_moves=400)
    # split the log into steps with the restatement and look for a long G applied with block moves
    cur, at, t, found = start.copy(), 0, 0, 0
    while at < len(moves):
        want = step_ref(x, y, cur, K.view(np.int32), 4096, t)
        got = moves[at:at + len(want)]
        assert [key(m) for m in got] == [key(m) for m in want[:len(got)]], t
        found += len(want) > 1 and span(want[0]) > SPAN
        cur = replay(cur, got)
        at += len(got)
        t += 1
    assert found > 0


@pytest.mark.gpu
@pytest.mark.parametrize("n", [13, 257, 2048])
def test_gpu_half_block_is_gpu_or_opt_n(ctx, n):
    import teeline_b200 as T
    x, y = O.gen_uniform(n, 40 + n)
    prob = make_problem(ctx, x, y, "f32", 8)
    for start in (prob.nn_tour(3), O.shuffle_tour(n, n)):
        tn, sn, mn = prob.local_search(T.ALGO_OR_OPT_NEIGHBOR, start, log_cap=1 << 14)
        tm, sm, mm = prob.local_search(T.ALGO_OR_OPT_NEIGHBOR_MULTI, start, log_cap=1 << 14)
        assert mm == mn and (tm == tn).all() and (sm.moves, sm.passes, sm.evals) == (sn.moves, sn.passes, sn.evals)


@pytest.mark.gpu
@pytest.mark.parametrize("block", [None, "64"])
def test_gpu_budgets_resume_and_log_cap(ctx, monkeypatch, block):
    import teeline_b200 as T
    if block:
        monkeypatch.setenv("TL_MULTI_BLOCK", block)
    B = int(block) if block else T.OR_MULTI_BLOCK
    n = 20000
    x, y = O.gen_uniform(n, 11 * n)
    P = O.Problem(x, y)
    prob = make_problem(ctx, x, y, "f32", 8)
    K = prob.knn(8)
    start = O.nn_tour(P, 3)
    full_t, fst, full_m, _ = NL.or_opt_nl_multi(P, start, K, B, nthreads=16, log_cap=1 << 20)
    first = len(step_ref(x, y, start, K.view(np.int32), B, 0))
    assert first >= 2  # the first step applies several moves, so the budgets below cut it
    for m in (1, 2, first - 1, first, first + 1, fst.moves // 2, fst.moves - 1):
        t, st, mv = prob.local_search(T.ALGO_OR_OPT_NEIGHBOR_MULTI, start, max_moves=m, log_cap=1 << 20)
        assert same_moves(mv, full_m[:m]) and int(st.moves) == m and st.converged == 0, m
        assert (t.astype(np.int64) == replay(start, full_m[:m])).all()
    # two session runs with cumulative budgets a and a + b against the oracle resumed with step0
    for a, b in ((2, first), (first + 3, 50), (fst.moves // 3, fst.moves // 3)):
        s = prob.session(T.ALGO_OR_OPT_NEIGHBOR_MULTI, start)
        s.run(a)
        s.run(a + b)
        ta, sa, ma, _ = NL.or_opt_nl_multi(P, start, K, B, max_moves=a, nthreads=16, log_cap=1 << 20)
        tb, sb, mb, _ = NL.or_opt_nl_multi(P, ta, K, B, step0=sa.passes, max_moves=b, nthreads=16, log_cap=1 << 20)
        st = s.stats()
        assert same_moves(s.log(1 << 20), ma + mb) and (s.tour().astype(np.int64) == tb).all()
        assert (int(st.moves), int(st.passes)) == (a + b, sa.passes + sb.passes)
        got = s.scan()  # G of the current tour, as Or-opt N's scan finds it
        want, _ = NL.or_opt_nl_scan(P, tb, K)
        assert key(got) == key(want)
        s.run(-1)
        assert s.stats().converged == 1 and s.scan() is None
        s.close()
    # a log shorter than the move count keeps the first entries
    t, st, mv = prob.local_search(T.ALGO_OR_OPT_NEIGHBOR_MULTI, start, log_cap=10)
    assert same_moves(mv, full_m[:10]) and int(st.moves) == fst.moves and (t.astype(np.int64) == full_t).all()


@pytest.mark.gpu
def test_gpu_small_and_errors(ctx):
    import teeline_b200 as T
    x, y = O.gen_uniform(50, 50)
    for n in (2, 3):
        small = T.Problem.euc2d(ctx, x[:n], y[:n])
        t, st, _ = small.local_search(T.ALGO_OR_OPT_NEIGHBOR_MULTI, np.arange(n)[::-1])
        assert t.tolist() == list(range(n)) and int(st.moves) == 0 and int(st.passes) == 0 and st.converged == 1
    ex = T.Problem.explicit(ctx, O.matrix_packed_f32(x, y), 50)
    with pytest.raises(T.TeelineError) as ei:
        ex.session(T.ALGO_OR_OPT_NEIGHBOR_MULTI, np.arange(50))
    assert ei.value.status == 3
    prob = T.Problem.euc2d(ctx, x, y)
    with pytest.raises(T.TeelineError) as ei:
        prob.session(T.ALGO_OR_OPT_NEIGHBOR_MULTI, np.arange(50), path=T.PATH_MATRIX)
    assert ei.value.status == 3
    s = prob.session(T.ALGO_OR_OPT_NEIGHBOR_MULTI, np.arange(50))
    with pytest.raises(T.TeelineError) as ei:
        s.set_shard(0, 2)
    assert ei.value.status == 3


@pytest.mark.gpu
def test_gpu_block_size_must_be_a_power_of_two_up_to_16384(ctx, monkeypatch):
    import teeline_b200 as T
    x, y = O.gen_uniform(50, 50)
    prob = T.Problem.euc2d(ctx, x, y)
    for bad in ("48", "1", "32768"):
        monkeypatch.setenv("TL_MULTI_BLOCK", bad)
        with pytest.raises(T.TeelineError) as ei:
            prob.session(T.ALGO_OR_OPT_NEIGHBOR_MULTI, np.arange(50))
        assert ei.value.status == 1
    monkeypatch.setenv("TL_MULTI_BLOCK", "16384")
    prob.session(T.ALGO_OR_OPT_NEIGHBOR_MULTI, np.arange(50)).close()


@pytest.mark.gpu
def test_gpu_million_cities_from_mode_nm_greedy(ctx):
    import teeline_b200 as T
    n = 1_000_000
    x, y = O.gen_uniform(n, n)
    # nint: converged, and the length falls by exactly the logged deltas
    prob = T.Problem.euc2d(ctx, x, y, T.DIST_NINT_I32)
    prob.set_candidates(8)
    g, _ = prob.greedy_tour()
    start = prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR_MULTI, g)[0]
    t, st, mv = prob.local_search(T.ALGO_OR_OPT_NEIGHBOR_MULTI, start, log_cap=1 << 22)
    assert st.converged == 1 and len(mv) == int(st.moves) and sorted(t.tolist()) == list(range(n))
    assert int(prob.tour_lengths(start)[0]) + int(sum(m[0] for m in mv)) == int(prob.tour_lengths(t)[0])
    assert prob.session(T.ALGO_OR_OPT_NEIGHBOR, t).scan() is None
    prob.close()
    # f32: GPU and oracle Or-opt N scans of the result find nothing, in fewer scans than GPU Or-opt N
    P = O.Problem(x, y)
    prob = T.Problem.euc2d(ctx, x, y)
    prob.set_candidates(8)
    K = prob.knn(8)
    g, _ = prob.greedy_tour()
    start = prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR_MULTI, g)[0]
    t, st, _ = prob.local_search(T.ALGO_OR_OPT_NEIGHBOR_MULTI, start)
    assert st.converged == 1 and sorted(t.tolist()) == list(range(n))
    assert prob.session(T.ALGO_OR_OPT_NEIGHBOR, t).scan() is None
    assert NL.or_opt_nl_scan(P, t, K, nthreads=16)[0] is None
    _, sn, _ = prob.local_search(T.ALGO_OR_OPT_NEIGHBOR, start)
    assert int(st.passes) < int(sn.passes)
    prob.close()


@pytest.mark.gpu
def test_gpu_cli_neighbor_multi(ctx, cli, tmp_path):
    import teeline_b200 as T
    inp = os.path.join(GOLDEN, "att532.tsp")
    ids, x, y = O.read_tsplib_coords(inp)
    P = O.Problem(x, y)
    K = O.knn(P, 8)
    tn, _, _, _ = NL.or_opt_nl_multi(P, O.nn_tour(P, 3), K, T.OR_MULTI_BLOCK)  # `solve` starts from the NN tour
    tg, _, _, _ = NL.two_opt_nl_multi(P, NL.greedy_lazy(x, y), K, T.MULTI_BLOCK)
    tp, _, _, _ = NL.or_opt_nl_multi(P, tg, K, T.OR_MULTI_BLOCK)
    cfg = tmp_path / "onm.toml"
    cfg.write_text("[[stage]]\nsolver = \"greedy_edge\"\n[stage.cuda]\ncandidates = 8\n"
                   "[[stage]]\nsolver = \"2opt\"\n[stage.cuda]\nmode = \"neighbor_multi\"\ncandidates = 8\n"
                   "[[stage]]\nsolver = \"or_opt\"\n[stage.cuda]\nmode = \"neighbor_multi\"\ncandidates = 8\n")
    for argv, want in ((["solve", "or_opt", "--mode", "neighbor_multi", "--candidates", "8"], tn),
                       (["pipeline", "--config", str(cfg)], tp)):
        rc, out, err = run([cli] + argv + ["-i", inp])
        assert rc == 0, err
        second = out.strip().split("\n")[1]
        assert [int(v) for v in second.split()] == [int(ids[p]) for p in want], argv
