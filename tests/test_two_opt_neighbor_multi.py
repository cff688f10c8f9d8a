"""Multi-move candidate-list 2-opt ("Mode NM", TL_ALGO_TWO_OPT_NEIGHBOR_MULTI).

CPU: the Mode NM oracle (oracle_nl) against Mode N's when one block covers the tour, against an independent
numpy restatement of a step, and on its own properties (disjoint moves, exact length change, Mode N local
optimum, budgets, thread count); the ABI and the CLI without a device.  GPU: the library bit for bit against
the oracle (move log, tour, moves / scans / evals) with the built block size and with small blocks, Mode N on
the GPU for n <= TL_MULTI_BLOCK/2, budgets and resumed sessions, 10^6 cities from the greedy tour, and the CLI.
The nint oracle needs the packed triangle, so nint runs stop at 10^4 cities against it."""
import os
import subprocess

import numpy as np
import pytest

import oracle as O
import oracle_nl as NL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def f32_bits(v):
    return np.float32(v).view(np.uint32)


def same_moves(got, want):
    """GPU log (f32 delta) against the oracle's (widened delta): (delta bits, i, j) per move."""
    return [(int(f32_bits(m[0])), m[1], m[2]) for m in got] == [(int(f32_bits(m[0])), m[1], m[2]) for m in want]


def replay(start, moves):
    cur = np.asarray(start).copy()
    for _, i, j, _, _ in moves:
        cur = O.swap_2opt(cur, i + 1, j)
    return cur


def oracle_problem(x, y, metric):
    return O.Problem(tri=O.matrix_packed_nint(x, y), n=len(x)) if metric == "nint" else O.Problem(x, y)


def step_ref(x, y, tour, K, block, t):
    """One Mode NM step restated with numpy (f32 metric): the moves it applies, in log order."""
    n = len(tour)
    tour = np.asarray(tour, dtype=np.int64)
    pos = np.empty(n, dtype=np.int64)
    pos[tour] = np.arange(n)
    i = np.repeat(np.arange(n), K.shape[1])
    b = K[tour].reshape(-1).astype(np.int64)
    keep = b >= 0
    i, j = i[keep], pos[b[keep]]
    lo, hi = np.minimum(i, j), np.maximum(i, j)
    ok = hi >= lo + 2
    lo, hi = lo[ok], hi[ok]
    pi = np.concatenate([lo[hi <= n - 2], lo[lo >= 1] - 1])
    pj = np.concatenate([hi[hi <= n - 2], hi[lo >= 1] - 1])

    def d(a, c):
        dx = (x[tour[a]] - x[tour[c]]).astype(np.float32)
        dy = (y[tour[a]] - y[tour[c]]).astype(np.float32)
        return np.sqrt(dx * dx + dy * dy, dtype=np.float32)

    delta = (d(pi, pj) + d(pi + 1, pj + 1)) - (d(pi, pi + 1) + d(pj, pj + 1))
    imp = delta < 0
    delta, pi, pj = delta[imp], pi[imp], pj[imp]
    if len(delta) == 0:
        return []
    order = np.lexsort((pj, pi, delta))
    delta, pi, pj = delta[order], pi[order], pj[order]
    gi, gj = pi[0], pj[0]
    off = (t % 2) * (block // 2)
    blk = (pi + off) // block
    inb = blk == (pj + 1 + off) // block
    _, first = np.unique(blk[inb], return_index=True)  # sorted by (delta, i, j): first per block is its best
    bi, bj, bd = pi[inb][first], pj[inb][first], delta[inb][first]
    acc = ~((bi == gi) & (bj == gj)) & ((bj < gi) | (bi > gj))
    rest = sorted(zip(bi[acc].tolist(), bj[acc].tolist(), bd[acc].tolist()))
    return [(float(delta[0]), int(gi), int(gj))] + [(float(dd), ii, jj) for ii, jj, dd in rest]


def next_pow2(v):
    return 1 << max(1, (v - 1).bit_length())


# ---- CPU: the oracle ------------------------------------------------------------------------------------

@pytest.mark.parametrize("n", list(range(4, 34)) + [1000])
@pytest.mark.parametrize("metric", ["f32", "nint"])
def test_oracle_one_block_is_mode_n(n, metric):
    x, y = O.gen_uniform(n, 500 + n)
    P = oracle_problem(x, y, metric)
    K = O.knn(O.Problem(x, y) if metric == "f32" else P, min(8, n - 1))
    start = O.shuffle_tour(n, 9 + n)
    tn, sn, mn = NL.two_opt_nl(P, start, K, log_cap=1 << 14)
    for block in (next_pow2(2 * n), 4 * next_pow2(2 * n)):
        tm, sm, mm, conv = NL.two_opt_nl_multi(P, start, K, block, log_cap=1 << 14)
        assert mm == mn and (tm == tn).all() and conv == 1
        assert (sm.moves, sm.passes, sm.evals) == (sn.moves, sn.passes, sn.evals)


@pytest.fixture(scope="module")
def inst20k():
    n = 20000
    x, y = O.gen_uniform(n, n)
    P = O.Problem(x, y)
    return x, y, P, O.knn(P, 8), NL.greedy_lazy(x, y)


@pytest.mark.parametrize("block", [256, 1024])
def test_oracle_properties_20k(inst20k, block):
    x, y, P, K, start = inst20k
    t, st, moves, conv = NL.two_opt_nl_multi(P, start, K, block, nthreads=8, log_cap=1 << 16)
    assert conv == 1 and st.moves == len(moves) and sorted(t.tolist()) == list(range(len(x)))
    # step by step against the numpy restatement: G first, then disjoint block bests by increasing i
    cur, at, steps = start.copy(), 0, 0
    while True:
        want = step_ref(x, y, cur, K, block, steps)
        if not want:
            break
        got = moves[at:at + len(want)]
        assert [(int(f32_bits(m[0])), m[1], m[2]) for m in got] == [(int(f32_bits(d)), i, j) for d, i, j in want], steps
        spans = sorted((i, j + 1) for _, i, j in want)
        assert all(a[1] <= b[0] for a, b in zip(spans, spans[1:]))  # at most an end position in common
        assert all(d < 0 for d, _, _ in want)
        cur = replay(cur, got)
        at += len(want)
        steps += 1
    assert at == len(moves) and st.passes == steps + 1 and (cur == t).all()
    assert NL.two_opt_nl_scan(P, t, K, nthreads=8)[0] is None
    assert steps < NL.two_opt_nl(P, start, K, nthreads=8)[1].passes
    # f32: the length falls by the logged deltas up to the rounding of each edge sum
    drop = O.tour_length(P, start) - O.tour_length(P, t)
    assert abs(drop + sum(m[0] for m in moves)) < 1e-3 * abs(drop)
    # budgets: the first m moves of the unbudgeted log, and the tour they give
    for m in (1, 2, 3, len(step_ref(x, y, start, K, block, 0)) - 1, 500, st.moves - 1):
        tb, sb, mb, cb = NL.two_opt_nl_multi(P, start, K, block, max_moves=m, nthreads=8, log_cap=1 << 16)
        assert mb == moves[:m] and sb.moves == m and cb == 0 and (tb == replay(start, moves[:m])).all()
    # thread count
    t1, s1, m1, _ = NL.two_opt_nl_multi(P, start, K, block, nthreads=1, log_cap=1 << 16)
    assert m1 == moves and (t1 == t).all() and (s1.passes, s1.evals) == (st.passes, st.evals)


def test_oracle_nint_length_exact_and_resume():
    n = 10000
    x, y = O.gen_uniform(n, 3 * n)
    P = oracle_problem(x, y, "nint")
    K = O.knn(P, 8)
    start = O.shuffle_tour(n, 5)
    t, st, moves, conv = NL.two_opt_nl_multi(P, start, K, 256, nthreads=8, log_cap=1 << 20)
    assert conv == 1 and all(m[0] < 0 and m[0] == int(m[0]) for m in moves)
    assert int(O.tour_length(P, start)) + int(sum(m[0] for m in moves)) == int(O.tour_length(P, t))
    assert NL.two_opt_nl_scan(P, t, K, nthreads=8)[0] is None
    # budget a at the end of a step, then b more from that tour with the step count carried over: the
    # unbudgeted log (a resumed search starts a new step, so a cut inside a step would not give it)
    a = next(a for a in range(777, 2000)
             if NL.two_opt_nl_multi(P, start, K, 256, max_moves=a + 1, nthreads=8)[1].passes >
             NL.two_opt_nl_multi(P, start, K, 256, max_moves=a, nthreads=8)[1].passes)
    b = 1234
    ta, sa, ma, _ = NL.two_opt_nl_multi(P, start, K, 256, max_moves=a, nthreads=8, log_cap=1 << 20)
    tb, sb, mb, _ = NL.two_opt_nl_multi(P, ta, K, 256, step0=sa.passes, max_moves=b, nthreads=8, log_cap=1 << 20)
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
    assert T.ALGO_TWO_OPT_NEIGHBOR_MULTI == 9 and T.MULTI_BLOCK == 4096
    hdr = open(os.path.join(ROOT, "include", "teeline_cuda.h")).read()
    assert "TL_ALGO_TWO_OPT_NEIGHBOR_MULTI = 9" in hdr and "#define TL_MULTI_BLOCK 4096" in hdr


def test_cli_without_device(cli, tmp_path):
    import torch
    rc, out, _ = run([cli, "solvers"])
    assert rc == 0 and "2opt --mode neighbor_multi" in out
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    inp = os.path.join(GOLDEN, "berlin52.tsp")
    rc, out, err = run([cli, "solve", "2opt", "--mode", "neighbor_multi", "--candidates", "8", "-i", inp])
    assert rc == 101 and out == "" and "no CPU fallback" in err
    cfg = tmp_path / "nm.toml"
    cfg.write_text("[[stage]]\nsolver = \"greedy_edge\"\n[[stage]]\nsolver = \"2opt\"\n[stage.cuda]\n"
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
    if name == "berlin52":
        _, x, y = O.read_tsplib_coords(os.path.join(GOLDEN, "berlin52.tsp"))
    elif name == "att532":
        _, x, y = O.read_tsplib_coords(os.path.join(GOLDEN, "att532.tsp"))
    else:
        x, y = O.gen_uniform(int(name), 7000 + int(name))
    return x, y


def gpu_vs_oracle(ctx, x, y, metric, k, start, block=None):
    import teeline_b200 as T
    n = len(x)
    prob = T.Problem.euc2d(ctx, x, y, T.DIST_NINT_I32 if metric == "nint" else T.DIST_F32_EXACT)
    P = O.Problem(x, y) if metric == "f32" else oracle_problem(x, y, metric)
    K = prob.knn(k)
    prob.set_candidates(k)
    cap = 1 << 20
    got_t, st, got_m = prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR_MULTI, start, log_cap=cap)
    want_t, wst, want_m, conv = NL.two_opt_nl_multi(P, start, K, block or T.MULTI_BLOCK, nthreads=16, log_cap=cap)
    assert same_moves(got_m, want_m), (n, metric, k)
    assert (got_t.astype(np.int64) == want_t).all()
    assert (int(st.moves), int(st.passes), int(st.evals)) == (wst.moves, wst.passes, wst.evals)
    assert st.converged == 1 == conv and st.path_used == T.PATH_RECOMPUTE
    return prob, got_t, wst


def starts(x, y, metric):
    return NL.greedy_lazy(x, y, metric), O.nn_tour(O.Problem(x, y), 3)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["4", "5", "6", "7", "13", "20", "33", "257", "1000", "berlin52", "att532"])
@pytest.mark.parametrize("metric", ["f32", "nint"])
def test_gpu_equals_oracle(ctx, name, metric):
    x, y = instance(name)
    for k in (5, 8, 10):
        for start in starts(x, y, metric):
            gpu_vs_oracle(ctx, x, y, metric, k, start)


@pytest.mark.gpu
@pytest.mark.parametrize("block", ["8", "64", "256"])
@pytest.mark.parametrize("n", [1000, 5000])
def test_gpu_equals_oracle_small_blocks(ctx, monkeypatch, block, n):
    """Many blocks: boundaries, both offsets and moves that straddle a boundary."""
    monkeypatch.setenv("TL_MULTI_BLOCK", block)
    x, y = O.gen_uniform(n, 3 * n)
    for metric in ("f32", "nint"):
        for start in starts(x, y, metric):
            gpu_vs_oracle(ctx, x, y, metric, 8, start, block=int(block))


@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["f32", "nint"])
def test_gpu_equals_oracle_10k(ctx, metric):
    x, y = O.gen_uniform(10000, 10000)
    for start in starts(x, y, metric):
        gpu_vs_oracle(ctx, x, y, metric, 8, start)


@pytest.mark.gpu
def test_gpu_equals_oracle_100k(ctx):
    x, y = O.gen_uniform(100_000, 100_000)
    gpu_vs_oracle(ctx, x, y, "f32", 8, NL.greedy_lazy(x, y))


@pytest.mark.gpu
def test_gpu_ties_on_a_lattice(ctx):
    side = 24
    q = np.arange(side * side)
    lattice = ((q % side).astype(np.float32), (q // side).astype(np.float32))
    for x, y in (lattice, O.gen_grid(900, 900)):
        for metric in ("f32", "nint"):
            for k in (3, 8):
                gpu_vs_oracle(ctx, x, y, metric, k, O.shuffle_tour(len(x), 3))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [13, 257, 2048])
def test_gpu_half_block_is_gpu_mode_n(ctx, n):
    import teeline_b200 as T
    x, y = O.gen_uniform(n, 40 + n)
    prob = T.Problem.euc2d(ctx, x, y)
    prob.set_candidates(8)
    for start in (prob.nn_tour(3), O.shuffle_tour(n, n)):
        tn, sn, mn = prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR, start, log_cap=1 << 14)
        tm, sm, mm = prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR_MULTI, start, log_cap=1 << 14)
        assert mm == mn and (tm == tn).all() and (sm.moves, sm.passes, sm.evals) == (sn.moves, sn.passes, sn.evals)


@pytest.mark.gpu
@pytest.mark.parametrize("block", [None, "64"])
def test_gpu_budgets_resume_and_log_cap(ctx, monkeypatch, block):
    import teeline_b200 as T
    if block:
        monkeypatch.setenv("TL_MULTI_BLOCK", block)
    B = int(block) if block else T.MULTI_BLOCK
    n = 20000
    x, y = O.gen_uniform(n, 11 * n)
    P = O.Problem(x, y)
    prob = T.Problem.euc2d(ctx, x, y)
    prob.set_candidates(8)
    K = prob.knn(8)
    start = O.nn_tour(P, 3)
    full_t, fst, full_m, _ = NL.two_opt_nl_multi(P, start, K, B, nthreads=8, log_cap=1 << 20)
    first = len(step_ref(x, y, start, K, B, 0))
    assert first >= 3  # the first step applies several moves, so the budgets below cut it
    for m in (1, 2, first - 1, first, first + 1, fst.moves // 2, fst.moves - 1):
        t, st, mv = prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR_MULTI, start, max_moves=m, log_cap=1 << 20)
        assert same_moves(mv, full_m[:m]) and int(st.moves) == m and st.converged == 0, m
        assert (t.astype(np.int64) == replay(start, full_m[:m])).all()
    # two session runs with cumulative budgets a and a + b against the oracle resumed with step0
    for a, b in ((2, first), (first + 3, 50), (fst.moves // 3, fst.moves // 3)):
        s = prob.session(T.ALGO_TWO_OPT_NEIGHBOR_MULTI, start)
        s.run(a)
        s.run(a + b)
        ta, sa, ma, _ = NL.two_opt_nl_multi(P, start, K, B, max_moves=a, nthreads=8, log_cap=1 << 20)
        tb, sb, mb, _ = NL.two_opt_nl_multi(P, ta, K, B, step0=sa.passes, max_moves=b, nthreads=8, log_cap=1 << 20)
        st = s.stats()
        assert same_moves(s.log(1 << 20), ma + mb) and (s.tour().astype(np.int64) == tb).all()
        assert (int(st.moves), int(st.passes)) == (a + b, sa.passes + sb.passes)
        first_scan = s.scan()  # G of the current tour, as Mode N's scan finds it
        want, _ = NL.two_opt_nl_scan(P, tb, K)
        assert (int(f32_bits(first_scan[0])), first_scan[1], first_scan[2]) == (int(f32_bits(want[0])), want[1], want[2])
        s.run(-1)
        assert s.stats().converged == 1 and s.scan() is None
        s.close()
    # a log shorter than the move count keeps the first entries
    t, st, mv = prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR_MULTI, start, log_cap=10)
    assert same_moves(mv, full_m[:10]) and int(st.moves) == fst.moves and (t.astype(np.int64) == full_t).all()


@pytest.mark.gpu
def test_gpu_small_and_errors(ctx):
    import teeline_b200 as T
    x, y = O.gen_uniform(50, 50)
    for n in (2, 3):
        small = T.Problem.euc2d(ctx, x[:n], y[:n])
        t, st, _ = small.local_search(T.ALGO_TWO_OPT_NEIGHBOR_MULTI, np.arange(n)[::-1])
        assert t.tolist() == list(range(n)) and int(st.moves) == 0 and int(st.passes) == 0 and st.converged == 1
    ex = T.Problem.explicit(ctx, O.matrix_packed_f32(x, y), 50)
    with pytest.raises(T.TeelineError) as ei:
        ex.session(T.ALGO_TWO_OPT_NEIGHBOR_MULTI, np.arange(50))
    assert ei.value.status == 3
    prob = T.Problem.euc2d(ctx, x, y)
    with pytest.raises(T.TeelineError) as ei:
        prob.session(T.ALGO_TWO_OPT_NEIGHBOR_MULTI, np.arange(50), path=T.PATH_MATRIX)
    assert ei.value.status == 3
    s = prob.session(T.ALGO_TWO_OPT_NEIGHBOR_MULTI, np.arange(50))
    with pytest.raises(T.TeelineError) as ei:
        s.set_shard(0, 2)
    assert ei.value.status == 3


@pytest.mark.gpu
def test_gpu_block_size_must_be_a_power_of_two(ctx, monkeypatch):
    import teeline_b200 as T
    x, y = O.gen_uniform(50, 50)
    prob = T.Problem.euc2d(ctx, x, y)
    for bad in ("48", "1", "131072"):
        monkeypatch.setenv("TL_MULTI_BLOCK", bad)
        with pytest.raises(T.TeelineError) as ei:
            prob.session(T.ALGO_TWO_OPT_NEIGHBOR_MULTI, np.arange(50))
        assert ei.value.status == 1


@pytest.mark.gpu
def test_gpu_million_cities_greedy_start(ctx):
    import teeline_b200 as T
    n = 1_000_000
    x, y = O.gen_uniform(n, n)
    # nint: the length falls by exactly the logged deltas
    prob = T.Problem.euc2d(ctx, x, y, T.DIST_NINT_I32)
    prob.set_candidates(8)
    start, _ = prob.greedy_tour()
    t, st, mv = prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR_MULTI, start, log_cap=1 << 22)
    assert st.converged == 1 and len(mv) == int(st.moves) and sorted(t.tolist()) == list(range(n))
    assert int(prob.tour_lengths(start)[0]) + int(sum(m[0] for m in mv)) == int(prob.tour_lengths(t)[0])
    assert prob.session(T.ALGO_TWO_OPT_NEIGHBOR, t).scan() is None
    # f32: the oracle's scan of the result, and fewer steps than Mode N
    P = O.Problem(x, y)
    prob = T.Problem.euc2d(ctx, x, y)
    prob.set_candidates(8)
    K = prob.knn(8)
    start, _ = prob.greedy_tour()
    t, st, mv = prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR_MULTI, start, log_cap=1 << 22)
    assert st.converged == 1 and sorted(t.tolist()) == list(range(n))
    assert prob.session(T.ALGO_TWO_OPT_NEIGHBOR, t).scan() is None
    assert NL.two_opt_nl_scan(P, t, K, nthreads=16)[0] is None
    def length64(tour):  # f64 sum of the f32 edge lengths
        a, b = tour, np.roll(tour, -1)
        dx, dy = (x[a] - x[b]).astype(np.float32), (y[a] - y[b]).astype(np.float32)
        return np.sqrt(dx * dx + dy * dy, dtype=np.float32).astype(np.float64).sum()

    drop = length64(start) - length64(t)
    assert abs(drop + sum(m[0] for m in mv)) < 1e-4 * drop
    _, sn, _ = prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR, start)
    assert int(st.passes) < int(sn.passes)


@pytest.mark.gpu
def test_gpu_cli_neighbor_multi(ctx, cli, tmp_path):
    import teeline_b200 as T
    inp = os.path.join(GOLDEN, "att532.tsp")
    ids, x, y = O.read_tsplib_coords(inp)
    P = O.Problem(x, y)
    K = O.knn(P, 8)
    tm, _, _, _ = NL.two_opt_nl_multi(P, O.nn_tour(P, 3), K, T.MULTI_BLOCK)  # `solve` starts from the NN tour
    g = NL.greedy_lazy(x, y)
    tg, _, _, _ = NL.two_opt_nl_multi(P, g, K, T.MULTI_BLOCK)
    tp, _, _ = NL.or_opt_nl(P, tg, K)
    cfg = tmp_path / "nm.toml"
    cfg.write_text("[[stage]]\nsolver = \"greedy_edge\"\n[stage.cuda]\ncandidates = 8\n"
                   "[[stage]]\nsolver = \"2opt\"\n[stage.cuda]\nmode = \"neighbor_multi\"\ncandidates = 8\n"
                   "[[stage]]\nsolver = \"or_opt\"\n[stage.cuda]\nmode = \"neighbor\"\ncandidates = 8\n")
    for argv, want in ((["solve", "2opt", "--mode", "neighbor_multi", "--candidates", "8"], tm),
                       (["pipeline", "--config", str(cfg)], tp)):
        rc, out, err = run([cli] + argv + ["-i", inp])
        assert rc == 0, err
        second = out.strip().split("\n")[1]
        assert [int(v) for v in second.split()] == [int(ids[p]) for p in want], argv
