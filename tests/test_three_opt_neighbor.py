"""Candidate-list best-improvement 3-opt ("3-opt N", TL_ALGO_THREE_OPT_NEIGHBOR).

CPU: the 3-opt N oracle (oracle_nl) against 3-opt's for k >= n-1 and on its own properties, the ABI and
the CLI without a device.  GPU: the library bit for bit against the oracle (move log, tour, moves /
scans / evals), GPU 3-opt for k >= n-1, every metric, ties, both relocation routes, budgets, 10^4 to
10^6 cities, errors and the CLI."""
import os
import subprocess

import numpy as np
import pytest

import oracle as O
import oracle_nl as NL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
CTA_SPAN = 4096  # kOrNlCtaSpan (csrc/kernels.cuh): longer spans are relocated by the apply grids


def f32_bits(v):
    return int(np.float32(v).view(np.uint32))


def key(moves):
    """(delta bits, i, j, k, case) per move: GPU logs carry f32 deltas, the oracle widened ones."""
    return [(f32_bits(m[0]),) + tuple(int(v) for v in m[1:5]) for m in moves]


def oracle_problem(x, y, metric):
    return O.Problem(tri=O.matrix_packed_nint(x, y), n=len(x)) if metric == "nint" else O.Problem(x, y)


def generated(tour, K, i, j, k):
    """Whether the rule generates the triple (i, j, k) on this tour, restated independently of the oracle:
    the three cut edges, in some order (e1, e2, e3), are an edge at c, an edge at b with b a candidate of
    c, and an edge at b' with b' a candidate of t, the other endpoint of the edge at b."""
    n = len(tour)
    ends = {e: (int(tour[e]), int(tour[(e + 1) % n])) for e in (i, j, k)}
    for e1, e2, e3 in ((i, j, k), (i, k, j), (j, i, k), (j, k, i), (k, i, j), (k, j, i)):
        for c in ends[e1]:
            for b in ends[e2]:
                if b not in K[c]:
                    continue
                t = ends[e2][1] if b == ends[e2][0] else ends[e2][0]
                if any(b2 in K[t] for b2 in ends[e3]):
                    return True
    return False


# ---- CPU: the oracle ------------------------------------------------------------------------------------

@pytest.mark.parametrize("n", [4, 5, 6, 7, 13, 20, 33])
@pytest.mark.parametrize("metric", ["f32", "nint"])
def test_oracle_all_candidates_is_three_opt(n, metric):
    x, y = O.gen_uniform(n, 100 + n)
    P = oracle_problem(x, y, metric)
    K = O.knn(O.Problem(x, y), n - 1)
    for start in (O.shuffle_tour(n, 7 + n), O.nn_tour(O.Problem(x, y), 3)):
        to, so, mo = O.three_opt(P, start, log_cap=1000)
        tn, sn, mn = NL.three_opt_nl(P, start, K, log_cap=1000)
        assert mn == mo and (tn == to).all() and (sn.moves, sn.passes) == (so.moves, so.passes)


def test_oracle_properties_1000():
    x, y = O.gen_uniform(1000, 1000)
    P = O.Problem(x, y)
    start = O.nn_tour(P, 3)
    K = O.knn(P, 8)
    Ks = [set(int(v) for v in row if v >= 0) for row in K]
    t, st, moves = NL.three_opt_nl(P, start, K, nthreads=8, log_cap=1 << 16)
    assert st.moves > 0 and st.passes == st.moves + 1 and sorted(t.tolist()) == list(range(1000))
    cur = start.copy()
    for m in moves:
        delta, i, j, k, case = m
        assert delta < 0 and 0 <= i < j < k < 1000 and not (i == 0 and k == 999) and 1 <= case <= 7
        assert generated(cur, Ks, i, j, k), m
        cur = O.three_opt_apply(cur, i, j, k, case)
    assert (cur == t).all()
    assert NL.three_opt_nl_scan(P, t, K, nthreads=8)[0] is None


# ---- CPU: ABI and CLI without a device --------------------------------------------------------------------

@pytest.fixture(scope="module")
def cli():
    from teeline_b200 import build as tb, build_host
    tb.build()
    return build_host.build()


def run(cmd):
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    return p.returncode, p.stdout, p.stderr


def test_abi_constant():
    import teeline_b200 as T
    assert T.ALGO_THREE_OPT_NEIGHBOR == 8
    hdr = open(os.path.join(ROOT, "include", "teeline_cuda.h")).read()
    assert "TL_ALGO_THREE_OPT_NEIGHBOR = 8" in hdr


def test_no_device_fails_loudly(cli):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    rc, out, err = run([cli, "solve", "3opt", "--mode", "neighbor", "--candidates", "8",
                        "-i", os.path.join(GOLDEN, "berlin52.tsp")])
    assert rc == 101 and out == "" and "no CPU fallback" in err


def test_cli_candidates_argument_and_solvers(cli, tmp_path):
    inp = os.path.join(GOLDEN, "berlin52.tsp")
    for bad in ("0", "33", "x", "-1"):
        rc, _, err = run([cli, "solve", "3opt", "--mode", "neighbor", "--candidates", bad, "-i", inp])
        assert rc == 2 and "--candidates" in err, (bad, err)
    rc, out, _ = run([cli, "solvers"])
    assert rc == 0 and "3opt --mode neighbor" in out
    f = tmp_path / "c.toml"
    f.write_text("[[stage]]\nsolver = \"3opt\"\n[stage.cuda]\nmode = \"neighbor\"\ncandidates = 33\n")
    rc, _, err = run([cli, "pipeline", "--config", str(f), "-i", inp])
    assert rc == 1 and "config: [cuda] candidates must be in 1..32" in err, err


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


def problem(ctx, x, y, metric):
    import teeline_b200 as T
    return T.Problem.euc2d(ctx, x, y, T.DIST_NINT_I32 if metric == "nint" else T.DIST_F32_EXACT)


def gpu_vs_oracle(ctx, x, y, metric, k, start, P=None, prob=None, max_moves=-1):
    """One local search on both sides.  max_moves bounds the oracle's time on long searches (the CPU
    oracle evaluates 8 n k^2 chains per scan); the run is then compared up to the budget."""
    import teeline_b200 as T
    prob = prob or problem(ctx, x, y, metric)
    P = P or oracle_problem(x, y, metric)
    K = prob.knn(k)
    prob.set_candidates(k)
    cap = 1 << 18
    got_t, st, got_m = prob.local_search(T.ALGO_THREE_OPT_NEIGHBOR, start, max_moves=max_moves, log_cap=cap)
    want_t, wst, want_m = NL.three_opt_nl(P, start, K, max_moves=max_moves, nthreads=16, log_cap=cap)
    assert key(got_m) == key(want_m), (len(x), metric, k)
    assert (got_t.astype(np.int64) == want_t).all()
    assert (int(st.moves), int(st.passes), int(st.evals)) == (wst.moves, wst.passes, wst.evals)
    assert st.converged == (1 if max_moves < 0 or wst.moves < max_moves else 0)
    assert st.path_used == T.PATH_RECOMPUTE
    return got_t, got_m


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["4", "5", "6", "7", "13", "33", "257", "1000", "berlin52", "att532"])
@pytest.mark.parametrize("metric", ["f32", "nint"])
def test_gpu_equals_oracle(ctx, name, metric):
    x, y = instance(name)
    n = len(x)
    Pf = O.Problem(x, y)
    P = oracle_problem(x, y, metric)
    prob = problem(ctx, x, y, metric)
    for k in (1, 3, 8, 32):
        for start in (O.nn_tour(Pf, 3), O.shuffle_tour(n, 11 + n)):
            # k = 32 from a shuffled start takes ~n moves of 8 n k^2 chains each on the CPU side
            gpu_vs_oracle(ctx, x, y, metric, k, start, P, prob, max_moves=150 if n >= 500 and k == 32 else -1)


def or_opt_n_optimum(prob, k):
    """The nn -> Mode N -> Or-opt N pipeline's result: 3-opt N's real input."""
    import teeline_b200 as T
    prob.set_candidates(k)
    t, _, _ = prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR, prob.nn_tour(3))
    t, st, _ = prob.local_search(T.ALGO_OR_OPT_NEIGHBOR, t)
    assert st.converged == 1
    return t


@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["f32", "nint"])
def test_gpu_equals_oracle_10k(ctx, metric):
    x, y = O.gen_uniform(10000, 10000)
    prob = problem(ctx, x, y, metric)
    gpu_vs_oracle(ctx, x, y, metric, 8, or_opt_n_optimum(prob, 8), prob=prob)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4, 5, 6, 7, 13, 20, 33])
@pytest.mark.parametrize("metric", ["f32", "nint"])
def test_gpu_all_candidates_is_gpu_three_opt(ctx, n, metric):
    import teeline_b200 as T
    x, y = O.gen_uniform(n, 300 + n)
    prob = problem(ctx, x, y, metric)
    prob.set_candidates(min(32, n - 1))
    for start in (O.shuffle_tour(n, 5 + n), O.nn_tour(O.Problem(x, y), 3)):
        # 3-opt runs on the recompute path for f32 and on the matrix path for nint
        to, so, mo = prob.local_search(T.ALGO_THREE_OPT, start, log_cap=1000)
        tn, sn, mn = prob.local_search(T.ALGO_THREE_OPT_NEIGHBOR, start, log_cap=1000)
        assert mn == mo and (tn == to).all() and (sn.moves, sn.passes) == (so.moves, so.passes)


def regime(x, y, metric):
    """The distance code these coordinates select (api.cu: coords_allow_fast_sqrt, coords_allow_grid_nint)."""
    c = np.abs(np.concatenate([x, y]).astype(np.float64))
    if metric == "f32":
        fast = bool(np.isfinite(c).all() and (c < 2.0 ** 62).all() and ((c == 0) | (c >= 2.0 ** -27)).all())
        return "f32-fast" if fast else "f32-safe"
    grid = (bool((np.floor(c) == c).all()) and bool((c <= 2.0 ** 22).all())
            and float(x.max()) - float(x.min()) <= 2.0 ** 20 and float(y.max()) - float(y.min()) <= 2.0 ** 20)
    return "nint-grid" if grid else "nint-f64"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["f32-fast", "f32-safe", "nint-grid", "nint-f64"])
def test_gpu_every_metric(ctx, name):
    n = 1500
    bx, by = O.gen_uniform(n, 31)
    metric = "nint" if name.startswith("nint") else "f32"
    if name == "f32-safe":
        x, y = np.ldexp(bx, -70), np.ldexp(by, -70)  # squared distances below 2^-101
    elif name == "nint-grid":
        x, y = O.gen_grid(n, 31)
    elif name == "nint-f64":
        x, y = bx * np.float32(37.3), by * np.float32(37.3)
    else:
        x, y = bx, by
    x, y = np.asarray(x, dtype=np.float32), np.asarray(y, dtype=np.float32)
    assert regime(x, y, metric) == name
    for k in (3, 8):
        for start in (O.nn_tour(O.Problem(x, y), 3), O.shuffle_tour(n, 9)):
            gpu_vs_oracle(ctx, x, y, metric, k, start)


@pytest.mark.gpu
@pytest.mark.parametrize("max_grid", [None, "2"])
def test_gpu_ties_on_a_lattice(ctx, monkeypatch, max_grid):
    if max_grid:
        monkeypatch.setenv("TL_MAX_GRID", max_grid)  # every thread walks many (position, slot) items
    side = 24
    q = np.arange(side * side)
    lattice = ((q % side).astype(np.float32), (q // side).astype(np.float32))
    for x, y in (lattice, O.gen_grid(900, 900)):
        for metric in ("f32", "nint"):
            for k in (3, 8):
                gpu_vs_oracle(ctx, x, y, metric, k, O.shuffle_tour(len(x), 3))


@pytest.mark.gpu
def test_gpu_both_relocation_routes(ctx):
    n = 10000
    x, y = O.gen_uniform(n, 4242)
    prob = problem(ctx, x, y, "f32")
    opt = or_opt_n_optimum(prob, 8).astype(np.int64).tolist()
    # carry runs of cities far from their place, including across position 0 and to position n-1:
    # 3-opt N brings them back with short and long spans [i+1, k]
    tour = opt
    for src, ln, dst in ((1000, 5, 9000), (2000, 3, 2300), (7000, 8, 100), (5000, 4, 5050), (9990, 10, 0),
                         (3000, 6, 9994), (50, 4, 6000)):
        run_ = tour[src:src + ln]
        del tour[src:src + ln]
        tour[dst:dst] = run_[::-1]
    start = np.array(tour, dtype=np.uint32)
    assert sorted(start.tolist()) == list(range(n))
    _, got_m = gpu_vs_oracle(ctx, x, y, "f32", 8, start, prob=prob)
    spans = [m[3] - m[1] for m in got_m]  # positions i+1 .. k
    assert min(spans) <= CTA_SPAN < max(spans), spans
    # spans next to position 0 (i = 0) and ending at n-1 (k = n-1: the closing edge and the wrap copy)
    assert any(m[1] == 0 for m in got_m) and any(m[3] == n - 1 for m in got_m), got_m


@pytest.mark.gpu
def test_gpu_budgets_scan_and_candidate_copy(ctx):
    import teeline_b200 as T
    x, y = O.gen_uniform(2000, 2000)
    P = O.Problem(x, y)
    prob = T.Problem.euc2d(ctx, x, y)
    start = O.nn_tour(P, 3)
    prob.set_candidates(5)
    K5 = prob.knn(5)
    want_t, wst, want_m = NL.three_opt_nl(P, start, K5, nthreads=16, log_cap=1 << 16)
    s = prob.session(T.ALGO_THREE_OPT_NEIGHBOR, start)
    prob.set_candidates(16)  # the session keeps its own copy of the k = 5 lists
    first = s.scan()
    assert key([first]) == key(want_m[:1])
    assert key([NL.three_opt_nl_scan(P, start, K5)[0]]) == key([first])
    for budget in (1, 7, 40, 41, 150):
        s.run(budget)
        assert int(s.stats().moves) == budget
    s.run(-1)
    st = s.stats()
    assert key(s.log(1 << 16)) == key(want_m) and (s.tour().astype(np.int64) == want_t).all()
    assert (int(st.moves), int(st.passes), int(st.evals)) == (wst.moves, wst.passes, wst.evals) and st.converged == 1
    assert s.scan() is None
    s.close()
    got_t, st16, _ = prob.local_search(T.ALGO_THREE_OPT_NEIGHBOR, start)  # the problem's lists are now k = 16
    want16 = NL.three_opt_nl(P, start, prob.knn(16), nthreads=16)
    assert (got_t.astype(np.int64) == want16[0]).all() and int(st16.moves) == want16[1].moves


@pytest.mark.gpu
def test_gpu_100k_after_or_opt_n(ctx):
    import teeline_b200 as T
    n = 100_000
    x, y = O.gen_uniform(n, n)
    P = O.Problem(x, y)
    prob = T.Problem.euc2d(ctx, x, y)
    start = or_opt_n_optimum(prob, 8)
    K = prob.knn(8)
    s = prob.session(T.ALGO_THREE_OPT_NEIGHBOR, start)
    s.run(200)
    _, _, want_m = NL.three_opt_nl(P, start, K, max_moves=200, nthreads=16, log_cap=200)
    assert key(s.log(200)) == key(want_m)
    s.run(-1)
    st = s.stats()
    t = s.tour()
    assert st.converged == 1 and sorted(t.tolist()) == list(range(n))
    assert np.float32(O.tour_length(P, t)) == prob.tour_lengths(t)[0]
    assert NL.three_opt_nl_scan(P, t, K, nthreads=16)[0] is None


@pytest.mark.gpu
def test_gpu_million_cities(ctx):
    import teeline_b200 as T
    n = 1_000_000
    x, y = O.gen_uniform(n, n)
    P = O.Problem(x, y)
    prob = T.Problem.euc2d(ctx, x, y)
    start = or_opt_n_optimum(prob, 8)
    K = prob.knn(8)
    s = prob.session(T.ALGO_THREE_OPT_NEIGHBOR, start)
    got = s.scan()
    want, _ = NL.three_opt_nl_scan(P, start, K, nthreads=16)
    assert key([got]) == key([want])
    s.run(1000)
    st = s.stats()
    log = s.log(1000)
    assert int(st.moves) == 1000 and len(log) == 1000
    cur = start.astype(np.int32)
    for m in log:
        delta, i, j, k, case = m
        ev = NL.three_opt_nl_eval(P, cur, i, j, k)  # the oracle's savings and case of this triple
        assert ev is not None and (f32_bits(ev[0]), ev[1]) == (f32_bits(delta), case), m
        cur = O.three_opt_apply(cur, i, j, k, case)
    assert (cur.astype(np.int64) == s.tour().astype(np.int64)).all()


@pytest.mark.gpu
def test_gpu_errors(ctx):
    import teeline_b200 as T
    x, y = O.gen_uniform(50, 50)
    prob = T.Problem.euc2d(ctx, x, y)
    tour = np.arange(50, dtype=np.uint32)
    ex = T.Problem.explicit(ctx, O.matrix_packed_f32(x, y), 50)
    with pytest.raises(T.TeelineError) as ei:
        ex.session(T.ALGO_THREE_OPT_NEIGHBOR, tour)
    assert ei.value.status == 3  # TL_ERR_UNSUPPORTED
    with pytest.raises(T.TeelineError) as ei:
        prob.session(T.ALGO_THREE_OPT_NEIGHBOR, tour, path=T.PATH_MATRIX)
    assert ei.value.status == 3
    s = prob.session(T.ALGO_THREE_OPT_NEIGHBOR, tour, path=T.PATH_RECOMPUTE)
    with pytest.raises(T.TeelineError) as ei:
        s.set_shard(0, 2)
    assert ei.value.status == 3
    s.set_shard(0, 1)
    s.close()
    with pytest.raises(T.TeelineError) as ei:
        prob.two_opt_batch(tour[None, :], algo=T.ALGO_THREE_OPT_NEIGHBOR)
    assert ei.value.status == 3
    for n in (2, 3):  # identity order, no scan, as 3-opt (three_opt.rs:25-28)
        small = T.Problem.euc2d(ctx, x[:n], y[:n])
        t, st, _ = small.local_search(T.ALGO_THREE_OPT_NEIGHBOR, np.arange(n)[::-1])
        assert t.tolist() == list(range(n)) and int(st.moves) == 0 and int(st.passes) == 0 and st.converged == 1


@pytest.mark.gpu
def test_gpu_cli_neighbor(ctx, cli, tmp_path):
    import teeline_b200 as T
    inp = os.path.join(GOLDEN, "att532.tsp")
    ids, x, y = O.read_tsplib_coords(inp)
    prob = T.Problem.euc2d(ctx, x, y)
    prob.set_candidates(8)
    nn = prob.nn_tour(3)
    t1, _, _ = prob.local_search(T.ALGO_THREE_OPT_NEIGHBOR, nn)
    t2, _, _ = prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR, nn)
    t2, _, _ = prob.local_search(T.ALGO_OR_OPT_NEIGHBOR, t2)
    t2, _, _ = prob.local_search(T.ALGO_THREE_OPT_NEIGHBOR, t2)
    want = [("%.5f" % prob.tour_lengths(t)[0], 0, [int(ids[p]) for p in t]) for t in (t1, t2)]
    cfg = tmp_path / "n.toml"
    cfg.write_text("[[stage]]\nsolver = \"nn\"\n"
                   "[[stage]]\nsolver = \"2opt\"\n[stage.cuda]\nmode = \"neighbor\"\ncandidates = 8\n"
                   "[[stage]]\nsolver = \"or_opt\"\n[stage.cuda]\nmode = \"neighbor\"\ncandidates = 8\n"
                   "[[stage]]\nsolver = \"3opt\"\n[stage.cuda]\nmode = \"neighbor\"\ncandidates = 8\n")
    runs = (["solve", "3opt", "--mode", "neighbor", "--candidates", "8"], ["pipeline", "--config", str(cfg)])
    for argv, w in zip(runs, want):
        rc, out, err = run([cli] + argv + ["-i", inp])
        assert rc == 0, err
        first, second = out.strip().split("\n")[:2]
        total, flag = first.split()
        assert (total, int(flag), [int(v) for v in second.split()]) == w, argv
