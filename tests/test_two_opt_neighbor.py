"""Candidate-list best-improvement 2-opt ("Mode N", TL_ALGO_TWO_OPT_NEIGHBOR).

CPU: the Mode N oracle (oracle_nl) against Mode B's for k >= n-1 and on its own properties, the
ABI and the CLI without a device.  GPU: the library bit for bit against the oracle (move log, tour,
moves / scans / evals), Mode B on the GPU for k >= n-1, ties, budgets, 10^5 and 10^6 cities, errors
and the CLI."""
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


def hilbert_order(x, y, bits=16):
    """Positions sorted along a Hilbert curve over the bounding box (a space-filling-curve start tour)."""
    side = 1 << bits
    def grid(v):
        lo, hi = float(v.min()), float(v.max())
        return np.minimum(((v - lo) / max(hi - lo, 1e-30) * (side - 1)).astype(np.int64), side - 1)
    gx, gy, d = grid(x), grid(y), np.zeros(len(x), dtype=np.int64)
    s = side >> 1
    while s > 0:
        rx = (gx & s) > 0
        ry = (gy & s) > 0
        d += s * s * ((3 * rx) ^ ry)
        flip = ~ry
        swap_x = np.where(flip & rx, s - 1 - gx, gx)
        swap_y = np.where(flip & rx, s - 1 - gy, gy)
        gx, gy = np.where(flip, swap_y, gx), np.where(flip, swap_x, gy)
        s >>= 1
    return np.argsort(d, kind="stable").astype(np.int32)


# ---- CPU: the oracle ------------------------------------------------------------------------------------

@pytest.mark.parametrize("n", [4, 5, 6, 7, 13, 20, 33])
def test_oracle_all_candidates_is_mode_b(n):
    x, y = O.gen_uniform(n, 100 + n)
    P = O.Problem(x, y)
    start = O.shuffle_tour(n, 7 + n)
    K = O.knn(P, n - 1)
    tb, sb, mb = O.two_opt_best(P, start, log_cap=1000)
    tn, sn, mn = NL.two_opt_nl(P, start, K, log_cap=1000)
    assert mn == mb and (tn == tb).all() and sn.moves == sb.moves and sn.passes == sb.passes


def test_oracle_properties_config2():
    x, y = O.gen_uniform(1000, 1000)  # BASELINE config 2
    P = O.Problem(x, y)
    start = O.nn_tour(P, 3)
    K = O.knn(P, 8)
    t, st, moves = NL.two_opt_nl(P, start, K, log_cap=4096)
    assert st.moves == 190 and st.passes == 191 and "%.5f" % np.float32(O.tour_length(P, t)) == "25217.68164"
    assert sorted(t.tolist()) == list(range(1000))
    cur = start.copy()
    for delta, i, j, _, _ in moves:
        assert delta < 0
        # one of the two new edges joins a city to one of its candidates
        new_edges = [(cur[i], cur[j]), (cur[i + 1], cur[j + 1])]
        assert any(b in K[a] or a in K[b] for a, b in new_edges)
        cur = O.swap_2opt(cur, i + 1, j)
    assert (cur == t).all()
    assert NL.two_opt_nl_scan(P, t, K)[0] is None


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
    assert T.ALGO_TWO_OPT_NEIGHBOR == 6 and T.CANDIDATES_DEFAULT == 8
    hdr = open(os.path.join(ROOT, "include", "teeline_cuda.h")).read()
    assert "TL_ALGO_TWO_OPT_NEIGHBOR = 6" in hdr and "#define TL_CANDIDATES_DEFAULT 8" in hdr


def test_no_device_fails_loudly(cli):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    import teeline_b200 as T
    with pytest.raises(T.TeelineError) as ei:
        T.Context(0)
    assert ei.value.status == 2  # TL_ERR_CUDA: no problem, no candidate lists, no Mode N session
    rc, out, err = run([cli, "solve", "2opt", "--mode", "neighbor", "--candidates", "8",
                        "-i", os.path.join(GOLDEN, "berlin52.tsp")])
    assert rc == 101 and out == "" and "no CPU fallback" in err


def test_cli_candidates_argument_and_toml(cli, tmp_path):
    inp = os.path.join(GOLDEN, "berlin52.tsp")
    for bad in ("0", "33", "x", "-1"):
        rc, _, err = run([cli, "solve", "2opt", "--mode", "neighbor", "--candidates", bad, "-i", inp])
        assert rc == 2 and "--candidates" in err, (bad, err)
    rc, out, _ = run([cli, "solvers"])
    assert rc == 0 and "2opt --mode neighbor" in out
    cases = {
        "candidates = 0\n": "config: [cuda] candidates must be in 1..32",
        "candidates = 33\n": "config: [cuda] candidates must be in 1..32",
        "k = 8\n": "config: unknown field `k` in [cuda] — valid: mode, path (strings), seed, candidates (integers)",
    }
    for k, (body, want) in enumerate(cases.items()):
        f = tmp_path / f"c{k}.toml"
        f.write_text("[[stage]]\nsolver = \"2opt\"\n[stage.cuda]\nmode = \"neighbor\"\n" + body)
        rc, _, err = run([cli, "pipeline", "--config", str(f), "-i", inp])
        assert rc == 1 and want in err, (body, err)


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


def gpu_vs_oracle(ctx, x, y, metric, k, start, check_evals=True):
    import teeline_b200 as T
    n = len(x)
    prob = T.Problem.euc2d(ctx, x, y, T.DIST_NINT_I32 if metric == "nint" else T.DIST_F32_EXACT)
    P = O.Problem(tri=O.matrix_packed_nint(x, y), n=n) if metric == "nint" else O.Problem(x, y)
    K = prob.knn(k)
    prob.set_candidates(k)
    cap = 1 << 16
    got_t, st, got_m = prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR, start, log_cap=cap)
    want_t, wst, want_m = NL.two_opt_nl(P, start, K, nthreads=8, log_cap=cap)
    assert same_moves(got_m, want_m), (n, metric, k)
    assert (got_t.astype(np.int64) == want_t).all()
    assert (int(st.moves), int(st.passes)) == (wst.moves, wst.passes)
    if check_evals:
        assert int(st.evals) == wst.evals
    assert st.converged == 1 and st.path_used == T.PATH_RECOMPUTE
    return prob, got_t


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["4", "5", "6", "7", "13", "33", "257", "1000", "berlin52", "att532"])
@pytest.mark.parametrize("metric", ["f32", "nint"])
def test_gpu_equals_oracle(ctx, name, metric):
    x, y = instance(name)
    n = len(x)
    Pf = O.Problem(x, y)
    for k in (1, 3, 8, 32):
        for start in (O.nn_tour(Pf, 3), O.shuffle_tour(n, 11 + n)):
            gpu_vs_oracle(ctx, x, y, metric, k, start)


@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["f32", "nint"])
def test_gpu_equals_oracle_10k(ctx, metric):
    x, y = O.gen_uniform(10000, 10000)
    gpu_vs_oracle(ctx, x, y, metric, 8, O.nn_tour(O.Problem(x, y), 3))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4, 5, 6, 7, 13, 20, 33])
def test_gpu_all_candidates_is_gpu_mode_b(ctx, n):
    import teeline_b200 as T
    x, y = O.gen_uniform(n, 300 + n)
    prob = T.Problem.euc2d(ctx, x, y)
    prob.set_candidates(min(32, n - 1))
    start = O.shuffle_tour(n, 5 + n)
    tb, sb, mb = prob.local_search(T.ALGO_TWO_OPT_BEST, start, log_cap=1000)
    tn, sn, mn = prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR, start, log_cap=1000)
    assert mn == mb and (tn == tb).all() and (sn.moves, sn.passes) == (sb.moves, sb.passes)


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
def test_gpu_budgets_scan_and_candidate_copy(ctx):
    import teeline_b200 as T
    x, y = O.gen_uniform(2000, 2000)
    P = O.Problem(x, y)
    prob = T.Problem.euc2d(ctx, x, y)
    start = O.nn_tour(P, 3)
    prob.set_candidates(5)
    K5 = prob.knn(5)
    want_t, wst, want_m = NL.two_opt_nl(P, start, K5, log_cap=1 << 16)
    s = prob.session(T.ALGO_TWO_OPT_NEIGHBOR, start)
    prob.set_candidates(16)  # the session keeps its own copy of the k = 5 lists
    first = s.scan()
    assert (int(f32_bits(first[0])), first[1], first[2]) == (int(f32_bits(want_m[0][0])), want_m[0][1], want_m[0][2])
    assert NL.two_opt_nl_scan(P, start, K5)[0][1:3] == first[1:3]
    for budget in (1, 7, 40, 41, 300):
        s.run(budget)
        assert int(s.stats().moves) == budget
    s.run(-1)
    st = s.stats()
    assert same_moves(s.log(1 << 16), want_m) and (s.tour().astype(np.int64) == want_t).all()
    assert (int(st.moves), int(st.passes), int(st.evals)) == (wst.moves, wst.passes, wst.evals) and st.converged == 1
    assert s.scan() is None
    s.close()
    # the problem's lists are now k = 16
    got_t, st16, _ = prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR, start)
    want16 = NL.two_opt_nl(P, start, prob.knn(16))
    assert (got_t.astype(np.int64) == want16[0]).all() and int(st16.moves) == want16[1].moves


@pytest.mark.gpu
def test_gpu_100k_nn_start(ctx):
    import teeline_b200 as T
    n = 100_000
    x, y = O.gen_uniform(n, n)
    P = O.Problem(x, y)
    prob = T.Problem.euc2d(ctx, x, y)
    K = prob.knn(8)
    rng = np.random.default_rng(1)
    for c in rng.choice(n, 1000, replace=False):
        dx = (x - x[c]).astype(np.float32)
        dy = (y - y[c]).astype(np.float32)
        d = np.sqrt(dx * dx + dy * dy, dtype=np.float32)
        d[c] = np.inf
        order = np.lexsort((np.arange(n), d))[:8]
        assert (K[c] == order).all(), c
    start = prob.nn_tour(3)
    prob.set_candidates(8)
    s = prob.session(T.ALGO_TWO_OPT_NEIGHBOR, start)
    s.run(2000)
    _, _, want_m = NL.two_opt_nl(P, start, K, max_moves=2000, nthreads=16, log_cap=2000)
    assert same_moves(s.log(2000), want_m)
    s.run(-1)
    st = s.stats()
    t = s.tour()
    assert st.converged == 1 and sorted(t.tolist()) == list(range(n))
    assert np.float32(O.tour_length(P, t)) == prob.tour_lengths(t)[0]
    assert NL.two_opt_nl_scan(P, t, K, nthreads=16)[0] is None


@pytest.mark.gpu
def test_gpu_million_cities_hilbert_start(ctx):
    import teeline_b200 as T
    n = 1_000_000
    x, y = O.gen_uniform(n, n)
    P = O.Problem(x, y)
    prob = T.Problem.euc2d(ctx, x, y)
    prob.set_candidates(8)
    K = prob.knn(8)
    start = hilbert_order(x, y)
    s = prob.session(T.ALGO_TWO_OPT_NEIGHBOR, start)
    got = s.scan()
    want, _ = NL.two_opt_nl_scan(P, start, K, nthreads=16)
    assert (int(f32_bits(got[0])), got[1], got[2]) == (int(f32_bits(want[0])), want[1], want[2])
    s.run(-1)
    assert s.stats().converged == 1
    t = s.tour()
    assert sorted(t.tolist()) == list(range(n))
    assert NL.two_opt_nl_scan(P, t, K, nthreads=16)[0] is None


@pytest.mark.gpu
def test_gpu_errors(ctx):
    import teeline_b200 as T
    x, y = O.gen_uniform(50, 50)
    prob = T.Problem.euc2d(ctx, x, y)
    tour = np.arange(50, dtype=np.uint32)
    for k in (0, 33):
        with pytest.raises(T.TeelineError) as ei:
            prob.set_candidates(k)
        assert ei.value.status == 1  # TL_ERR_INVALID
    ex = T.Problem.explicit(ctx, O.matrix_packed_f32(x, y), 50)
    with pytest.raises(T.TeelineError) as ei:
        ex.set_candidates(8)
    assert ei.value.status == 3
    with pytest.raises(T.TeelineError) as ei:
        ex.session(T.ALGO_TWO_OPT_NEIGHBOR, tour)
    assert ei.value.status == 3
    with pytest.raises(T.TeelineError) as ei:
        prob.session(T.ALGO_TWO_OPT_NEIGHBOR, tour, path=T.PATH_MATRIX)
    assert ei.value.status == 3
    s = prob.session(T.ALGO_TWO_OPT_NEIGHBOR, tour, path=T.PATH_RECOMPUTE)
    with pytest.raises(T.TeelineError) as ei:
        s.set_shard(0, 2)
    assert ei.value.status == 3
    s.set_shard(0, 1)
    with pytest.raises(T.TeelineError) as ei:
        prob.two_opt_batch(tour[None, :], algo=T.ALGO_TWO_OPT_NEIGHBOR)
    assert ei.value.status == 3
    for n in (2, 3):
        small = T.Problem.euc2d(ctx, x[:n], y[:n])
        t, st, _ = small.local_search(T.ALGO_TWO_OPT_NEIGHBOR, np.arange(n)[::-1])
        assert t.tolist() == list(range(n))[::-1] and int(st.moves) == 0 and st.converged == 1


@pytest.mark.gpu
def test_gpu_cli_neighbor(ctx, cli, tmp_path):
    import teeline_b200 as T
    inp = os.path.join(GOLDEN, "att532.tsp")
    ids, x, y = O.read_tsplib_coords(inp)
    prob = T.Problem.euc2d(ctx, x, y)
    prob.set_candidates(8)
    t, _, _ = prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR, prob.nn_tour(3))
    want = ("%.5f" % prob.tour_lengths(t)[0], 0, [int(ids[p]) for p in t])
    cfg = tmp_path / "n.toml"
    cfg.write_text("[[stage]]\nsolver = \"nn\"\n[[stage]]\nsolver = \"2opt\"\n[stage.cuda]\nmode = \"neighbor\"\n"
                   "candidates = 8\n")
    for argv in (["solve", "2opt", "--mode", "neighbor", "--candidates", "8"], ["pipeline", "--config", str(cfg)]):
        rc, out, err = run([cli] + argv + ["-i", inp])
        assert rc == 0, err
        first, second = out.strip().split("\n")[:2]
        total, flag = first.split()
        assert (total, int(flag), [int(v) for v in second.split()]) == want, argv
