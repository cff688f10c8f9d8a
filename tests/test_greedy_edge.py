"""The greedy-edge constructor (tl_greedy_tour, kernel K9).

CPU: the two oracles (all edges sorted + union-find, and Bentley's lazy greedy on a grid) agree bit for bit,
the emission rule, and the CLI without a device.  GPU: the tour equals the lazy oracle position for position
in every metric regime from 2 to 10^6 cities, for every list width, on a chain that takes one edge per round,
with its stats and lists; EXPLICIT problems are refused; the CLI and a TOML greedy -> Mode N pipeline."""
import math
import os
import subprocess

import numpy as np
import pytest

import oracle as O
import oracle_nl as NL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def family(name, n, seed=1):
    """Coordinates (x, y) and the metric ("f32" or "nint") of a test family with about n cities."""
    rng = np.random.default_rng(seed + n)
    if name == "uniform":
        x, y = O.gen_uniform(n, seed + n)
        return x, y, "f32"
    if name == "clustered":
        c = rng.uniform(0, 1000, size=(max(n // 50, 1), 2))
        p = c[rng.integers(0, len(c), n)] + rng.normal(0, 8, size=(n, 2))
        return p[:, 0].astype(np.float32), p[:, 1].astype(np.float32), "f32"
    if name in ("lattice", "shuffled_lattice"):
        side = max(int(np.ceil(np.sqrt(n))), 1)
        g = np.arange(side, dtype=np.float32) * 10
        X, Y = np.meshgrid(g, g)
        x, y = X.ravel()[:n], Y.ravel()[:n]
        if name == "shuffled_lattice":
            perm = rng.permutation(n)
            x, y = x[perm], y[perm]
        return np.ascontiguousarray(x), np.ascontiguousarray(y), "f32"
    if name == "twins":  # every city three times: zero distances
        x, y = O.gen_uniform((n + 2) // 3, seed + n)
        return np.repeat(x, 3)[:n].copy(), np.repeat(y, 3)[:n].copy(), "f32"
    if name == "nint_grid":
        x, y = O.gen_grid(n, seed + n)
        return x, y, "nint"
    if name == "nint_frac":  # fractional coordinates: the f64 nint metric
        x, y = O.gen_uniform(n, seed + n)
        return x, y, "nint"
    if name == "tiny":  # nonzero |c| < 2^-27: the IEEE-safe f32 metric
        x, y = O.gen_uniform(n, seed + n)
        return np.ldexp(x, -40).astype(np.float32), np.ldexp(y, -40).astype(np.float32), "f32"
    raise ValueError(name)


FAMILIES = ["uniform", "clustered", "lattice", "shuffled_lattice", "twins", "nint_grid", "nint_frac", "tiny"]


def chain(n):
    """Cities on a line with growing gaps: every city's nearest city is its left neighbour, so only one
    edge at a time is the best of both its ends."""
    x = np.cumsum(np.arange(n, dtype=np.float64)).astype(np.float32)  # gaps 1, 2, 3, ...: exact in f32
    return x, np.zeros(n, dtype=np.float32)


def emission_ok(x, y, metric, tour):
    """The emission rule: the identity order for n <= 3, else a permutation that starts at 0 and then goes to
    the lower of 0's two neighbours."""
    n = len(tour)
    if n <= 3:
        return list(tour) == list(range(n))
    if tour[0] != 0 or tour[1] > tour[-1]:
        return False
    return sorted(int(v) for v in tour) == list(range(n))


# ---- CPU: the oracles ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", FAMILIES)
def test_oracles_agree_small(name):
    for n in range(1, 13):
        x, y, metric = family(name, n)
        a = NL.greedy_brute(x, y, metric)
        b = NL.greedy_lazy(x, y, metric)
        assert (a == b).all(), (name, n)
        assert emission_ok(x, y, metric, a), (name, n, a)


@pytest.mark.parametrize("name", FAMILIES)
def test_oracles_agree_3000(name):
    x, y, metric = family(name, 3000)
    a = NL.greedy_brute(x, y, metric)
    b = NL.greedy_lazy(x, y, metric)
    assert (a == b).all(), name
    assert emission_ok(x, y, metric, a)


def test_oracles_agree_on_the_chain():
    x, y = chain(2000)
    a = NL.greedy_brute(x, y)
    assert (a == NL.greedy_lazy(x, y)).all()
    # the greedy takes every gap in turn and closes the line: 0, 1, ..., n-1
    assert a.tolist() == list(range(2000))


def test_emission_rule():
    for n in (1, 2, 3):  # the identity order
        x, y = O.gen_uniform(n, 5)
        for f in (NL.greedy_brute, NL.greedy_lazy):
            assert f(x[::-1].copy(), y[::-1].copy()).tolist() == list(range(n))
    # four cities on a square's corners, far apart pairwise: the tour starts 0, then 0's lower neighbour
    x = np.array([0, 10, 10, 0], dtype=np.float32)
    y = np.array([0, 0, 11, 11], dtype=np.float32)
    assert NL.greedy_brute(x, y).tolist() == [0, 1, 2, 3]
    x, y = O.gen_uniform(500, 9)
    t = NL.greedy_brute(x, y)
    assert t[0] == 0 and t[1] < t[-1]


def test_brute_is_sequential_greedy_restated():
    """The brute-force oracle against a Python restatement at 60 cities, both metrics."""
    for metric in ("f32", "nint"):
        x, y = O.gen_uniform(60, 11) if metric == "f32" else O.gen_grid(60, 11)
        n = len(x)
        dist = (lambda a, b: float(np.float32(O.dist_f32(x[a], y[a], x[b], y[b])))) if metric == "f32" else \
            (lambda a, b: float(int(math.sqrt((float(x[a]) - float(x[b])) ** 2 + (float(y[a]) - float(y[b])) ** 2) + 0.5)))
        edges = sorted((dist(a, b), a, b) for b in range(n) for a in range(b))
        deg, comp, adj = [0] * n, list(range(n)), [[] for _ in range(n)]
        for _, a, b in edges:
            if deg[a] < 2 and deg[b] < 2 and comp[a] != comp[b]:
                old = comp[b]
                comp = [comp[a] if c == old else c for c in comp]
                deg[a] += 1
                deg[b] += 1
                adj[a].append(b)
                adj[b].append(a)
        e = [v for v in range(n) if deg[v] < 2]
        adj[e[0]].append(e[1])
        adj[e[1]].append(e[0])
        t = [0, min(adj[0])]
        while len(t) < n:
            a, b = adj[t[-1]]
            t.append(b if a == t[-2] else a)
        assert NL.greedy_brute(x, y, metric).tolist() == t, metric


# ---- CPU: CLI without a device ------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def cli():
    from teeline_b200 import build as tb, build_host
    tb.build()
    return build_host.build()


def run(cmd):
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    return p.returncode, p.stdout, p.stderr


def test_solvers_lists_greedy_edge(cli):
    rc, out, _ = run([cli, "solvers"])
    assert rc == 0 and "greedy_edge" in out


def test_no_device_fails_loudly(cli):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    rc, out, err = run([cli, "solve", "greedy_edge", "-i", os.path.join(GOLDEN, "berlin52.tsp")])
    assert rc == 101 and out == "" and "no CPU fallback" in err


# ---- GPU ----------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def ctx():
    import teeline_b200 as T
    c = T.Context(0)
    yield c
    c.close()


def problem(ctx, x, y, metric):
    import teeline_b200 as T
    return T.Problem.euc2d(ctx, x, y, T.DIST_NINT_I32 if metric == "nint" else T.DIST_F32_EXACT)


def gpu_equals_oracle(ctx, x, y, metric, k=None):
    prob = problem(ctx, x, y, metric)
    if k is not None:
        prob.set_candidates(k)
    got, st = prob.greedy_tour()
    want = NL.greedy_lazy(x, y, metric)
    assert (got.astype(np.int64) == want).all(), (len(x), metric, k)
    return prob, got, st


@pytest.mark.gpu
@pytest.mark.parametrize("name", FAMILIES)
def test_gpu_equals_oracle_small(ctx, name):
    for n in range(2, 13):
        x, y, metric = family(name, n)
        gpu_equals_oracle(ctx, x, y, metric)


@pytest.mark.gpu
@pytest.mark.parametrize("name", FAMILIES)
@pytest.mark.parametrize("n", [1000, 10_000, 100_000])
def test_gpu_equals_oracle(ctx, name, n):
    x, y, metric = family(name, n)
    gpu_equals_oracle(ctx, x, y, metric)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["uniform", "nint_grid", "nint_frac", "tiny"])
def test_gpu_million_cities(ctx, name):
    x, y, metric = family(name, 1_000_000)
    _, t, st = gpu_equals_oracle(ctx, x, y, metric)
    assert int(st.moves) == 1_000_000 and st.converged == 1


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["uniform", "shuffled_lattice", "nint_grid"])
def test_gpu_list_width_does_not_change_the_tour(ctx, name):
    x, y, metric = family(name, 20_000)
    want = NL.greedy_lazy(x, y, metric)
    for k in (None, 1, 2, 8, 32):
        _, got, _ = gpu_equals_oracle(ctx, x, y, metric, k)
        assert (got.astype(np.int64) == want).all()


@pytest.mark.gpu
def test_gpu_chain_one_edge_per_round(ctx):
    n = 3000
    x, y = chain(n)
    _, t, st = gpu_equals_oracle(ctx, x, y, "f32")
    assert t.tolist() == list(range(n))
    assert int(st.passes) >= n - 2  # one edge per round: the rounds are reported


@pytest.mark.gpu
def test_gpu_explicit_unsupported(ctx):
    import teeline_b200 as T
    x, y = O.gen_uniform(50, 50)
    ex = T.Problem.explicit(ctx, O.matrix_packed_f32(x, y), 50)
    with pytest.raises(T.TeelineError) as ei:
        ex.greedy_tour()
    assert ei.value.status == 3  # TL_ERR_UNSUPPORTED


@pytest.mark.gpu
def test_gpu_stats_and_default_lists(ctx):
    import teeline_b200 as T
    x, y = O.gen_uniform(50_000, 77)
    prob = problem(ctx, x, y, "f32")
    l0 = ctx.launches
    t1, st1 = prob.greedy_tour()
    l1 = ctx.launches
    t2, st2 = prob.greedy_tour()
    l2 = ctx.launches
    assert (t1 == t2).all()
    assert int(st1.moves) == 50_000 and st1.converged == 1 and st1.device_ms > 0
    assert int(st1.passes) == int(st2.passes) > 0
    # the first call built the default lists (one k-NN launch) and kept them: the second call reuses them
    assert int(st1.launches) == l1 - l0 and int(st2.launches) == l2 - l1 == int(st1.launches) - 1
    # the kept lists are TL_CANDIDATES_DEFAULT wide: a Mode N search on them is the oracle's on knn(8)
    P = O.Problem(x, y)
    got, _, gm = prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR, t1, max_moves=300, log_cap=300)
    want, _, wm = NL.two_opt_nl(P, t1, prob.knn(T.CANDIDATES_DEFAULT), max_moves=300, nthreads=16, log_cap=300)
    assert [m[1:3] for m in gm] == [m[1:3] for m in wm] and (got.astype(np.int64) == want).all()
    for n in (2, 3):  # identity order, no device rounds
        small = problem(ctx, x[:n], y[:n], "f32")
        t, st = small.greedy_tour()
        assert t.tolist() == list(range(n)) and int(st.moves) == n and int(st.passes) == 0


@pytest.mark.gpu
def test_gpu_cli_and_pipeline(ctx, cli, tmp_path):
    import teeline_b200 as T
    inp = os.path.join(GOLDEN, "berlin52.tsp")
    ids, x, y = O.read_tsplib_coords(inp)
    P = O.Problem(x, y)
    g = NL.greedy_lazy(x, y)
    prob = problem(ctx, x, y, "f32")
    t2, _, _ = NL.two_opt_nl(P, g, prob.knn(T.CANDIDATES_DEFAULT))
    want = [("%.5f" % np.float32(O.tour_length(P, t)), 0, [int(ids[p]) for p in t]) for t in (g, t2)]
    cfg = tmp_path / "g.toml"
    cfg.write_text("[[stage]]\nsolver = \"greedy_edge\"\n"
                   "[[stage]]\nsolver = \"2opt\"\n[stage.cuda]\nmode = \"neighbor\"\n")
    for argv, w in zip((["solve", "greedy_edge"], ["pipeline", "--config", str(cfg)]), want):
        rc, out, err = run([cli] + argv + ["-i", inp])
        assert rc == 0, err
        first, second = out.strip().split("\n")[:2]
        total, flag = first.split()
        assert (total, int(flag), [int(v) for v in second.split()]) == w, argv
