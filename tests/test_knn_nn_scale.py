"""k-NN candidate lists and the nearest-neighbour tour at 10^4 to 10^6 cities, against an exact reference.

Candidate-list 2-opt and Or-opt run on the lists `knn_kernel` builds (K5, csrc/k5_knn.cu) and start from the
tour `nn_tour_kernel` builds.  The oracle's k-NN and NN tour are O(n^2), so above a few thousand cities the
other test files hand the library's own lists to the search oracles: a wrong list would be searched the same
way on both sides.  Here `knn_ref` gives an exact reference at any size, and the kernels are compared with it
where their launch shape changes:
  - `launch_knn_k` runs 64-thread CTAs below 148 * 128 = 18 944 cities, 128 from there and 256 from
    148 * 256 = 37 888; the K = 4 / 8 / 16 / 32 templates serve k up to their width;
  - `nn_tour_heads` keeps the first ks list entries of every city in shared memory: ks = 16 up to 6 375
    cities, 15 down to 4 up to 25 206, and none from 25 207 (the walk then reads every list from global
    memory); steps whose 32 listed neighbours are all visited take the block-wide argmin."""
import functools
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
from scipy.spatial import cKDTree

import oracle as O
import oracle_nl as NL

NCPU = max(1, min(16, os.cpu_count() or 1))
KS = (4, 8, 16, 17, 32)  # every template at its full width, and k = 17 of the 32-wide one


# ---- the reference ----------------------------------------------------------------------------------------

def keys(x, y, q, c, metric):
    """The distance of q to c bit for bit as the oracle computes it: tlo_dist_f32 (five f32 roundings, no
    FMA) or tlo_dist_nint (f64, truncated after + 0.5)."""
    if metric == "f32":
        dx = x[q] - x[c]
        dy = y[q] - y[c]
        dx2, dy2 = dx * dx, dy * dy
        # the margin below assumes every nonzero square is a normal f32
        tiny = np.finfo(np.float32).tiny
        assert (((dx2 == 0) | (dx2 >= tiny)) & ((dy2 == 0) | (dy2 >= tiny))).all()
        return np.sqrt(dx2 + dy2)
    xd = x[q].astype(np.float64) - x[c].astype(np.float64)
    yd = y[q].astype(np.float64) - y[c].astype(np.float64)
    return (np.sqrt(xd * xd + yd * yd) + 0.5).astype(np.int64)


def knn_ref(x, y, k, metric, extra=8):
    """For every city the first k other cities in (distance, index) order, padded with -1 as O.knn pads.

    A KD-tree query in f64 for k + extra neighbours gives a superset, re-keyed exactly by `keys`.  A row is
    accepted once the tree's farthest returned city is provably farther than any city whose key could equal
    the k-th key: every city left out then has a larger key.  Rows that fail are queried again with twice
    as many neighbours, up to all n."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    y = np.ascontiguousarray(y, dtype=np.float32)
    n = len(x)
    out = np.full((n, k), -1, dtype=np.int64)
    k = min(k, n - 1)
    if k <= 0:
        return out
    pts = np.stack([x, y], 1).astype(np.float64)
    tree = cKDTree(pts)
    todo = np.arange(n)
    kp = k + extra
    while len(todo):
        kq = min(kp + 1, n)  # + 1: the query city itself
        dd, ii = tree.query(pts[todo], k=kq, workers=-1)
        dd, ii = dd.reshape(len(todo), kq), ii.reshape(len(todo), kq)
        q = np.broadcast_to(todo[:, None], ii.shape)
        d = keys(x, y, q, ii, metric)
        d = np.where(ii == q, np.inf if metric == "f32" else np.iinfo(np.int64).max, d)
        order = np.lexsort((ii, d), axis=-1)
        ii, d = np.take_along_axis(ii, order, 1), np.take_along_axis(d, order, 1)
        kth = d[:, k - 1].astype(np.float64)
        # f32 keys carry a relative error below 2^-22 for normal squares; nint(d) > key once d > key + 0.5
        bound = kth * (1 + 2.0 ** -20) if metric == "f32" else (kth + 0.5) * (1 + 2.0 ** -40)
        ok = (kq == n) | (dd[:, -1] > bound)
        out[todo[ok], :k] = ii[ok, :k]
        todo = todo[~ok]
        kp *= 2
    return out


def regime(x, y, metric):
    """The distance code these coordinates select, restating api.cu (coords_allow_fast_sqrt,
    coords_allow_grid_nint)."""
    c = np.abs(np.concatenate([x, y]).astype(np.float64))
    if metric == "f32":
        fast = bool(np.isfinite(c).all() and (c < 2.0 ** 62).all() and ((c == 0) | (c >= 2.0 ** -27)).all())
        return "f32-fast" if fast else "f32-safe"
    grid = (bool((np.floor(c) == c).all()) and bool((c <= 2.0 ** 22).all())
            and float(x.max()) - float(x.min()) <= 2.0 ** 20 and float(y.max()) - float(y.min()) <= 2.0 ** 20)
    return "nint-grid" if grid else "nint-f64"


# ---- instances --------------------------------------------------------------------------------------------

def lattice(n):
    """n cities row by row on an integer lattice about sqrt(n) wide: equal distances everywhere."""
    side = int(np.ceil(np.sqrt(n)))
    q = np.arange(n)
    return (q % side).astype(np.float32), (q // side).astype(np.float32)


def shuffled_lattice(n):
    """The lattice with its cities in a seeded random order.  Walked row by row, the NN tour of the ordered
    lattice always finds a listed neighbour unvisited; in this order it does not, and the block-wide argmin
    then meets equal distances held by different warps."""
    x, y = lattice(n)
    p = np.random.default_rng(1).permutation(n)
    return x[p], y[p]


def with_twins(x, y):
    """Cities n-100..n-1 copy cities 0..99 and cities 100..119 all sit on city 100: zero distances."""
    x, y = x.copy(), y.copy()
    n = len(x)
    x[n - 100:], y[n - 100:] = x[:100], y[:100]
    x[100:120], y[100:120] = x[100], y[100]
    return x, y


# name: (metric, regime it must select)
INSTANCES = {
    "uniform": ("f32", "f32-fast"),
    "lattice": ("f32", "f32-fast"),
    "shuffled": ("f32", "f32-fast"),
    "twins": ("f32", "f32-fast"),
    "tiny": ("f32", "f32-safe"),  # the exact 2^-40 image of `uniform`
    "grid": ("nint", "nint-grid"),
    "frac": ("nint", "nint-f64"),
}


def coords(name, n):
    bx, by = O.gen_uniform(n, n)
    if name == "uniform":
        return bx, by
    if name == "lattice":
        return lattice(n)
    if name == "shuffled":
        return shuffled_lattice(n)
    if name == "twins":
        return with_twins(bx, by)
    if name == "tiny":
        return np.ldexp(bx, -40), np.ldexp(by, -40)
    if name == "grid":
        return O.gen_grid(n, n)
    if name == "frac":
        return bx * np.float32(37.3), by * np.float32(37.3)
    raise KeyError(name)


@functools.lru_cache(maxsize=None)
def instance(name, n):
    """(x, y, metric, reference 32-NN lists): the lists for k < 32 are their k-prefixes."""
    metric, want = INSTANCES[name]
    x, y = coords(name, n)
    assert regime(x, y, metric) == want, (name, n)
    return x, y, metric, knn_ref(x, y, 32, metric).astype(np.int32)


def oracle_problem(x, y, metric):
    return O.Problem(tri=O.matrix_packed_nint(x, y), n=len(x)) if metric == "nint" else O.Problem(x, y)


def f32_bits(v):
    return int(np.float32(v).view(np.uint32))


def signed(lists):
    """GPU lists (uint32, UINT32_MAX padding) as int64 with -1 padding."""
    return np.asarray(lists).view(np.int32).astype(np.int64)


# ---- CPU: the premises -------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", list(INSTANCES))
def test_reference_equals_oracle(name):
    """knn_ref is O.knn at 3000 cities for every k, also when nearly every row needs a wider query."""
    metric, want = INSTANCES[name]
    x, y = coords(name, 3000)
    assert regime(x, y, metric) == want
    P = oracle_problem(x, y, metric)
    ref32 = knn_ref(x, y, 32, metric)
    for k in (1, 4, 5, 8, 9, 16, 17, 31, 32):
        want_k = O.knn(P, k)
        assert (knn_ref(x, y, k, metric) == want_k).all(), k
        assert (knn_ref(x, y, k, metric, extra=0) == want_k).all(), k
        assert (ref32[:, :k] == want_k).all(), k
    if name == "lattice":
        assert int(x.max()) == 54  # the 55-wide lattice
    if name == "tiny":
        bx, by = coords("uniform", 3000)
        assert (x == np.ldexp(bx, -40)).all() and (ref32 == knn_ref(bx, by, 32, "f32")).all()


@pytest.mark.parametrize("metric", ["f32", "nint"])
def test_reference_pads_like_oracle(metric):
    for n in (2, 3, 5, 9, 33):
        x, y = O.gen_uniform(n, 50 + n)
        P = oracle_problem(x, y, metric)
        for k in (1, 4, 8, 32):
            assert (knn_ref(x, y, k, metric) == O.knn(P, k)).all(), (n, k)


@pytest.mark.parametrize("name", ["uniform", "lattice", "twins"])
def test_reference_by_brute_force_100k(name):
    """Sampled rows of the 10^5-city reference against a brute force over every city."""
    metric = INSTANCES[name][0]
    x, y = coords(name, 100_000)
    ref = knn_ref(x, y, 32, metric)
    n = len(x)
    rows = np.random.default_rng(5).choice(n, 300, replace=False)
    if name == "twins":
        rows = np.concatenate([rows, np.arange(95, 125), np.arange(n - 5, n)])
    for q in rows:
        d = keys(x, y, np.full(n, q), np.arange(n), metric).astype(np.float64)
        d[q] = np.inf
        assert (ref[q] == np.lexsort((np.arange(n), d))[:32]).all(), q


def test_nn_tour_head_boundaries():
    """The sizes the NN-tour tests use straddle the list-head regimes (nn_tour_heads, k5_knn.cu)."""
    def heads(n, kk=32):
        room = 200 * 1024 - (n + 31) // 32 * 4
        ks = min(16, kk, room // (2 * n))
        return ks if ks >= 4 and n <= 65535 else 0
    assert [heads(n) for n in (6375, 6376, 10000, 20226, 20227, 25206, 25207, 40000)] == [16, 15, 10, 5, 4, 4, 0, 0]


def check_nn_walk(x, y, metric, ref, tour, sample=500):
    """The NN tour's rule at every step: the next city is the first unvisited entry of the reference 32-NN
    list, and where all 32 are visited, the nearest unvisited city with ties to the lower index (checked by
    brute force on a seeded sample of those steps).  Returns the number of steps of the second kind."""
    n = len(x)
    tour = np.asarray(tour).astype(np.int64)
    assert tour[0] == 0 and (np.sort(tour) == np.arange(n)).all()
    when = np.empty(n, dtype=np.int64)
    when[tour] = np.arange(n)  # the step at which each city is visited
    steps = np.arange(n - 1)
    lists = ref[tour[:-1]]
    open_ = when[lists] > steps[:, None]
    listed = open_.any(axis=1)
    first = lists[steps, np.argmax(open_, axis=1)]
    bad = np.flatnonzero(listed & (first != tour[1:]))
    assert len(bad) == 0, bad[:5].tolist()
    rest = np.flatnonzero(~listed)
    for t in np.random.default_rng(3).choice(rest, min(sample, len(rest)), replace=False):
        cand = tour[t + 1:]
        d = keys(x, y, np.full(len(cand), tour[t]), cand, metric)
        assert cand[np.lexsort((cand, d))[0]] == tour[t + 1], int(t)
    return len(rest)


@pytest.mark.parametrize("name", ["uniform", "shuffled"])
def test_nn_walk_check_passes_the_oracle_tour(name):
    x, y = coords(name, 3000)
    ref = knn_ref(x, y, 32, "f32")
    tour = O.nn_tour(O.Problem(x, y), 3)
    assert check_nn_walk(x, y, "f32", ref, tour, sample=10**6) > 0
    bad = tour.copy()
    bad[[1000, 2000]] = bad[[2000, 1000]]
    with pytest.raises(AssertionError):
        check_nn_walk(x, y, "f32", ref, bad, sample=10**6)


# ---- GPU: k-NN -------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def T():
    import teeline_b200 as T
    return T


@pytest.fixture(scope="module")
def ctx(T):
    c = T.Context(0)
    yield c
    c.close()


def problem(T, ctx, x, y, metric):
    return T.Problem.euc2d(ctx, x, y, T.DIST_NINT_I32 if metric == "nint" else T.DIST_F32_EXACT)


def check_knn(prob, ref, ks, what):
    full = signed(prob.knn(32))
    assert (full == ref).all(), (what, 32, np.argwhere(full != ref)[:5].tolist())
    for k in ks:
        got = signed(prob.knn(k))
        assert (got == ref[:, :k]).all(), (what, k, np.argwhere(got != ref[:, :k])[:5].tolist())
        assert (got == full[:, :k]).all(), (what, k)  # the prefix rule


@pytest.mark.gpu
@pytest.mark.parametrize("n", [18943, 18944, 37887, 37888])
def test_knn_cta_shapes(T, ctx, n):
    """Both sides of the 64 -> 128 and 128 -> 256 thread switches; 18 943 and 37 887 end in a partial
    1024-city tile."""
    x, y, metric, ref = instance("uniform", n)
    check_knn(problem(T, ctx, x, y, metric), ref, KS, n)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["uniform", "tiny", "grid", "frac", "twins"])
def test_knn_100k_every_metric(T, ctx, name):
    n = 100_000
    x, y, metric, ref = instance(name, n)
    assert n % 1024
    prob = problem(T, ctx, x, y, metric)
    check_knn(prob, ref, KS, name)
    if name == "tiny":
        assert (ref == instance("uniform", n)[3]).all()
    if name == "twins":
        assert (ref[100, :19] == np.arange(101, 120)).all() and ref[n - 1, 0] == 99


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["uniform", "lattice", "shuffled"])
def test_knn_million(T, ctx, name):
    """10^6 cities: uniform, and the 1000 x 1000 lattice in two city orders, where every list ends inside a
    shell of ties."""
    x, y, metric, ref = instance(name, 1_000_000)
    check_knn(problem(T, ctx, x, y, metric), ref, (8,), name)


@pytest.mark.gpu
def test_knn_padding_small_n(T, ctx):
    for n in (2, 3, 5, 9, 33):
        x, y = O.gen_uniform(n, 50 + n)
        for metric in ("f32", "nint"):
            prob = problem(T, ctx, x, y, metric)
            for k in (1, 4, 8, 16, 17, 32):
                assert (signed(prob.knn(k)) == knn_ref(x, y, k, metric)).all(), (n, metric, k)


def explicit_triangles(n):
    x, y = O.gen_uniform(n, 77)
    tri = O.matrix_packed_f32(x, y)
    # distances 0..56 only: long runs of equal keys in every list and in the NN tour's argmin
    return {"f32": tri, "ties": np.floor(tri / np.float32(25)).astype(np.float32)}


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["f32", "ties"])
def test_knn_explicit_3000(T, ctx, which):
    """knn_packed_kernel over 12 CTAs of 256 threads."""
    n = 3000
    tri = explicit_triangles(n)[which]
    P = O.Problem(tri=tri, n=n)
    prob = T.Problem.explicit(ctx, tri, n)
    for k in KS:
        assert (signed(prob.knn(k)) == O.knn(P, k)).all(), k


# ---- GPU: the NN tour ------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_nn_tour_equals_oracle_across_head_regimes(T, ctx):
    """Uniform instances on both sides of every list-head boundary, and a shuffled lattice without heads
    (about 500 of its steps take the block-wide argmin, some 40 of them between equal distances); 40 000
    cities also take the 256-thread k-NN shape.  The oracle tours run in threads (ctypes drops the GIL)."""
    cases = [("uniform", n) for n in (6375, 6376, 20227, 25206, 25207, 40000)] + [("shuffled", 25207)]
    data = {c: coords(*c) for c in cases}
    for (name, n), (x, y) in data.items():
        assert regime(x, y, "f32") == "f32-fast"
    with ThreadPoolExecutor(max_workers=min(len(cases), NCPU)) as ex:
        want = {c: ex.submit(O.nn_tour, O.Problem(*data[c]), 3) for c in cases}
        got = {c: problem(T, ctx, *data[c], "f32").nn_tour(3) for c in cases}
        for c in cases:
            w = want[c].result()
            g = got[c].astype(np.int64)
            assert (g == w).all(), (c, int(np.argmax(g != w)))


@pytest.mark.gpu
def test_nn_tour_without_heads_10k(T, ctx, monkeypatch):
    x, y = O.gen_uniform(10_000, 10_000)
    prob = problem(T, ctx, x, y, "f32")
    monkeypatch.delenv("TL_NN_NO_HEADS", raising=False)
    with_heads = prob.nn_tour(3)
    monkeypatch.setenv("TL_NN_NO_HEADS", "1")
    without = prob.nn_tour(3)
    assert (with_heads == without).all()
    assert (without.astype(np.int64) == O.nn_tour(O.Problem(x, y), 3)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["f32", "ties"])
def test_nn_tour_explicit_3000(T, ctx, which):
    n = 3000
    tri = explicit_triangles(n)[which]
    got = T.Problem.explicit(ctx, tri, n).nn_tour(3)
    assert (got.astype(np.int64) == O.nn_tour(O.Problem(tri=tri, n=n), 3)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["uniform", "shuffled"])
def test_nn_tour_million_by_property(T, ctx, name):
    """At 10^6 cities the oracle's O(n^2) walk is out of reach: every step is checked by the rule itself."""
    x, y, metric, ref = instance(name, 1_000_000)
    tour = problem(T, ctx, x, y, metric).nn_tour(3)
    rest = check_nn_walk(x, y, metric, ref, tour)
    print(f"\n{name}: {rest} of {len(x) - 1} steps find every listed neighbour visited")
    assert rest > 0


# ---- GPU: the large-n searches on lists that do not come from the GPU ---------------------------------------

@pytest.mark.gpu
def test_searches_on_reference_lists_100k(T, ctx):
    """Mode N and Or-opt N on the library's own lists make the oracle's moves on the reference lists."""
    x, y, metric, ref = instance("uniform", 100_000)
    P = O.Problem(x, y)
    prob = problem(T, ctx, x, y, metric)
    prob.set_candidates(8)
    K = ref[:, :8]
    start = prob.nn_tour(3)
    budget = 2000
    for algo, search in ((T.ALGO_TWO_OPT_NEIGHBOR, NL.two_opt_nl), (T.ALGO_OR_OPT_NEIGHBOR, NL.or_opt_nl)):
        s = prob.session(algo, start)
        s.run(budget)
        got = s.log(budget)
        _, _, want = search(P, start, K, max_moves=budget, nthreads=NCPU, log_cap=budget)
        s.close()
        assert len(want) == budget
        assert [(f32_bits(m[0]),) + tuple(m[1:]) for m in got] == [(f32_bits(m[0]),) + tuple(m[1:]) for m in want], algo

