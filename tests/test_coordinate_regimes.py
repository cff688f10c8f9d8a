"""The search kernels in every coordinate regime, bit for bit against the CPU oracle.

The coordinates of a problem decide which distance code a kernel runs (api.cu, session.cu):
  - f32 metric, fast sqrt (`EucPol<true>`, Mode N / k-NN metric 0, Mode R `ref_persistent_kernel<0, .>`)
    when every nonzero |c| is in [2^-27, 2^62); IEEE-safe sqrt (`EucPol<false>`, metric 1) otherwise;
  - screening (`dist_f32_screen`) in the recompute scans, persistent Mode R and the batch engines only
    for fast-sqrt problems with dmax >= 2^-20 and TL_NO_SCREEN unset;
  - TSPLIB nint: `dist_nint_grid` for integer coordinates with axis ranges up to 2^20 and without
    TL_NINT_F64, `dist_nint` in f64 otherwise (Mode N metric 3, persistent Mode R metric 3).

Every instance below is built to land in one regime, and every test asserts that it does before it
compares anything.  Power-of-two scalings of an instance (`tiny`, `huge`) must make exactly the moves
of the unscaled one, with deltas scaled by the same power: that is checked without the oracle at sizes
the oracle cannot afford."""
import os

import numpy as np
import pytest

import oracle as O
import oracle_nl as NL

NCPU = max(1, min(16, os.cpu_count() or 1))
CAP = 1 << 16


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def f32_bits(v):
    return int(np.float32(v).view(np.uint32))


def log_key(moves, scale=0):
    """(delta bits, positions...) per move; deltas as f32, optionally times 2^scale."""
    return [(f32_bits(np.ldexp(np.float32(m[0]), scale)),) + tuple(m[1:]) for m in moves]


# ---- instances and their regimes ---------------------------------------------------------------------

def regime(x, y, kind, env=None):
    """The distance code a problem of these coordinates selects, restating api.cu and session.cu:
    (metric, screened) with metric one of f32-fast, f32-safe, nint-grid, nint-f64."""
    env = os.environ if env is None else env
    x = np.asarray(x, dtype=np.float32)
    y = np.asarray(y, dtype=np.float32)
    c = np.abs(np.concatenate([x, y]).astype(np.float64))
    # coords_allow_fast_sqrt: finite, below 2^62, and every nonzero |c| at least 2^-27
    fast = bool(np.isfinite(c).all() and (c < 2.0 ** 62).all() and ((c == 0) | (c >= 2.0 ** -27)).all())
    screen = False
    if fast:
        dx = float(x.max()) - float(x.min())
        dy = float(y.max()) - float(y.min())
        dmax = np.float32(np.sqrt(dx * dx + dy * dy) * (1.0 + 1e-6))
        screen = bool(dmax >= np.float32(2.0 ** -20)) and "TL_NO_SCREEN" not in env
    if kind == "f32":
        return ("f32-fast" if fast else "f32-safe"), screen
    # coords_allow_grid_nint: integers, |c| <= 2^22, both axis ranges <= 2^20
    grid = ("TL_NINT_F64" not in env and bool(np.isfinite(c).all()) and bool((np.floor(c) == c).all())
            and bool((c <= 2.0 ** 22).all()) and float(x.max()) - float(x.min()) <= 2.0 ** 20
            and float(y.max()) - float(y.min()) <= 2.0 ** 20)
    return ("nint-grid" if grid else "nint-f64"), screen


def with_twins(x, y):
    """Cities n-100..n-1 copy cities 0..99 and cities 100..119 all sit on city 100: zero-length edges."""
    x, y = x.copy(), y.copy()
    n = len(x)
    x[n - 100:], y[n - 100:] = x[:100], y[:100]
    x[100:120], y[100:120] = x[100], y[100]
    return x, y


# name: (kind, environment, regime it must select)
INSTANCES = {
    "base": ("f32", {}, ("f32-fast", True)),
    "tiny": ("f32", {}, ("f32-safe", False)),
    "deep": ("f32", {}, ("f32-safe", False)),
    "huge": ("f32", {}, ("f32-safe", False)),
    "narrow": ("f32", {}, ("f32-fast", False)),
    "noscreen": ("f32", {"TL_NO_SCREEN": "1"}, ("f32-fast", False)),
    "twins": ("f32", {}, ("f32-fast", True)),
    "twins_deep": ("f32", {}, ("f32-safe", False)),
    "one_site": ("f32", {}, ("f32-fast", False)),
    "two_sites": ("f32", {}, ("f32-fast", True)),
    "grid": ("nint", {}, ("nint-grid", True)),
    "half": ("nint", {}, ("nint-f64", True)),
    "wide": ("nint", {}, ("nint-f64", True)),
    "frac": ("nint", {}, ("nint-f64", True)),
    "grid64": ("nint", {"TL_NINT_F64": "1"}, ("nint-f64", True)),
    "twins_nint": ("nint", {}, ("nint-grid", True)),
    "twins_frac": ("nint", {}, ("nint-f64", True)),
}
# the exact 2^s images of `base`
SCALE = {"tiny": -40, "huge": 53}


def coords(name, n, seed=None):
    """Coordinates of instance `name` at about n cities (one_site and two_sites have 64)."""
    seed = n if seed is None else seed
    if name in ("one_site", "two_sites"):
        n = 64
    bx, by = O.gen_uniform(n, seed)
    if name in ("base", "noscreen"):
        return bx, by
    if name in SCALE:
        return np.ldexp(bx, SCALE[name]), np.ldexp(by, SCALE[name])
    if name == "deep":
        return np.ldexp(bx, -70), np.ldexp(by, -70)
    if name == "narrow":
        off = np.float32(2.0 ** -26)
        return off + np.ldexp(bx, -40), off + np.ldexp(by, -40)
    if name == "twins":
        return with_twins(bx, by)
    if name == "twins_deep":
        tx, ty = with_twins(bx, by)
        return np.ldexp(tx, -70), np.ldexp(ty, -70)
    if name == "one_site":
        return np.full(n, bx[0], np.float32), np.full(n, by[0], np.float32)
    if name == "two_sites":
        k = np.arange(n) % 2
        return bx[k], by[k]
    gx, gy = O.gen_grid(n, seed)
    if name in ("grid", "grid64", "twins_nint"):
        return with_twins(gx, gy) if name == "twins_nint" else (gx, gy)
    if name == "half":
        gx = gx.copy()
        gx[1::2] += np.float32(0.5)  # shifting every city would leave every difference an integer
        return gx, gy
    if name == "wide":
        rng = np.random.default_rng(seed)
        return (rng.integers(0, 4_000_000, n).astype(np.float32), rng.integers(0, 1000, n).astype(np.float32))
    if name == "frac":
        return bx * np.float32(37.3), by * np.float32(37.3)
    if name == "twins_frac":
        return with_twins(bx * np.float32(37.3), by * np.float32(37.3))
    raise KeyError(name)


def oracle_problem(x, y, kind):
    return O.Problem(tri=O.matrix_packed_nint(x, y), n=len(x)) if kind == "nint" else O.Problem(x, y)


def starts(P, n, budget):
    """name -> (start tour, move budget): the NN tour to the local optimum, a shuffled tour for
    `budget` moves (the oracle's full search from it would take minutes)."""
    return {"nn": (O.nn_tour(P, 3), -1), "shuffled": (O.shuffle_tour(n, 11 + n), budget)}


# ---- CPU: the premises ----------------------------------------------------------------------------------

def test_regimes_and_exact_images_on_the_oracle():
    """Every instance is in its regime, and the oracle itself makes the moves of `base` on its exact
    2^-40 and 2^53 images, with every delta scaled by the same power of two."""
    for name, (kind, env, want) in INSTANCES.items():
        for n in (300, 2000):
            x, y = coords(name, n)
            assert regime(x, y, kind, env) == want, (name, n)
    x, y = coords("deep", 1000)
    d2 = (x[:, None].astype(np.float32) - x[None, :]) ** 2 + (y[:, None].astype(np.float32) - y[None, :]) ** 2
    d2 = d2[np.triu_indices(1000, 1)]
    assert d2.max() < np.float32(2.0 ** -101) and (d2 < np.finfo(np.float32).tiny).mean() > 0.02  # subnormal
    tx, _ = coords("twins", 300)
    assert (tx[200:] == tx[:100]).all() and (tx[100:120] == tx[100]).all()

    n = 300
    bx, by = coords("base", n)
    Pb = O.Problem(bx, by)
    start = O.shuffle_tour(n, 5)
    want = {"best": O.two_opt_best(Pb, start, log_cap=CAP), "ref": O.two_opt_ref(Pb, start, log_cap=CAP),
            "nl": NL.two_opt_nl(Pb, start, O.knn(Pb, 8), log_cap=CAP)}
    assert len(want["best"][2]) > 200
    for name, s in SCALE.items():
        x, y = coords(name, n)
        assert (x == np.ldexp(bx, s)).all() and (np.ldexp(x, -s) == bx).all()
        P = O.Problem(x, y)
        assert (O.knn(P, 8) == O.knn(Pb, 8)).all() and (O.nn_tour(P, 3) == O.nn_tour(Pb, 3)).all()
        got = {"best": O.two_opt_best(P, start, log_cap=CAP), "ref": O.two_opt_ref(P, start, log_cap=CAP),
               "nl": NL.two_opt_nl(P, start, O.knn(P, 8), log_cap=CAP)}
        for algo, (wt, wst, wm) in want.items():
            gt, gst, gm = got[algo]
            assert log_key(gm) == log_key(wm, s), (name, algo)
            assert (gt == wt).all() and (gst.moves, gst.passes, gst.evals) == (wst.moves, wst.passes, wst.evals)


# ---- GPU ------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def T():
    import teeline_b200 as T
    return T


@pytest.fixture(scope="module")
def ctx(T):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    c = T.Context(0)
    yield c
    c.close()


@pytest.fixture
def inst(T, ctx, monkeypatch):
    """make(name, n) -> (x, y, device problem, oracle problem), with the instance's environment set."""
    def make(name, n, seed=None):
        kind, env, want = INSTANCES[name]
        for k in ("TL_NO_SCREEN", "TL_NINT_F64", "TL_BATCH_ENGINE", "TL_BATCH_CLUSTER"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        x, y = coords(name, n, seed)
        assert regime(x, y, kind) == want, name
        prob = T.Problem.euc2d(ctx, x, y, T.DIST_NINT_I32 if kind == "nint" else T.DIST_F32_EXACT)
        return x, y, prob, oracle_problem(x, y, kind)
    return make


def same_search(got, want, what, max_moves=-1, evals=True):
    """A library search (tour, Stats, log) against the oracle's (tour, stats, log)."""
    gt, gst, gm = got
    wt, wst, wm = want
    assert log_key(gm) == log_key(wm), what
    assert (gt.astype(np.int64) == wt).all(), what
    assert (int(gst.moves), int(gst.passes)) == (wst.moves, wst.passes), what
    if evals:
        assert int(gst.evals) == wst.evals, what
    assert bool(gst.converged) == (max_moves < 0 or wst.moves < max_moves), what


def unsupported(T, call):
    with pytest.raises(T.TeelineError) as ei:
        call()
    assert ei.value.status == 3  # TL_ERR_UNSUPPORTED


ALL = list(INSTANCES)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ALL)
def test_matrix_knn_nn_tour_and_lengths(T, inst, name):
    kind = INSTANCES[name][0]
    x, y, prob, P = inst(name, 1000)
    n = len(x)
    if kind == "nint":
        assert (prob.matrix_packed() == O.matrix_packed_nint(x, y)).all()
    else:
        assert (bits(prob.matrix_packed()) == bits(O.matrix_packed_f32(x, y))).all()
    for k in (1, 7, 32):
        assert (prob.knn(k).astype(np.int64) == O.knn(P, k)).all(), k
    nn = prob.nn_tour(3)
    assert (nn.astype(np.int64) == O.nn_tour(P, 3)).all()
    tours = np.stack([nn] + [O.shuffle_tour(n, s) for s in range(1, 6)])
    want = O.tour_lengths(P, tours)
    if kind == "nint":
        assert (prob.tour_lengths(tours) == want.astype(np.int64)).all()
        return
    assert (bits(prob.tour_lengths(tours, T.LEN_EXACT)) == bits(want.astype(np.float32))).all()
    # FAST sums in another order: against a float64 sum of the same f32 edges
    tri = O.matrix_packed_f32(x, y).astype(np.float64)
    nxt = np.roll(tours, -1, axis=1)
    a, b = np.minimum(tours, nxt).astype(np.int64), np.maximum(tours, nxt).astype(np.int64)
    edges = tri[b * (b - 1) // 2 + a]  # packed order: (a, b) with a < b at b(b-1)/2 + a
    np.testing.assert_allclose(prob.tour_lengths(tours, T.LEN_FAST), edges.sum(axis=1), rtol=1e-5, atol=0)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ALL)
def test_mode_b_cyclic_and_cached(T, inst, name):
    """Mode B and cyclic Mode B on both paths, cached Mode B on both paths, and one scan of each."""
    kind = INSTANCES[name][0]
    x, y, prob, P = inst(name, 1000)
    paths = (T.PATH_RECOMPUTE, T.PATH_MATRIX) if kind == "f32" else (T.PATH_MATRIX,)
    for sname, (start, mm) in starts(P, len(x), 100).items():
        for cyclic in (False, True):
            algo = T.ALGO_TWO_OPT_BEST_CYCLIC if cyclic else T.ALGO_TWO_OPT_BEST
            want = O.two_opt_best(P, start, cyclic=cyclic, max_moves=mm, nthreads=NCPU, log_cap=CAP)
            want_scan = O.two_opt_best_scan(P, start, cyclic=cyclic, nthreads=NCPU)
            for path in paths:
                what = (sname, cyclic, path)
                got = prob.local_search(algo, start, path=path, max_moves=mm, log_cap=CAP)
                assert got[1].path_used == path, what
                same_search(got, want, what, mm)
                s = prob.session(algo, start, path)
                scan = s.scan()
                assert (scan is None) == (want_scan is None), what
                if scan is not None:
                    assert log_key([scan]) == log_key([want_scan]), what
                s.close()
                if not cyclic:
                    got = prob.local_search(T.ALGO_TWO_OPT_BEST_CACHED, start, path=path, max_moves=mm, log_cap=CAP)
                    same_search(got, want, ("cached",) + what, mm, evals=False)
                    s = prob.session(T.ALGO_TWO_OPT_BEST_CACHED, start, path)
                    unsupported(T, s.scan)
                    s.close()
            if kind == "nint":
                unsupported(T, lambda: prob.local_search(algo, start, path=T.PATH_RECOMPUTE))
                unsupported(T, lambda: prob.local_search(T.ALGO_TWO_OPT_BEST_CACHED, start, path=T.PATH_RECOMPUTE))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ALL)
def test_mode_r_persistent(T, inst, name):
    """Mode R on PATH_AUTO: the persistent cluster kernel (a few launches for the whole search)."""
    x, y, prob, P = inst(name, 1000)
    for sname, (start, _) in starts(P, len(x), -1).items():
        want = O.two_opt_ref(P, start, log_cap=CAP)
        got = prob.local_search(T.ALGO_TWO_OPT_REF, start, log_cap=CAP)
        assert int(got[1].launches) < 16, sname
        same_search(got, want, sname)
        s = prob.session(T.ALGO_TWO_OPT_REF, start)
        unsupported(T, s.scan)
        s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ALL)
def test_mode_n(T, inst, name):
    """Candidate-list 2-opt against the Mode N oracle on the library's own k-NN lists."""
    x, y, prob, P = inst(name, 2000)
    for k in (1, 8, 32):
        prob.set_candidates(k)
        K = prob.knn(k)
        assert (K.astype(np.int64) == O.knn(P, k)).all(), k
        for sname, (start, mm) in starts(P, len(x), 300).items():
            want = NL.two_opt_nl(P, start, K, max_moves=mm, nthreads=NCPU, log_cap=CAP)
            got = prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR, start, max_moves=mm, log_cap=CAP)
            assert got[1].path_used == T.PATH_RECOMPUTE
            same_search(got, want, (k, sname), mm)
            s = prob.session(T.ALGO_TWO_OPT_NEIGHBOR, start)
            scan, want_scan = s.scan(), NL.two_opt_nl_scan(P, start, K, nthreads=NCPU)[0]
            assert (scan is None) == (want_scan is None) and (scan is None or log_key([scan]) == log_key([want_scan]))
            s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ALL)
def test_or_opt(T, inst, name):
    kind = INSTANCES[name][0]
    x, y, prob, P = inst(name, 300)
    paths = (T.PATH_RECOMPUTE, T.PATH_MATRIX) if kind == "f32" else (T.PATH_MATRIX,)
    for sname, (start, mm) in starts(P, len(x), 60).items():
        want = O.or_opt(P, start, max_moves=mm, log_cap=CAP)
        want_scan = O.or_opt_find_best(P, start)
        for path in paths:
            got = prob.local_search(T.ALGO_OR_OPT, start, path=path, max_moves=mm, log_cap=CAP)
            same_search(got, want, (sname, path), mm)
            s = prob.session(T.ALGO_OR_OPT, start, path)
            scan = s.scan()
            assert (scan is None) == (want_scan is None) and (scan is None or log_key([scan]) == log_key([want_scan]))
            s.close()
        if kind == "nint":
            unsupported(T, lambda: prob.local_search(T.ALGO_OR_OPT, start, path=T.PATH_RECOMPUTE))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ALL)
def test_three_opt(T, inst, name):
    kind = INSTANCES[name][0]
    x, y, prob, P = inst(name, 120)
    paths = (T.PATH_RECOMPUTE, T.PATH_MATRIX) if kind == "f32" else (T.PATH_MATRIX,)
    for sname, (start, mm) in starts(P, len(x), 40).items():
        # a budget from the NN tour too: on `twins` the reference 3-opt cycles between two moves of equal
        # f32 gain forever
        mm = mm if mm > 0 else 60
        want = O.three_opt(P, start, max_moves=mm, nthreads=NCPU, log_cap=CAP)
        want_scan, _ = O.three_opt_find_best(P, start, nthreads=NCPU)
        for path in paths:
            got = prob.local_search(T.ALGO_THREE_OPT, start, path=path, max_moves=mm, log_cap=CAP)
            same_search(got, want, (sname, path), mm)
            s = prob.session(T.ALGO_THREE_OPT, start, path)
            scan = s.scan()
            assert (scan is None) == (want_scan is None) and (scan is None or log_key([scan]) == log_key([want_scan]))
            s.close()


ENGINES = ("pop", "cta", "cluster2", "cluster4", "cluster8", "auto")


def set_engine(monkeypatch, engine):
    monkeypatch.delenv("TL_BATCH_ENGINE", raising=False)
    monkeypatch.delenv("TL_BATCH_CLUSTER", raising=False)
    if engine == "pop":
        monkeypatch.setenv("TL_BATCH_ENGINE", "pop")
    elif engine != "auto":
        monkeypatch.setenv("TL_BATCH_ENGINE", "cta")
        monkeypatch.setenv("TL_BATCH_CLUSTER", "1" if engine == "cta" else engine[len("cluster"):])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ALL)
def test_batch_engines(T, inst, monkeypatch, name):
    kind = INSTANCES[name][0]
    x, y, prob, P = inst(name, 300)
    n = len(x)
    tours = np.stack([O.nn_tour(P, 3)] + [O.shuffle_tour(n, s) for s in range(1, 8)])
    if kind == "nint":
        unsupported(T, lambda: prob.two_opt_batch(tours))
        return
    want = [O.two_opt_best(P, t, nthreads=NCPU) for t in tours]
    for engine in ENGINES:
        set_engine(monkeypatch, engine)
        got, st, lengths = prob.two_opt_batch(tours)
        for b, (wt, _, _) in enumerate(want):
            assert (got[b].astype(np.int64) == wt).all(), (engine, b)
            assert f32_bits(lengths[b]) == f32_bits(O.tour_length(P, wt)), (engine, b)
        assert (int(st.moves), int(st.passes), int(st.evals)) == tuple(
            sum(getattr(w[1], f) for w in want) for f in ("moves", "passes", "evals")), engine
        assert st.converged == 1, engine


# ---- GPU: exact images and knobs at sizes the oracle cannot afford -------------------------------------------

def search_key(got, scale=0):
    t, st, mv = got
    return log_key(mv, scale), t.tolist(), (int(st.moves), int(st.passes), int(st.evals), int(st.converged))


def check_images(runs):
    """runs: name -> key built with the instance's scale; every one equals base's."""
    for name, key in runs.items():
        assert key == runs["base"], name


@pytest.mark.gpu
def test_exact_images_mode_b_and_cached_10k(T, inst):
    """Mode B (recompute, screened / unscreened / IEEE-safe) and cached Mode B at n = 10 000."""
    runs = {}
    for name in ("base", "noscreen", "tiny", "huge"):
        x, y, prob, _ = inst(name, 10000)
        nn = prob.nn_tour(3)
        if name == "base":
            start = nn
        assert (nn == start).all(), name
        s = -SCALE.get(name, 0)  # scale the instance's deltas back to base's
        runs[name] = [search_key(prob.local_search(a, start, path=T.PATH_RECOMPUTE, log_cap=CAP), s)
                      for a in (T.ALGO_TWO_OPT_BEST, T.ALGO_TWO_OPT_BEST_CACHED)]
    assert runs["base"][0][2][0] > 1000
    check_images(runs)


@pytest.mark.gpu
def test_exact_images_mode_r_per_step_14500(T, inst):
    """Mode R beyond kRefPersistMaxN: the launch-per-step kernel in both sqrt regimes."""
    runs = {}
    for name in ("base", "tiny", "huge"):
        x, y, prob, _ = inst(name, 14500)
        if name == "base":
            start = prob.nn_tour(3)
        got = prob.local_search(T.ALGO_TWO_OPT_REF, start, log_cap=CAP)
        assert int(got[1].launches) > 1000, name
        runs[name] = search_key(got, -SCALE.get(name, 0))
    check_images(runs)


@pytest.mark.gpu
def test_exact_images_batch_pop_13000(T, inst, monkeypatch):
    runs = {}
    for name in ("base", "noscreen", "tiny", "huge"):
        x, y, prob, _ = inst(name, 13000)
        if name == "base":
            tours = np.stack([prob.nn_tour(3)] + [O.shuffle_tour(13000, s) for s in (1, 2, 3)])
        set_engine(monkeypatch, "pop")
        got, st, lengths = prob.two_opt_batch(tours, max_moves=2000)
        s = -SCALE.get(name, 0)
        runs[name] = (got.tolist(), bits(np.ldexp(lengths, s)).tolist(),
                      (int(st.moves), int(st.passes), int(st.evals), int(st.converged)))
    assert runs["base"][2][0] > 3 * 2000
    check_images(runs)


@pytest.mark.gpu
def test_exact_images_mode_n_100k(T, inst):
    runs = {}
    for name in ("base", "tiny", "huge"):
        x, y, prob, _ = inst(name, 100_000)
        if name == "base":
            start = prob.nn_tour(3)
        prob.set_candidates(8)
        got = prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR, start, log_cap=CAP)
        runs[name] = (prob.knn(8).tolist(), search_key(got, -SCALE.get(name, 0)))
    assert runs["base"][1][2][3] == 1
    check_images(runs)


def all_outputs(T, prob, kind, monkeypatch):
    """Every output of the kernels that have a screened / unscreened or a grid / f64 instantiation."""
    n = prob.n
    nn = prob.nn_tour(3)
    out = {"matrix": prob.matrix_packed().tobytes(), "knn": prob.knn(8).tolist(), "nn": nn.tolist()}
    out["best"] = search_key(prob.local_search(T.ALGO_TWO_OPT_BEST, nn, max_moves=300, log_cap=CAP))
    out["cyclic"] = search_key(prob.local_search(T.ALGO_TWO_OPT_BEST_CYCLIC, nn, max_moves=300, log_cap=CAP))
    out["cached"] = search_key(prob.local_search(T.ALGO_TWO_OPT_BEST_CACHED, nn, max_moves=300, log_cap=CAP))
    out["ref"] = search_key(prob.local_search(T.ALGO_TWO_OPT_REF, nn, log_cap=CAP))
    prob.set_candidates(8)
    out["nl"] = search_key(prob.local_search(T.ALGO_TWO_OPT_NEIGHBOR, nn, log_cap=CAP))
    out["or"] = search_key(prob.local_search(T.ALGO_OR_OPT, nn, max_moves=30, log_cap=CAP))
    if kind == "f32":
        tours = np.stack([nn] + [O.shuffle_tour(n, s) for s in (1, 2, 3)])
        for engine in ("pop", "cta", "auto"):
            set_engine(monkeypatch, engine)
            got, st, lengths = prob.two_opt_batch(tours, max_moves=100)
            out["batch-" + engine] = (got.tolist(), bits(lengths).tolist(), (int(st.moves), int(st.evals)))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("pair", [("base", "noscreen"), ("grid", "grid64")])
def test_knobs_leave_every_output_unchanged(T, inst, monkeypatch, pair):
    """TL_NO_SCREEN switches the screened kernels to their unscreened instantiations and TL_NINT_F64
    the integer nint kernels to the f64 ones: neither may change any output."""
    outs = []
    for name in pair:
        x, y, prob, _ = inst(name, 5000)
        outs.append(all_outputs(T, prob, INSTANCES[name][0], monkeypatch))
    assert outs[0]["ref"][2][3] == 1
    for key in outs[0]:
        assert outs[0][key] == outs[1][key], key
