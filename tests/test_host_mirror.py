"""The C++ host mirror of the reference interface (teeline_b200/host/) and its `teeline` CLI stand-in.

CPU tests: the binaries build, config/argument errors match the reference's messages and exit
codes (src/config.rs:82-153, teeline-cli/src/main.rs), and no device call is reachable without a
GPU.  GPU tests: the reference's published goldens through the CLI, and the library-level API
(DistanceMatrix::{distances,nearest,tour_length}, build_candidates, solve_with_context with a
progress sink) against the oracle."""
import json
import os
import subprocess
import zlib

import numpy as np
import pytest

import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def bins():
    from teeline_b200 import build as tb, build_host
    tb.build()
    cli = build_host.build()
    return cli, build_host.SELFTEST


def run(cmd, stdin=None, cwd=None):
    p = subprocess.run(cmd, capture_output=True, text=True, input=stdin, timeout=600, cwd=cwd)
    return p.returncode, p.stdout, p.stderr


# ---- CPU: surface, errors, exit codes ---------------------------------------------------------------

def test_cli_builds_and_lists_solvers(bins):
    rc, out, _ = run([bins[0], "solvers"])
    assert rc == 0 and "2opt" in out and "or_opt" in out and "nn" in out


def test_cli_convert_discopt_fixture(bins, tmp_path):
    """`teeline convert` on the reference's DiscOpt fixture (tests/e2e/convert.bats:18-31;
    writer format src/tsp/convert.rs:32-45: tab, 1-based id, Rust `{}` floats)."""
    cli = bins[0]
    rc, _, err = run([cli, "convert", "-i", os.path.join(GOLDEN, "tiny5_discopt"), "-o", str(tmp_path)])
    assert rc == 0, err
    out = tmp_path / "tiny5_discopt.tsp"
    assert out.read_text() == ("NAME: tiny5_discopt\nTYPE: TSP\nCOMMENT: converted from DiscOpt dataset tiny5_discopt\n"
                               "DIMENSION: 5\nEDGE_WEIGHT_TYPE: EUC_2D\nNODE_COORD_SECTION\n"
                               "\t1 0 0\n\t2 10 0\n\t3 10 10\n\t4 0 10\n\t5 5 5\nEOF\n")
    rc, _, _ = run([cli, "convert", "-i", "/nonexistent/file"], cwd=tmp_path)  # default output: ./data/discopt
    assert rc != 0
    frac = tmp_path / "frac.txt"
    frac.write_text("3\n0.5 1e3\n\n-2.25 0.1\n7 8\n")
    rc, _, _ = run([cli, "convert", "-i", str(frac), "-o", str(tmp_path / "x.tsp")])
    assert rc == 0 and "\t1 0.5 1000\n\t2 -2.25 0.1\n\t3 7 8\n" in (tmp_path / "x.tsp").read_text()
    bad = tmp_path / "bad.txt"
    bad.write_text("2\n1 2\n3\n")
    rc, _, err = run([cli, "convert", "-i", str(bad), "-o", str(tmp_path)])
    assert rc == 1 and "missing y" in err


def test_cli_config_errors_match_reference_messages(bins, tmp_path):
    cli = bins[0]
    inp = os.path.join(GOLDEN, "berlin52.tsp")
    rc, _, err = run([cli, "pipeline", "--config", os.path.join(GOLDEN, "pipeline_unknown_key.toml"), "-i", inp])
    assert rc == 1 and "config: unknown field `epoch` — valid stage fields: solver, sa, ga, cs, fpa, fourier, lk, som, aco, heuristic" in err
    cases = {
        "": "config: missing [[stage]] array — at least one stage is required",
        "stage = 3\n": "config: `stage` must be an array of tables ([[stage]])",
        "[[stage]]\nfoo = 1\n": "config: [[stage]] entry 0 missing required `solver` field",
        "[[stage]]\nsolver = 7\n": "config: [[stage]] entry 0: `solver` must be a string",
        "[[stage]]\nsolver = \"warp\"\n": "config: [[stage]] entry 0: unknown solver `warp`",
        "[[stage]]\nsolver = \"2opt\"\n[stage.sa]\ncooling_rate = 0.5\n": "config: stage 0 (2opt): `[stage.sa]` is not valid for this solver",
        "[[stage]]\nsolver = \"sa\"\n[stage.heuristic]\nepochs = 5\n": "config: stage 0 (sa): `[stage.heuristic]` is not valid for this solver",
        "[[stage]]\nsolver = \"nn\"\n[stage.heuristic]\nn_nearest = 0\n": "n_nearest must be >= 1",
        "[[stage]]\nsolver = \"nn\"\n[stage.heuristic]\nepochs = \"x\"\n": "config: `epochs` must be an integer, got \"x\"",
        "[[stage]]\nsolver = \"nn\"\n[stage.heuristic]\nspeed = 1\n": "config: unknown field `speed` in [heuristic] — valid: epochs, platoo_epochs, n_nearest, verbose",
        "[[stage]]\nsolver = \"nn\"\nheuristic = 4\n": "config: `heuristic` must be a table",
        "[[stage]\nsolver = \"nn\"\n": "config: TOML parse error",
    }
    for k, (src, want) in enumerate(cases.items()):
        f = tmp_path / f"c{k}.toml"
        f.write_text(src)
        rc, _, err = run([cli, "pipeline", "--config", str(f), "-i", inp])
        assert rc == 1 and want in err, (src, err)


def test_cli_population_option_errors_match_reference_messages(bins, tmp_path):
    """[stage.aco] / [stage.ga] tables and the matching CLI flags: AcoOptions / GAOptions from_toml and
    validate (src/tsp/mod.rs:1114-1196, 832-890), same messages."""
    cli = bins[0]
    inp = os.path.join(GOLDEN, "berlin52.tsp")
    cases = {
        "[[stage]]\nsolver = \"aco\"\n[stage.aco]\nalpha = -1.0\n": "alpha must be >= 0 (got -1)",
        "[[stage]]\nsolver = \"aco\"\n[stage.aco]\nbeta = 7\n": "beta must be in [0, 6] (got 7)",
        "[[stage]]\nsolver = \"aco\"\n[stage.aco]\nevaporation_rate = 1.0\n": "evaporation_rate must be in (0, 1) (got 1)",
        "[[stage]]\nsolver = \"aco\"\n[stage.aco]\nnum_ants = 0\n": "num_ants must be >= 1",
        "[[stage]]\nsolver = \"aco\"\n[stage.aco]\nants = 3\n":
            "config: unknown field `ants` in [aco] — valid: epochs, platoo_epochs, n_nearest, verbose, alpha, beta, evaporation_rate, num_ants",
        "[[stage]]\nsolver = \"aco\"\n[stage.aco]\nalpha = \"x\"\n": "config: `aco.alpha` must be a float, got \"x\"",
        "[[stage]]\nsolver = \"ga\"\n[stage.ga]\nmutation_probability = 1.5\n": "mutation_probability must be in [0, 1] (got 1.5)",
        "[[stage]]\nsolver = \"ga\"\n[stage.ga]\nn_elite = \"many\"\n": "config: `ga.n_elite` must be an integer, got \"many\"",
        "[[stage]]\nsolver = \"ga\"\n[stage.ga]\nelite = 1\n":
            "config: unknown field `elite` in [ga] — valid: epochs, platoo_epochs, n_nearest, verbose, mutation_probability, n_elite",
        "[[stage]]\nsolver = \"ga\"\n[stage.aco]\nalpha = 1.0\n": "config: stage 0 (ga): `[stage.aco]` is not valid for this solver",
    }
    for k, (src, want) in enumerate(cases.items()):
        f = tmp_path / f"p{k}.toml"
        f.write_text(src)
        rc, _, err = run([cli, "pipeline", "--config", str(f), "-i", inp])
        assert rc == 1 and want in err, (src, err)
    rc, _, err = run([cli, "solve", "aco", "--beta", "9", "-i", inp])
    assert rc == 1 and "beta must be in [0, 6] (got 9)" in err
    rc, _, err = run([cli, "solve", "ga", "--mutation_probability", "2", "-i", inp])
    assert rc == 1 and "mutation_probability must be in [0, 1] (got 2)" in err


def test_cli_argument_errors(bins):
    cli = bins[0]
    inp = os.path.join(GOLDEN, "berlin52.tsp")
    rc, _, err = run([cli, "pipeline", "-i", inp])
    assert rc == 1 and "one of --config <PATH> or --steps <SOLVERS> is required" in err
    rc, _, err = run([cli, "pipeline", "--steps", "nn,bogus", "-i", inp])
    assert rc == 1 and "unknown solver at --steps position 1: 'bogus'" in err
    rc, _, err = run([cli, "pipeline", "--steps", "nn", "--config", "x.toml", "-i", inp])
    assert rc == 1 and "--config and --steps are mutually exclusive" in err
    rc, _, err = run([cli, "solve", "2opt", "-i", "/nonexistent/file.tsp"])
    assert rc == 1 and "input file not found" in err
    rc, _, err = run([cli, "solve", "warp", "-i", inp])
    assert rc == 2
    rc, _, err = run([cli, "solve", "2opt", "--n_nearest", "0", "-i", inp])
    assert rc == 1 and "n_nearest must be >= 1" in err
    rc, _, err = run([cli, "solve", "2opt"], stdin="NAME: x\nTYPE: ATSP\nEOF\n")
    assert rc == 1 and "ATSP (asymmetric TSP) is not supported" in err
    rc, _, err = run([cli, "solve", "2opt"], stdin="garbage line\n")
    assert rc == 1 and "Failed to extract meta data on line." in err


@pytest.mark.skipif(os.path.exists("/dev/nvidiactl"), reason="needs a box WITHOUT a GPU")
def test_cli_has_no_cpu_fallback(bins):
    rc, out, err = run([bins[0], "solve", "2opt", "-i", os.path.join(GOLDEN, "berlin52.tsp")])
    assert rc == 101 and out == "" and "no CPU fallback" in err


# ---- GPU: goldens through the CLI ------------------------------------------------------------------------

def parse_cli(out):
    first, second = out.strip().split("\n")[:2]
    total, flag = first.split()
    return total, int(flag), [int(t) for t in second.split()]


def ids_and_problem(name):
    ids, x, y = O.read_tsplib_coords(os.path.join(GOLDEN, name))
    return ids, O.Problem(x, y)


@pytest.mark.gpu
def test_cli_goldens_berlin52(bins):
    cli = bins[0]
    inp = os.path.join(GOLDEN, "berlin52.tsp")
    ids, P = ids_and_problem("berlin52.tsp")
    nn = O.nn_tour(P, 3)
    # G1: `teeline solve nn` (bench/baseline-solvers.tsv:2-6)
    rc, out, _ = run([cli, "solve", "nn", "-i", inp])
    assert rc == 0 and parse_cli(out) == ("8980.91797", 0, [int(ids[p]) for p in nn])
    # G5: `teeline solve 2opt` = nn -> 2opt (README.md:385); `fast` preset is the same pipeline
    want = [int(ids[p]) for p in O.two_opt_ref(P, nn)[0]]
    for argv in (["solve", "2opt"], ["solve", "fast"], ["solve", "two_opt"], ["pipeline", "--steps", "nn,2opt"],
                 ["pipeline", "--config", os.path.join(GOLDEN, "pipeline_nn_2opt.toml")]):
        rc, out, _ = run([cli] + argv + ["-i", inp])
        assert rc == 0 and parse_cli(out) == ("8384.18848", 0, want), argv
    # G4: `--no-seed` starts from input order (docs/benchmarks.md:28)
    rc, out, _ = run([cli, "solve", "2opt", "--no-seed", "-i", inp])
    assert rc == 0 and parse_cli(out)[0] == "9368.31836"
    # G6: `teeline solve or_opt` (docs/benchmarks.md:48)
    rc, out, _ = run([cli, "solve", "or_opt", "-i", inp])
    assert rc == 0 and parse_cli(out) == ("8097.47607", 0, [int(ids[p]) for p in O.or_opt(P, nn)[0]])
    # G7: `teeline solve 3opt` = nn -> 3opt (docs/benchmarks.md:29)
    rc, out, _ = run([cli, "solve", "3opt", "-i", inp])
    assert rc == 0 and parse_cli(out) == ("7742.64697", 0, [int(ids[p]) for p in O.three_opt(P, nn)[0]])
    # stdin input + JSON output (main.rs:694-707)
    rc, out, _ = run([cli, "solve", "2opt", "--output-format", "json"], stdin=open(inp).read())
    obj = json.loads(out)
    assert rc == 0 and obj["route"] == want and obj["optimized"] is False and abs(obj["cost"] - 8384.18848) < 1e-3
    # the matrix path and the best-improvement extension
    rc, out, _ = run([cli, "solve", "2opt", "--path", "matrix", "-i", inp])
    assert rc == 0 and parse_cli(out) == ("8384.18848", 0, want)
    rc, out, _ = run([cli, "solve", "2opt_best", "-i", inp])
    tb = O.two_opt_best(P, nn)[0]
    assert rc == 0 and parse_cli(out) == ("%.5f" % O.tour_length(P, tb), 0, [int(ids[p]) for p in tb])


@pytest.mark.gpu
def test_cli_population_solvers(bins, tmp_path):
    """`teeline solve aco|ga` (= shuffle -> solver, main.rs:387-397) and a [[stage]] pipeline with
    [stage.aco] / [stage.ga] tables: a valid tour whose printed cost is its exact-order length; the
    same seed gives the same run; nn -> aco never ends worse than its warm start (ant_colony.rs:358-381)."""
    cli = bins[0]
    inp = os.path.join(GOLDEN, "berlin52.tsp")
    ids, P = ids_and_problem("berlin52.tsp")
    pos = {int(c): k for k, c in enumerate(ids)}

    def check(argv):
        rc, out, err = run([cli] + argv + ["-i", inp])
        assert rc == 0, err
        total, flag, route = parse_cli(out)
        assert sorted(route) == sorted(int(c) for c in ids) and flag == 0
        assert total == "%.5f" % O.tour_length(P, [pos[c] for c in route])
        return float(total), route

    a1 = check(["solve", "aco", "--seed", "3"])
    assert a1 == check(["solve", "aco", "--seed", "3"]) and a1[0] < 7542 * 1.25
    g1 = check(["solve", "ga", "--seed", "3", "--epochs", "2000"])
    assert g1 == check(["solve", "ga", "--seed", "3", "--epochs", "2000"]) and g1[0] < 7542 * 1.6
    assert g1 != check(["solve", "ga", "--seed", "4", "--epochs", "2000"])
    cfg = tmp_path / "pop.toml"
    cfg.write_text("[[stage]]\nsolver = \"nn\"\n[[stage]]\nsolver = \"aco\"\n[stage.aco]\nepochs = 40\nnum_ants = 10\n"
                   "[stage.cuda]\nseed = 5\n[[stage]]\nsolver = \"ga\"\n[stage.ga]\nepochs = 300\nn_elite = 2\n")
    total, _ = check(["pipeline", "--config", str(cfg)])
    assert total <= 8980.91797  # nn's G1 length: aco keeps its warm start as the incumbent, ga seeds it as an elite
    # the same stages against the oracle port, stage by stage
    nn = O.nn_tour(P, 3)
    t_aco, _, _ = O.aco(P, 5, init_tour=nn, epochs=40, num_ants=10)
    t_ga, c_ga, _ = O.ga(P, 0, init_tour=t_aco, epochs=300, n_elite=2)
    assert total == float("%.5f" % c_ga)


@pytest.mark.gpu
def test_cli_discopt_to_solve(bins, tmp_path):
    """DiscOpt input end to end: `teeline convert` then `teeline solve 2opt|or_opt` on the result
    (src/tsp/convert.rs -> src/tsp/tsplib.rs -> the accelerated stages), against the oracle."""
    cli = bins[0]
    rc, _, err = run([cli, "convert", "-i", os.path.join(GOLDEN, "tiny5_discopt"), "-o", str(tmp_path)])
    assert rc == 0, err
    inp = str(tmp_path / "tiny5_discopt.tsp")
    ids, x, y = O.read_tsplib_coords(inp)
    assert ids.tolist() == [1, 2, 3, 4, 5] and x.tolist() == [0, 10, 10, 0, 5] and y.tolist() == [0, 0, 10, 10, 5]
    P = O.Problem(x, y)
    nn = O.nn_tour(P, 3)
    for name, want in (("nn", nn), ("2opt", O.two_opt_ref(P, nn)[0]), ("or_opt", O.or_opt(P, nn)[0])):
        rc, out, err = run([cli, "solve", name, "-i", inp])
        assert rc == 0 and parse_cli(out) == ("%.5f" % O.tour_length(P, want), 0, [int(ids[p]) for p in want]), (name, err)
    # a 200-city DiscOpt file with fractional coordinates
    rng = np.random.default_rng(5)
    pts = (rng.random((200, 2)) * 1000).astype(np.float32)
    src = tmp_path / "rand200"
    src.write_text("200\n" + "".join(f"{a!r} {b!r}\n" for a, b in pts.tolist()))
    rc, _, err = run([cli, "convert", "-i", str(src), "-o", str(tmp_path / "rand200.tsp")])
    assert rc == 0, err
    ids, x, y = O.read_tsplib_coords(str(tmp_path / "rand200.tsp"))
    assert (x == pts[:, 0]).all() and (y == pts[:, 1]).all()  # the shortest round-trip decimals parse back exactly
    P = O.Problem(x, y)
    want = O.two_opt_ref(P, O.nn_tour(P, 3))[0]
    rc, out, _ = run([cli, "solve", "2opt", "-i", str(tmp_path / "rand200.tsp")])
    assert rc == 0 and parse_cli(out) == ("%.5f" % O.tour_length(P, want), 0, [int(ids[p]) for p in want])


@pytest.mark.gpu
def test_cli_att532_nn_golden_and_warning(bins):
    inp = os.path.join(GOLDEN, "att532.tsp")
    rc, out, _ = run([bins[0], "solve", "nn", "-i", inp])  # G2: ATT header is treated as EUC_2D
    assert rc == 0 and parse_cli(out)[0] == "112099.42188"
    rc, out, err = run([bins[0], "pipeline", "--steps", "2opt,nn", "-i", os.path.join(GOLDEN, "berlin52.tsp")])
    assert rc == 0 and "warning: nn at stage 1 discards the warm-start seed from the previous stage" in err
    assert parse_cli(out)[0] == "8980.91797"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["gr17.tsp", "ring6_explicit.tsp", "burma14.tsp"])
def test_cli_explicit_and_geo_instances(bins, name):
    """EXPLICIT (FULL_MATRIX / LOWER_DIAG_ROW) and GEO instances: matrix path only."""
    rc, out, err = run([bins[0], "solve", "2opt", "-i", os.path.join(GOLDEN, name)])
    assert rc == 0, err
    total, flag, route = parse_cli(out)
    n = len(route)
    assert sorted(route) == list(range(1, n + 1)) and flag == 0
    rc2, out2, _ = run([bins[0], "solve", "or_opt", "-i", os.path.join(GOLDEN, name)])
    assert rc2 == 0 and sorted(parse_cli(out2)[2]) == list(range(1, n + 1))
    if name == "gr17.tsp":  # tests/solvers_integration.rs:368-386: 2-opt < 1.5 x optimal (2085)
        assert float(total) < 1.5 * 2085


# ---- GPU: library-level API against the oracle ------------------------------------------------------------

def fnv(bits):
    h = 1469598103934665603
    for b in bits.tolist():
        h = ((h ^ b) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return "%016x" % h


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["berlin52.tsp", "a280.tsp"])
def test_host_library_api(bins, name):
    rc, out, err = run([bins[1], os.path.join(GOLDEN, name)])
    assert rc == 0, err
    got = json.loads(out)
    ids, P = ids_and_problem(name)
    n = len(ids)
    _, x, y = O.read_tsplib_coords(os.path.join(GOLDEN, name))
    tri = O.matrix_packed_f32(x, y)
    assert got["n"] == n and got["matrix_len"] == n * (n - 1) // 2 and got["matrix_fnv"] == fnv(tri.view(np.uint32))
    d = np.float32(O.distance(P, 0, n - 1)).view(np.uint32)
    assert got["d_first_last_bits"] == [int(d), int(d)] and got["d_unknown_is_none"] is True
    knn5 = O.knn(P, 5)
    knn3 = O.knn(P, 3)
    assert got["nearest_k3_first"] == [int(ids[q]) for q in knn3[0]]
    assert got["nearest_k5_last"] == [int(ids[q]) for q in knn5[n - 1]]
    assert got["candidates_first"] == [int(ids[q]) for q in knn5[0]] and got["candidates_last"] == got["nearest_k5_last"]
    assert got["nearest_unknown_len"] == 0
    ident = np.arange(n)
    assert got["len_identity_bits"] == int(np.float32(O.tour_length(P, ident)).view(np.uint32))
    assert got["len_unknown_id"] == 0.0
    assert got["len_batch_bits"] == [int(np.float32(O.tour_length(P, t)).view(np.uint32)) for t in (ident, ident[::-1].copy())]
    nn = O.nn_tour(P, 3)
    if name == "berlin52.tsp":
        assert got["nn_route"] == [int(ids[p]) for p in nn]
        assert (got["nn_total"], got["two_opt_total"], got["or_opt_total"], got["two_opt_noseed_total"]) == \
            ("8980.91797", "8384.18848", "8097.47607", "9368.31836")
    else:
        nn = np.array([list(ids).index(i) for i in got["nn_route"]])  # a280 has exact ties (nondeterministic in the reference)
        assert sorted(got["nn_route"]) == sorted(int(i) for i in ids)
    t_ref, st_ref, _ = O.two_opt_ref(P, nn)
    assert got["two_opt_route"] == [int(ids[p]) for p in t_ref]
    # one PathUpdate for the start tour + one per applied move, then Done (two_opt.rs:22-24,53-56,63-65)
    assert got["two_opt_updates"] == st_ref.moves + 1 and got["two_opt_dones"] == 1 and got["two_opt_last_update_is_final"]
    t_or, st_or, _ = O.or_opt(P, nn)
    assert got["or_opt_route"] == [int(ids[p]) for p in t_or] and got["or_opt_updates"] == st_or.moves + 1
    assert got["or_opt_last_total_bits"] == got["or_opt_total_bits"]  # or_opt.rs:62-67 sends the tour length
    t_best = O.two_opt_best(P, nn)[0]
    assert got["two_opt_best_route"] == [int(ids[p]) for p in t_best]
    assert got["sa_is_err"] is True and got["n_nearest_zero_error"] == "n_nearest must be >= 1"
    assert got["validate_dup"] == "tour contains invalid or duplicate city IDs"
