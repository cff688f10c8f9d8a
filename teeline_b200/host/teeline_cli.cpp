// teeline_cli.cpp -- stand-in for `teeline solve|pipeline|convert|solvers` (teeline-cli/src/main.rs) over the
// C++ host mirror, for the solvers on the accelerated path.  Same argument names, same stdout
// format ("{total:.5} {0|1}\n<ids...>\n", main.rs:645-652; JSON object :694-707), same auto-expansion
// (`solve 2opt` = nn -> 2opt unless --no-seed, main.rs:387-397), same exit codes for config errors.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <sstream>
#include <string>
#include <vector>

#include "teeline_host.hpp"

using namespace teeline;
using namespace teeline::tsp;

namespace {

struct Args {
    std::string cmd, solver, input, output, config, output_format = "text", distance_type, mode, path;
    std::vector<std::string> steps;
    bool no_seed = false, verbose = false;
    std::optional<size_t> epochs, platoo_epochs, n_nearest, n_elite, num_ants;
    std::optional<float> mutation_probability, alpha, beta, evaporation_rate;
    uint64_t seed = 0; // extension: Philox key of the population solvers
    uint32_t candidates = 0; // extension: k of `--mode neighbor` (0 = the library's default)
};

[[noreturn]] void die(const std::string &msg, int code = 1)
{
    std::fprintf(stderr, "error: %s\n", msg.c_str());
    std::exit(code);
}

std::vector<std::string> split(const std::string &s, char sep)
{
    std::vector<std::string> v;
    std::string t;
    std::istringstream is(s);
    while (std::getline(is, t, sep))
        if (!t.empty()) v.push_back(t);
    return v;
}

Args parse_args(int argc, char **argv)
{
    Args a;
    if (argc < 2) die("usage: teeline <solve|pipeline|convert|solvers> ...", 2);
    a.cmd = argv[1];
    for (int k = 2; k < argc; ++k) {
        const std::string s = argv[k];
        auto next = [&](const char *name) -> std::string {
            if (k + 1 >= argc) die(std::string("a value is required for '") + name + "'", 2);
            return argv[++k];
        };
        if (s == "-i" || s == "--input") a.input = next("--input");
        else if ((s == "-o" || s == "--output") && a.cmd == "convert") a.output = next("--output");
        else if (s == "--no-seed") a.no_seed = true;
        else if (s == "-v" || s == "--verbose") a.verbose = true;
        else if (s == "--output-format") a.output_format = next("--output-format");
        else if (s == "--distance-type") a.distance_type = next("--distance-type");
        else if (s == "--config") a.config = next("--config");
        else if (s == "--steps") { for (auto &t : split(next("--steps"), ',')) a.steps.push_back(t); }
        else if (s == "--epochs") a.epochs = std::strtoull(next("--epochs").c_str(), nullptr, 10);
        else if (s == "--platoo_epochs") a.platoo_epochs = std::strtoull(next("--platoo_epochs").c_str(), nullptr, 10);
        else if (s == "--n_nearest") a.n_nearest = std::strtoull(next("--n_nearest").c_str(), nullptr, 10);
        else if (s == "--n_elite") a.n_elite = std::strtoull(next("--n_elite").c_str(), nullptr, 10);
        else if (s == "--mutation_probability") a.mutation_probability = std::strtof(next("--mutation_probability").c_str(), nullptr);
        else if (s == "--alpha") a.alpha = std::strtof(next("--alpha").c_str(), nullptr);
        else if (s == "--beta") a.beta = std::strtof(next("--beta").c_str(), nullptr);
        else if (s == "--evaporation-rate") a.evaporation_rate = std::strtof(next("--evaporation-rate").c_str(), nullptr);
        else if (s == "--num-ants") a.num_ants = std::strtoull(next("--num-ants").c_str(), nullptr, 10);
        else if (s == "--seed") a.seed = std::strtoull(next("--seed").c_str(), nullptr, 10);
        else if (s == "--mode") a.mode = next("--mode");  // extension: ref | best | best_cyclic | neighbor | neighbor_multi (or_opt: neighbor | neighbor_multi, 3opt: neighbor)
        else if (s == "--candidates") { // extension: k nearest candidates of --mode neighbor, 1..32
            const std::string v = next("--candidates");
            char *end = nullptr;
            const unsigned long long k = std::strtoull(v.c_str(), &end, 10);
            if (v.empty() || *end || k < 1 || k > 32)
                die("invalid value '" + v + "' for '--candidates <K>': must be an integer in 1..32", 2);
            a.candidates = (uint32_t)k;
        }
        else if (s == "--path") a.path = next("--path");  // extension: auto | matrix | recompute
        else if (!s.empty() && s[0] != '-' && a.cmd == "solve" && a.solver.empty()) a.solver = s;
        else die("unexpected argument '" + s + "' found", 2);
    }
    return a;
}

AppOptions options_from_args(const Args &a)
{
    AppOptions o;
    HeuristicOptions h;
    if (a.epochs) h.epochs = *a.epochs;
    if (a.platoo_epochs) h.platoo_epochs = *a.platoo_epochs;
    if (a.n_nearest) h.n_nearest = *a.n_nearest;
    h.verbose = a.verbose;
    auto v = h.validate();
    if (v.is_err()) die(v.error);
    o.heuristic = h;
    // AcoOptions::from_cli / GAOptions::from_cli (mod.rs:1198-1240, 892-905): the solver's own defaults
    // (ACO: 150 epochs) unless a flag is given
    AcoOptions aco;
    if (a.epochs) aco.heuristic.epochs = *a.epochs;
    if (a.platoo_epochs) aco.heuristic.platoo_epochs = *a.platoo_epochs;
    if (a.alpha) aco.alpha = *a.alpha;
    if (a.beta) aco.beta = *a.beta;
    if (a.evaporation_rate) aco.evaporation_rate = *a.evaporation_rate;
    if (a.num_ants) aco.num_ants = *a.num_ants;
    auto av = aco.validate();
    if (av.is_err()) die(av.error);
    o.aco = aco;
    GAOptions ga;
    ga.heuristic = h;
    if (a.mutation_probability) ga.mutation_probability = *a.mutation_probability;
    if (a.n_elite) ga.n_elite = *a.n_elite;
    auto gv = ga.validate();
    if (gv.is_err()) die(gv.error);
    o.ga = ga;
    o.cuda_seed = a.seed;
    o.cuda_mode = a.mode;
    o.cuda_path = a.path;
    o.cuda_candidates = a.candidates;
    return o;
}

void print_solution(const Solution &tour, bool optimized)
{
    std::printf("%.5f %d\n", tour.total, optimized ? 1 : 0);
    for (size_t id : tour.route()) std::printf("%zu ", id);
    std::printf("\n");
}

void print_solution_json(const Solution &tour, bool optimized)
{
    std::printf("{\"cost\":%.9g,\"optimized\":%s,\"route\":[", tour.total, optimized ? "true" : "false");
    for (size_t k = 0; k < tour.route().size(); ++k) std::printf("%s%zu", k ? "," : "", tour.route()[k]);
    std::printf("]}\n");
}

int run_stages(const std::vector<std::pair<Solvers, AppOptions>> &stage_configs, const Args &a)
{
    std::vector<Solvers> solvers;
    for (auto &sc : stage_configs) solvers.push_back(sc.first);
    for (const std::string &w : pipeline::stage_warnings(solvers)) std::fprintf(stderr, "warning: %s\n", w.c_str());

    Result<tsplib::TspLibData> data = Result<tsplib::TspLibData>::err("");
    if (!a.input.empty()) {
        std::ifstream probe(a.input);
        if (!probe) die("input file not found: " + a.input);
        data = tsplib::read_from_file(a.input);
    } else {
        std::stringstream ss;
        ss << std::cin.rdbuf();
        data = tsplib::read_from_str(ss.str());
    }
    if (data.is_err()) die(data.error);
    tsplib::TspLibData d = std::move(data.unwrap());
    if (!a.distance_type.empty()) {
        auto dt = parse_distance_type(a.distance_type);
        if (dt.is_err()) die("--distance-type: " + dt.error);
        d.distance_type = dt.unwrap();
    }
    auto dm = d.distance_matrix();
    if (dm.is_err()) {
        std::fprintf(stderr, "Error building distance matrix: %s\n", dm.error.c_str());
        return 1;
    }
    std::vector<pipeline::PipelineStage> stages;
    for (auto &sc : stage_configs) {
        pipeline::PipelineStage st;
        st.solver = sc.first;
        st.options = sc.second;
        st.problem = TspProblem{d.cities, dm.unwrap()}; // the device problem is shared, not cloned per stage
        stages.push_back(std::move(st));
    }
    auto tour = pipeline::run_pipeline(stages);
    if (tour.is_err()) {
        std::fprintf(stderr, "solver failed: %s\n", tour.error.c_str());
        return 101; // the reference panics here (`.expect("solver failed")`)
    }
    if (a.output_format == "json") print_solution_json(tour.unwrap(), false);
    else print_solution(tour.unwrap(), false);
    return 0;
}

int run_solve(const Args &a)
{
    if (a.solver.empty()) die("the following required arguments were not provided: <solver>", 2);
    std::vector<Solvers> steps;
    if (a.solver == "fast") steps = {Solvers::NearestNeighbor, Solvers::TwoOpt}; // main.rs:354-369
    else if (a.solver == "classic") steps = {Solvers::NearestNeighbor, Solvers::TwoOpt, Solvers::SimulatedAnnealing};
    else if (a.solver == "thorough") steps = {Solvers::NearestNeighbor, Solvers::ThreeOpt, Solvers::SimulatedAnnealing};
    else {
        auto s = find_solver(a.solver);
        if (s.is_err()) die("invalid value '" + a.solver + "' for '<solver>'", 2);
        if (!a.no_seed && auto_expand_with_nn(s.unwrap())) steps = {Solvers::NearestNeighbor, s.unwrap()};
        else if (!a.no_seed && auto_expand_with_shuffle(s.unwrap())) steps = {Solvers::RandomShuffle, s.unwrap()};
        else steps = {s.unwrap()};
    }
    std::vector<std::pair<Solvers, AppOptions>> cfg;
    for (Solvers s : steps) cfg.push_back({s, options_from_args(a)});
    return run_stages(cfg, a);
}

int run_pipeline_cmd(const Args &a)
{
    if (!a.config.empty() && !a.steps.empty()) die("--config and --steps are mutually exclusive — provide one or the other");
    if (!a.config.empty()) {
        std::ifstream f(a.config);
        if (!f) die("config: cannot read " + a.config);
        std::stringstream ss;
        ss << f.rdbuf();
        auto cfg = config::load_pipeline_config(ss.str(), AppOptions{});
        if (cfg.is_err()) die(cfg.error);
        return run_stages(cfg.unwrap(), a);
    }
    if (a.steps.empty()) die("one of --config <PATH> or --steps <SOLVERS> is required");
    std::vector<std::pair<Solvers, AppOptions>> cfg;
    for (size_t i = 0; i < a.steps.size(); ++i) {
        auto s = find_solver(a.steps[i]);
        if (s.is_err()) die("unknown solver at --steps position " + std::to_string(i) + ": '" + a.steps[i] + "'");
        cfg.push_back({s.unwrap(), options_from_args(a)});
    }
    return run_stages(cfg, a);
}

// `teeline convert -i <DiscOpt file> [-o <file or dir>]` (teeline-cli/src/main.rs:532-562, single-file form)
int run_convert(const Args &a)
{
    if (a.input.empty()) die("the following required arguments were not provided: --input <PATH>", 2);
    std::string out = a.output.empty() ? "./data/discopt" : a.output;
    std::string stem = a.input.substr(a.input.find_last_of('/') == std::string::npos ? 0 : a.input.find_last_of('/') + 1);
    const size_t dot = stem.find_last_of('.');
    if (dot != std::string::npos && dot != 0) stem = stem.substr(0, dot);
    // an output without extension (or an existing directory) is a directory: <out>/<stem>.tsp
    const std::string leaf = out.substr(out.find_last_of('/') == std::string::npos ? 0 : out.find_last_of('/') + 1);
    const bool has_ext = leaf.find('.') != std::string::npos && leaf.find_last_of('.') != 0;
    if (!has_ext) {
        std::string cmd = "mkdir -p '" + out + "'";
        if (std::system(cmd.c_str()) != 0) die("cannot create " + out);
        out += "/" + stem + ".tsp";
    }
    auto r = tsp::convert::convert_file(a.input, out);
    if (r.is_err()) die(r.error);
    return 0;
}

int run_solvers()
{
    std::printf("solvers on the accelerated (CUDA, sm_100a) path of this build:\n");
    std::printf("  nn | nearest_neighbor        nearest-neighbour constructor (nearest_neighbor.rs)\n");
    std::printf("  gec | greedy_edge            greedy-edge constructor (greedy_edge.rs), --candidates K\n");
    std::printf("  2opt | two_opt               first-improvement 2-opt, bit-exact with two_opt.rs\n");
    std::printf("  2opt_best | two_opt_best     best-improvement 2-opt (extension)\n");
    std::printf("  2opt --mode neighbor         candidate-list best-improvement 2-opt, --candidates K (extension)\n");
    std::printf("  2opt --mode neighbor_multi   candidate-list 2-opt, many disjoint moves per step, --candidates K (extension)\n");
    std::printf("  or_opt | or-opt              Or-opt, bit-exact with or_opt.rs\n");
    std::printf("  or_opt --mode neighbor       candidate-list best-improvement Or-opt, --candidates K (extension)\n");
    std::printf("  or_opt --mode neighbor_multi candidate-list Or-opt, many disjoint moves per step, --candidates K (extension)\n");
    std::printf("  3opt | three_opt             best-improvement 3-opt, bit-exact with three_opt.rs\n");
    std::printf("  3opt --mode neighbor         candidate-list best-improvement 3-opt, --candidates K (extension)\n");
    std::printf("presets: fast (nn,2opt)\n");
    return 0;
}

} // namespace

int main(int argc, char **argv)
{
    try {
        const Args a = parse_args(argc, argv);
        if (a.cmd == "solve") return run_solve(a);
        if (a.cmd == "pipeline") return run_pipeline_cmd(a);
        if (a.cmd == "solvers") return run_solvers();
        if (a.cmd == "convert") return run_convert(a);
        die("unrecognized subcommand '" + a.cmd + "'", 2);
    } catch (const std::exception &e) { // the reference would panic: exit code 101
        std::fprintf(stderr, "thread 'main' panicked: %s\n", e.what());
        return 101;
    }
}
