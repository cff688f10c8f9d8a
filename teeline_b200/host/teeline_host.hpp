// teeline_host.hpp -- C++ host mirror of the reference's interface for the accelerated path.
//
// The reference (timgluz/teeline @ cd06a10) is Rust; this image has no cargo/rustc, so the host
// side above the C ABI (include/teeline_cuda.h) is written in C++ with the SAME names, argument
// meaning and error behaviour as the Rust items it mirrors.  Everything numeric is delegated to
// libteeline_cuda.so; this layer only marshals (city ids <-> matrix positions, exactly as
// DistanceMatrix::{city_id2pos,pos2city_id} do) and keeps the reference's orchestration:
//
//   KDPoint                      src/tsp/kdtree.rs:248-295
//   DistanceType, Solvers        src/tsp/mod.rs:165-182, :48-72, :559-590
//   DistanceMatrix               src/tsp/distance_matrix.rs:87-297
//   TspProblem, Solution         src/tsp/mod.rs:1732-1814
//   HeuristicOptions, AppOptions src/tsp/mod.rs:597-683, :1586-1596
//   ProgressMessage              src/tsp/progress.rs:3-11
//   two_opt::solve / or_opt::solve / three_opt::solve / nearest_neighbor::solve
//                                src/tsp/two_opt.rs:7-67, or_opt.rs:19-74, three_opt.rs:16-52,
//                                nearest_neighbor.rs:8-76
//   solve_with_context, solve_problem, validate_tour, find_solver
//                                src/tsp/mod.rs:1620-1723
//   pipeline::*                  src/tsp/pipeline.rs:11-132
//   config::load_pipeline_config src/config.rs:11-153
//   tsplib::read_from_*          src/tsp/tsplib.rs:84-377
//
// Rust `Result<T, String>` becomes `Result<T>` (value or error string); a Rust panic
// (`expect`, no CPU fallback when the device call fails) becomes a thrown `std::runtime_error`.
#pragma once

#include <cstddef>
#include <cstdint>
#include <functional>
#include <map>
#include <memory>
#include <optional>
#include <stdexcept>
#include <ostream>
#include <string>
#include <unordered_map>
#include <utility>
#include <variant>
#include <vector>

namespace teeline {

template <typename T>
struct Result {
    std::optional<T> value;
    std::string error;
    static Result ok(T v) { Result r; r.value = std::move(v); return r; }
    static Result err(std::string e) { Result r; r.error = std::move(e); return r; }
    bool is_ok() const { return value.has_value(); }
    bool is_err() const { return !value.has_value(); }
    T &unwrap()
    {
        if (!value) throw std::runtime_error("called `Result::unwrap()` on an `Err` value: " + error);
        return *value;
    }
};

namespace tsp {

// ---- src/tsp/kdtree.rs:248-295 ---------------------------------------------------------------
struct KDPoint {
    size_t id = 0;
    float coords[2] = {0.f, 0.f};
    static KDPoint new_with_id(size_t id, float x, float y) { KDPoint p; p.id = id; p.coords[0] = x; p.coords[1] = y; return p; }
    float x() const { return coords[0]; }
    float y() const { return coords[1]; }
};

// ---- src/tsp/mod.rs:165-182 --------------------------------------------------------------------
enum class DistanceType { Euc2D, Explicit, Geo };
Result<DistanceType> parse_distance_type(const std::string &s);

// ---- src/tsp/mod.rs:48-72, 559-590 -------------------------------------------------------------
enum class Solvers {
    AntColony, BellmanKarp, BranchBound, Christofides, Savings, CuckooSearch, FlowerPollination, Fourier,
    LinKernighan, NearestNeighbor, GeneticAlgorithm, GravitationalSearch, GreedyEdge, OrOpt,
    ParticleSwarmOptimization, RandomShuffle, SimulatedAnnealing, KohonenSom, StochasticHill, TabuSearch,
    ThreeOpt, TwoOpt,
    TwoOptBest, // extension (no Rust twin): best-improvement 2-opt, aliases "2opt_best" | "two_opt_best"
    Unspecified
};
Result<Solvers> find_solver(const std::string &name);   // "unknown solver: {name}"
const char *solver_name(Solvers s);
bool auto_expand_with_nn(Solvers s);                     // mod.rs:129-139
bool auto_expand_with_shuffle(Solvers s);                // mod.rs:144-157
bool is_accelerated(Solvers s);                          // the solvers this build implements

// ---- src/tsp/progress.rs ---------------------------------------------------------------------
struct ProgressMessage {
    enum Kind { PathUpdate, CityChange, Done } kind = Done;
    std::vector<size_t> route; // PathUpdate
    float total = 0.f;         // PathUpdate
    size_t city = 0;           // CityChange
};
using ProgressSender = std::function<void(const ProgressMessage &)>; // mpsc::Sender<ProgressMessage>

// ---- src/tsp/mod.rs:1817-1890 ------------------------------------------------------------------
struct NearestItem { KDPoint point; float distance; };
struct NearestResult {
    KDPoint target;
    size_t max_size = 0;
    std::vector<NearestItem> items;
    const std::vector<NearestItem> &nearest() const { return items; }
};

// ---- src/tsp/distance_matrix.rs:87-297 -----------------------------------------------------------
// Device-resident: build() uploads the coordinates (K1 on demand), new_explicit() uploads a packed
// triangle.  distances()/distance_by_pos() pull the packed triangle to the host once, lazily.
class DistanceMatrix {
  public:
    DistanceMatrix();
    ~DistanceMatrix();
    DistanceMatrix(const DistanceMatrix &);            // Clone: shares the device problem
    DistanceMatrix &operator=(const DistanceMatrix &);

    static Result<DistanceMatrix> from_cities(const std::vector<KDPoint> &cities);
    static Result<DistanceMatrix> build(const std::vector<KDPoint> &cities, DistanceType dt);
    // DistanceMatrix::new: packed strict lower triangle + cities in position order
    static DistanceMatrix new_explicit(size_t n, std::vector<float> distances, const std::vector<KDPoint> &cities);

    size_t num_cities() const;
    size_t len() const;                                  // n(n-1)/2
    const std::vector<float> &distances() const;         // distance_matrix.rs:171-173 (bit-identical)
    std::optional<float> distance_by_pos(size_t a, size_t b) const;       // :177-191
    std::optional<float> distance_between(size_t id1, size_t id2) const;  // :197-212
    float tour_length(const std::vector<size_t> &path_ids) const;         // :221-231 (unknown id -> 0.0)
    float tour_length_by_pos(const std::vector<size_t> &path_pos) const;  // :235-245
    // batch variant for population fitness (GA/ACO): tours are city ids, batch x n row-major
    std::vector<float> tour_lengths(const std::vector<size_t> &tours_ids, size_t batch) const;
    std::optional<size_t> pos2city_id(size_t pos) const;                  // :251-253
    std::optional<size_t> city_id2pos(size_t id) const;                   // :255-257
    NearestResult nearest(const KDPoint &target, size_t n) const;         // :259-280
    bool has_coordinates() const; // false for EXPLICIT problems: matrix path only

    struct Impl;
    std::shared_ptr<Impl> impl; // opaque: owns tl_ctx / tl_problem
};

// lin_kernighan::build_candidates (src/tsp/lin_kernighan.rs:12-27): candidates[city.id] = k nearest ids
std::vector<std::vector<size_t>> build_candidates(const std::vector<KDPoint> &cities, const DistanceMatrix &dm, size_t k);

// ---- src/tsp/mod.rs:1732-1814 ----------------------------------------------------------------------
struct TspProblem {
    std::vector<KDPoint> cities;
    DistanceMatrix distances;
};

class Solution {
  public:
    float total = 0.f;
    Solution() = default;
    Solution(const std::vector<size_t> &route, const TspProblem &problem);
    static Solution from_parts(const std::vector<size_t> &route, const std::vector<KDPoint> &cities,
                               const DistanceMatrix &distances);
    size_t len() const { return route_.size(); }
    bool is_empty() const { return route_.empty(); }
    const std::vector<size_t> &route() const { return route_; }
    const std::vector<KDPoint> &cities() const { return cities_; }
    const KDPoint *get_by_city_id(size_t id) const;

  private:
    std::vector<size_t> route_;
    std::vector<KDPoint> cities_;
    std::unordered_map<size_t, size_t> cities_idx_;
};

// ---- options: a minimal TOML value model (what `toml::Table` gives the reference) ---------------
struct TomlValue;
using TomlTable = std::vector<std::pair<std::string, TomlValue>>; // insertion-ordered
struct TomlValue {
    std::variant<std::monostate, std::string, int64_t, double, bool, std::shared_ptr<TomlTable>,
                 std::shared_ptr<std::vector<TomlValue>>> v;
    const std::string *as_str() const { return std::get_if<std::string>(&v); }
    const int64_t *as_integer() const { return std::get_if<int64_t>(&v); }
    const double *as_float() const { return std::get_if<double>(&v); }
    const bool *as_bool() const { return std::get_if<bool>(&v); }
    const TomlTable *as_table() const { auto p = std::get_if<std::shared_ptr<TomlTable>>(&v); return p ? p->get() : nullptr; }
    const std::vector<TomlValue> *as_array() const { auto p = std::get_if<std::shared_ptr<std::vector<TomlValue>>>(&v); return p ? p->get() : nullptr; }
    std::string display() const; // how `{v}` prints in the reference's error messages
};
Result<TomlTable> parse_toml(const std::string &source);
const TomlValue *toml_get(const TomlTable &t, const std::string &key);

struct HeuristicOptions { // mod.rs:597-683
    size_t epochs = 10000, platoo_epochs = 500, n_nearest = 3;
    bool verbose = false;
    static Result<HeuristicOptions> from_toml(const TomlTable &table);
    Result<bool> validate() const; // "n_nearest must be >= 1"
};

struct AcoOptions { // mod.rs:1083-1200; its own epochs = 150, platoo_epochs = 20 defaults
    HeuristicOptions heuristic{150, 20, 3, false};
    float alpha = 1.0f, beta = 2.0f, evaporation_rate = 0.5f;
    size_t num_ants = 25;
    static Result<AcoOptions> from_toml(const TomlTable &table);
    Result<bool> validate() const;
};

struct GAOptions { // mod.rs:816-905
    HeuristicOptions heuristic;
    float mutation_probability = 0.001f;
    size_t n_elite = 3;
    static Result<GAOptions> from_toml(const TomlTable &table);
    Result<bool> validate() const;
};

struct AppOptions { // mod.rs:1586-1596; only the sub-tables this path consumes are modelled
    std::optional<HeuristicOptions> heuristic;
    std::optional<AcoOptions> aco;
    std::optional<GAOptions> ga;
    // extension table [stage.cuda] (never required): mode = "ref"|"best"|"best_cyclic"|"neighbor"|"neighbor_multi"
    // (or_opt: "neighbor"|"neighbor_multi", 3opt: "neighbor"), path = "auto"|"matrix"|"recompute",
    // seed = <integer> (the population solvers' Philox key; the reference's RNG is unseeded),
    // candidates = <integer> (modes "neighbor" and "neighbor_multi": k of the candidate lists, 1..32;
    // 0 = TL_CANDIDATES_DEFAULT)
    std::string cuda_mode, cuda_path;
    uint64_t cuda_seed = 0;
    uint32_t cuda_candidates = 0;
};

// ---- solvers (same free-function convention as the reference) ------------------------------------
namespace two_opt {
Solution solve(const TspProblem &problem, const HeuristicOptions &opts, const ProgressSender *progress_tx,
               const std::vector<size_t> *init_tour);
// extension: best-improvement mode / explicit path selection ("ref"|"best"|"best_cyclic"|"neighbor"|"neighbor_multi",
// "auto"|"matrix"|"recompute"); candidates: k of modes "neighbor" and "neighbor_multi" (0 = the library's default)
Solution solve_with(const TspProblem &problem, const std::string &mode, const std::string &path,
                    const ProgressSender *progress_tx, const std::vector<size_t> *init_tour,
                    uint32_t candidates = 0);
}
namespace or_opt {
Solution solve(const TspProblem &problem, const HeuristicOptions &opts, const ProgressSender *progress_tx,
               const std::vector<size_t> *init_tour);
// extension: mode "neighbor" runs candidate-list Or-opt and mode "neighbor_multi" its multi-move form, with
// k = candidates (0 = the library's default); any other mode runs solve()'s Or-opt
Solution solve_with(const TspProblem &problem, const std::string &mode, const ProgressSender *progress_tx,
                    const std::vector<size_t> *init_tour, uint32_t candidates = 0);
}
namespace three_opt { // src/tsp/three_opt.rs:16-52
Solution solve(const TspProblem &problem, const HeuristicOptions &opts, const ProgressSender *progress_tx,
               const std::vector<size_t> *init_tour);
// extension: mode "neighbor" runs candidate-list 3-opt with k = candidates (0 = the library's default);
// any other mode runs solve()'s 3-opt
Solution solve_with(const TspProblem &problem, const std::string &mode, const ProgressSender *progress_tx,
                    const std::vector<size_t> *init_tour, uint32_t candidates = 0);
}
namespace nearest_neighbor {
Solution solve(const TspProblem &problem, const HeuristicOptions &opts, const ProgressSender *progress_tx,
               const std::vector<size_t> *init_tour);
}
namespace ant_colony { // src/tsp/ant_colony.rs:92-239; `seed` keys the Philox stream (extension)
Solution solve(const TspProblem &problem, const AcoOptions &opts, const ProgressSender *progress_tx,
               const std::vector<size_t> *init_tour, uint64_t seed = 0);
}
namespace genetic_algorithm { // src/tsp/genetic_algorithm.rs:16-44
Solution solve(const TspProblem &problem, const GAOptions &opts, const ProgressSender *progress_tx,
               const std::vector<size_t> *init_tour, uint64_t seed = 0);
}
namespace greedy_edge { // src/tsp/greedy_edge.rs: the greedy-edge tour (tl_greedy_tour); the seed is ignored.
// opts.cuda_candidates (1..32, 0 = keep the problem's lists) sets the width of the candidate lists first
Solution solve(const TspProblem &problem, const AppOptions &opts, const ProgressSender *progress_tx,
               const std::vector<size_t> *init_tour);
}
namespace random_shuffle { // src/tsp/random_shuffle.rs: a shuffled order of the city ids (splitmix64-seeded here)
Solution solve(const TspProblem &problem, uint64_t seed = 0);
}

Result<bool> validate_tour(const std::vector<size_t> &tour, const std::vector<KDPoint> &cities); // mod.rs:1620-1634
Result<Solution> solve_problem(Solvers solver, const TspProblem &problem, const AppOptions &opts);  // :1647-1653
Result<Solution> solve_with_context(Solvers solver, const TspProblem &problem, const AppOptions &opts,
                                    const ProgressSender *progress_tx, const std::vector<size_t> *init_tour);

// ---- src/tsp/pipeline.rs ----------------------------------------------------------------------------
namespace pipeline {
struct StageOutcome { Solution solution; uint64_t duration_ms = 0; };
struct PipelineStage {
    Solvers solver;
    AppOptions options;
    TspProblem problem;
    const ProgressSender *progress_tx = nullptr;
    Result<Solution> solve(const std::vector<size_t> *init_tour) const;
};
Result<std::vector<StageOutcome>> run_pipeline_stages(const std::vector<PipelineStage> &stages);
Result<Solution> run_pipeline(const std::vector<PipelineStage> &stages);
std::vector<std::string> stage_warnings(const std::vector<Solvers> &solvers);
}

// ---- src/tsp/tsplib.rs ------------------------------------------------------------------------------
namespace tsplib {
struct TspLibData {
    std::string name, comment;
    std::vector<KDPoint> cities;
    size_t dimension = 0;
    std::optional<std::vector<float>> raw_distances;
    DistanceType distance_type = DistanceType::Euc2D;
    bool has_explicit_weights() const { return raw_distances.has_value(); }
    Result<DistanceMatrix> distance_matrix() const; // tsplib.rs:84-98
};
Result<TspLibData> read_from_file(const std::string &path);
Result<TspLibData> read_from_str(const std::string &input);
}

// DiscOpt (Coursera "Discrete Optimization") coordinate files -> TSPLIB, src/tsp/convert.rs:6-66
namespace convert {
Result<std::vector<std::pair<float, float>>> parse_discopt(const std::string &input);         // convert.rs:6-29
void write_tsplib(const std::string &name, const std::vector<std::pair<float, float>> &coords,
                  std::ostream &writer);                                                        // convert.rs:32-45
Result<bool> convert_file(const std::string &input_path, const std::string &output_path);     // convert.rs:49-66
} // namespace convert

} // namespace tsp

// ---- src/config.rs ----------------------------------------------------------------------------------
namespace config {
Result<std::vector<std::pair<tsp::Solvers, tsp::AppOptions>>> load_pipeline_config(const std::string &source,
                                                                                   const tsp::AppOptions &base);
}

} // namespace teeline
