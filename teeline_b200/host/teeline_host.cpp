// teeline_host.cpp -- implementation of the C++ host mirror (see teeline_host.hpp).
// Every numeric result comes from libteeline_cuda.so through include/teeline_cuda.h; there is no
// CPU fallback: a failing device call throws, like the reference's `.expect(..)` panics.
#include "teeline_host.hpp"

#include <algorithm>
#include <cctype>
#include <chrono>
#include <charconv>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <set>
#include <sstream>

#include "../../include/teeline_cuda.h"

namespace teeline {
namespace tsp {

namespace {

[[noreturn]] void panic(const std::string &what)
{
    throw std::runtime_error(what + ": " + tl_last_error());
}
void check(tl_status s, const char *what)
{
    if (s != TL_OK) panic(what);
}

std::string upper(std::string s)
{
    for (char &c : s) c = (char)std::toupper((unsigned char)c);
    return s;
}
std::string lower(std::string s)
{
    for (char &c : s) c = (char)std::tolower((unsigned char)c);
    return s;
}
std::string trim(const std::string &s)
{
    size_t a = 0, b = s.size();
    while (a < b && std::isspace((unsigned char)s[a])) ++a;
    while (b > a && std::isspace((unsigned char)s[b - 1])) --b;
    return s.substr(a, b - a);
}

} // namespace

// ---- DistanceType / Solvers -----------------------------------------------------------------------

Result<DistanceType> parse_distance_type(const std::string &s)
{
    const std::string u = upper(s);
    if (u == "EUC_2D" || u == "EUC2D") return Result<DistanceType>::ok(DistanceType::Euc2D);
    if (u == "EXPLICIT") return Result<DistanceType>::ok(DistanceType::Explicit);
    if (u == "GEO") return Result<DistanceType>::ok(DistanceType::Geo);
    return Result<DistanceType>::err("unsupported distance type: " + u);
}

namespace {
struct SolverAlias { const char *alias; Solvers s; };
const SolverAlias kAliases[] = {
    {"aco", Solvers::AntColony}, {"ant_colony", Solvers::AntColony},
    {"bhk", Solvers::BellmanKarp}, {"bellman_karp", Solvers::BellmanKarp},
    {"branch_bound", Solvers::BranchBound},
    {"christofides", Solvers::Christofides}, {"chr", Solvers::Christofides},
    {"sav", Solvers::Savings}, {"savings", Solvers::Savings},
    {"cs", Solvers::CuckooSearch}, {"cuckoo_search", Solvers::CuckooSearch},
    {"fpa", Solvers::FlowerPollination}, {"flower_pollination", Solvers::FlowerPollination},
    {"fourier", Solvers::Fourier},
    {"lk", Solvers::LinKernighan}, {"lin_kernighan", Solvers::LinKernighan},
    {"nn", Solvers::NearestNeighbor}, {"nearest_neighbor", Solvers::NearestNeighbor},
    {"ga", Solvers::GeneticAlgorithm}, {"genetic_algorithm", Solvers::GeneticAlgorithm},
    {"gsa", Solvers::GravitationalSearch}, {"gravitational_search", Solvers::GravitationalSearch},
    {"gec", Solvers::GreedyEdge}, {"greedy_edge", Solvers::GreedyEdge},
    {"pso", Solvers::ParticleSwarmOptimization}, {"particle_swarm", Solvers::ParticleSwarmOptimization},
    {"shuffle", Solvers::RandomShuffle}, {"random_shuffle", Solvers::RandomShuffle},
    {"sa", Solvers::SimulatedAnnealing}, {"simulated_annealing", Solvers::SimulatedAnnealing},
    {"som", Solvers::KohonenSom}, {"kohonen", Solvers::KohonenSom}, {"kohonen_som", Solvers::KohonenSom},
    {"stochastic_hill", Solvers::StochasticHill},
    {"tabu", Solvers::TabuSearch}, {"tabu_search", Solvers::TabuSearch},
    {"or_opt", Solvers::OrOpt}, {"or-opt", Solvers::OrOpt},
    {"3opt", Solvers::ThreeOpt}, {"three_opt", Solvers::ThreeOpt},
    {"2opt", Solvers::TwoOpt}, {"two_opt", Solvers::TwoOpt},
    {"2opt_best", Solvers::TwoOptBest}, {"two_opt_best", Solvers::TwoOptBest},
};
} // namespace

Result<Solvers> find_solver(const std::string &name)
{
    for (const SolverAlias &a : kAliases)
        if (name == a.alias) return Result<Solvers>::ok(a.s);
    return Result<Solvers>::err("unknown solver: " + name);
}

const char *solver_name(Solvers s)
{
    switch (s) {
    case Solvers::AntColony: return "AntColony";
    case Solvers::BellmanKarp: return "BellmanKarp";
    case Solvers::BranchBound: return "BranchBound";
    case Solvers::Christofides: return "Christofides";
    case Solvers::Savings: return "Savings";
    case Solvers::CuckooSearch: return "CuckooSearch";
    case Solvers::FlowerPollination: return "FlowerPollination";
    case Solvers::Fourier: return "Fourier";
    case Solvers::LinKernighan: return "LinKernighan";
    case Solvers::NearestNeighbor: return "NearestNeighbor";
    case Solvers::GeneticAlgorithm: return "GeneticAlgorithm";
    case Solvers::GravitationalSearch: return "GravitationalSearch";
    case Solvers::GreedyEdge: return "GreedyEdge";
    case Solvers::OrOpt: return "OrOpt";
    case Solvers::ParticleSwarmOptimization: return "ParticleSwarmOptimization";
    case Solvers::RandomShuffle: return "RandomShuffle";
    case Solvers::SimulatedAnnealing: return "SimulatedAnnealing";
    case Solvers::KohonenSom: return "KohonenSom";
    case Solvers::StochasticHill: return "StochasticHill";
    case Solvers::TabuSearch: return "TabuSearch";
    case Solvers::ThreeOpt: return "ThreeOpt";
    case Solvers::TwoOpt: return "TwoOpt";
    case Solvers::TwoOptBest: return "TwoOptBest";
    default: return "Unspecified";
    }
}

bool auto_expand_with_nn(Solvers s)
{
    return s == Solvers::TwoOpt || s == Solvers::ThreeOpt || s == Solvers::TabuSearch || s == Solvers::BranchBound ||
           s == Solvers::LinKernighan || s == Solvers::OrOpt || s == Solvers::TwoOptBest;
}
bool auto_expand_with_shuffle(Solvers s)
{
    return s == Solvers::SimulatedAnnealing || s == Solvers::StochasticHill || s == Solvers::GeneticAlgorithm ||
           s == Solvers::GravitationalSearch || s == Solvers::ParticleSwarmOptimization ||
           s == Solvers::CuckooSearch || s == Solvers::FlowerPollination || s == Solvers::Fourier ||
           s == Solvers::AntColony;
}
bool is_accelerated(Solvers s)
{
    return s == Solvers::NearestNeighbor || s == Solvers::GreedyEdge || s == Solvers::TwoOpt || s == Solvers::OrOpt ||
           s == Solvers::TwoOptBest ||
           s == Solvers::ThreeOpt || s == Solvers::AntColony || s == Solvers::GeneticAlgorithm ||
           s == Solvers::RandomShuffle;
}

// ---- DistanceMatrix ----------------------------------------------------------------------------------

struct DistanceMatrix::Impl {
    tl_ctx *ctx = nullptr;
    tl_problem *prob = nullptr;
    size_t n = 0;
    bool coords = false;
    std::vector<KDPoint> cities;                 // position order (CityTable: pos -> KDPoint)
    std::unordered_map<size_t, size_t> city_idx; // id -> pos
    mutable std::vector<float> items;            // packed triangle, fetched lazily
    mutable bool have_items = false;
    mutable std::map<size_t, std::vector<uint32_t>> knn_cache;
    ~Impl()
    {
        if (prob) tl_problem_destroy(prob);
        if (ctx) tl_ctx_destroy(ctx);
    }
};

DistanceMatrix::DistanceMatrix() = default;
DistanceMatrix::~DistanceMatrix() = default;
DistanceMatrix::DistanceMatrix(const DistanceMatrix &) = default;
DistanceMatrix &DistanceMatrix::operator=(const DistanceMatrix &) = default;

namespace {

int device_ordinal()
{
    const char *e = std::getenv("TEELINE_CUDA_DEVICE");
    return e ? std::atoi(e) : 0;
}

// geo_distance, src/tsp/distance_matrix.rs:59-75 (TSPLIB GEO, f64, floor, stored as f32).  GEO is not
// on the accelerated path: the values are produced here once and uploaded as an explicit triangle.
float geo_distance(const KDPoint &p1, const KDPoint &p2)
{
    const double PI = 3.14159265358979323846264338327950288;
    auto to_rad = [&](float x) {
        const double deg = (double)std::trunc(x);
        const double min = (double)(x - std::trunc(x));
        return PI * (deg + 5.0 * min / 3.0) / 180.0;
    };
    const double lat1 = to_rad(p1.coords[0]), lon1 = to_rad(p1.coords[1]);
    const double lat2 = to_rad(p2.coords[0]), lon2 = to_rad(p2.coords[1]);
    const double q1 = std::cos(lon1 - lon2), q2 = std::cos(lat1 - lat2), q3 = std::cos(lat1 + lat2);
    const double RRR = 6378.388;
    return (float)std::floor(RRR * std::acos(0.5 * ((1.0 + q1) * q2 - (1.0 - q1) * q3)) + 1.0);
}

std::shared_ptr<DistanceMatrix::Impl> make_impl(const std::vector<KDPoint> &cities)
{
    auto im = std::make_shared<DistanceMatrix::Impl>();
    im->n = cities.size();
    im->cities = cities;
    for (size_t i = 0; i < cities.size(); ++i) im->city_idx[cities[i].id] = i;
    check(tl_ctx_create(device_ordinal(), &im->ctx), "tl_ctx_create");
    return im;
}

} // namespace

Result<DistanceMatrix> DistanceMatrix::from_cities(const std::vector<KDPoint> &cities)
{
    return build(cities, DistanceType::Euc2D);
}

Result<DistanceMatrix> DistanceMatrix::build(const std::vector<KDPoint> &cities, DistanceType dt)
{
    const size_t n = cities.size();
    if (n < 2) return Result<DistanceMatrix>::err("distance matrix requires at least 2 points");
    if (dt == DistanceType::Explicit)
        return Result<DistanceMatrix>::err("cannot build distance matrix from coordinates for EXPLICIT type — use "
                                           "DistanceMatrix::new() with precomputed distances");
    if (dt == DistanceType::Geo) {
        std::vector<float> tri;
        tri.reserve(n * (n - 1) / 2);
        for (size_t i = 0; i < n; ++i)
            for (size_t j = 0; j < i; ++j) tri.push_back(geo_distance(cities[i], cities[j]));
        return Result<DistanceMatrix>::ok(new_explicit(n, std::move(tri), cities));
    }
    DistanceMatrix dm;
    dm.impl = make_impl(cities);
    dm.impl->coords = true;
    std::vector<float> x(n), y(n);
    for (size_t i = 0; i < n; ++i) {
        x[i] = cities[i].coords[0];
        y[i] = cities[i].coords[1];
    }
    check(tl_problem_create_euc2d(dm.impl->ctx, (uint32_t)n, x.data(), y.data(), TL_DIST_F32_EXACT, &dm.impl->prob),
          "tl_problem_create_euc2d");
    return Result<DistanceMatrix>::ok(std::move(dm));
}

DistanceMatrix DistanceMatrix::new_explicit(size_t n, std::vector<float> distances, const std::vector<KDPoint> &cities)
{
    // the reference asserts both (distance_matrix.rs:99-108)
    if (n != cities.size()) throw std::runtime_error("city_idx size differs from n cities");
    if (distances.size() != n * (n - 1) / 2)
        throw std::runtime_error("distances length " + std::to_string(distances.size()) + " != n*(n-1)/2=" +
                                 std::to_string(n * (n - 1) / 2) + " for n=" + std::to_string(n));
    DistanceMatrix dm;
    dm.impl = make_impl(cities);
    dm.impl->coords = false;
    check(tl_problem_create_explicit(dm.impl->ctx, (uint32_t)n, distances.data(), &dm.impl->prob),
          "tl_problem_create_explicit");
    dm.impl->items = std::move(distances);
    dm.impl->have_items = true;
    return dm;
}

size_t DistanceMatrix::num_cities() const { return impl ? impl->n : 0; }
size_t DistanceMatrix::len() const { return impl ? impl->n * (impl->n - 1) / 2 : 0; }
bool DistanceMatrix::has_coordinates() const { return impl && impl->coords; }

const std::vector<float> &DistanceMatrix::distances() const
{
    if (!impl->have_items) {
        impl->items.resize(len());
        check(tl_dist_matrix_packed(impl->prob, impl->items.data()), "tl_dist_matrix_packed");
        impl->have_items = true;
    }
    return impl->items;
}

std::optional<float> DistanceMatrix::distance_by_pos(size_t a, size_t b) const
{
    if (a >= impl->n || b >= impl->n) return std::nullopt;
    if (a == b) return 0.0f;
    const size_t from = std::max(a, b), to = std::min(a, b);
    return distances()[from * (from - 1) / 2 + to];
}

std::optional<float> DistanceMatrix::distance_between(size_t id1, size_t id2) const
{
    const auto p1 = city_id2pos(id1), p2 = city_id2pos(id2);
    if (!p1 || !p2) return std::nullopt;
    return distance_by_pos(*p1, *p2);
}

std::optional<size_t> DistanceMatrix::pos2city_id(size_t pos) const
{
    if (pos >= impl->n) return std::nullopt;
    return impl->cities[pos].id;
}
std::optional<size_t> DistanceMatrix::city_id2pos(size_t id) const
{
    auto it = impl->city_idx.find(id);
    if (it == impl->city_idx.end()) return std::nullopt;
    return it->second;
}

float DistanceMatrix::tour_length_by_pos(const std::vector<size_t> &path) const
{
    if (path.size() < 2) return 0.0f;
    // K4 evaluates full tours of n positions; shorter or repeating paths (allowed by the reference)
    // are not on the accelerated path and take the reference's own loop over the packed triangle
    if (path.size() != impl->n) {
        float total = distance_by_pos(path.back(), path[0]).value_or(0.0f);
        for (size_t k = 0; k + 1 < path.size(); ++k) total += distance_by_pos(path[k], path[k + 1]).value_or(0.0f);
        return total;
    }
    std::vector<uint32_t> t(path.size());
    for (size_t k = 0; k < path.size(); ++k) t[k] = path[k] > 0xfffffffeull ? 0xffffffffu : (uint32_t)path[k];
    float out = 0.0f;
    check(tl_tour_lengths(impl->prob, t.data(), 1, TL_LEN_EXACT, &out), "tl_tour_lengths");
    return out;
}

float DistanceMatrix::tour_length(const std::vector<size_t> &path) const
{
    if (path.size() < 2) return 0.0f;
    std::vector<size_t> pos(path.size());
    for (size_t k = 0; k < path.size(); ++k) {
        const auto p = city_id2pos(path[k]);
        if (!p) return 0.0f; // unknown city id
        pos[k] = *p;
    }
    return tour_length_by_pos(pos);
}

std::vector<float> DistanceMatrix::tour_lengths(const std::vector<size_t> &tours_ids, size_t batch) const
{
    const size_t n = impl->n;
    if (tours_ids.size() != batch * n) throw std::runtime_error("tour_lengths: tours must be batch x n city ids");
    std::vector<uint32_t> t(batch * n);
    for (size_t k = 0; k < t.size(); ++k) {
        const auto p = city_id2pos(tours_ids[k]);
        t[k] = p ? (uint32_t)*p : 0xffffffffu; // unknown id -> that tour's length is 0.0
    }
    std::vector<float> out(batch);
    check(tl_tour_lengths(impl->prob, t.data(), batch, TL_LEN_EXACT, out.data()), "tl_tour_lengths");
    return out;
}

NearestResult DistanceMatrix::nearest(const KDPoint &target, size_t n) const
{
    NearestResult res;
    res.target = target;
    res.max_size = n;
    const auto pos = city_id2pos(target.id);
    if (!pos || n == 0) return res; // unknown target -> empty result, no panic
    auto it = impl->knn_cache.find(n);
    if (it == impl->knn_cache.end()) {
        std::vector<uint32_t> knn(impl->n * n);
        check(tl_knn(impl->prob, (uint32_t)n, knn.data()), "tl_knn");
        it = impl->knn_cache.emplace(n, std::move(knn)).first;
    }
    for (size_t t = 0; t < n; ++t) {
        const uint32_t q = it->second[*pos * n + t];
        if (q == 0xffffffffu) break;
        res.items.push_back(NearestItem{impl->cities[q], *distance_by_pos(*pos, q)});
    }
    return res;
}

std::vector<std::vector<size_t>> build_candidates(const std::vector<KDPoint> &cities, const DistanceMatrix &dm, size_t k)
{
    const size_t n = cities.size();
    k = std::min(k, n > 0 ? n - 1 : 0);
    size_t max_id = 0;
    for (const KDPoint &c : cities) max_id = std::max(max_id, c.id);
    std::vector<std::vector<size_t>> cand(max_id + 1);
    if (k == 0) return cand;
    std::vector<uint32_t> knn(n * k);
    check(tl_knn(dm.impl->prob, (uint32_t)k, knn.data()), "tl_knn");
    for (size_t pos = 0; pos < n; ++pos)
        for (size_t t = 0; t < k; ++t) {
            const uint32_t q = knn[pos * k + t];
            if (q != 0xffffffffu) cand[cities[pos].id].push_back(cities[q].id);
        }
    return cand;
}

// ---- Solution ------------------------------------------------------------------------------------------

Solution::Solution(const std::vector<size_t> &route, const TspProblem &problem)
{
    *this = from_parts(route, problem.cities, problem.distances);
}

Solution Solution::from_parts(const std::vector<size_t> &route, const std::vector<KDPoint> &cities,
                              const DistanceMatrix &distances)
{
    Solution s;
    s.total = distances.tour_length(route); // exact-order f32 sum (K4 EXACT), mod.rs:1776-1789
    s.route_ = route;
    s.cities_ = cities;
    for (size_t i = 0; i < cities.size(); ++i) s.cities_idx_[cities[i].id] = i;
    return s;
}

const KDPoint *Solution::get_by_city_id(size_t id) const
{
    auto it = cities_idx_.find(id);
    return it == cities_idx_.end() ? nullptr : &cities_[it->second];
}

// ---- solvers ----------------------------------------------------------------------------------------------

namespace {

std::vector<size_t> ids_of(const std::vector<KDPoint> &cities)
{
    std::vector<size_t> v(cities.size());
    for (size_t i = 0; i < cities.size(); ++i) v[i] = cities[i].id;
    return v;
}

std::vector<uint32_t> to_positions(const std::vector<size_t> &path, const DistanceMatrix &dm, const char *who)
{
    std::vector<uint32_t> t(path.size());
    for (size_t k = 0; k < path.size(); ++k) {
        const auto p = dm.city_id2pos(path[k]);
        if (!p) throw std::runtime_error(std::string(who) + ": invalid city pair"); // the reference's expect()
        t[k] = (uint32_t)*p;
    }
    return t;
}

std::vector<size_t> to_ids(const std::vector<uint32_t> &tour, const DistanceMatrix &dm)
{
    std::vector<size_t> v(tour.size());
    for (size_t k = 0; k < tour.size(); ++k) v[k] = *dm.pos2city_id(tour[k]);
    return v;
}

int path_code(const std::string &path)
{
    if (path.empty() || path == "auto") return TL_PATH_AUTO;
    if (path == "matrix") return TL_PATH_MATRIX;
    if (path == "recompute") return TL_PATH_RECOMPUTE;
    throw std::runtime_error("unknown path `" + path + "` (auto | matrix | recompute)");
}

// Runs one local search on the device and replays the reference's progress messages from the
// returned move log (two_opt.rs:22-24,53-56,63-65; or_opt.rs:40-42,62-71).
Solution run_local_search(const TspProblem &problem, int algo, int path, const ProgressSender *tx,
                          const std::vector<size_t> &start_ids, const char *who)
{
    const DistanceMatrix &dm = problem.distances;
    std::vector<uint32_t> tour = to_positions(start_ids, dm, who);
    if (tour.size() != dm.num_cities()) throw std::runtime_error(std::string(who) + ": init_tour must visit every city once");
    if (tx) {
        ProgressMessage m;
        m.kind = ProgressMessage::PathUpdate;
        m.route = start_ids;
        m.total = 0.0f;
        (*tx)(m);
    }
    // the candidate-list searches serve instances whose packed triangle cannot come to the host (2 TB at
    // 10^6 cities), and the per-move progress values of two_opt.rs and or_opt.rs need it: only the start
    // and the result are sent
    const bool replay = tx && algo != TL_ALGO_TWO_OPT_NEIGHBOR && algo != TL_ALGO_OR_OPT_NEIGHBOR &&
                        algo != TL_ALGO_THREE_OPT_NEIGHBOR && algo != TL_ALGO_TWO_OPT_NEIGHBOR_MULTI &&
                        algo != TL_ALGO_OR_OPT_NEIGHBOR_MULTI;
    std::vector<tl_move> log(replay ? (size_t)1 << 20 : 0);
    tl_stats st{};
    std::vector<uint32_t> before = tour;
    check(tl_local_search(dm.impl->prob, algo, path, tour.data(), -1, &st, log.empty() ? nullptr : log.data(), log.size()),
          who);
    if (tx && !replay) {
        ProgressMessage m;
        m.kind = ProgressMessage::PathUpdate;
        m.route = to_ids(tour, dm);
        m.total = 0.0f;
        (*tx)(m);
        ProgressMessage done;
        done.kind = ProgressMessage::Done;
        (*tx)(done);
    }
    if (replay) {
        std::vector<uint32_t> cur = before;
        const size_t n = cur.size();
        for (size_t k = 0; k < std::min<size_t>(st.moves, log.size()); ++k) {
            const tl_move &mv = log[k];
            ProgressMessage m;
            m.kind = ProgressMessage::PathUpdate;
            if (algo == TL_ALGO_THREE_OPT) { // apply_3opt, three_opt.rs:182-218; send_path sends 0.0
                std::vector<uint32_t> s1(cur.begin() + mv.i + 1, cur.begin() + mv.j + 1);
                std::vector<uint32_t> s2(cur.begin() + mv.j + 1, cur.begin() + mv.k + 1);
                const int kase = mv.seg_len;
                if (kase == 1 || kase == 3 || kase == 5 || kase == 7) std::reverse(s1.begin(), s1.end());
                if (kase == 2 || kase == 3 || kase == 6 || kase == 7) std::reverse(s2.begin(), s2.end());
                const std::vector<uint32_t> &a = kase >= 4 ? s2 : s1, &b = kase >= 4 ? s1 : s2;
                std::copy(a.begin(), a.end(), cur.begin() + mv.i + 1);
                std::copy(b.begin(), b.end(), cur.begin() + mv.i + 1 + a.size());
                m.total = 0.0f;
            } else if (algo == TL_ALGO_OR_OPT) {
                std::vector<uint32_t> seg(cur.begin() + mv.i, cur.begin() + mv.i + mv.seg_len);
                cur.erase(cur.begin() + mv.i, cur.begin() + mv.i + mv.seg_len);
                const size_t at = mv.j >= mv.i + mv.seg_len ? mv.j - mv.seg_len + 1 : mv.j + 1;
                if (mv.reversed) std::reverse(seg.begin(), seg.end());
                cur.insert(cur.begin() + at, seg.begin(), seg.end());
                std::vector<size_t> pos(cur.begin(), cur.end());
                m.total = dm.tour_length_by_pos(pos); // or_opt.rs:64-66 sends the tour length
            } else {
                // two_opt.rs:53-56 sends new_distance = d(p_i,p_j) + d(p_i+1,p_j+1)
                m.total = *dm.distance_by_pos(cur[mv.i], cur[mv.j]) + *dm.distance_by_pos(cur[mv.i + 1], cur[(mv.j + 1) % n]);
                std::reverse(cur.begin() + mv.i + 1, cur.begin() + mv.j + 1);
            }
            m.route = to_ids(cur, dm);
            (*tx)(m);
        }
        ProgressMessage done;
        done.kind = ProgressMessage::Done;
        (*tx)(done);
    }
    return Solution::from_parts(to_ids(tour, dm), problem.cities, dm);
}

} // namespace

namespace two_opt {

Solution solve_with(const TspProblem &problem, const std::string &mode, const std::string &path,
                    const ProgressSender *progress_tx, const std::vector<size_t> *init_tour, uint32_t candidates)
{
    int algo;
    if (mode.empty() || mode == "ref") algo = TL_ALGO_TWO_OPT_REF;
    else if (mode == "best") algo = TL_ALGO_TWO_OPT_BEST;
    else if (mode == "best_cyclic") algo = TL_ALGO_TWO_OPT_BEST_CYCLIC;
    else if (mode == "neighbor") algo = TL_ALGO_TWO_OPT_NEIGHBOR;
    else if (mode == "neighbor_multi") algo = TL_ALGO_TWO_OPT_NEIGHBOR_MULTI;
    else throw std::runtime_error("unknown 2-opt mode `" + mode + "` (ref | best | best_cyclic | neighbor | neighbor_multi)");
    if ((algo == TL_ALGO_TWO_OPT_NEIGHBOR || algo == TL_ALGO_TWO_OPT_NEIGHBOR_MULTI) && candidates)
        check(tl_problem_set_candidates(problem.distances.impl->prob, candidates), "two_opt");
    const std::vector<size_t> start = init_tour ? *init_tour : ids_of(problem.cities); // two_opt.rs:18-20
    return run_local_search(problem, algo, path_code(path), progress_tx, start, "two_opt");
}

Solution solve(const TspProblem &problem, const HeuristicOptions &, const ProgressSender *progress_tx,
               const std::vector<size_t> *init_tour)
{
    // the reference ignores HeuristicOptions here (two_opt.rs:9 `_opts`)
    return solve_with(problem, "ref", "auto", progress_tx, init_tour);
}

} // namespace two_opt

namespace or_opt {

Solution solve_with(const TspProblem &problem, const std::string &mode, const ProgressSender *progress_tx,
                    const std::vector<size_t> *init_tour, uint32_t candidates)
{
    const int algo = mode == "neighbor"         ? TL_ALGO_OR_OPT_NEIGHBOR
                     : mode == "neighbor_multi" ? TL_ALGO_OR_OPT_NEIGHBOR_MULTI
                                                : TL_ALGO_OR_OPT;
    // n < 4: identity order, seed ignored, no progress messages (or_opt.rs:31-34)
    if (problem.cities.size() < 4) return Solution::from_parts(ids_of(problem.cities), problem.cities, problem.distances);
    if (algo != TL_ALGO_OR_OPT && candidates)
        check(tl_problem_set_candidates(problem.distances.impl->prob, candidates), "or_opt");
    const std::vector<size_t> start = init_tour ? *init_tour : ids_of(problem.cities);
    return run_local_search(problem, algo, TL_PATH_AUTO, progress_tx, start, "or_opt");
}

Solution solve(const TspProblem &problem, const HeuristicOptions &, const ProgressSender *progress_tx,
               const std::vector<size_t> *init_tour)
{
    return solve_with(problem, "", progress_tx, init_tour);
}

} // namespace or_opt

namespace three_opt {

Solution solve_with(const TspProblem &problem, const std::string &mode, const ProgressSender *progress_tx,
                    const std::vector<size_t> *init_tour, uint32_t candidates)
{
    const int algo = mode == "neighbor" ? TL_ALGO_THREE_OPT_NEIGHBOR : TL_ALGO_THREE_OPT;
    // n < 4: identity order, seed ignored, no progress messages (three_opt.rs:25-28)
    if (problem.cities.size() < 4) return Solution::from_parts(ids_of(problem.cities), problem.cities, problem.distances);
    if (algo == TL_ALGO_THREE_OPT_NEIGHBOR && candidates)
        check(tl_problem_set_candidates(problem.distances.impl->prob, candidates), "three_opt");
    const std::vector<size_t> start = init_tour ? *init_tour : ids_of(problem.cities);
    return run_local_search(problem, algo, TL_PATH_AUTO, progress_tx, start, "three_opt");
}

Solution solve(const TspProblem &problem, const HeuristicOptions &, const ProgressSender *progress_tx,
               const std::vector<size_t> *init_tour)
{
    return solve_with(problem, "", progress_tx, init_tour);
}

} // namespace three_opt

namespace nearest_neighbor {

Solution solve(const TspProblem &problem, const HeuristicOptions &opts, const ProgressSender *progress_tx,
               const std::vector<size_t> *)
{
    const DistanceMatrix &dm = problem.distances;
    std::vector<uint32_t> tour(dm.num_cities());
    check(tl_nn_tour(dm.impl->prob, (uint32_t)opts.n_nearest, tour.data()), "nearest_neighbor");
    const std::vector<size_t> path = to_ids(tour, dm);
    if (progress_tx) { // nearest_neighbor.rs:32-34,41-43,67-73: a PathUpdate per appended city
        std::vector<size_t> partial;
        for (size_t k = 0; k < path.size(); ++k) {
            if (k > 0) {
                ProgressMessage c;
                c.kind = ProgressMessage::CityChange;
                c.city = path[k - 1];
                (*progress_tx)(c);
            }
            partial.push_back(path[k]);
            ProgressMessage m;
            m.kind = ProgressMessage::PathUpdate;
            m.route = partial;
            (*progress_tx)(m);
        }
        ProgressMessage done;
        done.kind = ProgressMessage::Done;
        (*progress_tx)(done);
    }
    return Solution::from_parts(path, problem.cities, dm);
}

} // namespace nearest_neighbor

namespace {

// PathUpdate(best) + Done, what the population solvers send at the end (ant_colony.rs:241-247,
// genetic_algorithm.rs:33-41); per-epoch updates are not replayed
void send_final(const ProgressSender *tx, const std::vector<size_t> &route, float total)
{
    if (!tx) return;
    ProgressMessage m;
    m.kind = ProgressMessage::PathUpdate;
    m.route = route;
    m.total = total;
    (*tx)(m);
    ProgressMessage done;
    done.kind = ProgressMessage::Done;
    (*tx)(done);
}

} // namespace

namespace ant_colony {

Solution solve(const TspProblem &problem, const AcoOptions &o, const ProgressSender *tx, const std::vector<size_t> *init_tour,
               uint64_t seed)
{
    const DistanceMatrix &dm = problem.distances;
    std::vector<uint32_t> init, best(dm.num_cities());
    if (init_tour) init = to_positions(*init_tour, dm, "ant_colony");
    tl_aco_options co{o.alpha, o.beta, o.evaporation_rate, (uint32_t)o.num_ants, (uint32_t)o.heuristic.epochs, 0u, seed};
    float cost = 0.0f;
    check(tl_aco(dm.impl->prob, &co, init_tour ? init.data() : nullptr, best.data(), &cost, nullptr), "ant_colony");
    const std::vector<size_t> route = to_ids(best, dm);
    send_final(tx, route, cost);
    return Solution::from_parts(route, problem.cities, dm);
}

} // namespace ant_colony

namespace genetic_algorithm {

Solution solve(const TspProblem &problem, const GAOptions &o, const ProgressSender *tx, const std::vector<size_t> *init_tour,
               uint64_t seed)
{
    const DistanceMatrix &dm = problem.distances;
    std::vector<uint32_t> init, best(dm.num_cities());
    if (init_tour) init = to_positions(*init_tour, dm, "genetic_algorithm");
    tl_ga_options go{o.mutation_probability, (uint32_t)o.n_elite, (uint32_t)o.heuristic.epochs, 0u, seed};
    float cost = 0.0f;
    check(tl_ga(dm.impl->prob, &go, init_tour ? init.data() : nullptr, best.data(), &cost, nullptr), "genetic_algorithm");
    const std::vector<size_t> route = to_ids(best, dm);
    send_final(tx, route, cost);
    return Solution::from_parts(route, problem.cities, dm);
}

} // namespace genetic_algorithm

namespace greedy_edge {

Solution solve(const TspProblem &problem, const AppOptions &opts, const ProgressSender *tx, const std::vector<size_t> *)
{
    // greedy_edge.rs builds its tour from the instance alone: the seed is ignored (stage_warnings says so)
    const DistanceMatrix &dm = problem.distances;
    if (opts.cuda_candidates) check(tl_problem_set_candidates(dm.impl->prob, opts.cuda_candidates), "greedy_edge");
    std::vector<uint32_t> tour(dm.num_cities());
    check(tl_greedy_tour(dm.impl->prob, tour.data(), nullptr), "greedy_edge");
    const std::vector<size_t> route = to_ids(tour, dm);
    Solution s = Solution::from_parts(route, problem.cities, dm);
    send_final(tx, route, s.total);
    return s;
}

} // namespace greedy_edge

namespace random_shuffle {

Solution solve(const TspProblem &problem, uint64_t seed)
{
    std::vector<size_t> ids = ids_of(problem.cities);
    uint64_t state = seed ^ 0x9E3779B97F4A7C15ull;
    auto next = [&state]() { // splitmix64
        uint64_t z = (state += 0x9E3779B97F4A7C15ull);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        return z ^ (z >> 31);
    };
    for (size_t i = ids.size(); i > 1; --i) std::swap(ids[i - 1], ids[(size_t)(next() % i)]);
    return Solution::from_parts(ids, problem.cities, problem.distances);
}

} // namespace random_shuffle

Result<bool> validate_tour(const std::vector<size_t> &tour, const std::vector<KDPoint> &cities)
{
    if (tour.size() != cities.size())
        return Result<bool>::err("tour length " + std::to_string(tour.size()) + " != cities length " +
                                 std::to_string(cities.size()));
    std::set<size_t> a, b(tour.begin(), tour.end());
    for (const KDPoint &c : cities) a.insert(c.id);
    if (a != b) return Result<bool>::err("tour contains invalid or duplicate city IDs");
    return Result<bool>::ok(true);
}

Result<Solution> solve_with_context(Solvers solver, const TspProblem &problem, const AppOptions &opts,
                                    const ProgressSender *tx, const std::vector<size_t> *init_tour)
{
    const HeuristicOptions h = opts.heuristic.value_or(HeuristicOptions{});
    auto v = h.validate();
    if (v.is_err()) return Result<Solution>::err(v.error);
    switch (solver) {
    case Solvers::NearestNeighbor: return Result<Solution>::ok(nearest_neighbor::solve(problem, h, tx, init_tour));
    case Solvers::GreedyEdge: return Result<Solution>::ok(greedy_edge::solve(problem, opts, tx, init_tour));
    case Solvers::OrOpt:
        if (opts.cuda_mode == "neighbor" || opts.cuda_mode == "neighbor_multi")
            return Result<Solution>::ok(or_opt::solve_with(problem, opts.cuda_mode, tx, init_tour, opts.cuda_candidates));
        return Result<Solution>::ok(or_opt::solve(problem, h, tx, init_tour));
    case Solvers::ThreeOpt:
        if (opts.cuda_mode == "neighbor")
            return Result<Solution>::ok(three_opt::solve_with(problem, "neighbor", tx, init_tour, opts.cuda_candidates));
        return Result<Solution>::ok(three_opt::solve(problem, h, tx, init_tour));
    case Solvers::TwoOpt:
        if (opts.cuda_mode.empty() && opts.cuda_path.empty())
            return Result<Solution>::ok(two_opt::solve(problem, h, tx, init_tour));
        return Result<Solution>::ok(
            two_opt::solve_with(problem, opts.cuda_mode, opts.cuda_path, tx, init_tour, opts.cuda_candidates));
    case Solvers::TwoOptBest:
        return Result<Solution>::ok(two_opt::solve_with(problem, "best", opts.cuda_path, tx, init_tour));
    case Solvers::AntColony: { // mod.rs:1706-1711: options validated, then ant_colony::solve
        const AcoOptions o = opts.aco.value_or(AcoOptions{});
        auto av = o.validate();
        if (av.is_err()) return Result<Solution>::err(av.error);
        return Result<Solution>::ok(ant_colony::solve(problem, o, tx, init_tour, opts.cuda_seed));
    }
    case Solvers::GeneticAlgorithm: {
        GAOptions o = opts.ga.value_or(GAOptions{});
        if (!opts.ga && opts.heuristic) o.heuristic = *opts.heuristic; // CLI --epochs reaches the GA this way
        auto gv = o.validate();
        if (gv.is_err()) return Result<Solution>::err(gv.error);
        return Result<Solution>::ok(genetic_algorithm::solve(problem, o, tx, init_tour, opts.cuda_seed));
    }
    case Solvers::RandomShuffle: return Result<Solution>::ok(random_shuffle::solve(problem, opts.cuda_seed));
    case Solvers::Unspecified: return Result<Solution>::err("solver not specified");
    default:
        return Result<Solution>::err(std::string("solver ") + solver_name(solver) +
                                     " is outside the accelerated path of this build (nn, greedy_edge, 2opt, or_opt, 3opt, aco, ga)");
    }
}

Result<Solution> solve_problem(Solvers solver, const TspProblem &problem, const AppOptions &opts)
{
    return solve_with_context(solver, problem, opts, nullptr, nullptr);
}

// ---- options --------------------------------------------------------------------------------------------

std::string TomlValue::display() const
{
    if (auto s = as_str()) return "\"" + *s + "\"";
    if (auto i = as_integer()) return std::to_string(*i);
    if (auto f = as_float()) {
        std::ostringstream o;
        o << *f;
        std::string t = o.str();
        if (t.find_first_of(".en") == std::string::npos) t += ".0";
        return t;
    }
    if (auto b = as_bool()) return *b ? "true" : "false";
    if (as_table()) return "{ .. }";
    if (as_array()) return "[ .. ]";
    return "";
}

const TomlValue *toml_get(const TomlTable &t, const std::string &key)
{
    for (const auto &kv : t)
        if (kv.first == key) return &kv.second;
    return nullptr;
}

Result<HeuristicOptions> HeuristicOptions::from_toml(const TomlTable &table)
{
    HeuristicOptions h;
    for (const auto &kv : table) {
        const std::string &k = kv.first;
        const TomlValue &v = kv.second;
        if (k == "epochs" || k == "platoo_epochs" || k == "n_nearest") {
            const int64_t *i = v.as_integer();
            if (!i) return Result<HeuristicOptions>::err("config: `" + k + "` must be an integer, got " + v.display());
            (k == "epochs" ? h.epochs : k == "platoo_epochs" ? h.platoo_epochs : h.n_nearest) = (size_t)*i;
        } else if (k == "verbose") {
            const bool *b = v.as_bool();
            if (!b) return Result<HeuristicOptions>::err("config: `verbose` must be a bool, got " + v.display());
            h.verbose = *b;
        } else {
            return Result<HeuristicOptions>::err("config: unknown field `" + k +
                                                 "` in [heuristic] — valid: epochs, platoo_epochs, n_nearest, verbose");
        }
    }
    auto v = h.validate();
    if (v.is_err()) return Result<HeuristicOptions>::err(v.error);
    return Result<HeuristicOptions>::ok(h);
}

Result<bool> HeuristicOptions::validate() const
{
    if (n_nearest == 0) return Result<bool>::err("n_nearest must be >= 1");
    return Result<bool>::ok(true);
}

namespace {

// `{}` of an f32 in the reference's messages: shortest round-trip decimal; %g is enough for the values users type
std::string fmt_f32(float v)
{
    char b[64];
    std::snprintf(b, sizeof b, "%g", v);
    return b;
}

// parse_f32 (mod.rs:1602-1607): a float, or an integer widened
bool toml_f32(const TomlValue &v, float &out)
{
    if (const double *d = v.as_float()) { out = (float)*d; return true; }
    if (const int64_t *i = v.as_integer()) { out = (float)*i; return true; }
    return false;
}

// the four HeuristicOptions keys every population table accepts; returns 0 = not one of them, 1 = ok, -1 = error
int heuristic_key(const std::string &k, const TomlValue &v, HeuristicOptions &h, std::string &err)
{
    if (k == "epochs" || k == "platoo_epochs" || k == "n_nearest") {
        const int64_t *i = v.as_integer();
        if (!i || *i < 0) { err = "config: `" + k + "` must be a non-negative integer, got " + v.display(); return -1; }
        (k == "epochs" ? h.epochs : k == "platoo_epochs" ? h.platoo_epochs : h.n_nearest) = (size_t)*i;
        return 1;
    }
    if (k == "verbose") {
        const bool *b = v.as_bool();
        if (!b) { err = "config: `verbose` must be a bool, got " + v.display(); return -1; }
        h.verbose = *b;
        return 1;
    }
    return 0;
}

} // namespace

Result<bool> AcoOptions::validate() const // mod.rs:1114-1153
{
    if (!std::isfinite(alpha) || alpha < 0.0f) return Result<bool>::err("alpha must be >= 0 (got " + fmt_f32(alpha) + ")");
    if (!(beta >= 0.0f && beta <= 6.0f)) return Result<bool>::err("beta must be in [0, 6] (got " + fmt_f32(beta) + ")");
    if (!std::isfinite(evaporation_rate) || evaporation_rate <= 0.0f || evaporation_rate >= 1.0f)
        return Result<bool>::err("evaporation_rate must be in (0, 1) (got " + fmt_f32(evaporation_rate) + ")");
    if (num_ants == 0) return Result<bool>::err("num_ants must be >= 1");
    return Result<bool>::ok(true);
}

Result<AcoOptions> AcoOptions::from_toml(const TomlTable &table) // mod.rs:1155-1196
{
    AcoOptions a;
    for (const auto &kv : table) {
        const std::string &k = kv.first;
        std::string err;
        const int hk = heuristic_key(k, kv.second, a.heuristic, err);
        if (hk < 0) return Result<AcoOptions>::err(err);
        if (hk > 0) continue;
        if (k == "alpha" || k == "beta" || k == "evaporation_rate") {
            float f;
            if (!toml_f32(kv.second, f))
                return Result<AcoOptions>::err("config: `aco." + k + "` must be a float, got " + kv.second.display());
            (k == "alpha" ? a.alpha : k == "beta" ? a.beta : a.evaporation_rate) = f;
        } else if (k == "num_ants") {
            const int64_t *i = kv.second.as_integer();
            if (!i || *i < 0)
                return Result<AcoOptions>::err("config: `aco.num_ants` must be a non-negative integer, got " + kv.second.display());
            a.num_ants = (size_t)*i;
        } else {
            return Result<AcoOptions>::err("config: unknown field `" + k +
                                           "` in [aco] — valid: epochs, platoo_epochs, n_nearest, verbose, alpha, beta, "
                                           "evaporation_rate, num_ants");
        }
    }
    auto v = a.validate();
    if (v.is_err()) return Result<AcoOptions>::err(v.error);
    return Result<AcoOptions>::ok(a);
}

Result<bool> GAOptions::validate() const // mod.rs:832-845
{
    auto h = heuristic.validate();
    if (h.is_err()) return h;
    if (!std::isfinite(mutation_probability) || mutation_probability < 0.0f || mutation_probability > 1.0f)
        return Result<bool>::err("mutation_probability must be in [0, 1] (got " + fmt_f32(mutation_probability) + ")");
    return Result<bool>::ok(true);
}

Result<GAOptions> GAOptions::from_toml(const TomlTable &table) // mod.rs:847-890
{
    GAOptions g;
    for (const auto &kv : table) {
        const std::string &k = kv.first;
        std::string err;
        const int hk = heuristic_key(k, kv.second, g.heuristic, err);
        if (hk < 0) return Result<GAOptions>::err(err);
        if (hk > 0) continue;
        if (k == "mutation_probability") {
            if (!toml_f32(kv.second, g.mutation_probability))
                return Result<GAOptions>::err("config: `ga.mutation_probability` must be a float, got " + kv.second.display());
        } else if (k == "n_elite") {
            const int64_t *i = kv.second.as_integer();
            if (!i) return Result<GAOptions>::err("config: `ga.n_elite` must be an integer, got " + kv.second.display());
            g.n_elite = (size_t)*i;
        } else {
            return Result<GAOptions>::err("config: unknown field `" + k +
                                          "` in [ga] — valid: epochs, platoo_epochs, n_nearest, verbose, mutation_probability, n_elite");
        }
    }
    auto v = g.validate();
    if (v.is_err()) return Result<GAOptions>::err(v.error);
    return Result<GAOptions>::ok(g);
}

// ---- pipeline ---------------------------------------------------------------------------------------------

namespace pipeline {

Result<Solution> PipelineStage::solve(const std::vector<size_t> *init_tour) const
{
    return solve_with_context(solver, problem, options, progress_tx, init_tour);
}

Result<std::vector<StageOutcome>> run_pipeline_stages(const std::vector<PipelineStage> &stages)
{
    using R = Result<std::vector<StageOutcome>>;
    if (stages.empty()) return R::err("pipeline has no stages");
    std::optional<std::vector<size_t>> seed;
    std::vector<StageOutcome> outcomes;
    for (const PipelineStage &stage : stages) {
        if (seed) {
            auto ok = validate_tour(*seed, stage.problem.cities);
            if (ok.is_err()) {
                std::fprintf(stderr, "WARN pipeline: invalid seed (%s); using default seeding\n", ok.error.c_str());
                seed.reset();
            }
        }
        const auto t0 = std::chrono::steady_clock::now();
        auto sol = stage.solve(seed ? &*seed : nullptr);
        if (sol.is_err()) return R::err(sol.error);
        const auto ms = std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now() - t0).count();
        auto ok = validate_tour(sol.unwrap().route(), stage.problem.cities);
        if (ok.is_err()) return R::err(std::string("stage ") + solver_name(stage.solver) + " invalid tour: " + ok.error);
        seed = sol.unwrap().route();
        outcomes.push_back(StageOutcome{std::move(sol.unwrap()), (uint64_t)ms});
    }
    return R::ok(std::move(outcomes));
}

Result<Solution> run_pipeline(const std::vector<PipelineStage> &stages)
{
    auto r = run_pipeline_stages(stages);
    if (r.is_err()) return Result<Solution>::err(r.error);
    return Result<Solution>::ok(std::move(r.unwrap().back().solution));
}

std::vector<std::string> stage_warnings(const std::vector<Solvers> &solvers)
{
    std::vector<std::string> w;
    const size_t last = solvers.empty() ? 0 : solvers.size() - 1;
    for (size_t i = 0; i < solvers.size(); ++i) {
        const std::string at = std::to_string(i);
        if (i > 0) {
            if (solvers[i] == Solvers::NearestNeighbor)
                w.push_back("nn at stage " + at + " discards the warm-start seed from the previous stage");
            else if (solvers[i] == Solvers::GreedyEdge)
                w.push_back("greedy_edge at stage " + at + " discards the warm-start seed from the previous stage (it "
                            "always rebuilds from scratch)");
            else if (solvers[i] == Solvers::Savings)
                w.push_back("savings at stage " + at + " discards the warm-start seed from the previous stage (it "
                            "always rebuilds from scratch)");
        }
        if (i != last) {
            if (solvers[i] == Solvers::BellmanKarp)
                w.push_back("BellmanKarp at stage " + at + " ignores the warm-start seed entirely (the exact DP has no use "
                            "for a partial/seed tour) and its optimal result will be superseded by later stages");
            else if (solvers[i] == Solvers::BranchBound)
                w.push_back("BranchBound at stage " + at + " only uses the warm-start seed to prime its pruning bound, not "
                            "as a tour to refine, and its optimal result will be superseded by later stages");
        }
    }
    return w;
}

} // namespace pipeline

// ---- tsplib ------------------------------------------------------------------------------------------------

namespace tsplib {

namespace {

bool parse_f32(const std::string &tok, float &out)
{
    if (tok.empty()) return false;
    char *end = nullptr;
    const float v = std::strtof(tok.c_str(), &end);
    if (end == tok.c_str() || *end != '\0') return false;
    out = v;
    return true;
}

std::vector<std::string> split_ws(const std::string &s)
{
    std::vector<std::string> v;
    std::istringstream is(s);
    std::string t;
    while (is >> t) v.push_back(t);
    return v;
}

bool starts_with_number(const std::string &line)
{
    const auto toks = split_ws(line);
    float f;
    return !toks.empty() && parse_f32(toks[0], f);
}

// ^[A-Z_]\w*$ on the upper-cased line (tsplib.rs:21-22)
bool is_state_marker(const std::string &line)
{
    if (line.empty() || !(std::isupper((unsigned char)line[0]) || line[0] == '_')) return false;
    for (char c : line)
        if (!(std::isalnum((unsigned char)c) || c == '_')) return false;
    return true;
}

// ^(\w+)\s*:\s*(.+)$ (tsplib.rs:23-24)
bool key_value(const std::string &line, std::string &key, std::string &val)
{
    size_t k = 0;
    while (k < line.size() && (std::isalnum((unsigned char)line[k]) || line[k] == '_')) ++k;
    if (k == 0) return false;
    size_t p = k;
    while (p < line.size() && std::isspace((unsigned char)line[p])) ++p;
    if (p >= line.size() || line[p] != ':') return false;
    ++p;
    while (p < line.size() && std::isspace((unsigned char)line[p])) ++p;
    if (p >= line.size()) return false;
    key = line.substr(0, k);
    val = line.substr(p);
    return true;
}

Result<std::vector<float>> pack_weights(const std::string &fmt, const std::vector<float> &tok, size_t n)
{
    using R = Result<std::vector<float>>;
    std::vector<float> out;
    if (fmt == "FULL_MATRIX") {
        if (tok.size() != n * n)
            return R::err("FULL_MATRIX: expected " + std::to_string(n * n) + " tokens, got " + std::to_string(tok.size()));
        for (size_t i = 1; i < n; ++i)
            for (size_t j = 0; j < i; ++j) out.push_back(tok[i * n + j]);
    } else if (fmt == "UPPER_ROW") {
        const size_t expected = n * (n - 1) / 2;
        if (tok.size() != expected)
            return R::err("UPPER_ROW: expected " + std::to_string(expected) + " tokens, got " + std::to_string(tok.size()));
        std::vector<float> m(n * n, 0.0f);
        size_t idx = 0;
        for (size_t i = 0; i + 1 < n; ++i)
            for (size_t j = i + 1; j < n; ++j) {
                m[i * n + j] = m[j * n + i] = tok[idx++];
            }
        for (size_t i = 1; i < n; ++i)
            for (size_t j = 0; j < i; ++j) out.push_back(m[i * n + j]);
    } else if (fmt == "LOWER_DIAG_ROW") {
        const size_t expected = n * (n + 1) / 2;
        if (tok.size() != expected)
            return R::err("LOWER_DIAG_ROW: expected " + std::to_string(expected) + " tokens, got " +
                          std::to_string(tok.size()));
        size_t idx = 0;
        for (size_t i = 0; i < n; ++i) {
            out.insert(out.end(), tok.begin() + idx, tok.begin() + idx + i);
            idx += i + 1;
        }
    } else {
        return R::err("Unsupported EDGE_WEIGHT_FORMAT: " + fmt);
    }
    return R::ok(std::move(out));
}

Result<TspLibData> process_lines(std::istream &in)
{
    using R = Result<TspLibData>;
    enum State { Start, Insection, Outsection, End } state = Start;
    std::string section;
    std::map<std::string, std::string> meta;
    std::vector<KDPoint> cities;
    std::vector<float> weights;
    size_t line_no = 1;
    std::string raw;
    while (std::getline(in, raw)) {
        const std::string line = upper(trim(raw));
        ++line_no;
        if (state == End) break;
        if (is_state_marker(line)) { // tsplib.rs:161-164, next_state :324-337
            if (line == "EOF") state = End;
            else { state = Insection; section = line; }
            continue;
        }
        if (state == Start) {
            std::string k, v;
            if (!key_value(line, k, v)) return R::err("Failed to extract meta data on line." + std::to_string(line_no));
            meta[k] = v;
        } else if (state == Insection && (section == "NODE_COORD_SECTION" || section == "DISPLAY_DATA_SECTION")) {
            if (!starts_with_number(line)) return R::err("Failed to extract coordinates on line." + std::to_string(line_no));
            const auto toks = split_ws(line);
            KDPoint p;
            p.id = (size_t)std::strtoull(toks[0].c_str(), nullptr, 10);
            std::vector<float> c;
            for (size_t t = 1; t < toks.size(); ++t) {
                float f;
                if (!parse_f32(toks[t], f)) return R::err("Error on line." + std::to_string(line_no) + " - invalid number");
                c.push_back(f);
            }
            p.coords[0] = c.size() > 0 ? c[0] : 0.0f;
            p.coords[1] = c.size() > 1 ? c[1] : 0.0f;
            cities.push_back(p);
        } else if (state == Insection && section == "EDGE_WEIGHT_SECTION") {
            for (const std::string &t : split_ws(line)) {
                float f;
                if (parse_f32(t, f)) weights.push_back(f);
            }
        }
    }
    if (meta.count("TYPE") && trim(meta["TYPE"]) == "ATSP") return R::err("ATSP (asymmetric TSP) is not supported");
    TspLibData d;
    if (meta.count("EDGE_WEIGHT_TYPE")) { // unknown types (ATT!) silently fall back to EUC_2D, tsplib.rs:199-202
        auto dt = parse_distance_type(trim(meta["EDGE_WEIGHT_TYPE"]));
        if (dt.is_ok()) d.distance_type = dt.unwrap();
    }
    if (meta.count("DIMENSION")) d.dimension = (size_t)std::strtoull(trim(meta["DIMENSION"]).c_str(), nullptr, 10);
    if (!weights.empty()) {
        auto packed = pack_weights(meta.count("EDGE_WEIGHT_FORMAT") ? trim(meta["EDGE_WEIGHT_FORMAT"]) : "", weights, d.dimension);
        if (packed.is_err()) return R::err(packed.error);
        d.raw_distances = std::move(packed.unwrap());
    }
    if (cities.empty() && d.raw_distances) { // grid placeholder coordinates, tsplib.rs:257-262
        const size_t cols = (size_t)std::ceil(std::sqrt((double)d.dimension));
        for (size_t i = 0; i < d.dimension; ++i) cities.push_back(KDPoint::new_with_id(i + 1, (float)(i % cols), (float)(i / cols)));
    }
    if (cities.empty() && !d.raw_distances) return R::err("Found no valid city coordinates");
    d.name = lower(meta.count("NAME") ? meta["NAME"] : "unspecified");
    d.comment = lower(meta.count("COMMENT") ? meta["COMMENT"] : "unspecified");
    d.cities = std::move(cities);
    return R::ok(std::move(d));
}

} // namespace

Result<DistanceMatrix> TspLibData::distance_matrix() const
{
    if (raw_distances) return Result<DistanceMatrix>::ok(DistanceMatrix::new_explicit(cities.size(), *raw_distances, cities));
    return DistanceMatrix::build(cities, distance_type);
}

Result<TspLibData> read_from_file(const std::string &path)
{
    std::ifstream f(path);
    if (!f) return Result<TspLibData>::err("tsplib: failed to read file");
    return process_lines(f);
}

Result<TspLibData> read_from_str(const std::string &input)
{
    std::istringstream s(input);
    return process_lines(s);
}

} // namespace tsplib

// ---- convert: DiscOpt coordinate files (src/tsp/convert.rs) --------------------------------------------------

namespace convert {

namespace {

// Rust's `{}` for f32: the shortest decimal that round-trips, never in exponent form
std::string f32_display(float v)
{
    char buf[128];
    auto r = std::to_chars(buf, buf + sizeof buf, v, std::chars_format::fixed);
    return std::string(buf, r.ptr);
}

// Rust's str::parse::<f32>: the whole token must be a float literal (no trailing junk, no hex)
bool parse_rust_f32(const std::string &tok, float &out)
{
    if (tok.empty()) return false;
    for (char ch : tok)
        if (ch == 'x' || ch == 'X') return false;
    char *end = nullptr;
    const float v = std::strtof(tok.c_str(), &end);
    if (end == tok.c_str() || *end != '\0') return false;
    out = v;
    return true;
}

} // namespace

// skip the first line (city count), then one `x y` pair per non-empty line (convert.rs:6-29)
Result<std::vector<std::pair<float, float>>> parse_discopt(const std::string &input)
{
    using R = Result<std::vector<std::pair<float, float>>>;
    std::vector<std::pair<float, float>> coords;
    std::istringstream is(input);
    std::string line;
    bool first = true;
    while (std::getline(is, line)) {
        if (first) { first = false; continue; }
        std::istringstream ls(line);
        std::string xs, ys;
        if (!(ls >> xs)) continue; // blank line
        float x = 0.f, y = 0.f;
        if (!parse_rust_f32(xs, x)) return R::err("invalid float literal");
        if (!(ls >> ys)) return R::err("missing y");
        if (!parse_rust_f32(ys, y)) return R::err("invalid float literal");
        coords.emplace_back(x, y);
    }
    if (coords.empty()) return R::err("no coordinates found");
    return R::ok(std::move(coords));
}

void write_tsplib(const std::string &name, const std::vector<std::pair<float, float>> &coords, std::ostream &w)
{
    w << "NAME: " << name << "\n";
    w << "TYPE: TSP\n";
    w << "COMMENT: converted from DiscOpt dataset " << name << "\n";
    w << "DIMENSION: " << coords.size() << "\n";
    w << "EDGE_WEIGHT_TYPE: EUC_2D\n";
    w << "NODE_COORD_SECTION\n";
    for (size_t i = 0; i < coords.size(); ++i)
        w << "\t" << (i + 1) << " " << f32_display(coords[i].first) << " " << f32_display(coords[i].second) << "\n";
    w << "EOF\n";
}

Result<bool> convert_file(const std::string &input_path, const std::string &output_path)
{
    std::ifstream in(input_path);
    if (!in) return Result<bool>::err("No such file or directory (os error 2)");
    std::stringstream ss;
    ss << in.rdbuf();
    auto coords = parse_discopt(ss.str());
    if (coords.is_err()) return Result<bool>::err(coords.error);
    // NAME = the input file stem
    std::string stem = input_path.substr(input_path.find_last_of('/') == std::string::npos ? 0 : input_path.find_last_of('/') + 1);
    const size_t dot = stem.find_last_of('.');
    if (dot != std::string::npos && dot != 0) stem = stem.substr(0, dot);
    std::ofstream out(output_path);
    if (!out) return Result<bool>::err("cannot create " + output_path);
    write_tsplib(stem, coords.unwrap(), out);
    return Result<bool>::ok(true);
}

} // namespace convert

// ---- a minimal TOML reader (the subset the reference's pipeline configs use) ---------------------------------

namespace {

struct TomlParser {
    const std::string &src;
    size_t pos = 0;
    int line = 1;
    explicit TomlParser(const std::string &s) : src(s) {}

    std::string fail(const std::string &msg) const { return "TOML parse error at line " + std::to_string(line) + ": " + msg; }
    void skip_inline_ws()
    {
        while (pos < src.size() && (src[pos] == ' ' || src[pos] == '\t')) ++pos;
    }
    void skip_comment()
    {
        if (pos < src.size() && src[pos] == '#')
            while (pos < src.size() && src[pos] != '\n') ++pos;
    }
    bool parse_key(std::string &key)
    {
        skip_inline_ws();
        key.clear();
        if (pos < src.size() && (src[pos] == '"' || src[pos] == '\'')) {
            const char q = src[pos++];
            while (pos < src.size() && src[pos] != q && src[pos] != '\n') key += src[pos++];
            if (pos >= src.size() || src[pos] != q) return false;
            ++pos;
            return true;
        }
        while (pos < src.size() && (std::isalnum((unsigned char)src[pos]) || src[pos] == '_' || src[pos] == '-')) key += src[pos++];
        return !key.empty();
    }
    bool parse_value(TomlValue &out, std::string &err)
    {
        skip_inline_ws();
        if (pos >= src.size()) { err = fail("missing value"); return false; }
        const char c = src[pos];
        if (c == '"' || c == '\'') {
            ++pos;
            std::string s;
            while (pos < src.size() && src[pos] != c && src[pos] != '\n') {
                if (c == '"' && src[pos] == '\\' && pos + 1 < src.size()) {
                    const char e = src[pos + 1];
                    s += e == 'n' ? '\n' : e == 't' ? '\t' : e;
                    pos += 2;
                } else {
                    s += src[pos++];
                }
            }
            if (pos >= src.size() || src[pos] != c) { err = fail("unterminated string"); return false; }
            ++pos;
            out.v = s;
            return true;
        }
        if (c == '[') { // inline array
            ++pos;
            auto arr = std::make_shared<std::vector<TomlValue>>();
            for (;;) {
                while (pos < src.size() && (std::isspace((unsigned char)src[pos]) || src[pos] == ',')) { if (src[pos] == '\n') ++line; ++pos; }
                if (pos < src.size() && src[pos] == ']') { ++pos; break; }
                TomlValue v;
                if (!parse_value(v, err)) return false;
                arr->push_back(v);
            }
            out.v = arr;
            return true;
        }
        std::string tok;
        while (pos < src.size() && !std::isspace((unsigned char)src[pos]) && src[pos] != '#' && src[pos] != ',' && src[pos] != ']') tok += src[pos++];
        if (tok == "true" || tok == "false") { out.v = (tok == "true"); return true; }
        std::string clean;
        for (char ch : tok) if (ch != '_') clean += ch;
        if (clean.empty()) { err = fail("missing value"); return false; }
        char *end = nullptr;
        if (clean.find_first_of(".eE") == std::string::npos || clean == "inf" || clean == "nan") {
            const long long i = std::strtoll(clean.c_str(), &end, 10);
            if (end && *end == '\0') { out.v = (int64_t)i; return true; }
        }
        const double f = std::strtod(clean.c_str(), &end);
        if (end && *end == '\0') { out.v = f; return true; }
        err = fail("invalid value `" + tok + "`");
        return false;
    }
};

TomlTable *descend(TomlTable *t, const std::string &key, bool array_elem, std::string &err)
{
    for (auto &kv : *t) {
        if (kv.first != key) continue;
        if (auto tp = std::get_if<std::shared_ptr<TomlTable>>(&kv.second.v)) return tp->get();
        if (auto ap = std::get_if<std::shared_ptr<std::vector<TomlValue>>>(&kv.second.v)) {
            if ((*ap)->empty()) { err = "empty array of tables `" + key + "`"; return nullptr; }
            if (array_elem) return nullptr; // caller appends
            auto tp = std::get_if<std::shared_ptr<TomlTable>>(&(*ap)->back().v);
            return tp ? tp->get() : nullptr;
        }
        err = "key `" + key + "` is not a table";
        return nullptr;
    }
    auto nt = std::make_shared<TomlTable>();
    TomlValue v;
    v.v = nt;
    t->push_back({key, v});
    return nt.get();
}

} // namespace

Result<TomlTable> parse_toml(const std::string &source)
{
    using R = Result<TomlTable>;
    TomlTable root;
    TomlTable *cur = &root;
    TomlParser p(source);
    while (p.pos < source.size()) {
        p.skip_inline_ws();
        if (p.pos >= source.size()) break;
        const char c = source[p.pos];
        if (c == '\n') { ++p.line; ++p.pos; continue; }
        if (c == '\r') { ++p.pos; continue; }
        if (c == '#') { p.skip_comment(); continue; }
        if (c == '[') {
            const bool arr = p.pos + 1 < source.size() && source[p.pos + 1] == '[';
            p.pos += arr ? 2 : 1;
            std::vector<std::string> parts;
            for (;;) {
                std::string k;
                if (!p.parse_key(k)) return R::err(p.fail("invalid table header"));
                parts.push_back(k);
                p.skip_inline_ws();
                if (p.pos < source.size() && source[p.pos] == '.') { ++p.pos; continue; }
                break;
            }
            if (source.compare(p.pos, arr ? 2 : 1, arr ? "]]" : "]") != 0) return R::err(p.fail("invalid table header"));
            p.pos += arr ? 2 : 1;
            TomlTable *t = &root;
            std::string err;
            for (size_t i = 0; i < parts.size(); ++i) {
                const bool last = i + 1 == parts.size();
                if (last && arr) {
                    std::shared_ptr<std::vector<TomlValue>> a;
                    for (auto &kv : *t)
                        if (kv.first == parts[i]) {
                            auto ap = std::get_if<std::shared_ptr<std::vector<TomlValue>>>(&kv.second.v);
                            if (!ap) return R::err(p.fail("key `" + parts[i] + "` is not an array of tables"));
                            a = *ap;
                        }
                    if (!a) {
                        a = std::make_shared<std::vector<TomlValue>>();
                        TomlValue v;
                        v.v = a;
                        t->push_back({parts[i], v});
                    }
                    auto nt = std::make_shared<TomlTable>();
                    TomlValue ev;
                    ev.v = nt;
                    a->push_back(ev);
                    t = nt.get();
                } else {
                    t = descend(t, parts[i], false, err);
                    if (!t) return R::err(p.fail(err.empty() ? "invalid table path" : err));
                }
            }
            cur = t;
            p.skip_inline_ws();
            p.skip_comment();
            continue;
        }
        std::string key;
        if (!p.parse_key(key)) return R::err(p.fail("expected a key"));
        p.skip_inline_ws();
        if (p.pos >= source.size() || source[p.pos] != '=') return R::err(p.fail("expected `=` after key `" + key + "`"));
        ++p.pos;
        TomlValue v;
        std::string err;
        if (!p.parse_value(v, err)) return R::err(err);
        if (toml_get(*cur, key)) return R::err(p.fail("duplicate key `" + key + "`"));
        cur->push_back({key, v});
        p.skip_inline_ws();
        p.skip_comment();
        if (p.pos < source.size() && source[p.pos] != '\n' && source[p.pos] != '\r') return R::err(p.fail("unexpected text after value"));
    }
    return R::ok(std::move(root));
}

} // namespace tsp

// ---- config (src/config.rs:23-153) -------------------------------------------------------------------------------

namespace config {

using tsp::AppOptions;
using tsp::Solvers;
using tsp::TomlTable;
using tsp::TomlValue;

namespace {

Result<AppOptions> provide(const TomlTable &table, AppOptions base)
{
    static const char *kSub[] = {"sa", "ga", "cs", "fpa", "fourier", "lk", "som", "aco"};
    for (const auto &kv : table) {
        const std::string &key = kv.first;
        if (key == "solver") continue;
        bool known_sub = false;
        for (const char *s : kSub) known_sub = known_sub || key == s;
        if (key == "aco" || key == "ga") {
            const TomlTable *t = kv.second.as_table();
            if (!t) return Result<AppOptions>::err("config: `" + key + "` must be a table");
            if (key == "aco") {
                auto a = tsp::AcoOptions::from_toml(*t);
                if (a.is_err()) return Result<AppOptions>::err(a.error);
                base.aco = a.unwrap();
            } else {
                auto g = tsp::GAOptions::from_toml(*t);
                if (g.is_err()) return Result<AppOptions>::err(g.error);
                base.ga = g.unwrap();
            }
        } else if (known_sub) { // validated as tables; their solvers are outside this build's path
            if (!kv.second.as_table()) return Result<AppOptions>::err("config: `" + key + "` must be a table");
        } else if (key == "heuristic") {
            const TomlTable *t = kv.second.as_table();
            if (!t) return Result<AppOptions>::err("config: `heuristic` must be a table");
            auto h = tsp::HeuristicOptions::from_toml(*t);
            if (h.is_err()) return Result<AppOptions>::err(h.error);
            base.heuristic = h.unwrap();
        } else if (key == "cuda") { // extension table of this build, never required
            const TomlTable *t = kv.second.as_table();
            if (!t) return Result<AppOptions>::err("config: `cuda` must be a table");
            for (const auto &ckv : *t) {
                const std::string *s = ckv.second.as_str();
                const int64_t *iv = ckv.second.as_integer();
                if (ckv.first == "mode" && s) base.cuda_mode = *s;
                else if (ckv.first == "path" && s) base.cuda_path = *s;
                else if (ckv.first == "seed" && iv) base.cuda_seed = (uint64_t)*iv;
                else if (ckv.first == "candidates" && iv) {
                    if (*iv < 1 || *iv > 32) return Result<AppOptions>::err("config: [cuda] candidates must be in 1..32");
                    base.cuda_candidates = (uint32_t)*iv;
                }
                else return Result<AppOptions>::err("config: unknown field `" + ckv.first + "` in [cuda] — valid: mode, path (strings), seed, candidates (integers)");
            }
        } else {
            return Result<AppOptions>::err("config: unknown field `" + key +
                                           "` — valid stage fields: solver, sa, ga, cs, fpa, fourier, lk, som, aco, heuristic");
        }
    }
    return Result<AppOptions>::ok(std::move(base));
}

} // namespace

Result<std::vector<std::pair<Solvers, AppOptions>>> load_pipeline_config(const std::string &source, const AppOptions &base)
{
    using R = Result<std::vector<std::pair<Solvers, AppOptions>>>;
    auto root = tsp::parse_toml(source);
    if (root.is_err()) return R::err("config: " + root.error);
    const TomlValue *stage = tsp::toml_get(root.unwrap(), "stage");
    if (!stage) return R::err("config: missing [[stage]] array — at least one stage is required");
    const std::vector<TomlValue> *arr = stage->as_array();
    if (!arr) return R::err("config: `stage` must be an array of tables ([[stage]])");
    if (arr->empty()) return R::err("config: [[stage]] list is empty — at least one stage is required");
    std::vector<std::pair<Solvers, AppOptions>> stages;
    for (size_t i = 0; i < arr->size(); ++i) {
        const std::string at = std::to_string(i);
        const TomlTable *table = (*arr)[i].as_table();
        if (!table) return R::err("config: [[stage]] entry " + at + " is not a table");
        const TomlValue *sv = tsp::toml_get(*table, "solver");
        if (!sv) return R::err("config: [[stage]] entry " + at + " missing required `solver` field");
        const std::string *name = sv->as_str();
        if (!name) return R::err("config: [[stage]] entry " + at + ": `solver` must be a string");
        auto solver = tsp::find_solver(*name);
        if (solver.is_err()) return R::err("config: [[stage]] entry " + at + ": unknown solver `" + *name + "`");
        auto opts = provide(*table, base);
        if (opts.is_err()) return R::err(opts.error);
        const Solvers s = solver.unwrap();
        const std::pair<const char *, bool> belongs[] = {
            {"sa", s == Solvers::SimulatedAnnealing}, {"ga", s == Solvers::GeneticAlgorithm},
            {"cs", s == Solvers::CuckooSearch}, {"fpa", s == Solvers::FlowerPollination},
            {"fourier", s == Solvers::Fourier}, {"lk", s == Solvers::LinKernighan},
            {"som", s == Solvers::KohonenSom}, {"aco", s == Solvers::AntColony},
            {"heuristic", !(s == Solvers::SimulatedAnnealing || s == Solvers::GeneticAlgorithm || s == Solvers::CuckooSearch ||
                            s == Solvers::FlowerPollination || s == Solvers::Fourier || s == Solvers::LinKernighan ||
                            s == Solvers::KohonenSom || s == Solvers::AntColony)},
        };
        for (const auto &b : belongs)
            if (tsp::toml_get(*table, b.first) && !b.second)
                return R::err("config: stage " + at + " (" + *name + "): `[stage." + b.first + "]` is not valid for this solver");
        stages.push_back({s, std::move(opts.unwrap())});
    }
    return R::ok(std::move(stages));
}

} // namespace config
} // namespace teeline
