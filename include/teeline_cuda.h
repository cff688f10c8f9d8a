/*
 * teeline_cuda.h -- C ABI of libteeline_cuda.so (sm_100a / B200).
 *
 * This is the drop-in boundary for the data-parallel local-search hot path of
 * timgluz/teeline (reference @ cd06a10).  The reference has no FFI layer; the
 * seam is its solver-function convention
 *     pub fn solve(&TspProblem, &HeuristicOptions, Option<&Sender<ProgressMessage>>,
 *                  Option<&[usize]>) -> Solution          (src/tsp/two_opt.rs:7-12,
 *                                                          src/tsp/or_opt.rs:19-24)
 * plus DistanceMatrix::{build,tour_length,tour_length_by_pos,nearest}
 * (src/tsp/distance_matrix.rs:122-153,221-245,259-280) and
 * lin_kernighan::build_candidates (src/tsp/lin_kernighan.rs:12-27).  Each entry
 * point below names the reference function body it replaces.  INTEGRATION.md
 * shows the Rust `extern "C"` block + build.rs a maintainer would add.
 *
 * Conventions
 *  - Every pointer argument is a HOST pointer owned by the caller; the library
 *    copies in and out.  Handles are opaque and owned by the library.
 *  - Cities are addressed by POSITION 0..n-1 (index into the coordinate arrays,
 *    i.e. DistanceMatrix's `pos`), never by TSPLIB id.  The shim translates ids
 *    with city_id2pos / pos2city_id (distance_matrix.rs:251-257).
 *  - Every function returns tl_status (0 = OK).  tl_last_error() returns a
 *    thread-local message for the last failure.  Nothing throws across the ABI.
 *  - There is no CPU fallback: without a CUDA device every call fails with
 *    TL_ERR_CUDA.
 *  - Re-entrant: no global mutable state; one CUDA stream per tl_ctx; calls on
 *    different contexts may run concurrently from different host threads.
 */
#ifndef TEELINE_CUDA_H
#define TEELINE_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef int32_t tl_status;
enum {
    TL_OK = 0,
    TL_ERR_INVALID = 1,     /* bad argument (null pointer, n < 2, tour not a permutation, ...) */
    TL_ERR_CUDA = 2,        /* CUDA runtime / driver error, or no device                        */
    TL_ERR_UNSUPPORTED = 3, /* e.g. recompute path on an EXPLICIT problem                       */
    TL_ERR_NOMEM = 4,       /* n^2 matrix does not fit device memory                             */
    TL_ERR_NCCL = 5
};

typedef struct tl_ctx tl_ctx;
typedef struct tl_problem tl_problem;
typedef struct tl_session tl_session;

/* distance kinds */
enum {
    TL_DIST_F32_EXACT = 0, /* reference metric: un-rounded f32 sqrt(dx*dx+dy*dy), kdtree.rs:291-295 */
    TL_DIST_NINT_I32 = 1   /* TSPLIB nint(sqrt(.)) in f64 -> int32 (no reference twin)              */
};

/* local-search algorithms */
enum {
    TL_ALGO_TWO_OPT_REF = 0,         /* "Mode R": first-improvement, two_opt.rs:26-61 (bit-exact) */
    TL_ALGO_TWO_OPT_BEST = 1,        /* "Mode B": best-improvement, same neighbourhood            */
    TL_ALGO_TWO_OPT_BEST_CYCLIC = 2, /* Mode B incl. closing edge (two-opt-algo.ts:71-99)         */
    TL_ALGO_OR_OPT = 3,              /* or_opt.rs:80-184 (best-improvement, bit-exact)            */
    TL_ALGO_THREE_OPT = 4,           /* three_opt.rs:16-218 (best-improvement over triples, bit-exact) */
    TL_ALGO_TWO_OPT_BEST_CACHED = 5, /* Mode B, the same moves and tour as TL_ALGO_TWO_OPT_BEST, but a step only
                                        re-evaluates the pairs the previous move changed (cached row minima):
                                        the fast way to the local optimum; stats.evals counts the pairs actually
                                        computed.  Not shardable, no tl_session_scan / time_scans. */
    TL_ALGO_TWO_OPT_NEIGHBOR = 6,    /* "Mode N": Mode B's move and delta over the pairs that create an edge to
                                        one of a city's k nearest neighbours (see tl_problem_set_candidates):
                                        a step costs O(n k) instead of O(n^2), for 10^5..10^6 cities.
                                        Coordinate problems (F32_EXACT, NINT_I32), TL_PATH_AUTO / RECOMPUTE;
                                        stats.evals counts the generated pairs.  Not shardable, not batched. */
    TL_ALGO_OR_OPT_NEIGHBOR = 7,     /* "Or-opt N": TL_ALGO_OR_OPT's move, delta, forbidden window and tie order
                                        over the moves that create an edge between a segment endpoint and one
                                        of its k nearest neighbours (see tl_problem_set_candidates): a step
                                        costs O(n k) instead of O(n^2).  Same problems, paths and limits as
                                        Mode N; n < 4 returns the identity order with no scan, as
                                        TL_ALGO_OR_OPT does. */
    TL_ALGO_THREE_OPT_NEIGHBOR = 8,  /* "3-opt N": TL_ALGO_THREE_OPT's triples, costs, case choice and tie order
                                        over the triples that the first two candidate edges of a sequential
                                        3-exchange generate (see tl_problem_set_candidates): a step costs
                                        O(n k^2) instead of O(n^3).  Same problems, paths and limits as Or-opt N;
                                        n < 4 returns the identity order with no scan, as TL_ALGO_THREE_OPT
                                        does. */
    TL_ALGO_TWO_OPT_NEIGHBOR_MULTI = 9, /* "Mode NM": Mode N's pairs, deltas and order, but a step also applies the
                                        best improving pair of every block of TL_MULTI_BLOCK positions that is
                                        disjoint from Mode N's move (see tl_problem_set_candidates): far fewer
                                        steps to a Mode N local optimum.  Same problems, paths and limits as
                                        Mode N; n < 4 returns the identity order with no scan. */
    TL_ALGO_OR_OPT_NEIGHBOR_MULTI = 10 /* "Or-opt NM": Or-opt N's moves, deltas, threshold and order, but a step also
                                        applies the best move of every block of TL_OR_MULTI_BLOCK positions that does
                                        not touch Or-opt N's move (see tl_problem_set_candidates): far fewer steps
                                        to an Or-opt N local optimum.  Same problems, paths and limits as Or-opt N;
                                        n < 4 returns the identity order with no scan. */
};

/* Mode NM's block size in positions (a power of two).  Among 256, 1024 and 4096, 4096 took the fewest steps and
 * the least time to the optimum of 10^6-city greedy and NN tours on a B200 at a 1000 W power limit (5010 steps,
 * 0.71 s from greedy; profiles/r05e_two_opt_neighbor_multi_timing.json, DESIGN.md section 5).  Instances of a
 * few blocks (about 2*10^4 cities) take fewer steps with smaller blocks. */
#define TL_MULTI_BLOCK 4096
/* Or-opt NM's block size in positions (a power of two, at most 16384).  Among 1024, 4096 and 16384, 16384 took the
 * fewest steps and the least time from the Mode NM optima of 10^6-city greedy and NN tours on a B200 at a 1000 W
 * power limit (1176 steps, 0.28 s from greedy against 0.37 s for 4096; profiles/r05f_or_opt_neighbor_multi_timing.json,
 * DESIGN.md section 5).  At 10^5 cities 4096 took half the time of 16384. */
#define TL_OR_MULTI_BLOCK 16384

/* where distances come from during the scan */
enum {
    TL_PATH_AUTO = 0,     /* matrix for EXPLICIT and NINT_I32 problems, recompute for F32_EXACT coordinates */
    TL_PATH_MATRIX = 1,   /* n x n matrix in HBM, tour-ordered, re-permuted as the tour fragments */
    TL_PATH_RECOMPUTE = 2 /* distances recomputed from tour-ordered coordinates (bit-identical)   */
};

/* tour-length modes */
enum {
    TL_LEN_EXACT = 0, /* sequential f32 sum, closing edge first (distance_matrix.rs:235-245) */
    TL_LEN_FAST = 1   /* pairwise f64 reduction of the same f32 edge lengths                  */
};

typedef struct {
    float delta;      /* f32 delta of the applied move (exact int value for NINT_I32)          */
    uint32_t i, j;    /* 2-opt: path[i+1..=j] reversed.  Or-opt: segment start, insert-after j.
                         3-opt: the first two cut positions                                     */
    uint8_t seg_len;  /* Or-opt: 1..3; 3-opt: reconnection case 1..7; 0 for 2-opt              */
    uint8_t reversed; /* Or-opt: segment re-inserted reversed                                  */
    uint16_t pad;
    uint32_t k;       /* 3-opt: the third cut position; 0 otherwise                            */
} tl_move;

typedef struct {
    uint64_t passes;    /* Mode R: outer `while improved` iterations; otherwise full scans     */
    uint64_t moves;     /* applied moves                                                       */
    uint64_t evals;     /* candidate moves whose delta was computed                            */
    uint64_t launches;  /* CUDA kernels launched by the call                                   */
    uint64_t repermutes;/* matrix path: how many times the matrix was re-laid in tour order    */
    double device_ms;   /* CUDA-event time from first to last kernel of the call               */
    int32_t converged;  /* 1 = local optimum reached, 0 = stopped by max_moves                  */
    int32_t path_used;  /* TL_PATH_MATRIX or TL_PATH_RECOMPUTE                                  */
} tl_stats;

/* ---- context ---------------------------------------------------------------- */

/* device: CUDA ordinal.  The context owns one non-blocking stream. */
tl_status tl_ctx_create(int32_t device, tl_ctx **out);
/* Same, but launch everything on a caller-owned cudaStream_t (passed as void*), so
 * that the caller's own CUDA events bracket the library's kernels. */
tl_status tl_ctx_create_on_stream(int32_t device, void *cuda_stream, tl_ctx **out);
void tl_ctx_destroy(tl_ctx *ctx);
tl_status tl_ctx_sync(tl_ctx *ctx);
const char *tl_last_error(void);
const char *tl_version(void);
/* kernels launched by this context since creation (bench.py's gpu_launches) */
uint64_t tl_ctx_launch_count(const tl_ctx *ctx);

/* Multi-GPU (one process per GPU).  Rank 0 makes the id, the host runtime
 * (torch.distributed) broadcasts it, every rank attaches (collective call).  Attaching
 * also maps every rank's 1 KB "mailbox" into every other process (cudaIpc over NVLink):
 * a sharded Mode B step then exchanges the per-rank best records INSIDE the scan kernel
 * (peer stores + polling by the last CTA, csrc/shard_exchange.cuh) and applies the move in
 * the same launch.  If peers cannot be mapped (or TL_SHARD_TRANSPORT=nccl) the step is
 * scan -> ncclAllGather -> apply kernel instead; results are identical. */
#define TL_NCCL_ID_BYTES 128
tl_status tl_nccl_unique_id(uint8_t id_out[TL_NCCL_ID_BYTES]);
tl_status tl_ctx_attach_nccl(tl_ctx *ctx, const uint8_t id[TL_NCCL_ID_BYTES], int32_t rank,
                             int32_t world);

/* ---- problem ------------------------------------------------------------------ */

/* Replaces DistanceMatrix::build for EUC_2D (distance_matrix.rs:122-153; call site
 * tsplib.rs:84-98): uploads the coordinates; matrices are built on demand. */
tl_status tl_problem_create_euc2d(tl_ctx *ctx, uint32_t n, const float *x, const float *y,
                                  int32_t dist_kind, tl_problem **out);
/* EXPLICIT / GEO problems: DistanceMatrix::new with precomputed distances
 * (distance_matrix.rs:96-115); packed strict lower triangle, idx = hi(hi-1)/2+lo. */
tl_status tl_problem_create_explicit(tl_ctx *ctx, uint32_t n, const float *packed_tri,
                                     tl_problem **out);
void tl_problem_destroy(tl_problem *p);

/* DistanceMatrix::distances() (distance_matrix.rs:171-173): the packed triangle,
 * n(n-1)/2 values, bit-identical to the reference's Vec<f32>. */
tl_status tl_dist_matrix_packed(tl_problem *p, float *out);
tl_status tl_dist_matrix_packed_i32(tl_problem *p, int32_t *out); /* NINT_I32 problems */

/* DistanceMatrix::nearest for every city at once / build_candidates
 * (distance_matrix.rs:259-297, lin_kernighan.rs:12-27): out is n*k positions,
 * ascending distance, ties by lower position, rows padded with UINT32_MAX. */
tl_status tl_knn(tl_problem *p, uint32_t k, uint32_t *out);

/* Candidate lists for TL_ALGO_TWO_OPT_NEIGHBOR[_MULTI], TL_ALGO_OR_OPT_NEIGHBOR[_MULTI] and TL_ALGO_THREE_OPT_NEIGHBOR,
 * built
 * on the device by
 * tl_knn's kernel and kept with the problem (they depend on the instance only, like
 * lin_kernighan::build_candidates, lin_kernighan.rs:12-27).  K[c] = the first k entries of tl_knn(k)
 * for city c; padded slots (k > n-1) are skipped.
 *
 * Mode N: for every position i and slot s, with b = K[p_i][s], j = pos[b], lo = min(i, j),
 * hi = max(i, j), the search generates the pairs (lo, hi) (the candidate edge is the move's first new
 * edge) and (lo-1, hi-1) (its second new edge); a pair counts if it lies in Mode B's neighbourhood
 * 0 <= i, i+2 <= j <= n-2.  A step applies the argmin of (delta, i, j) over them with strict '< 0',
 * exactly as TL_ALGO_TWO_OPT_BEST; with k >= n-1 the moves are Mode B's.
 *
 * Or-opt N: with f = p_i, l = p_i+s-1, x = p_j, y = p_(j+1)%n, for every position q, c = p_q, slot t,
 * b = K[c][t] and r = pos[b], the search generates the Or-opt moves (segment [i, i+s-1] inserted
 * between x and y) whose new edge is (c, b):
 *   (f, x) forward:  i = q,     j = r,           s = 1..3
 *   (l, y) forward:  i = q-s+1, j = (r-1) mod n, s = 1..3
 *   (l, x) reversed: i = q-s+1, j = r,           s = 2..3
 *   (f, y) reversed: i = q,     j = (r-1) mod n, s = 2..3
 * A move counts if it is legal for TL_ALGO_OR_OPT (n > s+1, 0 <= i, i+s <= n, j != prev(i), j outside
 * [i, i+s-1]); its delta is TL_ALGO_OR_OPT's in the same rounding order, and a step applies the minimum
 * of (delta, s, i, j, reversed) below Or-opt's threshold (-1e-3 in f32, 0 for NINT_I32), as
 * TL_ALGO_OR_OPT's first-found scan does.  stats.evals counts the generated legal moves, forward and
 * reversed separately, duplicates included.  With k >= n-1 every legal move is generated, so the moves
 * are TL_ALGO_OR_OPT's.
 *
 * 3-opt N: cut edge e (0 <= e <= n-1) joins p_e and p_(e+1)%n; TL_ALGO_THREE_OPT's triple (i, j, k) with
 * i < j < k removes edges i, j and k.  Following the first two candidate edges of a sequential
 * 3-exchange, for every position q, c = p_q:
 *   1. every slot s1 with b = K[c][s1] not padding, r = pos[b];
 *   2. each e2 in {(r-1) mod n, r}; t = the other endpoint of edge e2: p_(r+1)%n when e2 = r, p_(r-1)%n
 *      otherwise;
 *   3. every slot s2 with b' = K[t][s2] not padding, r' = pos[b'];
 *   4. each e1 in {(q-1) mod n, q} and e3 in {(r'-1) mod n, r'}: if e1, e2 and e3 are distinct, sorted
 *      into i < j < k, the triple counts unless i = 0 and k = n-1 (TL_ALGO_THREE_OPT's skip).
 * At most 8 triples per (q, s1, s2), 8 n k^2 per step.  Evaluation is TL_ALGO_THREE_OPT's: orig and
 * cost1..cost7 are its left-to-right sums in the metric's value type, the triple's case is the first
 * minimal cost among those below orig, and savings = orig - cost.  A step applies the counted triple with
 * the largest savings > 0, ties to the lowest (i, j, k); duplicates carry the same key.  stats.evals
 * counts every counted triple, duplicates included.  With k >= n-1 every triple is generated (q = i+1,
 * b = p_j, e2 = j, t = p_j+1, b' = p_k, e1 = i, e3 = k), so the moves are TL_ALGO_THREE_OPT's.
 *
 * Mode NM: Mode N's generated pairs, deltas and (delta, i, j) order with strict '< 0'.  Step t (t = the steps
 * the session has applied so far, 0 for the first step of a tl_local_search call) works on the tour as it stood
 * at the start of the step:
 *   1. G = Mode N's move, the argmin over all generated improving pairs; none: converged (Mode N's stop).
 *   2. With B = TL_MULTI_BLOCK and o = (t mod 2) * B/2, position q lies in block floor((q + o) / B).  A pair
 *      (i, j) is in-block when i and j+1 lie in the same block (so does every position it reads or writes);
 *      a block's best is the argmin of (delta, i, j) over its in-block generated improving pairs.
 *   3. The step applies G and every block best (i, j) other than G with j < i_G or i > j_G.  These share no
 *      edge with G or with one another, so their start-of-step deltas are their real deltas.
 *   4. They are logged G first, then by increasing i, each with its start-of-step delta.  stats.moves counts
 *      logged moves, stats.passes scans and stats.evals generated pairs, as in Mode N.
 *   5. max_moves >= 0: a step applies the first max_moves - moves of its moves in log order, and the search
 *      stops with converged = 0.  A budget of m gives the first m moves of the unbudgeted log; a later
 *      tl_session_run starts a new step with a fresh scan.
 * With n <= B/2 every pair is in-block at both offsets and the moves are Mode N's; at convergence Mode N's scan
 * finds no improving pair.  tl_session_scan and tl_session_time_scans scan for G as Mode N does.
 *
 * Or-opt NM: Or-opt N's generated moves, legality, deltas, threshold and (delta, s, i, j, reversed) order.  Step t
 * (t = the steps the session has applied so far) works on the tour as it stood at the start of the step:
 *   1. G = Or-opt N's move, the minimum over all generated legal moves below the threshold; none: converged
 *      (Or-opt N's stop).
 *   2. The hull of a move (i, s, j, reversed) is [a0, a1] with a0 = min(i-1, j), a1 = max(i+s, j+1).  A move wraps
 *      when it touches the closing edge: i = 0, i+s = n or j = n-1.  Every position its delta reads is in the hull,
 *      and so is every position its relocation writes (the relocated span is [a0+1, a1-1], and a1 gets a new
 *      entering edge); the cities at a0 and a1 do not move.
 *   3. With B = TL_OR_MULTI_BLOCK and o = (t mod 2) * B/2, position q lies in block floor((q + o) / B).  A move that
 *      does not wrap is in-block when a0 and a1 lie in the same block; a block's best is the minimum, in Or-opt N's
 *      order, over its in-block generated legal moves below the threshold.
 *   4. If G wraps, the step applies G alone.  Otherwise it applies G and every block best with a1 <= g0 or a0 >= g1,
 *      [g0, g1] being G's hull.  Hulls of different blocks are disjoint, and a block best shares at most an end
 *      position with G, which keeps its city and whose entering edge only one of the two rewrites: every
 *      start-of-step delta is the move's real delta, and applying the moves one after another in log order gives
 *      the same tour.
 *   5. They are logged G first, then by increasing block (so by increasing i), each with its start-of-step delta.
 *      stats.moves counts logged moves, stats.passes scans and stats.evals generated legal moves, as in Or-opt N.
 *   6. max_moves >= 0: as in Mode NM, a step applies the first max_moves - moves of its moves in log order and the
 *      search stops with converged = 0; a later tl_session_run starts a new step with a fresh scan.
 * With n <= B/2 every move that does not wrap is in-block at both offsets, so the moves are Or-opt N's (and, with
 * k >= n-1, TL_ALGO_OR_OPT's).  tl_session_scan and tl_session_time_scans scan for G as Or-opt N does.  Or-opt NM
 * needs B <= 16384: the TL_MULTI_BLOCK environment variable, which also sets its block size, must then be a power of
 * two in 2..16384 (TL_ERR_INVALID otherwise).
 *
 * 1 <= k <= 32 (TL_ERR_INVALID otherwise); EXPLICIT problems: TL_ERR_UNSUPPORTED.  A session copies
 * the lists when it is created, so later calls do not affect it.  Without a call, the first session
 * of any of these algorithms builds TL_CANDIDATES_DEFAULT lists.  Memory is O(n k): nothing n^2 is allocated. */
#define TL_CANDIDATES_DEFAULT 8
tl_status tl_problem_set_candidates(tl_problem *p, uint32_t k);

/* nearest_neighbor::solve (nearest_neighbor.rs:22-70), start at position 0. */
tl_status tl_nn_tour(tl_problem *p, uint32_t k, uint32_t *tour_out);

/* greedy_edge::solve (src/tsp/greedy_edge.rs): the greedy-edge tour over ALL n(n-1)/2 edges, built on the
 * device from the candidate lists (kernel K9).  Edge (a, b) with a < b (positions) has the key (d(a, b), a, b),
 * d in the problem's metric as tl_knn compares it (f32; NINT_I32 values are exact there), compared
 * lexicographically, so no two edges tie.  Taking the edges in key order, an edge is accepted when both
 * endpoints have degree < 2 and lie in different fragments; after n-1 accepted edges the two endpoints of the
 * Hamiltonian path are joined.  The result is this tour whatever the candidate lists are: k changes the speed
 * only.  tour_out[0] = 0, tour_out[1] = the lower-positioned of city 0's two tour neighbours, then the cycle
 * (n <= 3: the identity order).
 * Uses the problem's candidate lists; without any, builds TL_CANDIDATES_DEFAULT lists and keeps them with the
 * problem, as the first candidate-list session does.  Cities whose listed neighbours are all taken get lists
 * rebuilt over the cities still free.  EXPLICIT problems: TL_ERR_UNSUPPORTED.  Nothing n^2 is allocated.
 * stats (nullable): passes = device rounds, moves = accepted edges including the closing one, repermutes =
 * list rebuilds, launches, device_ms, converged = 1. */
tl_status tl_greedy_tour(tl_problem *p, uint32_t *tour_out, tl_stats *stats);

/* DistanceMatrix::tour_length_by_pos for a batch (distance_matrix.rs:235-245; GA
 * fitness genetic_algorithm.rs:112-124; ACO ant_colony.rs:138,221).  tours is
 * batch x n positions, row-major.  out_f32[b] (F32 problems) / out_i64[b] (NINT). */
tl_status tl_tour_lengths(tl_problem *p, const uint32_t *tours, size_t batch, int32_t mode,
                          float *out_f32);
tl_status tl_tour_lengths_i64(tl_problem *p, const uint32_t *tours, size_t batch, int64_t *out);

/* ---- local search, one call ------------------------------------------------------ */

/* Replaces the body of two_opt::solve (two_opt.rs:17-61) / or_opt::solve
 * (or_opt.rs:31-74) / three_opt::solve (three_opt.rs:24-52).  tour_inout: n positions, start tour in, local optimum out.
 * max_moves < 0: run to the local optimum.  log (nullable) receives the applied
 * moves in order, up to log_cap. */
tl_status tl_local_search(tl_problem *p, int32_t algo, int32_t path, uint32_t *tour_inout,
                          int64_t max_moves, tl_stats *stats, tl_move *log, size_t log_cap);

/* Independent local searches over a batch of start tours (multi-start / GA
 * population): tours_inout is batch x n.  lengths_out (nullable): exact-order length
 * of each result.  Only TL_ALGO_TWO_OPT_BEST[_CYCLIC] on coordinate problems. */
tl_status tl_two_opt_batch(tl_problem *p, int32_t algo, uint32_t *tours_inout, size_t batch,
                           int64_t max_moves, tl_stats *stats, float *lengths_out);

/* ---- Ant System (population solver, SURVEY.md section 8(f) row N4) ------------------------------- */

/* Replaces the body of ant_colony::solve (src/tsp/ant_colony.rs:92-239): roulette construction of
 * num_ants tours per epoch over tau^alpha * eta^beta, evaporate-and-floor, per-ant deposits,
 * incumbent update; tour costs are the exact-order sums of tl_tour_lengths.  The reference draws
 * from an unseeded RNG; here every draw is Philox4x32-10(seed; step, ant, epoch), so a run is
 * reproducible.  Option defaults and validation follow AcoOptions (src/tsp/mod.rs:1083-1153).
 * init_tour (nullable): as `init_tour` of the reference (seeds the incumbent, tau0 = num_ants/cost
 * and one deposit); null: a Philox-shuffled start and tau0 = 1.  Coordinate (F32_EXACT) and
 * EXPLICIT problems. */
typedef struct {
    float alpha;            /* >= 0, default 1                     */
    float beta;             /* in [0, 6], default 2                */
    float evaporation_rate; /* in (0, 1), default 0.5              */
    uint32_t num_ants;      /* >= 1, default 25                    */
    uint32_t epochs;        /* default 150                         */
    uint32_t pad;
    uint64_t seed;
} tl_aco_options;
tl_status tl_aco(tl_problem *p, const tl_aco_options *opts, const uint32_t *init_tour, uint32_t *best_tour_out,
                 float *best_cost_out, tl_stats *stats);

/* ---- Genetic algorithm (population solver, SURVEY.md section 8(f) row N4) ----------------------- */

/* Replaces the body of genetic_algorithm::solve / solve_ga (src/tsp/genetic_algorithm.rs:16-107): a
 * population of n tours; per epoch a stable sort by fitness, n_elite elites, n/2 - n_elite pairs of
 * roulette-selected parents, ordered crossover (:140-176), fitness 1/tour_length (exact-order sum, as
 * tl_tour_lengths) taken before the optional reversal mutation; returns best() (:264-269) and its
 * exact-order length.  Every random draw is Philox4x32-10(seed; ...), so a run is reproducible.
 * Option defaults and validation follow GAOptions (src/tsp/mod.rs:816-846).  init_tour (nullable):
 * seeds max(n/5, 1) individuals (the tour itself and 2..=4-times mutated copies, :207-222), the rest
 * are shuffles.  Coordinate (F32_EXACT) and EXPLICIT problems; n up to what one CTA's shared memory
 * holds (about 7000 cities), TL_ERR_UNSUPPORTED beyond. */
typedef struct {
    float mutation_probability; /* in [0, 1], default 0.001 */
    uint32_t n_elite;           /* default 3                */
    uint32_t epochs;            /* default 10000            */
    uint32_t pad;
    uint64_t seed;
} tl_ga_options;
tl_status tl_ga(tl_problem *p, const tl_ga_options *opts, const uint32_t *init_tour, uint32_t *best_tour_out,
                float *best_cost_out, tl_stats *stats);

/* ---- local search, device-resident session (benchmarks, pipelines) ---------------- */

tl_status tl_session_create(tl_problem *p, int32_t algo, int32_t path, const uint32_t *tour,
                            tl_session **out);
void tl_session_destroy(tl_session *s);
/* Shard the move space: this session scans shard `index` of `count` and exchanges per-rank
 * bests with the other ranks after every scan (see tl_ctx_attach_nccl).  Every rank must
 * call it with its own rank and the world size, create/step its sharded sessions in the same
 * order, and step ONE sharded session at a time per context. */
tl_status tl_session_set_shard(tl_session *s, int32_t index, int32_t count);
/* One full scan without applying: the best move (found=0 when none improves). */
tl_status tl_session_scan(tl_session *s, tl_move *best, int32_t *found);
/* Launch the scan kernel `reps` times back to back (no apply, no cross-rank exchange) between
 * two CUDA events on the context's stream and return the average launch duration: the roofline
 * numerator.  A sharded session times its own share of the move space. */
tl_status tl_session_time_scans(tl_session *s, uint32_t reps, double *avg_ms);
/* Enqueue `steps` scan+apply iterations; does not synchronise. */
tl_status tl_session_enqueue(tl_session *s, uint32_t steps);
/* Run until the local optimum or max_moves, then synchronise. */
tl_status tl_session_run(tl_session *s, int64_t max_moves);
/* Synchronise and read back the current tour / statistics / move log. */
tl_status tl_session_tour(tl_session *s, uint32_t *tour_out);
tl_status tl_session_stats(tl_session *s, tl_stats *stats);
tl_status tl_session_log(tl_session *s, tl_move *log, size_t log_cap, size_t *n_out);

/* ---- diagnostics ------------------------------------------------------------------ */

/* Exhaustively compares the library's guarded fast sqrt with IEEE sqrt.rn over
 * every f32 bit pattern in [lo_bits, hi_bits]; returns the mismatch count. */
tl_status tl_selftest_sqrt(tl_ctx *ctx, uint32_t lo_bits, uint32_t hi_bits, uint64_t *mismatches);
/* FP32 issue microbenchmark for the recompute-path roofline: dependent-free FFMA
 * stream; returns lane-instructions per second. */
tl_status tl_microbench_fp32(tl_ctx *ctx, double *ffma_per_s, double *mufu_per_s);

#ifdef __cplusplus
}
#endif
#endif
