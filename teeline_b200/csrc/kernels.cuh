// kernels.cuh -- kernel-side types and host launcher prototypes (internal).
#pragma once
#include <optional>
#include <vector>

#include "common.cuh"
#include "shard_exchange.cuh"
#include "../../include/teeline_cuda.h"

namespace tl {

// ---------------------------------------------------------------------------
// 2-opt scan geometry (host-computed, passed by value)
// ---------------------------------------------------------------------------
// The (i,j) triangle is cut into BANDS of BW = 32*R consecutive diagonals
// k = j - i (k starts at 2, so no triangular mask is ever needed).  Band b has
// rows i = 0 .. jmax - K0_b.  Each band is cut into work items of `chunk` rows;
// a warp normally processes exactly one item (the host sizes `chunk` for that), in
// (i ascending, j ascending) order = the reference's order; when it has to take
// several, the (delta, i, j) comparison in the kernels' slow path keeps the argmin
// exact.  Items are numbered band major: item = first[b] + c for band b, row chunk c
// (row-chunk major was measured and is slower: profiles/r01g_probe.txt).
struct ScanGeom {
    int32_t n;
    int32_t jmax;       // n-2 (reference neighbourhood) or n-1 (cyclic)
    int32_t kmax;       // n-2
    int32_t nbands;
    int32_t chunk;      // rows per work item
    int32_t item_begin; // this launch scans items [item_begin, item_end)
    int32_t item_end;
    int32_t cyclic;
    float screen_margin; // recompute path: Dmax * kScreenMarginScale, < 0 disables screening
    // matrix path: warp w first scans the `run` consecutive items starting at item_begin + w * run
    // (clipped to dyn_begin); the items [dyn_begin, item_end) are handed out one at a time through
    // an atomic ticket to whichever warp finishes first (evens out the tail of the scan)
    int32_t run;
    int32_t dyn_begin;
};

// device-resident loop state, updated by the apply kernels
struct DevState {
    unsigned long long moves;
    unsigned long long scans;
    long long max_moves; // < 0: unlimited
    int32_t done;        // 1: converged or max_moves reached -> later launches are no-ops
    int32_t converged;
    // Mode R cursor
    int32_t cur_i, cur_j;
    int32_t improved_in_pass;
    int32_t window_rows;
    unsigned long long passes;
    unsigned long long found_key; // Mode R: (i << 32 | j) of the first improving pair, ~0 if none
    float last_delta;
    int32_t error; // 1: a sharded step timed out waiting for a peer's record (shard_exchange.cuh)
    unsigned long long computed; // cached Mode B (k2_two_opt_cached.cu): pairs whose delta was computed
};

// cached Mode B: what the next step has to re-evaluate (written by the previous step's tail)
struct CachedDesc {
    int32_t nfull;      // rows to rescan from scratch, listed in `fullrows`; -1: every row
    int32_t I, J;       // the move just applied: columns I .. J of the rows above changed
    int32_t npart_rows; // rows 0 .. npart_rows-1 re-evaluate those columns only
    int32_t active;     // CTAs of the launch that take part in the step
};


// Where a launch gets its distances from (selects the Policy instantiation, policy.cuh).
enum SrcKind { SRC_EUC_FAST = 0, SRC_EUC_SAFE = 1, SRC_MAT_F32 = 2, SRC_MAT_I32 = 3 };
struct Src {
    int kind = SRC_EUC_FAST;
    Pt *pts = nullptr;       // SRC_EUC_*
    Cs *cs = nullptr;        // SRC_MAT_*
    const void *M = nullptr; // slot-ordered n x ld matrix (f32 or i32)
    uint32_t ld = 0;
    bool is_int() const { return kind == SRC_MAT_I32; }
    void *records() const { return kind <= SRC_EUC_SAFE ? (void *)pts : (void *)cs; }
};
#define TL_DISPATCH_POL(src, ...)                                                             \
    switch ((src).kind) {                                                                     \
    case SRC_EUC_FAST: { EucPol<true> P{(src).pts}; __VA_ARGS__; } break;                      \
    case SRC_EUC_SAFE: { EucPol<false> P{(src).pts}; __VA_ARGS__; } break;                     \
    case SRC_MAT_F32: { MatPol<float> P{(src).cs, (const float *)(src).M, (src).ld}; __VA_ARGS__; } break; \
    default: { MatPol<int32_t> P{(src).cs, (const int32_t *)(src).M, (src).ld}; __VA_ARGS__; } break;      \
    }

// ---------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------
// Launch configuration with programmatic dependent launch (common.cuh: griddep_wait) in attr[0].  A
// caller that needs more attributes sets attr[1..] and raises numAttrs.
inline cudaLaunchConfig_t pdl_config(int grid, int threads, size_t smem, cudaLaunchAttribute *attr, cudaStream_t st)
{
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cfg;
}

void launch_k1_packed(const float2 *xy, uint32_t n, Metric metric, void *out, int sm_count, cudaStream_t st);
void launch_k1_square(const float2 *sxy, uint32_t n, uint32_t ld, Metric metric, void *out, cudaStream_t st);
void launch_k1_square_from_packed(const uint32_t *tri, const int32_t *slot_city, uint32_t n,
                                  uint32_t ld, uint32_t *out, cudaStream_t st);

// opt-in dynamic shared memory sizes for every kernel that needs > 48 KB
cudaError_t configure_all_kernels();

// K2 recompute path
#ifndef TL_SCAN_R
#define TL_SCAN_R 7
#endif
#ifndef TL_SCAN_TI
#define TL_SCAN_TI 128
#endif
#ifndef TL_SCAN_MINB
#define TL_SCAN_MINB 3
#endif
constexpr int kScanR = TL_SCAN_R;       // diagonals per lane (odd => conflict-free 128-bit LDS)
constexpr int kScanBW = 32 * kScanR;    // diagonals per band
constexpr int kScanTI = TL_SCAN_TI;     // max rows per staged tile
constexpr int kScanWarps = 8;           // warps per CTA
constexpr int kScanMinBlocks = TL_SCAN_MINB; // resident CTAs per SM the kernel is compiled for
size_t scan_recompute_smem_bytes();
cudaError_t scan_recompute_configure();
// fuse_apply: the last CTA reduces the per-CTA records and applies the move; with `shard` non-null it
// first exchanges this rank's record with every peer over NVLink (shard_exchange.cuh)
void launch_scan_recompute(Pt *pts, const ScanGeom &g, const int32_t *band_first, BestF *blockbest,
                           DevState *state, unsigned int *ticket, tl_move *log, uint64_t log_cap,
                           bool fuse_apply, const ShardComm *shard, int grid, bool fast, cudaStream_t st);
void launch_build_pts(const float2 *xy, const uint32_t *tour, uint32_t n, uint32_t npad, int cyclic,
                      bool fast, Pt *pts, cudaStream_t st);
void launch_apply_two_opt(const Src &src, const void *cand, int ncand, DevState *state, unsigned int *ticket,
                          tl_move *log, uint64_t log_cap, int grid, cudaStream_t st);
void launch_extract_tour(const Src &src, uint32_t n, uint32_t *tour, cudaStream_t st);

// K2 Mode R (reference-exact first improvement)
constexpr int kRefWindow0 = 8; // rows scanned per launch right after a hit
void launch_ref_step(const Src &src, uint32_t n, DevState *state, unsigned int *ticket, tl_move *log,
                     uint64_t log_cap, int grid, cudaStream_t st);
// persistent form: one thread-block cluster runs up to max_steps cursor steps from shared memory.
// f32 coordinate sessions, and nint matrix sessions of coordinate problems (xy = city-ordered
// coordinates: the entries are recomputed in the problem's metric, bit-equal to K1's).  metric: the
// session's metric, none for sessions that read f32 matrix entries (f32 matrix, EXPLICIT)
constexpr int kRefPersistMaxN = 14000;    // 16 bytes per position of the whole tour in one SM's shared memory
constexpr int kRefPersistMaxNInt = 11000; // 20 bytes per position (the matrix slot travels with the city)
int ref_persistent_cluster_size(std::optional<Metric> metric, uint32_t n);
void launch_ref_persistent(const Src &src, const float2 *xy, Metric metric, uint32_t n, DevState *state, tl_move *log,
                           uint64_t log_cap, uint32_t max_steps, int csize, float screen_margin, cudaStream_t st);

// K3 Or-opt (recompute path)
constexpr int kOrR = 8;          // columns per lane
constexpr int kOrTI = 96;        // max rows per staged tile
constexpr int kOrWarps = 8;
constexpr int kOrMinBlocks = 2;
size_t or_scan_smem_bytes();
cudaError_t or_scan_configure();
void launch_or_rowinfo(const Src &src, uint32_t n, uint32_t npad, void *info, const DevState *state,
                       unsigned int *work_ticket, cudaStream_t st);
// Order in which the Or-opt scan hands out its work items (column block cb x row chunk c, index
// cb * items_per_cb + c).  The tiles that touch the diagonal run the masked step and cost ~4x the
// others; taken late they ARE the tail of the scan (per-warp timeline: warps end between 114 and
// 223 us, mean 145), so the queue serves them first: in every column block the `near` chunks
// [near_first(cb), near_first(cb) + near) count as "near".  A rank that owns the items [begin, end)
// of the plain order takes ticket t < near_count as the (near_begin + t)-th near item of the whole
// instance and any later ticket as the (far_begin + t - near_count)-th other item -- a bijection
// onto [begin, end), so which items a rank scans does not change, only their order.  (One more
// masked tile is not "near": rows 0.. against the LAST column block, where j = n-1 is the position
// before i = 0.  An unsharded scan walks the other items from the last column block down so that
// this tile comes right after the near ones instead of at the very end.)
struct OrOrder {
    int chunk, items_per_cb, near; // rows per item; items per column block; near chunks per block
    int total;                     // items of this rank
    int near_begin, near_count, far_begin;
    int far_reversed_ncb; // > 0: unsharded scan over this many column blocks, far items taken last block first
    __host__ __device__ int near_first(int cb) const
    {
        const int j0 = cb * 32 * kOrR;
        const int a = j0 < 3 ? 0 : (j0 - 3) / chunk;
        return a < items_per_cb - near ? a : items_per_cb - near;
    }
    __host__ __device__ int near_before(int item) const // near items among the plain-order items [0, item)
    {
        const int cb = item / items_per_cb, c = item - cb * items_per_cb - near_first(cb);
        return cb * near + (c < 0 ? 0 : (c > near ? near : c));
    }
    __host__ __device__ void item_of_ticket(int t, int &cb, int &c) const
    {
        if (t < near_count) {
            const int q = near_begin + t;
            cb = q / near;
            c = near_first(cb) + (q - cb * near);
        } else {
            const int far = items_per_cb - near, q = far_begin + (t - near_count);
            cb = q / far;
            const int cc = q - cb * far;
            if (far_reversed_ncb > 0) cb = far_reversed_ncb - 1 - cb;
            c = cc < near_first(cb) ? cc : cc + near;
        }
    }
};
void launch_or_scan(const Src &src, const void *info, uint32_t n, const OrOrder &order, void *blockbest,
                    const DevState *state, unsigned int *work_ticket, int grid, cudaStream_t st);
void launch_or_apply(const Src &src, void *tmp, uint32_t n, const void *cand, int ncand, DevState *state,
                     unsigned int *ticket, tl_move *log, uint64_t log_cap, int grid, cudaStream_t st);

// K6 3-opt (three_opt.rs): row_first[i] = work items before row i (an item = row i x 32 values of j)
constexpr int kThreeWarps = 8;
constexpr int kThreeMinBlocks = 4;
void launch_three_scan(const Src &src, uint32_t n, const int32_t *row_first, int item_begin, int item_end,
                       void *blockbest, const DevState *state, unsigned int *work_ticket, int grid, cudaStream_t st);
void launch_three_apply(const Src &src, void *tmp, uint32_t n, const void *cand, int ncand, DevState *state,
                        unsigned int *ticket, tl_move *log, uint64_t log_cap, int grid, cudaStream_t st);

// K5 / N1
// tri non-null (EXPLICIT problems): distances from the packed triangle, else recomputed in `metric`
void launch_knn(const float2 *xy, const float *tri, uint32_t n, uint32_t k, Metric metric, uint32_t *out,
                cudaStream_t st);
size_t nn_tour_smem_bytes(uint32_t n);
cudaError_t nn_tour_configure();
void launch_nn_tour(const float2 *xy, const float *tri, uint32_t n, const uint32_t *knn, uint32_t kk,
                    Metric metric, uint32_t *tour, cudaStream_t st);

// K9 greedy edge (k9_greedy.cu): a round is the best kernel and the accept kernel; the accept kernel's last
// block ends the round in `status`, and later rounds of an enqueued batch return at once until the host acts
enum : uint32_t { kGreedyRun = 0, kGreedyStalled = 1, kGreedyDone = 2 };
struct GreedyState {
    uint32_t status;    // kGreedyRun; kGreedyStalled: the last round accepted nothing; kGreedyDone: two free cities
    uint32_t free;      // cities of degree < 2
    uint32_t round_acc; // edges accepted by the running round
    uint32_t ticket;
    unsigned long long rounds, accepted;
};
struct GreedyBufs {
    uint8_t *deg;
    uint32_t *adj;   // 2n: the two tour neighbours of every city
    uint32_t *other; // far endpoint of a free city's fragment
    float *bd;       // per free city: key distance of its best edge or bound
    uint32_t *bv;    // its partner, | kExhausted for a bound, UINT32_MAX for none
    uint32_t *oth;   // other[] as the best kernel saw it
    GreedyState *state;
};
constexpr uint32_t kGreedyRefreshK = 16; // width of the lists rebuilt over the free cities (>= 2)
void launch_greedy_init(uint32_t n, uint8_t *deg, uint32_t *other, GreedyState *gs, cudaStream_t st);
void launch_greedy_round(const float2 *xy, uint32_t n, Metric metric, const uint32_t *list, uint32_t k, GreedyBufs b,
                         int grid, cudaStream_t st);
size_t greedy_refresh_blocks(uint32_t n);
// the free cities' coordinates and positions in position order (3 launches); blockcnt: greedy_refresh_blocks(n)
void launch_greedy_compact(const float2 *xy, uint32_t n, const uint8_t *deg, uint32_t *blockcnt, float2 *cxy,
                           uint32_t *cidx, cudaStream_t st);
void launch_greedy_map(uint32_t F, uint32_t k, const uint32_t *cidx, const uint32_t *cknn, uint32_t *list, cudaStream_t st);
// closes the path and writes the tour; succ and dist hold 4n entries each.  Returns the launch count.
int launch_greedy_emit(uint32_t n, const uint8_t *deg, const uint32_t *other, uint32_t *adj, uint32_t *succ,
                       uint32_t *dist, uint32_t *tour, cudaStream_t st);

// K2 matrix path
constexpr int kMatR = 8;                 // diagonals per lane (strided by 32 => coalesced rows)
constexpr int kMatBW = 32 * kMatR;
constexpr int kMatTI = 64;
constexpr int kMatWarps = 8;
#ifndef TL_MAT_MINB
#define TL_MAT_MINB 3
#endif
constexpr int kMatMinBlocks = TL_MAT_MINB;
#ifndef TL_MAT_D
#define TL_MAT_D 4
#endif
constexpr int kMatD = TL_MAT_D;          // prefetch depth in row steps
constexpr int kMatPrefetchRows = 16;      // rows per warp prefetched into L2 before the grid dependency resolves
size_t scan_matrix_smem_bytes();
cudaError_t scan_matrix_configure();
#ifndef TL_MAT_PIN_MB
#define TL_MAT_PIN_MB 0
#endif
constexpr double kMatPinMB = TL_MAT_PIN_MB; // default size of the L2-resident part (0 = off until measured)
// L2 residency of a matrix larger than L2 (k2_two_opt_matrix.cu): either per-load eviction
// hints on the rows with slot < hint_rows, or a driver access-policy window over the first
// window_bytes of M (needs the persisting-L2 carve-out, session.cu); both 0 = plain streaming.
struct MatPin {
    int hint_rows = 0;
    size_t window_bytes = 0;
    float window_hit_ratio = 1.0f;
};
void launch_scan_matrix(const Src &src, const ScanGeom &g, const int32_t *band_first, void *blockbest,
                        DevState *state, unsigned int *ticket, tl_move *log, uint64_t log_cap, bool fuse_apply,
                        const ShardComm *shard, int grid, const MatPin &pin, cudaStream_t st);
// cs[q] = {slot = q, sp = M[q-1][q], city = tour[q]} (+ wrap copy at n when cyclic, -inf padding)
void launch_build_cs(const Src &src, const uint32_t *tour, uint32_t n, uint32_t npad, int cyclic, cudaStream_t st);
// slot-ordered scratch for (re)building the matrix in tour order: from `tour` (session start)
// or from the current records (re-permutation); also resets slot = position
void launch_gather_slots(const float2 *xy, const uint32_t *tour, const Cs *cs, uint32_t n, float2 *sxy,
                         int32_t *slot_city, cudaStream_t st);
void launch_reset_slots(const Src &src, uint32_t n, uint32_t npad, int cyclic, cudaStream_t st);

// K2 cached Mode B (k2_two_opt_cached.cu): one step = re-evaluate what the last move changed, reduce the
// row keys, apply
void launch_two_opt_cached_step(const Src &src, uint32_t n, int cyclic, unsigned long long *rowkey, CachedDesc *desc,
                                int *fullrows, DevState *state, unsigned int *ticket, tl_move *log, uint64_t log_cap,
                                int grid, cudaStream_t st);

// K2 candidate-list 2-opt, "Mode N" (k2_two_opt_neighbor.cu): distances recomputed in the problem's
// metric.  blockbest holds grid + 1 records: one per CTA and, at [grid], the step's pending long move
// for the apply grid (Mode N only).
constexpr int kNlThreads = 256;
constexpr int kNlMinBlocks = 2;
constexpr int kNlCtaSwaps = 2048; // segments of up to this many swapped pairs are reversed by the reducing CTA
// cyclic: Or-opt N's records (position 0 carries the closing edge, position n is the wrap copy)
void launch_nl_init(Metric metric, const float2 *xy, const uint32_t *tour, uint32_t n, uint32_t npad, bool cyclic,
                    Pt *pts, uint32_t *pos, cudaStream_t st);
// Multi-move candidate-list 2-opt, "Mode NM" (same file): Mode N's scan, plus one 64-bit key per block of
// 2^bshift positions (order-preserving delta bits << 32 | in-block offsets of i and j), re-armed to ~0 by
// the step's last CTA.  That CTA lists the accepted block moves (i, j) in `list` and leaves
// desc = {block moves to apply, pending long G's i, its j} (i = ~0: none) for the apply grid, which resets it.
// Multi-move Or-opt N, "Or-opt NM" (k3_or_opt_neighbor.cu), keeps the same buffers: its keys hold (s, i, j, rev)
// below the delta bits, `list` holds the accepted moves as Or-opt records (Best<V>) and
// desc = {block moves to apply, pending long G's i, j, aux}.
struct NlMulti {
    unsigned long long *keys; // nslots = ceil(n / 2^bshift) + 1
    void *list;               // nslots entries: uint2 (Mode NM) or 16-byte Or-opt records (Or-opt NM)
    uint32_t *desc;           // 4
    uint32_t bshift, nslots;
};
// multi (nullable): a fused scan also keeps Mode NM's block bests and ends the step as Mode NM
void launch_nl_scan(Metric metric, Pt *pts, uint32_t *pos, const uint32_t *cand, uint32_t k, uint32_t n, void *blockbest,
                    DevState *state, unsigned int *ticket, tl_move *log, uint64_t log_cap, bool fuse_apply, int grid,
                    cudaStream_t st, const NlMulti *multi = nullptr);
void launch_nl_apply(Metric metric, Pt *pts, uint32_t *pos, const void *pending, DevState *state, unsigned int *ticket,
                     tl_move *log, uint64_t log_cap, int grid, cudaStream_t st);
// Mode NM's apply grid: a pending long G cooperatively, each listed block move by one CTA
void launch_nlm_apply(Metric metric, Pt *pts, uint32_t *pos, const NlMulti &multi, unsigned int *ticket, int grid,
                      cudaStream_t st);

// K3 candidate-list Or-opt, "Or-opt N" (k3_or_opt_neighbor.cu): Mode N's records (cyclic), pos[] and
// lists.  blockbest holds grid + 1 records as in Mode N, blockcnt the grid per-CTA candidate counts;
// tmp stages the relocated span (npad records).
constexpr int kOrNlCtaSpan = 4096; // relocated spans of up to this many positions are moved by the reducing CTA
// multi (nullable): a fused scan also keeps Or-opt NM's block bests and ends the step as Or-opt NM
void launch_or_nl_scan(Metric metric, Pt *pts, uint32_t *pos, const uint32_t *cand, uint32_t k, uint32_t n, void *tmp,
                       void *blockbest, unsigned long long *blockcnt, DevState *state, unsigned int *ticket, tl_move *log,
                       uint64_t log_cap, bool fuse_apply, int grid, cudaStream_t st, const NlMulti *multi = nullptr);
void launch_or_nl_apply(Metric metric, Pt *pts, uint32_t *pos, void *tmp, uint32_t n, const void *pending,
                        DevState *state, unsigned int *ticket, tl_move *log, uint64_t log_cap, int grid, cudaStream_t st);
// Or-opt NM's apply grids (same file): a pending long G cooperatively and each listed block move by one CTA, every
// move staged in tmp from its first relocated position on; the last CTA resets multi.desc
void launch_or_nlm_apply(Metric metric, Pt *pts, uint32_t *pos, void *tmp, uint32_t n, const NlMulti &multi,
                         unsigned int *ticket, int grid, cudaStream_t st);

// K6 candidate-list 3-opt, "3-opt N" (k6_three_opt_neighbor.cu): Or-opt N's records, pos[], lists,
// buffers and relocation routes; its records carry the savings, as K6's do.
void launch_three_nl_scan(Metric metric, Pt *pts, uint32_t *pos, const uint32_t *cand, uint32_t k, uint32_t n, void *tmp,
                          void *blockbest, unsigned long long *blockcnt, DevState *state, unsigned int *ticket,
                          tl_move *log, uint64_t log_cap, bool fuse_apply, int grid, cudaStream_t st);
void launch_three_nl_apply(Metric metric, Pt *pts, uint32_t *pos, void *tmp, uint32_t n, const void *pending,
                           DevState *state, unsigned int *ticket, tl_move *log, uint64_t log_cap, int grid,
                           cudaStream_t st);

// K2-batch: one CTA per tour, tour records in shared memory
constexpr int kBatchR = 5;              // diagonals per thread group (odd => conflict-free LDS.128)
constexpr int kBatchMaxSmem = 200 * 1024;
size_t two_opt_batch_smem_bytes(uint32_t n);
size_t two_opt_batch_counter_bytes();
cudaError_t two_opt_batch_configure();
// launch configuration (threads per tour x resident CTAs per SM) for a batch of this size
int two_opt_batch_config(uint32_t n, uint64_t batch, int sm_count);
int two_opt_batch_grid(int cfg, uint32_t n, uint64_t batch, int sm_count, bool fast, bool screen);
// counters: {u64 moves, u64 scans, u32 next_tour, u32 unconverged}, zeroed by the caller;
// screen_margin < 0 disables screening (common.cuh: kScreenMarginScale)
// work items of one scan (full-width row chunks + the bands' tails as quarter-warp pieces), host copy
std::vector<unsigned char> two_opt_batch_item_table(uint32_t n, int cyclic, int cfg, int cl, int *nitems);
void launch_two_opt_batch(int cfg, const float2 *xy, uint32_t *tours, uint32_t n, uint64_t batch, int cyclic,
                          long long max_moves, float screen_margin, const void *items, int nitems, void *counters,
                          int grid, bool fast, cudaStream_t st);

// cluster per tour (small batches): returns the cluster size (1 = use the CTA-per-tour kernel) and its configuration
int two_opt_batch_cluster_plan(uint32_t n, uint64_t batch, int sm_count, int *cfg_out);
cudaError_t launch_two_opt_batch_cluster(int cfg, int cl, const float2 *xy, uint32_t *tours, uint32_t n, uint64_t batch,
                                         int cyclic, long long max_moves, float screen_margin, const void *items,
                                         int nitems, void *counters, bool fast, cudaStream_t st);

// K2-pop: population 2-opt scheduled at work-item granularity over the whole GPU (k2_two_opt_pop.cu)
constexpr int kPopR = 5;        // diagonals per lane (odd => conflict-free LDS.128)
constexpr int kPopTI = 96;      // rows per work item (default; TL_POP_CHUNK overrides up to kPopMaxTI)
constexpr int kPopMaxTI = 128;  // two tiles per warp: 8 x 2 x (2*128 + 162) x 16 B = 107 KB per CTA
constexpr int kPopWarps = 8;
constexpr int kPopMinBlocks = 3;
constexpr int kPopBandCap = 512; // band table entries in shared memory (n <= 65535)
struct __align__(32) PopTourCtl {
    uint32_t ticket;          // (unused since the FIFO scheduler)
    uint32_t done;            // items of the current scan completed
    unsigned long long best;  // min over the scan of (order-preserving delta bits << 32 | i*n + j); ~0 = none
    uint32_t moves;           // moves applied to this tour
    uint32_t state;           // 0 active, 1 converged, 2 stopped by max_moves
    uint32_t pad[2];
};
struct PopCounters {
    unsigned long long moves, scans;
    uint32_t active, unconverged;
    unsigned long long head;  // work-item slots handed out (slot / items_per_scan = FIFO entry)
    unsigned long long tail;  // FIFO entries published
    uint32_t error, pad;      // 1: the ring wrapped past an unread entry
};
size_t two_opt_pop_smem_bytes(int chunk);
cudaError_t two_opt_pop_configure();
uint32_t two_opt_pop_npad(uint32_t n);
bool two_opt_pop_supported(uint32_t n);
uint32_t two_opt_pop_queue_cap(uint64_t batch);
void launch_pop_init(const float2 *xy, const uint32_t *tours, uint32_t n, uint32_t npad, uint64_t batch, int cyclic,
                     bool fast, Pt *recs, PopTourCtl *ctl, PopCounters *ctr, unsigned long long *queue, uint32_t qcap,
                     int sm_count, cudaStream_t st);
void launch_pop_extract(const Pt *recs, uint32_t n, uint32_t npad, uint64_t batch, uint32_t *tours, int sm_count,
                        cudaStream_t st);
void launch_two_opt_pop(Pt *recs, PopTourCtl *ctl, PopCounters *ctr, uint32_t n, uint32_t npad, uint64_t batch,
                        int cyclic, long long max_moves, float screen_margin, int chunk, int nbands, int nitems,
                        const int32_t *band_first, unsigned long long *queue, uint32_t qcap, bool fast, int sm_count,
                        cudaStream_t st);

// K7: Ant System (k7_aco.cu)
void aco_philox_host(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4]);
int aco_stream_shuffle();
void launch_aco_eta(const float2 *xy, const float *tri, uint32_t n, bool fast, float beta, float *eta, int sm_count,
                    cudaStream_t st);
void launch_aco_fill(float *p, size_t count, float v, int sm_count, cudaStream_t st);
void launch_aco_weights(const float *ph, const float *eta, size_t count, float alpha, float *w, int sm_count,
                        cudaStream_t st);
void launch_aco_evaporate(float *ph, size_t count, float keep, float tau_min, int sm_count, cudaStream_t st);
cudaError_t launch_aco_construct(const float *w, const float *eta, uint32_t n, uint32_t ants, uint32_t epoch,
                                 uint64_t seed, uint32_t *tours, cudaStream_t st);
void launch_aco_update(float *ph, uint32_t n, const uint32_t *tours, const float *costs, uint32_t ants,
                       uint32_t *best_tour, float *best_cost, unsigned long long *improvements, cudaStream_t st);

// K8: GA population step (k8_ga.cu)
size_t ga_breed_smem_bytes(uint32_t n, uint32_t L);
cudaError_t launch_ga_init(const float2 *xy, const float *tri, uint32_t n, bool fast, const uint32_t *init,
                           uint32_t n_seeded, uint64_t seed, uint32_t *pop, float *fit, cudaStream_t st);
cudaError_t launch_ga_rank(const float *fit, uint32_t L, int *order, float *sfit, cudaStream_t st);
cudaError_t launch_ga_breed(const float2 *xy, const float *tri, uint32_t n, bool fast, uint32_t L, uint32_t ne,
                            uint32_t pairs, uint32_t epoch, uint64_t seed, float mutation_probability,
                            const uint32_t *pop, const int *order, const float *sfit, uint32_t *nxt, float *nfit,
                            unsigned long long *mutations, cudaStream_t st);
void launch_ga_best(const uint32_t *pop, const float *fit, uint32_t n, uint32_t L, uint32_t *best, cudaStream_t st);

// K4
void launch_tour_lengths_f32(const float2 *xy, const float *tri, uint32_t n, const uint32_t *tours,
                             uint64_t batch, bool fast_sqrt, bool fast_mode, float *out, int sm_count,
                             cudaStream_t st);
void launch_tour_lengths_nint(const float2 *xy, uint32_t n, const uint32_t *tours, uint64_t batch,
                              long long *out, int sm_count, cudaStream_t st);

// diagnostics
void launch_selftest_sqrt(uint32_t lo, uint32_t hi, unsigned long long *mismatch, int sm_count,
                          cudaStream_t st);
void launch_microbench_ffma(float *sink, int iters, int grid, cudaStream_t st);
void launch_microbench_mufu(float *sink, int iters, int grid, cudaStream_t st);

} // namespace tl
