// session.cu -- device-resident local-search sessions and the one-call wrappers.
//
// A session keeps the tour on the device in tour order (16-byte records, updated in place
// by the apply kernels) and runs  scan -> [all-gather] -> apply  iterations without host round
// trips: the apply step decides convergence on the device and later launches become no-ops,
// so the host only synchronises once per batch of steps.
//
// Two distance sources (policy.cuh): coordinate recompute (Pt records) and the slot-ordered
// n x ld matrix in HBM (Cs records).  The matrix is laid out in tour order when the session
// starts and re-laid every `repermute_every` steps, which keeps the 2-opt scan's row reads
// contiguous as reversals fragment the tour.
#include "host.hpp"

#include <algorithm>
#include <chrono>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

using namespace tl;

namespace tl {

cudaError_t configure_all_kernels()
{
    cudaError_t e = scan_recompute_configure();
    if (e == cudaSuccess) e = nn_tour_configure();
    if (e == cudaSuccess) e = or_scan_configure();
    if (e == cudaSuccess) e = scan_matrix_configure();
    if (e == cudaSuccess) e = two_opt_batch_configure();
    if (e == cudaSuccess) e = two_opt_pop_configure();
    return e;
}

} // namespace tl

struct tl_session {
    tl_problem *p = nullptr;
    tl_ctx *c = nullptr;
    int algo = 0;
    int path_used = TL_PATH_RECOMPUTE;
    uint32_t n = 0;
    int cyclic = 0;
    bool trivial = false; // n < 4: nothing to scan

    uint32_t npad = 0;
    Src src;                 // which policy the kernels run with, and its device pointers
    DevBuf<Pt> pts;          // recompute path: tour-ordered point records
    DevBuf<Cs> cs;           // matrix path: tour-ordered (slot, edge, city) records
    DevBuf<uint32_t> M;      // matrix path: n x ld distances (f32 bits or int32), slot order
    uint32_t ld = 0;
    DevBuf<float2> sxy;          // scratch: slot-ordered coordinates for (re)building M
    DevBuf<int32_t> slot_city;   // scratch: slot -> city for EXPLICIT problems
    int repermute_every = 0;     // matrix path: re-lay M in tour order every this many steps (0 = never)
    uint32_t steps_since_permute = 0;
    uint64_t repermutes = 0;
    MatPin pin;                  // matrix path: L2 residency of part of a matrix larger than L2

    DevBuf<unsigned char> tmp;     // Or-opt, Or-opt N, 3-opt N: relocated range staging (npad records of 16 B)
    DevBuf<unsigned char> rowinfo; // Or-opt: per-row removal gains (npad x 16 B)
    DevBuf<unsigned int> or_ticket; // Or-opt: work queue of the scan kernel
    int or_chunk = 0, or_items_per_cb = 0, or_item_begin = 0, or_item_end = 0;
    OrOrder or_order{};

    ScanGeom geom{};
    DevBuf<int32_t> band_first;
    int nitems = 0;
    int grid = 1;
    int shard_index = 0, shard_count = 1;
    bool use_mailbox = false; // sharded 2-opt: per-rank minima exchanged inside the scan kernel (shard_exchange.cuh)
    ShardComm comm{};

    // cached Mode B (TL_ALGO_TWO_OPT_BEST_CACHED is run as TL_ALGO_TWO_OPT_BEST with `cached` set)
    bool cached = false;
    DevBuf<unsigned long long> rowkey; // per-row minimum: order-preserving delta bits << 32 | j
    DevBuf<CachedDesc> cdesc;
    DevBuf<int> fullrows;

    // candidate-list searches (TL_ALGO_TWO_OPT_NEIGHBOR, TL_ALGO_OR_OPT_NEIGHBOR, TL_ALGO_THREE_OPT_NEIGHBOR):
    // Pt records plus pos[] and the session's own copy of the problem's candidate lists
    bool nl = false;
    DevBuf<uint32_t> pos;            // city -> position
    DevBuf<uint32_t> nl_cand;        // n x nl_k
    uint32_t nl_k = 0;
    DevBuf<unsigned long long> nl_cnt; // Or-opt N, 3-opt N: per-CTA counts of evaluated candidates
    // Mode NM and Or-opt NM (TL_ALGO_TWO_OPT_NEIGHBOR_MULTI, TL_ALGO_OR_OPT_NEIGHBOR_MULTI): per-block keys, the
    // step's accepted block moves, apply descriptor
    DevBuf<unsigned long long> nlm_keys;
    DevBuf<uint4> nlm_list;
    DevBuf<uint32_t> nlm_desc;
    NlMulti nlm{};
    int nlm_grid = 1; // the apply grid: fixed per session, since steps are queued without reading back

    DevBuf<BestF> cand; // shard_count * grid records (BestF and BestI have the same layout)
    DevBuf<DevState> state;
    DevBuf<unsigned int> ticket;
    DevBuf<tl_move> log;
    uint64_t log_cap = 0;

    DevState h{};
    uint64_t pairs_per_scan = 0;
    uint64_t launches0 = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // tl_session_run: pinned snapshots of the device state, read back asynchronously so that the
    // next batches of steps are already queued while the host looks at an earlier one
    DevState *h_snap = nullptr;
    cudaEvent_t ev_snap[3] = {nullptr, nullptr, nullptr};
    bool timing_open = false;
    double device_ms = 0.0;

    bool matrix() const { return path_used == TL_PATH_MATRIX; }
    // the candidate-list searches that relocate a span of positions (cyclic records, staging buffer, counts)
    bool nl_relocating() const
    {
        return algo == TL_ALGO_OR_OPT_NEIGHBOR || algo == TL_ALGO_THREE_OPT_NEIGHBOR || algo == TL_ALGO_OR_OPT_NEIGHBOR_MULTI;
    }
    // the multi-move candidate-list searches (block keys, list and descriptor)
    bool nl_multi() const { return algo == TL_ALGO_TWO_OPT_NEIGHBOR_MULTI || algo == TL_ALGO_OR_OPT_NEIGHBOR_MULTI; }
    bool int_values() const { return metric_is_int(p->metric); }
    // the metric the persistent Mode R kernel recomputes distances in; none when the session reads f32
    // matrix entries (f32 matrix and EXPLICIT sessions)
    std::optional<Metric> recompute_metric() const
    {
        return src.kind == SRC_MAT_F32 ? std::nullopt : std::optional<Metric>(p->metric);
    }
};

namespace {

// Work decomposition of the 2-opt diagonal bands (see kernels.cuh: ScanGeom).
void build_geometry(tl_session *s, std::vector<int32_t> &band_first_h)
{
    const int bw = s->matrix() ? kMatBW : kScanBW;
    const int warps = s->matrix() ? kMatWarps : kScanWarps;
    const int minb = s->matrix() ? kMatMinBlocks : kScanMinBlocks;
    const int n = (int)s->n;
    ScanGeom &g = s->geom;
    g.n = n;
    g.cyclic = s->cyclic;
    g.jmax = s->cyclic ? n - 1 : n - 2;
    g.kmax = n - 2;
    g.screen_margin = screen_margin(s->p);
    g.nbands = (g.kmax - 2) / bw + 1;
    auto H = [&](int b) { return g.jmax - (2 + b * bw) + 1; };
    // one work item per resident warp, times the shard count so that every rank of a sharded
    // scan still fills its GPU
    const int64_t target = (int64_t)s->c->sm_count * minb * warps * s->shard_count;
    auto items_for = [&](int chunk) {
        int64_t t = 0;
        for (int b = 0; b < g.nbands; ++b) t += (H(b) + chunk - 1) / chunk;
        return t;
    };
    int lo = 8, hi = std::max(8, H(0)); // >= 8 rows per item amortises the tile set-up
    while (lo < hi) {
        const int mid = (lo + hi) / 2;
        if (items_for(mid) <= target)
            hi = mid;
        else
            lo = mid + 1;
    }
    g.chunk = lo;
    band_first_h.assign(g.nbands + 1, 0);
    for (int b = 0; b < g.nbands; ++b) band_first_h[b + 1] = band_first_h[b] + (H(b) + g.chunk - 1) / g.chunk;
    s->nitems = band_first_h[g.nbands];
    const int64_t per = ((int64_t)s->nitems + s->shard_count - 1) / s->shard_count;
    g.item_begin = (int32_t)std::min<int64_t>(s->nitems, per * s->shard_index);
    g.item_end = (int32_t)std::min<int64_t>(s->nitems, per * (s->shard_index + 1));
    // matrix path: one static item per warp.  (Tried: cutting a warp's share into ~7 items and
    // handing the last 15-40 % out through an atomic ticket to even out the 28-36 us spread of the
    // CTAs' finishing times -- every short item restarts the load pipeline with two dependent
    // round trips, and the scan got 5 us SLOWER; profiles/r01t_probe_dynamic_tail.txt.)
    g.run = 1; // set below once the grid is known
    g.dyn_begin = g.item_end;
    // same grid on every rank so the all-gather is symmetric
    const int64_t blocks = (per + warps - 1) / warps;
    s->grid = (int)std::max<int64_t>(1, std::min<int64_t>(blocks, (int64_t)s->c->sm_count * minb));
    // test hook: a small grid makes every warp walk several work items
    if (const char *cap = getenv("TL_MAX_GRID")) s->grid = std::max(1, std::min(s->grid, atoi(cap)));
    g.run = (int32_t)std::max<int64_t>(1, (per + (int64_t)s->grid * warps - 1) / ((int64_t)s->grid * warps));
}

// Or-opt work decomposition: column blocks of 32*kOrR insertion edges x row chunks.
void build_or_geometry(tl_session *s)
{
    const int n = (int)s->n;
    const int cw = 32 * kOrR;
    const int ncb = (n + cw - 1) / cw;
    // ~3 items per resident warp (times the shard count): the scan kernel hands them out dynamically
    // (2 leaves a long tail; 4, 6, 8 and 12 are slower: every item re-stages its columns and restarts
    // the distance pipeline -- profiles/r01zx_or_items.txt)
    int per_warp = 3;
    if (const char *ev = getenv("TL_OR_ITEMS_PER_WARP")) per_warp = std::max(1, atoi(ev));
    const int64_t target = (int64_t)s->c->sm_count * kOrMinBlocks * kOrWarps * s->shard_count * per_warp;
    const int per_cb = (int)std::max<int64_t>(1, target / ncb);
    s->or_chunk = std::max(16, (n + per_cb - 1) / per_cb);
    s->or_items_per_cb = (n + s->or_chunk - 1) / s->or_chunk;
    s->nitems = ncb * s->or_items_per_cb; // <= ~(n/256) * max(n/16, target/ncb): fits int32 for every n that fits HBM
    const int64_t per = ((int64_t)s->nitems + s->shard_count - 1) / s->shard_count;
    s->or_item_begin = (int)std::min<int64_t>(s->nitems, per * s->shard_index);
    s->or_item_end = (int)std::min<int64_t>(s->nitems, per * (s->shard_index + 1));
    const int64_t blocks = (per + kOrWarps - 1) / kOrWarps;
    s->grid = (int)std::max<int64_t>(1, std::min<int64_t>(blocks, (int64_t)s->c->sm_count * kOrMinBlocks));
    // diagonal tiles first (kernels.cuh: OrOrder)
    OrOrder &o = s->or_order;
    o.chunk = s->or_chunk;
    o.items_per_cb = s->or_items_per_cb;
    o.near = std::min(o.items_per_cb, (cw + 3 + o.chunk - 1) / o.chunk + 2);
    if (getenv("TL_OR_PLAIN_ORDER")) o.near = o.items_per_cb; // every chunk "near": the plain cb-major order
    o.total = s->or_item_end - s->or_item_begin;
    o.near_begin = o.near_before(s->or_item_begin);
    o.near_count = (s->or_item_end >= s->nitems ? ncb * o.near : o.near_before(s->or_item_end)) - o.near_begin;
    o.far_begin = s->or_item_begin - o.near_begin;
    o.far_reversed_ncb = s->shard_count == 1 ? ncb : 0;
}

// 3-opt work decomposition: an item is row i x 32 consecutive j; row_first[i] = items before row i.
tl_status upload_three_geometry(tl_session *s)
{
    const int n = (int)s->n;
    // ~n^2/64 work items: the table is int32, so refuse instances whose count would not fit
    int64_t total_items = 0;
    for (int i = 0; i + 2 < n; ++i) total_items += (n - 2 - i + 31) / 32;
    if (total_items > INT32_MAX) {
        set_error("3-opt on n = %d needs %lld work items (> 2^31): not supported", n, (long long)total_items);
        return TL_ERR_UNSUPPORTED;
    }
    std::vector<int32_t> rf(n - 1, 0); // rows i = 0 .. n-3, plus the total
    for (int i = 0; i + 2 < n; ++i) rf[i + 1] = rf[i] + (n - 2 - i + 31) / 32;
    s->nitems = rf[n - 2];
    const int64_t per = ((int64_t)s->nitems + s->shard_count - 1) / s->shard_count;
    s->or_item_begin = (int)std::min<int64_t>(s->nitems, per * s->shard_index);
    s->or_item_end = (int)std::min<int64_t>(s->nitems, per * (s->shard_index + 1));
    const int64_t blocks = (per + kThreeWarps - 1) / kThreeWarps;
    s->grid = (int)std::max<int64_t>(1, std::min<int64_t>(blocks, (int64_t)s->c->sm_count * kThreeMinBlocks));
    TL_CUDA_TRY(s->band_first.alloc(rf.size()));
    TL_CUDA_TRY(cudaMemcpyAsync(s->band_first.p, rf.data(), rf.size() * 4, cudaMemcpyHostToDevice, s->c->stream));
    TL_CUDA_TRY(s->cand.alloc((size_t)s->grid * s->shard_count));
    TL_CUDA_TRY(cudaStreamSynchronize(s->c->stream)); // rf is a local
    return TL_OK;
}

tl_status upload_geometry(tl_session *s)
{
    if (s->algo == TL_ALGO_THREE_OPT) return upload_three_geometry(s);
    if (s->nl) {
        // resident CTAs walk the n*k (position, slot) items; one record per CTA plus the pending move
        const int64_t blocks = ceil_div64((int64_t)s->n * s->nl_k, kNlThreads);
        s->grid = (int)std::max<int64_t>(1, std::min<int64_t>(blocks, (int64_t)s->c->sm_count * kNlMinBlocks));
        if (const char *cap = getenv("TL_MAX_GRID")) s->grid = std::max(1, std::min(s->grid, atoi(cap)));
        TL_CUDA_TRY(s->cand.alloc((size_t)s->grid + 1));
        TL_CUDA_TRY(cudaMemsetAsync(s->cand.p, 0xff, ((size_t)s->grid + 1) * sizeof(BestF), s->c->stream)); // no move pending
        if (s->nl_relocating()) TL_CUDA_TRY(s->nl_cnt.alloc((size_t)s->grid));
        if (s->nl_multi()) {
            NlMulti &m = s->nlm;
            m.nslots = (uint32_t)((s->n + (1u << m.bshift) - 1) >> m.bshift) + 1;
            TL_CUDA_TRY(s->nlm_keys.alloc(m.nslots));
            TL_CUDA_TRY(s->nlm_list.alloc(m.nslots));
            TL_CUDA_TRY(s->nlm_desc.alloc(4));
            TL_CUDA_TRY(cudaMemsetAsync(s->nlm_keys.p, 0xff, (size_t)m.nslots * 8, s->c->stream)); // no key
            TL_CUDA_TRY(cudaMemsetAsync(s->nlm_desc.p, 0xff, 16, s->c->stream));
            TL_CUDA_TRY(cudaMemsetAsync(s->nlm_desc.p, 0, 4, s->c->stream)); // nothing to apply
            m.keys = s->nlm_keys.p;
            m.list = s->nlm_list.p;
            m.desc = s->nlm_desc.p;
            // one CTA per block move (up to two per SM), at least Mode N's (Or-opt N's) apply grid for a long G
            const uint32_t half_pairs = (s->n / 2 + 255) / 256;
            s->nlm_grid = (int)std::max<uint32_t>(std::min<uint32_t>(half_pairs, (uint32_t)s->c->sm_count),
                                                  std::min<uint32_t>(m.nslots, 2u * (uint32_t)s->c->sm_count));
            s->nlm_grid = std::max(1, s->nlm_grid);
        }
        return TL_OK;
    }
    if (s->algo == TL_ALGO_OR_OPT) {
        build_or_geometry(s);
        TL_CUDA_TRY(s->cand.alloc((size_t)s->grid * s->shard_count));
        return TL_OK;
    }
    std::vector<int32_t> bf;
    build_geometry(s, bf);
    TL_CUDA_TRY(s->band_first.alloc(bf.size()));
    TL_CUDA_TRY(cudaMemcpyAsync(s->band_first.p, bf.data(), bf.size() * 4, cudaMemcpyHostToDevice, s->c->stream));
    TL_CUDA_TRY(s->cand.alloc((size_t)s->grid * s->shard_count));
    TL_CUDA_TRY(cudaStreamSynchronize(s->c->stream)); // bf is a local
    return TL_OK;
}

tl_status push_state(tl_session *s)
{
    TL_CUDA_TRY(cudaMemcpyAsync(s->state.p, &s->h, sizeof(DevState), cudaMemcpyHostToDevice, s->c->stream));
    TL_CUDA_TRY(cudaStreamSynchronize(s->c->stream));
    return TL_OK;
}

tl_status pull_state(tl_session *s)
{
    TL_CUDA_TRY(cudaMemcpyAsync(&s->h, s->state.p, sizeof(DevState), cudaMemcpyDeviceToHost, s->c->stream));
    TL_CUDA_TRY(cudaStreamSynchronize(s->c->stream));
    return TL_OK;
}

// (Re)build the slot-ordered matrix: slot q holds the city at `tour[q]` (session start) or at
// the current position q (re-permutation, tour == nullptr).
void build_matrix(tl_session *s, const uint32_t *d_tour)
{
    tl_problem *p = s->p;
    cudaStream_t st = s->c->stream;
    if (p->kind == PK_EXPLICIT) {
        launch_gather_slots(nullptr, d_tour, s->cs.p, s->n, nullptr, s->slot_city.p, st);
        launch_k1_square_from_packed(reinterpret_cast<const uint32_t *>(p->d_tri), s->slot_city.p, s->n, s->ld,
                                     s->M.p, st);
    } else {
        launch_gather_slots(p->d_xy, d_tour, s->cs.p, s->n, s->sxy.p, nullptr, st);
        launch_k1_square(s->sxy.p, s->n, s->ld, p->metric, s->M.p, st);
        if (getenv("TL_K1_TIMING")) { // tuning aid: warm kernel time (CUDA events, 20 back-to-back launches) on stderr
            cudaEvent_t e0, e1;
            cudaEventCreate(&e0);
            cudaEventCreate(&e1);
            cudaEventRecord(e0, st);
            for (int r = 0; r < 20; ++r) launch_k1_square(s->sxy.p, s->n, s->ld, p->metric, s->M.p, st);
            cudaEventRecord(e1, st);
            cudaEventSynchronize(e1);
            float ms = 0.f;
            cudaEventElapsedTime(&ms, e0, e1);
            fprintf(stderr, "[tl] k1_square n=%u %s: %.2f us per launch, %.1f GB/s written\n", s->n, metric_name(p->metric),
                    ms / 20 * 1e3, (double)s->n * s->ld * 4.0 / (ms / 20 * 1e-3) / 1e9);
            cudaEventDestroy(e0);
            cudaEventDestroy(e1);
        }
    }
    s->c->launches += 2;
}

// A Mode B scan reads every upper-triangle element once and the next scan reads (almost) the same
// elements again.  When the matrix does not fit L2, keep a fixed part of it resident: the first
// `rows` physical rows, whose scanned part is about `pin_mb` MB.
//   TL_MAT_PIN_MB=<mb>      size of the resident part (0 disables; default kMatPinMB)
//   TL_MAT_PIN_MODE=hint    per-load L2 eviction hints (default)
//   TL_MAT_PIN_MODE=window  driver access-policy window + persisting-L2 carve-out
void configure_matrix_pin(tl_session *s, size_t matrix_bytes)
{
    s->pin = MatPin{};
    if (s->algo != TL_ALGO_TWO_OPT_BEST && s->algo != TL_ALGO_TWO_OPT_BEST_CYCLIC) return;
    int l2 = 0;
    cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, s->c->device);
    if (matrix_bytes / 2 <= (size_t)l2 * 3 / 4) return; // the scanned triangle already lives in L2
    double pin_mb = kMatPinMB;
    if (const char *ev = getenv("TL_MAT_PIN_MB")) pin_mb = atof(ev);
    if (pin_mb <= 0) return;
    // rows r of the scanned triangle hold (n - r) elements: smallest r0 with sum_{r<r0} 4 (n - r) >= pin bytes
    const double n = (double)s->n, want = pin_mb * 1048576.0 / 4.0;
    const double disc = n * n - 2.0 * want;
    const int rows = disc <= 0 ? (int)s->n : (int)std::ceil(n - std::sqrt(disc));
    const char *mode = getenv("TL_MAT_PIN_MODE");
    if (mode && !strcmp(mode, "window")) {
        int max_persist = 0, max_window = 0;
        cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, s->c->device);
        cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, s->c->device);
        if (getenv("TL_DEBUG_PIN"))
            fprintf(stderr, "[tl] L2 %d B, max persisting %d B, max window %d B, rows %d\n", l2, max_persist, max_window, rows);
        if (max_persist <= 0 || max_window <= 0) return;
        const size_t carve = std::min<size_t>((size_t)max_persist, (size_t)(pin_mb * 1048576.0));
        const cudaError_t le = cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve);
        if (getenv("TL_DEBUG_PIN")) fprintf(stderr, "[tl] set persisting carve-out %zu B: %s\n", carve, cudaGetErrorString(le));
        if (le != cudaSuccess) { cudaGetLastError(); return; }
        const size_t span = std::min<size_t>((size_t)rows * s->ld * 4, (size_t)max_window);
        s->pin.window_bytes = span;
        // the window spans whole rows (both triangles); only about pin_mb of it is ever touched
        s->pin.window_hit_ratio = 1.0f;
        if (const char *hr = getenv("TL_MAT_PIN_HIT")) s->pin.window_hit_ratio = (float)atof(hr);
    } else {
        s->pin.hint_rows = rows;
    }
}

void repermute(tl_session *s)
{
    build_matrix(s, nullptr);
    launch_reset_slots(s->src, s->n, s->npad, s->cyclic, s->c->stream);
    s->c->launches++;
    s->repermutes++;
    s->steps_since_permute = 0;
}

// fuse: let the 2-opt scan kernel's last CTA apply the move -- single-GPU stepping, and sharded
// stepping when the peers' mailboxes are mapped (the last CTA then exchanges the per-rank minima
// over NVLink before it applies the move)
tl_status launch_scan(tl_session *s, bool fuse, bool exchange = true)
{
    const bool fused = fuse && (s->shard_count == 1 || s->use_mailbox);
    const ShardComm *comm = (fused && s->shard_count > 1) ? &s->comm : nullptr;
    BestF *mine = s->cand.p + (size_t)s->shard_index * s->grid;
    cudaStream_t st = s->c->stream;
    if (s->algo == TL_ALGO_OR_OPT_NEIGHBOR || s->algo == TL_ALGO_OR_OPT_NEIGHBOR_MULTI) {
        launch_or_nl_scan(s->p->metric, s->pts.p, s->pos.p, s->nl_cand.p, s->nl_k, s->n, s->tmp.p, s->cand.p,
                          s->nl_cnt.p, s->state.p, s->ticket.p, s->log.p, s->log_cap, fuse, s->grid, st,
                          s->nl_multi() ? &s->nlm : nullptr);
        s->c->launches++;
    } else if (s->algo == TL_ALGO_THREE_OPT_NEIGHBOR) {
        launch_three_nl_scan(s->p->metric, s->pts.p, s->pos.p, s->nl_cand.p, s->nl_k, s->n, s->tmp.p, s->cand.p,
                             s->nl_cnt.p, s->state.p, s->ticket.p, s->log.p, s->log_cap, fuse, s->grid, st);
        s->c->launches++;
    } else if (s->nl) {
        launch_nl_scan(s->p->metric, s->pts.p, s->pos.p, s->nl_cand.p, s->nl_k, s->n, s->cand.p, s->state.p,
                       s->ticket.p, s->log.p, s->log_cap, fuse, s->grid, st, s->nl_multi() ? &s->nlm : nullptr);
        s->c->launches++;
    } else if (s->algo == TL_ALGO_THREE_OPT) {
        TL_CUDA_TRY(cudaMemsetAsync(s->or_ticket.p, 0, 4, st)); // re-arm the work queue
        launch_three_scan(s->src, s->n, s->band_first.p, s->or_item_begin, s->or_item_end, mine, s->state.p,
                          s->or_ticket.p, s->grid, st);
        s->c->launches++;
    } else if (s->algo == TL_ALGO_OR_OPT) {
        launch_or_rowinfo(s->src, s->n, s->npad, s->rowinfo.p, s->state.p, s->or_ticket.p, st);
        launch_or_scan(s->src, s->rowinfo.p, s->n, s->or_order, mine, s->state.p, s->or_ticket.p, s->grid, st);
        s->c->launches += 2;
    } else if (s->matrix()) {
        launch_scan_matrix(s->src, s->geom, s->band_first.p, mine, s->state.p, s->ticket.p, s->log.p, s->log_cap,
                           fused, comm, s->grid, s->pin, st);
        s->c->launches++;
    } else {
        launch_scan_recompute(s->pts.p, s->geom, s->band_first.p, mine, s->state.p, s->ticket.p, s->log.p,
                              s->log_cap, fused, comm, s->grid, s->src.kind == SRC_EUC_FAST, st);
        s->c->launches++;
    }
    if (s->shard_count > 1 && !comm && exchange) {
        if (!s->c->nccl_comm) { set_error("sharded session needs tl_ctx_attach_nccl first"); return TL_ERR_NCCL; }
        // in-place all-gather: every rank contributes its `grid` block records
        tl_status rc = nccl_all_gather_bytes(s->c->nccl_comm, mine, s->cand.p, (size_t)s->grid * sizeof(BestF), st);
        if (rc != TL_OK) return rc;
    }
    return TL_OK;
}

tl_status enqueue_steps(tl_session *s, uint32_t steps)
{
    if (s->trivial) return TL_OK;
    if (!s->timing_open) {
        TL_CUDA_TRY(cudaEventRecord(s->ev0, s->c->stream));
        s->timing_open = true;
    }
    cudaStream_t st = s->c->stream;
    // one thread per swapped pair, at most n/2 pairs
    const int apply_grid =
        (int)std::max<uint32_t>(1, std::min<uint32_t>((s->n / 2 + 255) / 256, (uint32_t)s->c->sm_count));
    if (s->algo == TL_ALGO_TWO_OPT_REF) {
        // coordinate problems whose records fit one SM's shared memory: the whole chain of `steps`
        // cursor steps in ONE launch of a thread-block cluster (k2_two_opt_ref.cu, persistent form)
        if (const int csize = ref_persistent_cluster_size(s->recompute_metric(), s->n)) {
            launch_ref_persistent(s->src, s->p->d_xy, s->p->metric, s->n, s->state.p, s->log.p, s->log_cap, steps, csize,
                                  screen_margin(s->p), st);
            s->c->launches += 1;
            TL_CUDA_TRY(cudaGetLastError());
            return TL_OK;
        }
        // one unit (row x 256 columns) per CTA: the first window (8 rows) is covered in one shot
        const int units0 = kRefWindow0 * (int)((s->n + 255) / 256);
        const int ref_grid = std::max(1, std::min(units0, s->c->sm_count * 4));
        for (uint32_t k = 0; k < steps; ++k) {
            launch_ref_step(s->src, s->n, s->state.p, s->ticket.p, s->log.p, s->log_cap, ref_grid, st);
            s->c->launches += 1;
        }
        TL_CUDA_TRY(cudaGetLastError());
        return TL_OK;
    }
    if (s->cached) {
        // a full grid for the steps that rescan many rows; a step's tail decides how many of these CTAs
        // the next step uses (the others leave at once)
        const int cgrid = s->c->sm_count * 8;
        for (uint32_t k = 0; k < steps; ++k) {
            launch_two_opt_cached_step(s->src, s->n, s->cyclic, s->rowkey.p, s->cdesc.p, s->fullrows.p, s->state.p,
                                       s->ticket.p, s->log.p, s->log_cap, cgrid, st);
            s->c->launches += 1;
        }
        TL_CUDA_TRY(cudaGetLastError());
        return TL_OK;
    }
    for (uint32_t k = 0; k < steps; ++k) {
        if (s->matrix() && s->algo != TL_ALGO_OR_OPT && s->algo != TL_ALGO_THREE_OPT && s->repermute_every > 0 &&
            s->steps_since_permute >= (uint32_t)s->repermute_every)
            repermute(s);
        tl_status rc = launch_scan(s, true);
        if (rc != TL_OK) return rc;
        s->steps_since_permute++;
        if (s->algo == TL_ALGO_OR_OPT_NEIGHBOR) { // a long span left pending by the scan's last CTA
            launch_or_nl_apply(s->p->metric, s->pts.p, s->pos.p, s->tmp.p, s->n, s->cand.p + s->grid, s->state.p,
                               s->ticket.p + 1, s->log.p, s->log_cap, apply_grid, st);
            s->c->launches += 2;
            continue;
        }
        if (s->algo == TL_ALGO_THREE_OPT_NEIGHBOR) { // as Or-opt N
            launch_three_nl_apply(s->p->metric, s->pts.p, s->pos.p, s->tmp.p, s->n, s->cand.p + s->grid, s->state.p,
                                  s->ticket.p + 1, s->log.p, s->log_cap, apply_grid, st);
            s->c->launches += 2;
            continue;
        }
        if (s->algo == TL_ALGO_OR_OPT_NEIGHBOR_MULTI) { // as Mode NM, with Or-opt N's two apply grids
            launch_or_nlm_apply(s->p->metric, s->pts.p, s->pos.p, s->tmp.p, s->n, s->nlm, s->ticket.p + 1, s->nlm_grid, st);
            s->c->launches += 2;
            continue;
        }
        if (s->nl_multi()) { // the step's block moves and a pending long G (none: the grid leaves at once)
            launch_nlm_apply(s->p->metric, s->pts.p, s->pos.p, s->nlm, s->ticket.p + 1, s->nlm_grid, st);
            s->c->launches++;
            continue;
        }
        if (s->nl) { // a long segment left pending by the scan's last CTA (none: the grid leaves at once)
            launch_nl_apply(s->p->metric, s->pts.p, s->pos.p, s->cand.p + s->grid, s->state.p, s->ticket.p + 1,
                            s->log.p, s->log_cap, apply_grid, st);
            s->c->launches++;
            continue;
        }
        if (s->algo == TL_ALGO_OR_OPT) {
            launch_or_apply(s->src, s->tmp.p, s->n, s->cand.p, s->grid * s->shard_count, s->state.p, s->ticket.p,
                            s->log.p, s->log_cap, apply_grid, st);
            s->c->launches += 2;
            continue;
        }
        if (s->algo == TL_ALGO_THREE_OPT) {
            launch_three_apply(s->src, s->tmp.p, s->n, s->cand.p, s->grid * s->shard_count, s->state.p, s->ticket.p,
                               s->log.p, s->log_cap, apply_grid, st);
            s->c->launches += 2;
            continue;
        }
        if (s->shard_count == 1 || s->use_mailbox) continue; // the scan kernel's last CTA applied the move
        launch_apply_two_opt(s->src, s->cand.p, s->grid * s->shard_count, s->state.p, s->ticket.p, s->log.p,
                             s->log_cap, apply_grid, st);
        s->c->launches++;
    }
    TL_CUDA_TRY(cudaGetLastError());
    return TL_OK;
}

tl_status close_timing(tl_session *s)
{
    if (!s->timing_open) return TL_OK;
    TL_CUDA_TRY(cudaEventRecord(s->ev1, s->c->stream));
    TL_CUDA_TRY(cudaEventSynchronize(s->ev1));
    float ms = 0.f;
    TL_CUDA_TRY(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
    s->device_ms += ms;
    s->timing_open = false;
    return TL_OK;
}

// host-side (delta, rank) reduction of the per-CTA records of one scan
// 3-opt records: delta = savings (larger is better), aux = k * 8 + case; ties to the lowest (i, j, k)
template <typename V>
bool reduce_host_three(const std::vector<Best<V>> &hc, tl_move *best)
{
    Best<V> v{(V)0, 0xffffffffu, 0xffffffffu, 0u};
    auto better = [](const Best<V> &a, const Best<V> &b) {
        if (a.delta != b.delta) return a.delta > b.delta;
        if (a.i != b.i) return a.i < b.i;
        if (a.j != b.j) return a.j < b.j;
        return (a.aux >> 3) < (b.aux >> 3);
    };
    for (const Best<V> &o : hc) {
        if (o.i == 0xffffffffu) continue;
        if (v.i == 0xffffffffu || better(o, v)) v = o;
    }
    if (v.i == 0xffffffffu) return false;
    if (best) *best = tl_move{-(float)v.delta, v.i, v.j, (uint8_t)(v.aux & 7u), 0, 0, v.aux >> 3};
    return true;
}

template <typename V>
bool reduce_host(const std::vector<Best<V>> &hc, bool or_opt, tl_move *best)
{
    Best<V> v{(V)0, 0xffffffffu, 0xffffffffu, 0u};
    auto rank_less = [&](const Best<V> &a, const Best<V> &b) {
        if (or_opt && (a.aux >> 1) != (b.aux >> 1)) return (a.aux >> 1) < (b.aux >> 1);
        if (a.i != b.i) return a.i < b.i;
        if (a.j != b.j) return a.j < b.j;
        return (a.aux & 1u) < (b.aux & 1u);
    };
    for (const Best<V> &o : hc) {
        if (o.i == 0xffffffffu) continue;
        if (v.i == 0xffffffffu || o.delta < v.delta || (o.delta == v.delta && rank_less(o, v))) v = o;
    }
    if (v.i == 0xffffffffu) return false;
    if (best) {
        if (or_opt)
            *best = tl_move{(float)v.delta, v.i, v.j, (uint8_t)((v.aux >> 1) + 1), (uint8_t)(v.aux & 1u), 0};
        else
            *best = tl_move{(float)v.delta, v.i, v.j, 0, 0, 0};
    }
    return true;
}

} // namespace

extern "C" {

tl_status tl_session_create(tl_problem *p, int32_t algo, int32_t path, const uint32_t *tour, tl_session **out)
{
    return tl::guarded([&]() -> tl_status {
    if (!p || !tour || !out) { set_error("tl_session_create: null argument"); return TL_ERR_INVALID; }
    *out = nullptr;
    const bool cached = algo == TL_ALGO_TWO_OPT_BEST_CACHED; // Mode B with cached row minima: runs as Mode B
    if (cached) algo = TL_ALGO_TWO_OPT_BEST;
    if (algo != TL_ALGO_TWO_OPT_BEST && algo != TL_ALGO_TWO_OPT_BEST_CYCLIC && algo != TL_ALGO_TWO_OPT_REF &&
        algo != TL_ALGO_OR_OPT && algo != TL_ALGO_THREE_OPT && algo != TL_ALGO_TWO_OPT_NEIGHBOR &&
        algo != TL_ALGO_OR_OPT_NEIGHBOR && algo != TL_ALGO_THREE_OPT_NEIGHBOR && algo != TL_ALGO_TWO_OPT_NEIGHBOR_MULTI &&
        algo != TL_ALGO_OR_OPT_NEIGHBOR_MULTI) {
        set_error("tl_session_create: unknown algo %d", algo);
        return TL_ERR_INVALID;
    }
    if (path != TL_PATH_AUTO && path != TL_PATH_MATRIX && path != TL_PATH_RECOMPUTE) {
        set_error("tl_session_create: unknown path %d", path);
        return TL_ERR_INVALID;
    }
    const bool nl = algo == TL_ALGO_TWO_OPT_NEIGHBOR || algo == TL_ALGO_OR_OPT_NEIGHBOR ||
                    algo == TL_ALGO_THREE_OPT_NEIGHBOR || algo == TL_ALGO_TWO_OPT_NEIGHBOR_MULTI ||
                    algo == TL_ALGO_OR_OPT_NEIGHBOR_MULTI;
    // Mode NM's and Or-opt NM's block size: TL_MULTI_BLOCK / TL_OR_MULTI_BLOCK, or the TL_MULTI_BLOCK environment
    // variable (a power of two in 2..65536, 2..16384 for Or-opt NM, whose keys hold s, i, j and rev in 31 bits) for
    // measuring other sizes
    uint32_t multi_block = algo == TL_ALGO_OR_OPT_NEIGHBOR_MULTI ? TL_OR_MULTI_BLOCK : TL_MULTI_BLOCK;
    if (const char *ev = getenv("TL_MULTI_BLOCK");
        ev && (algo == TL_ALGO_TWO_OPT_NEIGHBOR_MULTI || algo == TL_ALGO_OR_OPT_NEIGHBOR_MULTI)) {
        const long b = atol(ev), bmax = algo == TL_ALGO_OR_OPT_NEIGHBOR_MULTI ? 16384 : 65536;
        if (b < 2 || b > bmax || (b & (b - 1))) {
            set_error("TL_MULTI_BLOCK=%s: must be a power of two in 2..%ld", ev, bmax);
            return TL_ERR_INVALID;
        }
        multi_block = (uint32_t)b;
    }
    if (nl && (path == TL_PATH_MATRIX || p->kind == PK_EXPLICIT)) {
        // candidate-list searches are for instances whose n^2 matrix is the problem; both metrics are recomputed
        set_error(p->kind == PK_EXPLICIT ? "candidate-list search needs coordinates (EXPLICIT problem)"
                                         : "candidate-list search recomputes distances: TL_PATH_MATRIX is not supported");
        return TL_ERR_UNSUPPORTED;
    }
    // AUTO: recompute for f32 coordinate problems (bit-identical to the matrix and no n^2 memory),
    // matrix for EXPLICIT problems (placeholder coordinates, tsplib.rs:257-262) and the nint metric
    const bool want_matrix = !nl && (path == TL_PATH_MATRIX || (path == TL_PATH_AUTO && p->kind != PK_EUC_F32));
    if (!nl && !want_matrix && p->kind != PK_EUC_F32) {
        set_error(p->kind == PK_EXPLICIT ? "recompute path is illegal for EXPLICIT problems (no coordinates)"
                                         : "recompute path is not available for the NINT_I32 metric");
        return TL_ERR_UNSUPPORTED;
    }
    if (!tour_is_permutation(tour, p->n)) {
        set_error("tl_session_create: tour is not a permutation of 0..%u", p->n - 1);
        return TL_ERR_INVALID;
    }
    tl_ctx *c = p->ctx;
    DeviceGuard g(c);
    tl_session *s = new tl_session();
    s->p = p;
    s->c = c;
    s->algo = algo;
    s->cached = cached;
    s->nl = nl;
    while ((1u << s->nlm.bshift) < multi_block) ++s->nlm.bshift;
    s->path_used = want_matrix ? TL_PATH_MATRIX : TL_PATH_RECOMPUTE;
    s->n = p->n;
    s->cyclic = algo == TL_ALGO_TWO_OPT_BEST_CYCLIC || algo == TL_ALGO_OR_OPT || algo == TL_ALGO_THREE_OPT;
    s->trivial = p->n < 4;
    s->launches0 = c->launches;
    s->log_cap = 1u << 16;
    const uint64_t n = p->n;
    s->pairs_per_scan = s->trivial ? 0 : (s->cyclic ? n * (n - 3) / 2 : (n - 3) * (n - 2) / 2);
    if (algo == TL_ALGO_OR_OPT && !s->trivial) {
        // candidates per find_best_move: sum over s of (n-s+1)(n-s-1), doubled for s > 1 (fwd + rev)
        s->pairs_per_scan = 0;
        for (uint64_t sg = 1; sg <= 3; ++sg)
            if (n > sg + 1) s->pairs_per_scan += (n - sg + 1) * (n - sg - 1) * (sg > 1 ? 2 : 1);
    }
    if (algo == TL_ALGO_THREE_OPT && !s->trivial) {
        // triples i < j < k minus the skipped (i == 0, k == n-1) ones (three_opt.rs:79-83)
        s->pairs_per_scan = n * (n - 1) * (n - 2) / 6 - (n - 2);
    }
    // pad so that every staged window of a valid row stays in bounds for every kernel
    s->npad = p->n + std::max(std::max(kScanBW + kScanTI, kMatBW + kMatTI), 32 * kOrR + kOrR) + 64;

    auto fail = [&](tl_status rc) {
        tl_session_destroy(s);
        return rc;
    };
    // TL_DEBUG_TIMING: host wall time of the phases of this call on stderr
    const bool trace = getenv("TL_DEBUG_TIMING") != nullptr;
    auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double tc0 = trace ? now() : 0.0;
    double tc1 = tc0, tc2 = tc0, tc3 = tc0;
    if (want_matrix) {
        // The matrix is allocated FIRST: the pool usually holds the previous session's matrix block, and
        // the small buffers below would otherwise be carved out of it, so that the matrix no longer fits
        // and the pool has to grow by another n^2 block (8-30 ms per call in the end-to-end path).
        s->ld = (p->n + 31u) & ~31u;
        const size_t bytes = (size_t)p->n * s->ld * 4;
        void *cached = nullptr;
        size_t cached_bytes = 0;
        {   // take the block a previous session of this context left behind (host.hpp: mat_block)
            std::lock_guard<std::mutex> lk(c->pin_mu);
            cached = c->mat_block;
            cached_bytes = c->mat_bytes;
            c->mat_block = nullptr;
            c->mat_bytes = 0;
        }
        if (cached && cached_bytes >= bytes) {
            s->M.adopt(static_cast<uint32_t *>(cached), cached_bytes / 4);
        } else {
            if (cached) cudaFreeAsync(cached, c->stream); // too small: given back first
            // what a new block can come from: the driver's free memory plus what this context's pool
            // holds cached from earlier sessions (reserved but not in use)
            size_t free_b = 0, total_b = 0;
            cudaMemGetInfo(&free_b, &total_b);
            if (c->pool) {
                uint64_t reserved = 0, used = 0;
                if (cudaMemPoolGetAttribute(c->pool, cudaMemPoolAttrReservedMemCurrent, &reserved) == cudaSuccess &&
                    cudaMemPoolGetAttribute(c->pool, cudaMemPoolAttrUsedMemCurrent, &used) == cudaSuccess && reserved > used)
                    free_b += (size_t)(reserved - used);
            }
            free_b += cached_bytes;
            if (bytes > free_b - std::min<size_t>(free_b, (size_t)1 << 30)) {
                set_error("the %u x %u distance matrix (%.1f GB) does not fit device memory (%.1f GB free); "
                          "use TL_PATH_RECOMPUTE", p->n, s->ld, bytes / 1e9, free_b / 1e9);
                return fail(TL_ERR_NOMEM);
            }
            if (s->M.alloc((size_t)p->n * s->ld) != cudaSuccess) {
                cudaGetLastError();
                set_error("tl_session_create: matrix allocation failed");
                return fail(TL_ERR_NOMEM);
            }
        }
    }
    if (trace) tc1 = now();
    DevBuf<uint32_t> d_tour;
    if (d_tour.alloc(p->n) != cudaSuccess || s->state.alloc(1) != cudaSuccess || s->ticket.alloc(2) != cudaSuccess ||
        s->log.alloc(s->log_cap) != cudaSuccess || cudaEventCreate(&s->ev0) != cudaSuccess ||
        cudaEventCreate(&s->ev1) != cudaSuccess) {
        set_error("tl_session_create: device allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
        return fail(TL_ERR_NOMEM);
    }
    if ((algo == TL_ALGO_OR_OPT || algo == TL_ALGO_THREE_OPT) &&
        (s->tmp.alloc((size_t)s->npad * 16) != cudaSuccess || s->rowinfo.alloc((size_t)s->npad * 16) != cudaSuccess ||
         s->or_ticket.alloc(1) != cudaSuccess)) {
        set_error("tl_session_create: device allocation failed");
        return fail(TL_ERR_NOMEM);
    }
    if (s->nl_relocating() && s->tmp.alloc((size_t)s->npad * 16) != cudaSuccess) {
        set_error("tl_session_create: device allocation failed");
        return fail(TL_ERR_NOMEM);
    }
    if (cached && !s->trivial) {
        if (s->rowkey.alloc(p->n) != cudaSuccess || s->cdesc.alloc(1) != cudaSuccess || s->fullrows.alloc(p->n) != cudaSuccess) {
            set_error("tl_session_create: device allocation failed");
            return fail(TL_ERR_NOMEM);
        }
        // every row key "none", first step: rescan every row
        const CachedDesc d0{-1, 0, 0, 0, p->ctx->sm_count * 8};
        cudaError_t ce = cudaMemsetAsync(s->rowkey.p, 0xff, (size_t)p->n * 8, c->stream);
        if (ce == cudaSuccess) ce = cudaMemcpyAsync(s->cdesc.p, &d0, sizeof d0, cudaMemcpyHostToDevice, c->stream);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(c->stream); // d0 is a local
        if (ce != cudaSuccess) { set_error("tl_session_create: %s", cudaGetErrorString(ce)); return fail(TL_ERR_CUDA); }
    }
    // or_opt::solve and three_opt::solve ignore the seed and return identity order when n < 4
    // (or_opt.rs:31-34, three_opt.rs:25-28); so do Or-opt N and 3-opt N
    // (Mode NM and Or-opt NM too: new modes, defined with no scan for n < 4)
    const bool or_like = algo == TL_ALGO_OR_OPT || algo == TL_ALGO_THREE_OPT || s->nl_relocating() || s->nl_multi();
    std::vector<uint32_t> ident;
    if (or_like && s->trivial) {
        ident.resize(p->n);
        for (uint32_t k = 0; k < p->n; ++k) ident[k] = k;
        tour = ident.data();
    }
    if (trace) tc2 = now();
    cudaError_t e = cudaMemcpyAsync(d_tour.p, tour, (size_t)p->n * 4, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(s->ticket.p, 0, 8, c->stream);
    if (e != cudaSuccess) { set_error("tl_session_create: %s", cudaGetErrorString(e)); return fail(TL_ERR_CUDA); }

    if (want_matrix) {
        bool ok = s->cs.alloc(s->npad) == cudaSuccess;
        if (p->kind == PK_EXPLICIT)
            ok = ok && s->slot_city.alloc(p->n) == cudaSuccess;
        else
            ok = ok && s->sxy.alloc(p->n) == cudaSuccess;
        if (!ok) { set_error("tl_session_create: matrix allocation failed"); return fail(TL_ERR_NOMEM); }
        s->src.kind = p->kind == PK_EUC_NINT ? SRC_MAT_I32 : SRC_MAT_F32;
        s->src.cs = s->cs.p;
        s->src.M = s->M.p;
        s->src.ld = s->ld;
        build_matrix(s, d_tour.p);
        launch_build_cs(s->src, d_tour.p, p->n, s->npad, s->cyclic, c->stream);
        c->launches++;
        // re-lay the matrix in tour order only when it cannot live in L2 (gathers are cheap there)
        const size_t bytes = (size_t)p->n * s->ld * 4;
        s->repermute_every = bytes > ((size_t)96 << 20) ? 256 : 0;
        if (const char *ev = getenv("TL_REPERMUTE_EVERY")) s->repermute_every = atoi(ev);
        if (cached) s->repermute_every = 0; // a cached step reads a few rows, not the triangle
        configure_matrix_pin(s, bytes);
    } else if (nl) {
        if (!s->trivial && !p->d_cand) {
            tl_status rc = tl_problem_set_candidates(p, TL_CANDIDATES_DEFAULT);
            if (rc != TL_OK) return fail(rc);
        }
        s->nl_k = s->trivial ? 0 : p->cand_k;
        if (s->pts.alloc(s->npad) != cudaSuccess || s->pos.alloc(p->n) != cudaSuccess ||
            s->nl_cand.alloc((size_t)p->n * s->nl_k) != cudaSuccess) {
            set_error("tl_session_create: device allocation failed");
            return fail(TL_ERR_NOMEM);
        }
        if (s->nl_k) { // the session's own copy: later tl_problem_set_candidates calls do not reach it
            e = cudaMemcpyAsync(s->nl_cand.p, p->d_cand, (size_t)p->n * s->nl_k * 4, cudaMemcpyDeviceToDevice, c->stream);
            if (e != cudaSuccess) { set_error("tl_session_create: %s", cudaGetErrorString(e)); return fail(TL_ERR_CUDA); }
        }
        s->src.kind = SRC_EUC_SAFE; // tl_session_tour reads the city fields only
        s->src.pts = s->pts.p;
        launch_nl_init(p->metric, p->d_xy, d_tour.p, p->n, s->npad, s->nl_relocating(), s->pts.p, s->pos.p, c->stream);
        c->launches++;
    } else {
        if (s->pts.alloc(s->npad) != cudaSuccess) { set_error("tl_session_create: device allocation failed"); return fail(TL_ERR_NOMEM); }
        const bool fast = p->metric == Metric::F32_FAST;
        s->src.kind = fast ? SRC_EUC_FAST : SRC_EUC_SAFE;
        s->src.pts = s->pts.p;
        launch_build_pts(p->d_xy, d_tour.p, p->n, s->npad, s->cyclic, fast, s->pts.p, c->stream);
        c->launches++;
    }
    memset(&s->h, 0, sizeof s->h);
    s->h.max_moves = -1;
    s->h.cur_i = 0;
    s->h.cur_j = 2;
    s->h.window_rows = kRefWindow0;
    s->h.found_key = ~0ull;
    if (s->trivial) {
        // oracle/reference behaviour for n < 4: Mode B scans once and finds nothing; the reference
        // loop runs one empty pass for n == 3 and is skipped for n < 3 (two_opt.rs:17,29 underflow)
        s->h.done = 1;
        s->h.converged = 1;
        s->h.scans = or_like ? 0 : 1;
        s->h.passes = (p->n == 3) ? 1 : 0;
    }
    tl_status rc = push_state(s); // also waits for d_tour's consumers
    if (rc != TL_OK) return fail(rc);
    if (trace) tc3 = now();
    if (!s->trivial && algo != TL_ALGO_TWO_OPT_REF) {
        rc = upload_geometry(s);
        if (rc != TL_OK) return fail(rc);
    }
    if (trace)
        fprintf(stderr, "[tl] session_create: matrix block %.2f ms, buffers %.2f ms, build + state %.2f ms, geometry %.2f ms\n",
                tc1 - tc0, tc2 - tc1, tc3 - tc2, now() - tc3);
    if (cudaGetLastError() != cudaSuccess) { set_error("tl_session_create: kernel launch failed"); return fail(TL_ERR_CUDA); }
    *out = s;
    return TL_OK;
    });
}

void tl_session_destroy(tl_session *s)
{
    if (!s) return;
    DeviceGuard g(s->c);
    cudaStreamSynchronize(s->c->stream);
    if (s->ev0) cudaEventDestroy(s->ev0);
    if (s->ev1) cudaEventDestroy(s->ev1);
    for (cudaEvent_t e : s->ev_snap)
        if (e) cudaEventDestroy(e);
    if (s->h_snap) s->c->return_pinned(s->h_snap);
    if (s->M.p) { // keep the matrix block for the next session of this context (the larger one wins)
        tl_ctx *c = s->c;
        const size_t bytes = s->M.count * 4;
        void *drop = nullptr;
        {
            std::lock_guard<std::mutex> lk(c->pin_mu);
            if (!c->mat_block || bytes > c->mat_bytes) {
                drop = c->mat_block;
                c->mat_bytes = bytes;
                c->mat_block = s->M.detach();
            }
        }
        if (drop) cudaFreeAsync(drop, c->stream);
    }
    delete s;
}

tl_status tl_session_set_shard(tl_session *s, int32_t index, int32_t count)
{
    return tl::guarded([&]() -> tl_status {
    if (!s || count < 1 || index < 0 || index >= count) { set_error("tl_session_set_shard: bad arguments"); return TL_ERR_INVALID; }
    if (s->algo == TL_ALGO_TWO_OPT_REF) {
        if (count > 1) { set_error("Mode R does not shard (replicas only)"); return TL_ERR_UNSUPPORTED; }
        return TL_OK;
    }
    if (s->cached) {
        if (count > 1) { set_error("cached Mode B does not shard (a step touches a few rows)"); return TL_ERR_UNSUPPORTED; }
        return TL_OK;
    }
    if (s->nl) {
        if (count > 1) { set_error("candidate-list searches do not shard"); return TL_ERR_UNSUPPORTED; }
        return TL_OK;
    }
    DeviceGuard g(s->c);
    s->shard_index = index;
    s->shard_count = count;
    s->use_mailbox = false;
    tl_ctx *c = s->c;
    const bool two_opt_best = s->algo == TL_ALGO_TWO_OPT_BEST || s->algo == TL_ALGO_TWO_OPT_BEST_CYCLIC;
    const char *tr = getenv("TL_SHARD_TRANSPORT"); // "nccl": force the all-gather + apply-kernel path
    if (count > 1 && two_opt_best && c->p2p_ready && count == c->world && index == c->rank &&
        !(tr && !strcmp(tr, "nccl"))) {
        // One sharded session steps at a time per context; its records are tagged with an epoch so
        // that a mailbox slot left over from an earlier session can never look current.  Every 255
        // sessions the epochs are recycled behind a collective reset of the mailboxes.
        if (c->shard_epoch > 0 && c->shard_epoch % 255 == 0) {
            TL_CUDA_TRY(cudaStreamSynchronize(c->stream));
            tl_status rc = nccl_barrier(c);
            if (rc != TL_OK) return rc;
            TL_CUDA_TRY(cudaMemsetAsync(c->mailbox, 0, kMailboxBytes, c->stream));
            rc = nccl_barrier(c);
            if (rc != TL_OK) return rc;
        }
        s->comm = ShardComm{};
        for (int r = 0; r < count; ++r) s->comm.peer[r] = c->peer_mailbox[r];
        s->comm.rank = index;
        s->comm.world = count;
        s->comm.epoch = c->shard_epoch % 255 + 1;
        c->shard_epoch++;
        s->use_mailbox = true;
    }
    if (s->trivial) return TL_OK;
    return upload_geometry(s);
    });
}

tl_status tl_session_scan(tl_session *s, tl_move *best, int32_t *found)
{
    return tl::guarded([&]() -> tl_status {
    if (!s || !found) { set_error("tl_session_scan: null argument"); return TL_ERR_INVALID; }
    *found = 0;
    if (s->algo == TL_ALGO_TWO_OPT_REF) { set_error("tl_session_scan: Mode R has no whole-triangle scan"); return TL_ERR_UNSUPPORTED; }
    if (s->cached) { set_error("tl_session_scan: cached Mode B has no whole-triangle scan (use TL_ALGO_TWO_OPT_BEST)"); return TL_ERR_UNSUPPORTED; }
    if (s->trivial) return TL_OK;
    DeviceGuard g(s->c);
    tl_status rc = pull_state(s);
    if (rc != TL_OK) return rc;
    // a scan of a finished session is still a scan: lift the no-op flag for this launch
    const int was_done = s->h.done;
    if (was_done) { s->h.done = 0; rc = push_state(s); if (rc != TL_OK) return rc; }
    rc = launch_scan(s, false);
    if (rc != TL_OK) return rc;
    TL_CUDA_TRY(cudaGetLastError());
    std::vector<BestF> hc((size_t)s->grid * s->shard_count);
    TL_CUDA_TRY(cudaMemcpyAsync(hc.data(), s->cand.p, hc.size() * sizeof(BestF), cudaMemcpyDeviceToHost, s->c->stream));
    TL_CUDA_TRY(cudaStreamSynchronize(s->c->stream));
    if (was_done) { s->h.done = was_done; rc = push_state(s); if (rc != TL_OK) return rc; }
    bool any;
    const bool three = s->algo == TL_ALGO_THREE_OPT || s->algo == TL_ALGO_THREE_OPT_NEIGHBOR;
    const bool or_opt =
        s->algo == TL_ALGO_OR_OPT || s->algo == TL_ALGO_OR_OPT_NEIGHBOR || s->algo == TL_ALGO_OR_OPT_NEIGHBOR_MULTI;
    if (s->int_values()) {
        std::vector<BestI> hi(hc.size());
        memcpy(hi.data(), hc.data(), hc.size() * sizeof(BestF));
        any = three ? reduce_host_three(hi, best) : reduce_host(hi, or_opt, best);
    } else {
        any = three ? reduce_host_three(hc, best) : reduce_host(hc, or_opt, best);
    }
    *found = any ? 1 : 0;
    return TL_OK;
    });
}

tl_status tl_session_time_scans(tl_session *s, uint32_t reps, double *avg_ms)
{
    return tl::guarded([&]() -> tl_status {
    if (!s || !avg_ms || reps == 0) { set_error("tl_session_time_scans: bad arguments"); return TL_ERR_INVALID; }
    if (s->algo == TL_ALGO_TWO_OPT_REF) { set_error("tl_session_time_scans: Mode R has no whole-triangle scan"); return TL_ERR_UNSUPPORTED; }
    if (s->cached) { set_error("tl_session_time_scans: cached Mode B has no whole-triangle scan"); return TL_ERR_UNSUPPORTED; }
    *avg_ms = 0.0;
    if (s->trivial) return TL_OK;
    DeviceGuard g(s->c);
    tl_status rc = pull_state(s);
    if (rc != TL_OK) return rc;
    const int was_done = s->h.done;
    if (was_done) { s->h.done = 0; rc = push_state(s); if (rc != TL_OK) return rc; }
    cudaEvent_t a, b;
    TL_CUDA_TRY(cudaEventCreate(&a));
    TL_CUDA_TRY(cudaEventCreate(&b));
    rc = launch_scan(s, false, false); // warm; a sharded session times its own share of the scan, no exchange
    if (rc == TL_OK) {
        cudaEventRecord(a, s->c->stream);
        for (uint32_t r = 0; r < reps && rc == TL_OK; ++r) rc = launch_scan(s, false, false);
        cudaEventRecord(b, s->c->stream);
        cudaEventSynchronize(b);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, a, b);
        *avg_ms = (double)ms / reps;
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    if (rc != TL_OK) return rc;
    TL_CUDA_TRY(cudaGetLastError());
    if (was_done) { s->h.done = was_done; rc = push_state(s); }
    return rc;
    });
}

tl_status tl_session_enqueue(tl_session *s, uint32_t steps)
{
    return tl::guarded([&]() -> tl_status {
    if (!s) { set_error("tl_session_enqueue: null session"); return TL_ERR_INVALID; }
    DeviceGuard g(s->c);
    return enqueue_steps(s, steps);
    });
}

tl_status tl_session_run(tl_session *s, int64_t max_moves)
{
    return tl::guarded([&]() -> tl_status {
    if (!s) { set_error("tl_session_run: null session"); return TL_ERR_INVALID; }
    DeviceGuard g(s->c);
    tl_status rc = pull_state(s);
    if (rc != TL_OK) return rc;
    if (s->trivial || s->h.converged) return close_timing(s);
    s->h.max_moves = max_moves;
    s->h.done = (max_moves >= 0 && (long long)s->h.moves >= max_moves) ? 1 : 0;
    rc = push_state(s);
    if (rc != TL_OK) return rc;
    if (s->h.done) return close_timing(s);
    constexpr int kSlots = 3; // batches in flight: two are always queued behind the one the host waits for
    if (!s->h_snap) {
        static_assert(kSlots * sizeof(DevState) <= 512, "the state snapshots fit one pinned slot");
        s->h_snap = static_cast<DevState *>(s->c->borrow_pinned());
        if (!s->h_snap) { set_error("tl_session_run: pinned host allocation failed"); return TL_ERR_NOMEM; }
        for (cudaEvent_t &e : s->ev_snap) TL_CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    // Batches of steps are queued ahead of the host: batches k+1 and k+2 are already enqueued when
    // the host waits for the state snapshot taken after batch k, so the device does not idle on a
    // host round trip (or on a host thread that is late by a millisecond or two).  Steps queued
    // past convergence (or past max_moves, which the device checks itself) are no-op launches.
    // with a move budget every step applies exactly one move (or finds none and stops), so the host
    // knows how many steps are still worth queueing without looking at the device
    // (not so for Mode R, whose persistent kernel stops by itself, and Mode NM and Or-opt NM, whose steps apply
    // several moves: they get unbudgeted batches and the device stops at the budget)
    const bool budgeted = max_moves >= 0 && s->algo != TL_ALGO_TWO_OPT_REF && !s->nl_multi();
    int64_t budget = budgeted ? max_moves - (int64_t)s->h.moves : 0;
    auto issue = [&](int slot) -> tl_status {
        uint32_t batch = s->algo == TL_ALGO_TWO_OPT_REF ? 64 : 32;
        // Mode R, persistent form: a batch is one launch, so make it long (the kernel stops by itself
        // at convergence or at the move budget)
        if (s->algo == TL_ALGO_TWO_OPT_REF && ref_persistent_cluster_size(s->recompute_metric(), s->n)) batch = 1u << 20;
        if (budgeted) {
            batch = (uint32_t)std::min<int64_t>(256, budget);
            budget -= batch;
        }
        tl_status r = enqueue_steps(s, batch);
        if (r != TL_OK) return r;
        TL_CUDA_TRY(cudaMemcpyAsync(s->h_snap + slot, s->state.p, sizeof(DevState), cudaMemcpyDeviceToHost, s->c->stream));
        TL_CUDA_TRY(cudaEventRecord(s->ev_snap[slot], s->c->stream));
        return TL_OK;
    };
    int head = 0, queued = 0; // `queued` snapshots are outstanding, the oldest one in slot `head`
    for (;;) {
        while (queued < kSlots && (!budgeted || budget > 0)) {
            rc = issue((head + queued) % kSlots);
            if (rc != TL_OK) return rc;
            ++queued;
        }
        if (queued == 0) break; // budget spent and every snapshot seen
        TL_CUDA_TRY(cudaEventSynchronize(s->ev_snap[head]));
        s->h = s->h_snap[head];
        head = (head + 1) % kSlots;
        --queued;
        if (s->h.done) break;
    }
    while (queued > 0) { // the batches that were queued ahead
        TL_CUDA_TRY(cudaEventSynchronize(s->ev_snap[head]));
        s->h = s->h_snap[head];
        head = (head + 1) % kSlots;
        --queued;
    }
    rc = close_timing(s);
    if (rc == TL_OK && s->h.error) {
        set_error("sharded step: a peer's best-move record did not arrive (rank down or not stepping the same session)");
        return TL_ERR_NCCL;
    }
    return rc;
    });
}

tl_status tl_session_tour(tl_session *s, uint32_t *tour_out)
{
    return tl::guarded([&]() -> tl_status {
    if (!s || !tour_out) { set_error("tl_session_tour: null argument"); return TL_ERR_INVALID; }
    DeviceGuard g(s->c);
    DevBuf<uint32_t> d;
    TL_CUDA_TRY(d.alloc(s->n));
    launch_extract_tour(s->src, s->n, d.p, s->c->stream);
    s->c->launches++;
    TL_CUDA_TRY(cudaGetLastError());
    TL_CUDA_TRY(cudaMemcpyAsync(tour_out, d.p, (size_t)s->n * 4, cudaMemcpyDeviceToHost, s->c->stream));
    TL_CUDA_TRY(cudaStreamSynchronize(s->c->stream));
    return TL_OK;
    });
}

tl_status tl_session_stats(tl_session *s, tl_stats *stats)
{
    return tl::guarded([&]() -> tl_status {
    if (!s || !stats) { set_error("tl_session_stats: null argument"); return TL_ERR_INVALID; }
    DeviceGuard g(s->c);
    tl_status rc = pull_state(s);
    if (rc != TL_OK) return rc;
    rc = close_timing(s);
    if (rc != TL_OK) return rc;
    memset(stats, 0, sizeof *stats);
    stats->passes = s->algo == TL_ALGO_TWO_OPT_REF ? s->h.passes : s->h.scans;
    stats->moves = s->h.moves;
    stats->evals = (s->cached || s->nl) ? s->h.computed : stats->passes * s->pairs_per_scan;
    stats->launches = s->c->launches - s->launches0;
    stats->repermutes = s->repermutes;
    stats->device_ms = s->device_ms;
    stats->converged = s->h.converged;
    stats->path_used = s->path_used;
    if (s->h.error) {
        set_error("sharded step: a peer's best-move record did not arrive (rank down or not stepping the same session)");
        return TL_ERR_NCCL;
    }
    return TL_OK;
    });
}

tl_status tl_session_log(tl_session *s, tl_move *log, size_t log_cap, size_t *n_out)
{
    return tl::guarded([&]() -> tl_status {
    if (!s || !n_out) { set_error("tl_session_log: null argument"); return TL_ERR_INVALID; }
    DeviceGuard g(s->c);
    tl_status rc = pull_state(s);
    if (rc != TL_OK) return rc;
    const size_t have = (size_t)std::min<uint64_t>(s->h.moves, s->log_cap);
    const size_t cnt = std::min(have, log_cap);
    if (cnt && log) {
        TL_CUDA_TRY(cudaMemcpyAsync(log, s->log.p, cnt * sizeof(tl_move), cudaMemcpyDeviceToHost, s->c->stream));
        TL_CUDA_TRY(cudaStreamSynchronize(s->c->stream));
    }
    *n_out = cnt;
    return TL_OK;
    });
}

tl_status tl_local_search(tl_problem *p, int32_t algo, int32_t path, uint32_t *tour_inout, int64_t max_moves,
                          tl_stats *stats, tl_move *log, size_t log_cap)
{
    return tl::guarded([&]() -> tl_status {
    if (!p || !tour_inout) { set_error("tl_local_search: null argument"); return TL_ERR_INVALID; }
    tl_session *s = nullptr;
    const bool trace = getenv("TL_DEBUG_TIMING") != nullptr; // host wall time of each phase on stderr
    auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t0 = trace ? now() : 0.0;
    tl_status rc = tl_session_create(p, algo, path, tour_inout, &s);
    if (rc != TL_OK) return rc;
    const double t1 = trace ? now() : 0.0;
    if (log && log_cap > s->log_cap) {
        DeviceGuard g(s->c);
        if (s->log.alloc(log_cap) != cudaSuccess) {
            tl_session_destroy(s);
            set_error("tl_local_search: move log of %zu entries does not fit", log_cap);
            return TL_ERR_NOMEM;
        }
        s->log_cap = log_cap;
    }
    rc = tl_session_run(s, max_moves);
    const double t2 = trace ? now() : 0.0;
    if (rc == TL_OK) rc = tl_session_tour(s, tour_inout);
    if (rc == TL_OK && stats) rc = tl_session_stats(s, stats);
    if (rc == TL_OK && log) {
        size_t got = 0;
        rc = tl_session_log(s, log, log_cap, &got);
    }
    const double t3 = trace ? now() : 0.0;
    tl_session_destroy(s);
    if (trace)
        fprintf(stderr, "[tl] local_search: create %.2f ms, run %.2f ms, tour+stats+log %.2f ms, destroy %.2f ms\n",
                t1 - t0, t2 - t1, t3 - t2, now() - t3);
    return rc;
    });
}

// ---- batched multi-start 2-opt (GA / multi-start populations) ----------------------------------

tl_status tl_two_opt_batch(tl_problem *p, int32_t algo, uint32_t *tours_inout, size_t batch, int64_t max_moves,
                           tl_stats *stats, float *lengths_out)
{
    return tl::guarded([&]() -> tl_status {
    if (!p || (!tours_inout && batch)) { set_error("tl_two_opt_batch: null argument"); return TL_ERR_INVALID; }
    if (algo != TL_ALGO_TWO_OPT_BEST && algo != TL_ALGO_TWO_OPT_BEST_CYCLIC) {
        set_error("tl_two_opt_batch: only TL_ALGO_TWO_OPT_BEST[_CYCLIC] is batched");
        return TL_ERR_UNSUPPORTED;
    }
    if (p->kind != PK_EUC_F32) {
        set_error("tl_two_opt_batch: needs an F32_EXACT coordinate problem");
        return TL_ERR_UNSUPPORTED;
    }
    if (batch > 0xffffffffull) { set_error("tl_two_opt_batch: batch too large"); return TL_ERR_INVALID; }
    // Two engines with identical results.  The CTA-per-tour kernel (k2_two_opt_batch.cu) keeps a tour
    // in one CTA's shared memory for its whole search and is the faster one wherever it applies
    // (1024 x 1000: 401 vs 451 ms; 128 x 1000: 70 vs 109 ms, profiles/r02k_batch_phases.txt).  K2-pop
    // (k2_two_opt_pop.cu) schedules single work items of single scans over every warp of the GPU from
    // tour records in global memory: it takes over when a tour does not fit one CTA's shared memory
    // (n > ~12 000, up to 65 535).  TL_BATCH_ENGINE=pop|cta overrides.
    const bool fits_cta = two_opt_batch_smem_bytes(p->n) <= (size_t)kBatchMaxSmem;
    bool use_pop = !fits_cta && two_opt_pop_supported(p->n);
    if (const char *ev = getenv("TL_BATCH_ENGINE")) {
        if (!strcmp(ev, "cta")) use_pop = false;
        if (!strcmp(ev, "pop")) {
            if (!two_opt_pop_supported(p->n)) {
                set_error("tl_two_opt_batch: TL_BATCH_ENGINE=pop does not support n = %u", p->n);
                return TL_ERR_UNSUPPORTED;
            }
            use_pop = true;
        }
    }
    if (!use_pop && p->n >= 4 && two_opt_batch_smem_bytes(p->n) > (size_t)kBatchMaxSmem) {
        set_error("tl_two_opt_batch: n = %u is beyond both batched engines (65 535 cities); use tl_local_search per tour", p->n);
        return TL_ERR_UNSUPPORTED;
    }
    if (stats) memset(stats, 0, sizeof *stats);
    if (batch == 0) return TL_OK;
    for (size_t b = 0; b < batch; ++b) {
        if (!tour_is_permutation(tours_inout + b * p->n, p->n)) {
            set_error("tl_two_opt_batch: tour %zu is not a permutation of 0..%u", b, p->n - 1);
            return TL_ERR_INVALID;
        }
    }
    tl_ctx *c = p->ctx;
    DeviceGuard g(c);
    const uint32_t n = p->n;
    const bool cyclic = algo == TL_ALGO_TWO_OPT_BEST_CYCLIC;
    const bool fast = p->metric == Metric::F32_FAST;
    const uint64_t launches0 = c->launches;
    DevBuf<uint32_t> d_t;
    DevBuf<float> d_len;
    DevBuf<unsigned char> d_ctr;
    const size_t ctr_bytes = std::max(two_opt_batch_counter_bytes(), sizeof(PopCounters));
    if (d_t.alloc(batch * n) != cudaSuccess || d_len.alloc(batch) != cudaSuccess ||
        d_ctr.alloc(ctr_bytes) != cudaSuccess) {
        set_error("tl_two_opt_batch: device allocation failed");
        return TL_ERR_NOMEM;
    }
    struct { unsigned long long moves, scans; unsigned int next_tour, unconverged; unsigned long long phase[5]; } h{};
    cudaEvent_t e0, e1;
    TL_CUDA_TRY(cudaEventCreate(&e0));
    TL_CUDA_TRY(cudaEventCreate(&e1));
    cudaStream_t st = c->stream;
    cudaError_t e = cudaMemcpyAsync(d_t.p, tours_inout, batch * n * 4, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_ctr.p, 0, ctr_bytes, st);
    if (e == cudaSuccess) e = cudaEventRecord(e0, st);
    DevBuf<Pt> d_recs;
    DevBuf<unsigned char> d_items;
    DevBuf<PopTourCtl> d_ctl;
    DevBuf<int32_t> d_bands;
    DevBuf<unsigned long long> d_queue;
    if (e == cudaSuccess && n >= 4 && max_moves != 0) { // n < 4: nothing to scan, tours come back unchanged
        const float margin = screen_margin(p);
        if (use_pop) {
            std::vector<int32_t> bf;
            int chunk = 0;
            const int nitems = two_opt_pop_geometry(n, cyclic, &chunk, bf);
            const uint32_t npad = two_opt_pop_npad(n);
            const uint32_t qcap = two_opt_pop_queue_cap(batch);
            if (d_recs.alloc(batch * npad) != cudaSuccess || d_ctl.alloc(batch) != cudaSuccess ||
                d_bands.alloc(bf.size()) != cudaSuccess || d_queue.alloc(qcap) != cudaSuccess) {
                cudaGetLastError();
                cudaEventDestroy(e0);
                cudaEventDestroy(e1);
                set_error("tl_two_opt_batch: device allocation failed (%.1f MB of tour records)", batch * npad * 16.0 / 1e6);
                return TL_ERR_NOMEM;
            }
            e = cudaMemcpyAsync(d_bands.p, bf.data(), bf.size() * 4, cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st); // bf is a local
            launch_pop_init(p->d_xy, d_t.p, n, npad, batch, cyclic, fast, d_recs.p, d_ctl.p,
                            reinterpret_cast<PopCounters *>(d_ctr.p), d_queue.p, qcap, c->sm_count, st);
            launch_two_opt_pop(d_recs.p, d_ctl.p, reinterpret_cast<PopCounters *>(d_ctr.p), n, npad, batch, cyclic,
                               max_moves, margin, chunk, (int)bf.size() - 1, nitems, d_bands.p, d_queue.p, qcap,
                               fast, c->sm_count, st);
            launch_pop_extract(d_recs.p, n, npad, batch, d_t.p, c->sm_count, st);
            c->launches += 3;
        } else {
            int ccfg = 0;
            const int cl = two_opt_batch_cluster_plan(n, batch, c->sm_count, &ccfg);
            const int cfg = cl > 1 ? ccfg : two_opt_batch_config(n, batch, c->sm_count);
            int nitems = 0;
            const std::vector<unsigned char> items = two_opt_batch_item_table(n, cyclic, cfg, cl, &nitems);
            if (d_items.alloc(items.size()) != cudaSuccess) {
                cudaGetLastError();
                cudaEventDestroy(e0);
                cudaEventDestroy(e1);
                set_error("tl_two_opt_batch: device allocation failed");
                return TL_ERR_NOMEM;
            }
            e = cudaMemcpyAsync(d_items.p, items.data(), items.size(), cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st); // `items` is a local
            if (e != cudaSuccess) {
                // reported below
            } else if (cl > 1) { // fewer tours than CTA slots: a thread-block cluster per tour
                e = launch_two_opt_batch_cluster(cfg, cl, p->d_xy, d_t.p, n, batch, cyclic, max_moves, margin, d_items.p,
                                                 nitems, d_ctr.p, fast, st);
            } else {
                const int grid = two_opt_batch_grid(cfg, n, batch, c->sm_count, fast, margin >= 0.0f);
                launch_two_opt_batch(cfg, p->d_xy, d_t.p, n, batch, cyclic, max_moves, margin, d_items.p, nitems, d_ctr.p,
                                     grid, fast, st);
            }
            c->launches++;
        }
        if (e == cudaSuccess) e = cudaGetLastError();
    }
    if (e == cudaSuccess && lengths_out) {
        launch_tour_lengths_f32(p->d_xy, nullptr, n, d_t.p, batch, fast, false, d_len.p, c->sm_count, st);
        c->launches++;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaEventRecord(e1, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(tours_inout, d_t.p, batch * n * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && lengths_out) e = cudaMemcpyAsync(lengths_out, d_len.p, batch * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h, d_ctr.p, sizeof h, cudaMemcpyDeviceToHost, st);
    PopCounters hp{};
    if (e == cudaSuccess && use_pop) e = cudaMemcpyAsync(&hp, d_ctr.p, sizeof hp, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    float ms = 0.f;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (e != cudaSuccess) { set_error("tl_two_opt_batch: %s", cudaGetErrorString(e)); return TL_ERR_CUDA; }
    if (hp.error) { set_error("tl_two_opt_batch: work queue overrun (a worker stalled)"); return TL_ERR_CUDA; }
    if (!use_pop && h.phase[4] && getenv("TL_BATCH_PHASES")) // -DTL_TIMELINE builds only
        fprintf(stderr, "[tl] batch phases per CTA step (kcycles): scan %.2f  wait-cta %.2f  exchange %.2f  apply %.2f  (%llu CTA steps)\n",
                h.phase[0] / 1e3 / h.phase[4], h.phase[1] / 1e3 / h.phase[4], h.phase[2] / 1e3 / h.phase[4],
                h.phase[3] / 1e3 / h.phase[4], h.phase[4]);
    if (stats) {
        const uint64_t nn = n;
        const uint64_t pairs = n < 4 ? 0 : (cyclic ? nn * (nn - 3) / 2 : (nn - 3) * (nn - 2) / 2);
        // n < 4 mirrors the single-tour session: one empty scan per tour, converged
        stats->passes = n < 4 ? batch : h.scans;
        stats->moves = h.moves;
        stats->evals = stats->passes * pairs;
        stats->launches = c->launches - launches0;
        stats->device_ms = ms;
        stats->converged = h.unconverged == 0 ? 1 : 0;
        stats->path_used = TL_PATH_RECOMPUTE;
    }
    return TL_OK;
    });
}

} // extern "C"
