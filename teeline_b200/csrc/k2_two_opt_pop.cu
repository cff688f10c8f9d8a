// k2_two_opt_pop.cu -- K2-pop: best-improvement 2-opt over a POPULATION of tours, scheduled at
// work-item granularity over the whole GPU (multi-start / GA population, BASELINE config 5).
//
// Semantics per tour: exactly the Mode B loop of k2_two_opt.cu / k2_two_opt_batch.cu
// (SURVEY.md Appendix A "2-opt B"; neighbourhood of src/tsp/two_opt.rs:17,29,34; cyclic variant
// two-opt-algo.ts:71-99): argmin of the exact f32 delta, strict '<' from 0, lowest (i,j) on ties,
// reverse p[i+1..=j], until no move improves.
//
// Why a second batched kernel: k2_two_opt_batch.cu gives every tour ONE CTA for its whole search.
// That is ideal while tours >= CTA slots, but a population sharded over the 8 GPUs of a box leaves
// 128 tours for 148 SMs: SMs idle, CTA slots quantise (512 tours = 3.46 CTAs per SM run as 4), and
// the measured per-tour cost rises 0.395 -> 0.558 ms (profiles/r02c_batch_scaling_1gpu.json).  Here
// the unit of scheduling is one WORK ITEM of one scan of one tour (a band of 32*R diagonals x a
// chunk of rows, as in the single-tour kernels), and every warp of a persistent grid is a worker:
//
//   Open scans sit in a FIFO of tour ids (a ring in global memory; entry e carries its generation
//   e+1, so a slot is valid exactly when its generation matches -- no flags, no clearing).
//   worker loop:  slot = atomicAdd(head, 1); entry = slot / items_per_scan, item = slot % items_per_scan
//                 -> wait until entry `entry` has been published (workers that run ahead of the queue
//                 already sit on the entry they will serve, so a re-armed scan starts without any
//                 discovery latency) -> stage the item's tour-ordered records from global memory (L2)
//                 into the warp's shared-memory tile -> walk the diagonals (one new distance per
//                 move, screened like K2-B) -> publish the warp's best candidate with ONE 64-bit
//                 atomicMin on (order-preserving delta bits << 32 | i*n + j) -> count the item done.
//   the worker that completes the LAST item of a scan applies the move: reverses the segment in
//   the tour's global records (apply.cuh), bumps the move count and pushes the tour back
//   into the FIFO (or retires it when nothing improves / the move budget is spent).
//   (First version: per-tour tickets that idle workers polled, 32 tours per round -- the polling
//   storm of ~3500 warps on a few KB of L2 made a step take 340 us; profiles/r02d.)
//
// No CTA-wide or grid-wide barrier exists anywhere: tours advance independently, workers flow to
// whichever tours have open items, and the tail of the search (a few unconverged tours) still
// spreads each scan over ~60 warps instead of one SM.  Determinism: the argmin key carries the
// rank (i,j), and a scan's items are all complete before its move is applied, so the result does
// not depend on which worker did what.
//
// Roofline: FP32 issue, ~0.5 B/move of L2 traffic for staging; 15 flop/move as for K2-B.
#include "host.hpp"
#include "policy.cuh"
#include "apply.cuh"

#include <math_constants.h>

#include <algorithm>
#include <cstdlib>
#include <type_traits>
#include <vector>

namespace tl {

namespace {

constexpr int R = kPopR;
constexpr int BW = 32 * R;          // diagonals per band
constexpr int WARPS = kPopWarps;
// per-warp tile for items of at most `ti` rows: positions i0 .. i0+cnt and i0+K0 .. i0+K0+cnt+BW
__host__ __device__ constexpr int warp_pts(int ti) { return (ti + 1) + (ti + BW + 1); }

template <int N, typename F>
__device__ __forceinline__ void static_for(F &&f)
{
    if constexpr (N > 0) {
        static_for<N - 1>(f);
        f(std::integral_constant<int, N - 1>{});
    }
}

constexpr unsigned long long kNoKey = ~0ull;

// order-preserving map of an f32 onto u32 (smaller float -> smaller key)
__device__ __forceinline__ uint32_t f32_order_key(float f)
{
    const uint32_t b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float f32_from_order_key(uint32_t k)
{
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t *p)
{
    uint32_t v;
    asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_volatile_u32(uint32_t *p, uint32_t v)
{
    asm volatile("st.volatile.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_volatile_u64(const unsigned long long *p)
{
    unsigned long long v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_volatile_u64(unsigned long long *p, unsigned long long v)
{
    asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// tour-ordered records of every tour + control block (one launch, before the engine)
template <bool FAST>
__global__ void __launch_bounds__(256)
    pop_init_kernel(const float2 *__restrict__ xy, const uint32_t *__restrict__ tours, uint32_t n, uint32_t npad,
                    uint32_t batch, int cyclic, Pt *__restrict__ recs, PopTourCtl *__restrict__ ctl,
                    PopCounters *__restrict__ ctr, unsigned long long *__restrict__ queue, uint32_t qcap)
{
    // the FIFO starts with every tour's first scan open, in tour order; the rest of the ring is zero
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < qcap; q += gridDim.x * blockDim.x)
        queue[q] = q < batch ? (((unsigned long long)(q + 1u) << 32) | q) : 0ull;
    for (uint32_t b = blockIdx.x; b < batch; b += gridDim.x) {
        const uint32_t *tour = tours + (size_t)b * n;
        Pt *pts = recs + (size_t)b * npad;
        for (uint32_t q = threadIdx.x; q < npad; q += blockDim.x) {
            Pt p;
            if (q < n || (q == n && cyclic)) {
                const uint32_t c = tour[q == n ? 0 : q];
                const uint32_t cp = tour[q == 0 ? n - 1 : q - 1];
                const float2 a = __ldg(&xy[c]), bp = __ldg(&xy[cp]);
                p.x = a.x;
                p.y = a.y;
                p.city = (int32_t)c;
                p.sp = (q == 0 && !cyclic) ? 0.0f : dist_f32<FAST>(bp.x, bp.y, a.x, a.y);
            } else {
                p.x = 0.0f;
                p.y = 0.0f;
                p.city = -1;
                p.sp = -CUDART_INF_F; // delta = new - (s_i + -inf) = +inf: never selected
            }
            pts[q] = p;
        }
        if (threadIdx.x == 0) {
            PopTourCtl c{};
            c.best = kNoKey;
            ctl[b] = c;
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        ctr->moves = 0;
        ctr->scans = 0;
        ctr->active = batch;
        ctr->unconverged = 0;
        ctr->head = 0;
        ctr->tail = batch;
        ctr->error = 0;
    }
}

__global__ void __launch_bounds__(256)
    pop_extract_kernel(const Pt *__restrict__ recs, uint32_t n, uint32_t npad, uint32_t batch, uint32_t *__restrict__ tours)
{
    for (uint32_t b = blockIdx.x; b < batch; b += gridDim.x)
        for (uint32_t q = threadIdx.x; q < n; q += blockDim.x)
            tours[(size_t)b * n + q] = (uint32_t)recs[(size_t)b * npad + q].city;
}

__device__ __forceinline__ int find_band_pop(const int32_t *band_first, int nbands, int item)
{
    int lo = 0, hi = nbands - 1; // largest b with band_first[b] <= item
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (band_first[mid] <= item)
            lo = mid;
        else
            hi = mid - 1;
    }
    return lo;
}

// The worker that finished the last item of a scan: apply the move (or retire the tour) and re-arm.
template <bool FAST>
__device__ __noinline__ void pop_finish_scan(Pt *pts, PopTourCtl *ct, PopCounters *ctr, uint32_t tour, uint32_t n,
                                             long long max_moves, unsigned long long *queue, uint32_t qmask, int lane)
{
    __threadfence(); // acquire side of the done counter: every worker's atomicMin is visible
    unsigned long long key = 0;
    if (lane == 0) key = atomicAdd(&ct->best, 0ull); // L2 read of the reduced candidate
    key = __shfl_sync(0xffffffffu, key, 0);
    bool retire = false, converged = false;
    if (key == kNoKey) {
        retire = converged = true;
    } else {
        const uint32_t pair = (uint32_t)key;
        const uint32_t mi = pair / n, mj = pair - mi * n;
        reverse_segment_inplace(EucPol<FAST, true>{pts}, mi, mj, nullptr, (uint32_t)lane, 32u);
        __threadfence(); // every lane's stores before lane 0 re-opens the tour
        __syncwarp();
    }
    if (lane == 0) {
        const uint32_t moves = ld_volatile_u32(&ct->moves) + (converged ? 0u : 1u);
        st_volatile_u32(&ct->moves, moves);
        atomicAdd(&ctr->scans, 1ull);
        if (!converged) {
            atomicAdd(&ctr->moves, 1ull);
            if (max_moves >= 0 && (long long)moves >= max_moves) retire = true;
        }
        if (retire) {
            if (!converged) atomicAdd(&ctr->unconverged, 1u);
            st_volatile_u32(&ct->state, converged ? 1u : 2u);
            __threadfence();
            atomicSub(&ctr->active, 1u);
        } else {
            ct->best = kNoKey;
            ct->done = 0u;
            __threadfence(); // the reversed records and the re-armed counters before the scan re-opens
            const unsigned long long e = atomicAdd(&ctr->tail, 1ull);
            st_volatile_u64(&queue[(uint32_t)e & qmask], ((unsigned long long)((uint32_t)e + 1u) << 32) | tour);
        }
    }
    __syncwarp();
}

struct WalkResult {
    float best;
    uint32_t bi, bj;
    int improved;
};

// One work item: rows i0 .. i0+cnt-1 of a band, this lane's R diagonals starting at lane_k0.  srow
// and scl point into the warp's staged tile (scl = the lane's window into the column records).
// (best, bi, bj) in: the tour's best so far; out: this lane's best, `improved` if it found a better one.
template <bool FAST, bool SCREEN>
__device__ __noinline__ WalkResult pop_walk_item(const Pt *__restrict__ srow, const Pt *__restrict__ scl, int cnt,
                                                 int i0, int lane_k0, uint32_t n, int cyclic, float screen_margin,
                                                 float best, uint32_t bi, uint32_t bj)
{
    bool improved = false; // this worker found something better than what it started from
    float thr = SCREEN ? __fadd_rn(best, screen_margin) : best; // best + margin

    float E[R], wx[R], wy[R], ws[R];
    {
        const Pt rp0 = srow[0];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const Pt c = scl[r];
            E[r] = SCREEN ? dist_f32_screen(rp0.x, rp0.y, c.x, c.y) : dist_f32<FAST>(rp0.x, rp0.y, c.x, c.y);
            const Pt w = scl[r + 1];
            wx[r] = w.x;
            wy[r] = w.y;
            ws[r] = w.sp;
        }
    }
    auto step = [&](auto Uc, int tau) {
        constexpr int U = decltype(Uc)::value;
        const Pt rp = srow[tau + 1];                // (x,y) of i+1 and s_i, warp broadcast
        const Pt nx = scl[tau + R + 1];             // next window point
        float dl[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int ph = (r + U) % R;
            const float en = SCREEN ? dist_f32_screen(rp.x, rp.y, wx[ph], wy[ph])
                                    : dist_f32<FAST>(rp.x, rp.y, wx[ph], wy[ph]);
            const float cur_e = __fadd_rn(rp.sp, ws[ph]);
            const float nw = __fadd_rn(E[r], en);
            dl[r] = __fsub_rn(nw, cur_e);
            E[r] = en;
        }
        float m = dl[0];
#pragma unroll
        for (int r = 1; r < R; ++r) m = fminf(m, dl[r]);
        if (m <= thr) { // rare near a local optimum
            const uint32_t i = (uint32_t)(i0 + tau);
            const Pt pi = srow[tau];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const uint32_t j = i + (uint32_t)(lane_k0 + r);
                float d = dl[r];
                if (SCREEN) { // exact re-evaluation from the staged records
                    const Pt pj = scl[tau + r], pj1 = scl[tau + r + 1];
                    const float e1 = dist_f32<FAST>(pi.x, pi.y, pj.x, pj.y);
                    const float e2 = dist_f32<FAST>(rp.x, rp.y, pj1.x, pj1.y);
                    d = __fsub_rn(__fadd_rn(e1, e2), __fadd_rn(rp.sp, pj1.sp));
                }
                const bool excluded = cyclic && i == 0 && j == n - 1; // both edges share p_0
                if (d < 0.0f && !excluded && better_2opt(d, i, j, best, bi, bj)) {
                    best = d;
                    bi = i;
                    bj = j;
                    improved = true;
                    thr = SCREEN ? __fadd_rn(best, screen_margin) : best;
                }
            }
        }
        wx[U] = nx.x;
        wy[U] = nx.y;
        ws[U] = nx.sp;
    };
    int t = 0;
#pragma unroll 1
    for (; t + R <= cnt; t += R) static_for<R>([&](auto Uc) { step(Uc, t + decltype(Uc)::value); });
    static_for<R>([&](auto Uc) {
        if (t + decltype(Uc)::value < cnt) step(Uc, t + decltype(Uc)::value);
    });
    return WalkResult{best, bi, bj, improved ? 1 : 0};
}

// 16-byte asynchronous copy global -> shared that bypasses L1 (the records are rewritten by other SMs)
__device__ __forceinline__ void cp_async_cg16(void *dst_smem, const void *src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

struct ItemGeom {
    int K0, i0, cnt;
};
__device__ __forceinline__ ItemGeom item_geom(const int32_t *s_band, int nbands, int item, int chunk, int jmax)
{
    const int b = find_band_pop(s_band, nbands, item);
    ItemGeom g;
    g.K0 = 2 + b * BW;
    g.i0 = (item - s_band[b]) * chunk;
    g.cnt = min(chunk, jmax - g.K0 + 1 - g.i0); // rows 0 .. H-1 exist on the band's first diagonal
    return g;
}
// the item's tour-ordered records into a tile: rows i0 .. i0+cnt, columns i0+K0 .. i0+K0+cnt+BW
__device__ __forceinline__ void stage_item_async(const Pt *pts, const ItemGeom &g, Pt *srow, Pt *scol, int lane)
{
    for (int t = lane; t < g.cnt + 1; t += 32) cp_async_cg16(srow + t, pts + g.i0 + t);
    for (int t = lane; t < g.cnt + BW + 1; t += 32) cp_async_cg16(scol + t, pts + g.i0 + g.K0 + t);
    cp_async_commit();
}

// Every round trip to L2 that a worker makes between two items is exposed latency (measured: ~23 us
// of overhead per 64-row item against ~11 us of arithmetic when every item paid a claim, a queue
// look-up, a synchronous staging, two fences and a completion count; profiles/r02h).  So a worker
// claims a GROUP of consecutive slots with one atomic, publishes once per (group, tour), and
// prefetches the next item's tile with cp.async into the other half of its double buffer while it
// walks the current one.  The group size follows the amount of open work: many items per claim
// while there are many more open items than workers, one when few tours are left and each scan
// should spread over as many workers as possible.
template <bool FAST, bool SCREEN>
__global__ void __launch_bounds__(WARPS * 32, kPopMinBlocks)
    two_opt_pop_kernel(Pt *__restrict__ recs, PopTourCtl *__restrict__ ctl, PopCounters *__restrict__ ctr, uint32_t n,
                       uint32_t npad, uint32_t batch, int cyclic, long long max_moves, float screen_margin, int chunk,
                       int nbands, int nitems, const int32_t *__restrict__ band_first_g,
                       unsigned long long *__restrict__ queue, uint32_t qmask, int gmax)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wp = warp_pts(chunk);
    Pt *tile0 = reinterpret_cast<Pt *>(smem_raw) + (size_t)warp * 2 * wp; // two tiles per warp
    __shared__ int32_t s_band[kPopBandCap];
    for (int t = threadIdx.x; t <= nbands; t += blockDim.x) s_band[t] = __ldg(&band_first_g[t]);
    __syncthreads(); // the only CTA-wide barrier: from here on every warp is an independent worker

    const int jmax = cyclic ? (int)n - 1 : (int)n - 2;
    const uint32_t nworkers = gridDim.x * WARPS;

    for (;;) {
        // ---- claim a group of consecutive slots of the FIFO of open scans ------------------------------
        unsigned long long slot0 = 0;
        int G = 1;
        if (lane == 0) {
            // open work per worker, halved: leaves the other half to even out the end of the queue
            const unsigned long long open_items = (unsigned long long)ld_volatile_u32(&ctr->active) * (unsigned)nitems;
            G = (int)min((unsigned long long)gmax, max(1ull, open_items / (2ull * nworkers)));
            slot0 = atomicAdd(&ctr->head, (unsigned long long)G);
        }
        slot0 = __shfl_sync(0xffffffffu, slot0, 0);
        G = __shfl_sync(0xffffffffu, G, 0);

        unsigned long long cur_entry = ~0ull;
        uint32_t tour = 0;
        Pt *pts = nullptr;
        float best = 0.0f;
        uint32_t bi = 0xffffffffu, bj = 0xffffffffu;
        bool improved = false;
        unsigned int k_done = 0;
        int buf = 0;
        bool staged = false; // the current item's tile is already on its way (prefetched)
        bool quit = false;

        // publish what this worker found for `tour` and count its k_done items; the worker that
        // completes the scan applies the move
        auto flush = [&]() {
            if (k_done == 0) return;
            const bool any_improved = __any_sync(0xffffffffu, improved);
            warp_argmin_2opt(best, bi, bj);
            PopTourCtl *ct = &ctl[tour];
            unsigned int prev = 0;
            if (lane == 0) {
                // (a worker that found nothing better than what it started from has nothing to publish.
                // Tried: publishing from the walk's slow path the moment a lane improves -- the early
                // scans of a random tour then hammer one address per tour; 128 tours 128 -> 151 ms.)
                if (any_improved)
                    atomicMin(&ct->best, ((unsigned long long)f32_order_key(best) << 32) | (unsigned long long)(bi * n + bj));
                __threadfence(); // candidate before the count
                prev = atomicAdd(&ct->done, k_done);
            }
            prev = __shfl_sync(0xffffffffu, prev, 0);
            if (prev + k_done == (unsigned int)nitems)
                pop_finish_scan<FAST>(pts, ct, ctr, tour, n, max_moves, queue, qmask, lane);
            k_done = 0;
        };

        for (int gi = 0; gi < G; ++gi) {
            const unsigned long long slot = slot0 + (unsigned long long)gi;
            const unsigned long long entry = slot / (unsigned long long)nitems;
            const int item = (int)(slot - entry * (unsigned long long)nitems);
            if (entry != cur_entry) {
                flush();
                // wait for the entry to be published (a worker ahead of the queue waits on its own entry)
                const uint32_t gen = (uint32_t)entry + 1u;
                int status = 0; // 1 = got the tour, 2 = no tours left, 3 = ring overrun
                if (lane == 0) {
                    const unsigned long long *q = &queue[(uint32_t)entry & qmask];
                    for (unsigned int spin = 0; status == 0; ++spin) {
                        const unsigned long long w = ld_volatile_u64(q);
                        const uint32_t g = (uint32_t)(w >> 32);
                        if (g == gen) {
                            tour = (uint32_t)w;
                            status = 1;
                        } else if (g != 0u && (int32_t)(g - gen) > 0) {
                            status = 3; // the ring wrapped past an unread entry (a worker stalled for ~qcap scans)
                        } else {
                            if ((spin & 7u) == 7u && ld_volatile_u32(&ctr->active) == 0u) status = 2;
                            if (status == 0 && spin > 4u) __nanosleep(spin < 64u ? 100u : 400u);
                        }
                    }
                }
                status = __shfl_sync(0xffffffffu, status, 0);
                tour = __shfl_sync(0xffffffffu, tour, 0);
                if (status != 1) {
                    if (status == 3 && lane == 0) {
                        st_volatile_u32(&ctr->error, 1u);
                        st_volatile_u32(&ctr->active, 0u);
                    }
                    quit = true;
                    break;
                }
                __threadfence(); // the claim orders this worker's record loads after the publisher's release
                cur_entry = entry;
                pts = recs + (size_t)tour * npad;
                staged = false;
                // The running best of this worker starts at the tour's best so far (what other workers
                // have already published for this scan): a candidate has to beat -- or tie with, the
                // rank decides in the atomicMin -- that value anyway, and the rare exact re-evaluation
                // path of the walk is only entered for deltas within the screen margin of it.
                best = 0.0f;
                bi = bj = 0xffffffffu;
                improved = false;
            }
            // re-read the tour's published best before every item (the load overlaps the staging)
            unsigned long long seen = kNoKey;
            if (lane == 0) seen = ld_volatile_u64(&ctl[tour].best);
            const ItemGeom g = item_geom(s_band, nbands, item, chunk, jmax);
            Pt *srow = tile0 + buf * wp, *scol = srow + (chunk + 1);
            if (!staged) stage_item_async(pts, g, srow, scol, lane);
            seen = __shfl_sync(0xffffffffu, seen, 0);
            if (seen != kNoKey) {
                const float pb = f32_from_order_key((uint32_t)(seen >> 32));
                const uint32_t pair = (uint32_t)seen, pi_ = pair / n, pj_ = pair - pi_ * n;
                // somebody else's better candidate is only a stronger filter: ours would lose the
                // atomicMin anyway, so dropping it (and its `improved` flag) changes nothing
                if (better_2opt(pb, pi_, pj_, best, bi, bj)) {
                    best = pb;
                    bi = pi_;
                    bj = pj_;
                }
            }
            // prefetch the next item of the group when it belongs to the same scan
            staged = false;
            if (gi + 1 < G && item + 1 < nitems) {
                const ItemGeom gn = item_geom(s_band, nbands, item + 1, chunk, jmax);
                Pt *nrow = tile0 + (buf ^ 1) * wp;
                cp_async_wait_all(); // (the current tile first: wait_group counts whole groups)
                __syncwarp();
                stage_item_async(pts, gn, nrow, nrow + (chunk + 1), lane);
                staged = true;
            } else {
                cp_async_wait_all();
                __syncwarp();
            }
            // the walk itself lives in its own function: its register allocation (the R-point window,
            // the carried distances) must not compete with the scheduler's state
            const WalkResult wr = pop_walk_item<FAST, SCREEN>(srow, scol + lane * R, g.cnt, g.i0, g.K0 + lane * R, n,
                                                              cyclic, screen_margin, best, bi, bj);
            best = wr.best;
            bi = wr.bi;
            bj = wr.bj;
            improved = improved || wr.improved != 0;
            ++k_done;
            buf ^= 1;
            __syncwarp(); // everyone is done with this tile before it is refilled two items later
        }
        if (quit) break;
        flush();
    }
}

} // namespace

size_t two_opt_pop_smem_bytes(int chunk) { return (size_t)WARPS * 2 * warp_pts(chunk) * sizeof(Pt); }

cudaError_t two_opt_pop_configure()
{
    const int bytes = (int)std::min<size_t>(two_opt_pop_smem_bytes(kPopMaxTI), 200 * 1024);
    cudaError_t e = cudaFuncSetAttribute(two_opt_pop_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(two_opt_pop_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(two_opt_pop_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    return e;
}

uint32_t two_opt_pop_npad(uint32_t n) { return n + (uint32_t)BW + (uint32_t)kPopMaxTI + 8u; }

// Work decomposition of one scan (the same for every tour): bands of BW diagonals x chunks of rows.
// Returns the item count; band_first (nbands + 1 entries) is uploaded by the caller.
int two_opt_pop_geometry(uint32_t n, int cyclic, int *chunk_out, std::vector<int32_t> &band_first)
{
    const int jmax = cyclic ? (int)n - 1 : (int)n - 2;
    const int nbands = ((int)n - 3 + BW - 1) / BW;
    int chunk = kPopTI;
    if (const char *ev = getenv("TL_POP_CHUNK")) chunk = std::max(8, std::min(kPopMaxTI, atoi(ev)));
    band_first.assign(nbands + 1, 0);
    for (int b = 0; b < nbands; ++b) {
        const int H = jmax - (2 + b * BW) + 1;
        band_first[b + 1] = band_first[b] + (H + chunk - 1) / chunk;
    }
    *chunk_out = chunk;
    return band_first[nbands];
}

bool two_opt_pop_supported(uint32_t n)
{
    const int nbands = ((int)n - 3 + BW - 1) / BW;
    return n >= 4 && n <= 65535u && nbands + 1 <= kPopBandCap;
}

// ring capacity: a power of two, at least 4 entries per tour (at most one is ever open per tour)
uint32_t two_opt_pop_queue_cap(uint64_t batch)
{
    uint32_t cap = 1u << 16;
    while ((uint64_t)cap < 4 * batch) cap <<= 1;
    return cap;
}

void launch_pop_init(const float2 *xy, const uint32_t *tours, uint32_t n, uint32_t npad, uint64_t batch, int cyclic,
                     bool fast, Pt *recs, PopTourCtl *ctl, PopCounters *ctr, unsigned long long *queue, uint32_t qcap,
                     int sm_count, cudaStream_t st)
{
    const unsigned grid = (unsigned)std::min<uint64_t>(batch, (uint64_t)sm_count * 8);
    if (fast)
        pop_init_kernel<true><<<grid, 256, 0, st>>>(xy, tours, n, npad, (uint32_t)batch, cyclic, recs, ctl, ctr, queue, qcap);
    else
        pop_init_kernel<false><<<grid, 256, 0, st>>>(xy, tours, n, npad, (uint32_t)batch, cyclic, recs, ctl, ctr, queue, qcap);
}

void launch_pop_extract(const Pt *recs, uint32_t n, uint32_t npad, uint64_t batch, uint32_t *tours, int sm_count,
                        cudaStream_t st)
{
    const unsigned grid = (unsigned)std::min<uint64_t>(batch, (uint64_t)sm_count * 8);
    pop_extract_kernel<<<grid, 256, 0, st>>>(recs, n, npad, (uint32_t)batch, tours);
}

void launch_two_opt_pop(Pt *recs, PopTourCtl *ctl, PopCounters *ctr, uint32_t n, uint32_t npad, uint64_t batch,
                        int cyclic, long long max_moves, float screen_margin, int chunk, int nbands, int nitems,
                        const int32_t *band_first, unsigned long long *queue, uint32_t qcap, bool fast, int sm_count,
                        cudaStream_t st)
{
    const bool screen = fast && screen_margin >= 0.0f;
    auto kern = screen ? two_opt_pop_kernel<true, true>
                : fast ? two_opt_pop_kernel<true, false>
                       : two_opt_pop_kernel<false, false>;
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WARPS * 32, two_opt_pop_smem_bytes(chunk));
    if (per_sm < 1) per_sm = 1;
    // no more workers than there can ever be open items
    const uint64_t want = (batch * (uint64_t)nitems + WARPS - 1) / WARPS;
    const unsigned grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)sm_count * per_sm, want));
    int gmax = 16; // items per claim at most (TL_POP_GROUP overrides; 1 = one claim per item)
    if (const char *ev = getenv("TL_POP_GROUP")) gmax = std::max(1, std::min(64, atoi(ev)));
    kern<<<grid, WARPS * 32, two_opt_pop_smem_bytes(chunk), st>>>(recs, ctl, ctr, n, npad, (uint32_t)batch, cyclic, max_moves,
                                                             screen_margin, chunk, nbands, nitems, band_first, queue,
                                                             qcap - 1u, gmax);
}

} // namespace tl
