// k2_two_opt_batch.cu -- K2-batch: independent best-improvement 2-opt searches over a batch of
// start tours (multi-start / GA population, BASELINE config 5).
//
// Semantics per tour: exactly the Mode B loop of k2_two_opt.cu (SURVEY.md Appendix A "2-opt B",
// neighbourhood of src/tsp/two_opt.rs:17,29,34; cyclic variant two-opt-algo.ts:71-99):
//     loop { (delta,i,j) = argmin over the neighbourhood, strict '<' from 0, lowest (i,j) on ties;
//            none -> stop;  reverse p[i+1..=j] }
//
// How: ONE CTA PER TOUR, the whole search runs inside one kernel launch.  The tour lives in
// shared memory as tour-ordered 16-byte records (x, y, city, entering-edge length), so a scan
// touches no global memory at all; CTAs pull tours from a global ticket counter (tours converge
// after different move counts, so a static split would leave SMs idle at the tail).
// Scan: diagonals k = j - i again (one new distance per move), cut like the single-tour kernel
// into bands of 32*R diagonals x chunks of rows; the tail of a band (rows on which only a prefix of
// its diagonals is still inside the triangle) is tiled with quarter-warp pieces instead (BatchItem).
// The work items of one scan -- a table built on the host -- are handed to the CTA's warps through a
// shared-memory ticket (an item is ~60 rows, so a warp's last item costs a few percent of a scan,
// whatever n is).  A lane owns R consecutive diagonals and walks its rows with the (R+1)-point
// register window of k2_two_opt.cu, reading the records straight from shared memory: the lanes of a
// warp (of a quarter-warp in a tail item) sit on the same row i (broadcast LDS.128 of the row point)
// and on windows R records apart (odd R => conflict-free LDS.128).  The threshold below which a
// screened delta is re-evaluated exactly is shared by all threads working on the tour.
// Argmin: (delta, i, j) lexicographic as ONE 64-bit key, two REDUX and one shared-memory atomicMin per
// warp -- independent of which thread saw a candidate first.  Apply: the in-place reversal of
// apply.cuh on the shared-memory records.
//
// CLUSTER PER TOUR (two_opt_batch_cluster_kernel): when the batch has fewer tours than the GPU has
// CTA slots -- BASELINE config 5 sharded over 8 GPUs leaves 128 tours for 148 SMs -- a tour is a
// thread-block cluster of 2, 4 or 8 CTAs on different SMs.  Every CTA keeps its own replica of the
// tour records in shared memory; the work items of a scan are handed out from ONE ticket in the
// rank-0 CTA's shared memory (atom.shared::cluster over DSMEM, the next ticket fetched while the
// current item runs), so a CTA that shares its SM with other tours simply takes fewer items; the
// CTAs exchange their candidates with remote shared-memory stores and ONE cluster barrier per step,
// take the same lexicographic minimum and apply the same reversal to their replicas.  SMs freed by
// converged tours speed up the remaining ones (their CTAs get the issue slots), and the last tours
// run on several SMs instead of one -- which is what bounds strong scaling of a fixed population.
//
// Roofline: FP32 issue, ~0 bytes per move (the only global traffic is n x 4 B in and out per
// tour).  Algorithmic work 15 flop/move as for the single-tour recompute kernel.
#include "kernels.cuh"
#include "policy.cuh"
#include "apply.cuh"

#include <cooperative_groups.h>
#include <math_constants.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <type_traits>
#include <vector>

namespace tl {

namespace {

constexpr int R = kBatchR;
constexpr int BW = 32 * R; // diagonals per band

template <int N, typename F>
__device__ __forceinline__ void static_for(F &&f)
{
    if constexpr (N > 0) {
        static_for<N - 1>(f);
        f(std::integral_constant<int, N - 1>{});
    }
}

struct BatchCounters {
    unsigned long long moves, scans;
    unsigned int next_tour;
    unsigned int unconverged;
    // -DTL_TIMELINE builds: SM clock cycles summed over the CTAs' steps -- [0] warp 0 in the item loop,
    // [1] waiting for the CTA's other warps, [2] candidate exchange + cluster barrier, [3] apply, [4] steps
    unsigned long long phase[5];
};

#ifdef TL_TIMELINE
__device__ __forceinline__ unsigned long long gtime_b() { return (unsigned long long)clock64(); } // SM cycles
#define TL_PH(k) do { if (tid == 0) { const unsigned long long t_ = gtime_b(); ph[k] += t_ - tph; tph = t_; } } while (0)
#else
#define TL_PH(k) do { } while (0)
#endif

namespace cg = cooperative_groups;

// One work item of a scan (built on the host, batch_items below): four quarter-warp pieces that walk
// `cnt` rows together.  Quarter q (lanes 8q .. 8q+7) starts at row r0[q] on the diagonals k0[q] + 5*(lane & 7) + r.
// A full-width item has r0[q] equal and k0[q] = K0 + 40 q; the TAIL of a band -- the rows on which only a
// prefix of its 160 diagonals still lies inside the triangle -- is tiled with 40-row x 40-diagonal pieces
// instead, four pieces (of any bands) per item, so that a band costs ~3 k cells beyond the triangle
// instead of 12.8 k (18 % of a 1000-city scan with full-width rows).
struct __align__(16) BatchItem {
    int32_t k0[4];
    int32_t r0[4];
    int32_t cnt, pad[3];
};
constexpr int QD = 8 * R; // diagonals (and rows) of a quarter-warp piece

__device__ __forceinline__ void load_item(const BatchItem *__restrict__ items, int item, int lane, int &k0, int &r0, int &cnt)
{
    const int4 a = __ldg(reinterpret_cast<const int4 *>(items + item));
    const int4 b = __ldg(reinterpret_cast<const int4 *>(items + item) + 1);
    const int q = lane >> 3;
    k0 = (q == 0 ? a.x : q == 1 ? a.y : q == 2 ? a.z : a.w) + (lane & 7) * R;
    r0 = q == 0 ? b.x : q == 1 ? b.y : q == 2 ? b.z : b.w;
    cnt = __ldg(&items[item].cnt);
}

// tour-ordered records of one tour in shared memory (same layout and padding rules as build_pts_kernel)
template <bool FAST>
__device__ __forceinline__ void stage_tour(Pt *pts, const float2 *__restrict__ xy, const uint32_t *tour, uint32_t n,
                                           uint32_t npad, int cyclic, int tid, int nthreads)
{
    for (uint32_t q = tid; q < npad; q += nthreads) {
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
}

// One work item walked by one warp.
// SCREEN: as in k2_two_opt.cu -- the walk evaluates deltas with the screening distance and
// re-evaluates exactly (from the shared-memory records) whenever a candidate comes within the
// rigorous margin of the best known delta.  `shared_best` is the best exact delta any thread of the
// tour's CTA(s) has published in this scan (bit pattern of a non-positive float; more negative =
// larger as unsigned): a thread that only sees mediocre candidates stops paying for exact
// re-evaluations as soon as ANY thread has found a better one.  It only filters what is re-evaluated
// -- a candidate above (another candidate's exact delta + margin) cannot be the minimum nor tie with
// it -- so the result does not depend on when a thread sees an update.  publish(bits) is called with
// every new thread-best.
template <bool FAST, bool SCREEN, class Publish>
__device__ __forceinline__ void scan_item(const Pt *pts, uint32_t n, int cyclic, int k0, int r_begin, int cnt,
                                          float screen_margin, const volatile unsigned int *shared_best, Publish &&publish,
                                          float &best, uint32_t &bi, uint32_t &bj, float &thr)
{
    // k0: first diagonal of this lane; r_begin: its first row (equal across the warp for a full-width item)
    const Pt *srow = pts + r_begin;
    const Pt *scol = pts + r_begin + k0;

    float E[R], wx[R], wy[R], ws[R];
    {
        const Pt rp0 = srow[0];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const Pt c = scol[r];
            E[r] = SCREEN ? dist_f32_screen(rp0.x, rp0.y, c.x, c.y) : dist_f32<FAST>(rp0.x, rp0.y, c.x, c.y);
            const Pt w = scol[r + 1];
            wx[r] = w.x;
            wy[r] = w.y;
            ws[r] = w.sp;
        }
    }
    auto refresh = [&]() {
        const float cb = __uint_as_float(*shared_best);
        thr = fminf(thr, SCREEN ? __fadd_rn(cb, screen_margin) : cb);
    };
    auto step = [&](auto Uc, int tau) {
        constexpr int U = decltype(Uc)::value;
        const Pt rp = srow[tau + 1];     // (x,y) of i+1 and s_i: one address per warp (per quarter in a tail item)
        const Pt nx = scol[tau + R + 1]; // next window point
        float dl[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int ph = (r + U) % R;
            const float en = SCREEN ? dist_f32_screen(rp.x, rp.y, wx[ph], wy[ph])
                                    : dist_f32<FAST>(rp.x, rp.y, wx[ph], wy[ph]);
            const float cur = __fadd_rn(rp.sp, ws[ph]);
            const float nw = __fadd_rn(E[r], en);
            dl[r] = __fsub_rn(nw, cur);
            E[r] = en;
        }
        float m = dl[0];
#pragma unroll
        for (int r = 1; r < R; ++r) m = fminf(m, dl[r]);
        if (m <= thr) { // rare once any thread of the tour has seen a good candidate
            const Pt pi = srow[tau];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                if (!(dl[r] <= thr)) continue; // above the margin of a known candidate: cannot win or tie
                const uint32_t ii = (uint32_t)(r_begin + tau), jj = ii + (uint32_t)(k0 + r);
                float d = dl[r];
                if (SCREEN) { // exact re-evaluation from the shared-memory records
                    const Pt pj = scol[tau + r], pj1 = scol[tau + r + 1];
                    const float e1 = dist_f32<FAST>(pi.x, pi.y, pj.x, pj.y);
                    const float e2 = dist_f32<FAST>(rp.x, rp.y, pj1.x, pj1.y);
                    d = __fsub_rn(__fadd_rn(e1, e2), __fadd_rn(rp.sp, pj1.sp));
                }
                // the cyclic neighbourhood excludes (0, n-1): both edges share p_0
                const bool excluded = cyclic && ii == 0 && jj == n - 1;
                // items are not visited in (i,j) order: full lexicographic compare
                if (d < 0.0f && !excluded && better_2opt(d, ii, jj, best, bi, bj)) {
                    best = d;
                    bi = ii;
                    bj = jj;
                    thr = fminf(thr, SCREEN ? __fadd_rn(best, screen_margin) : best);
                    publish(__float_as_uint(d));
                }
            }
        }
        wx[U] = nx.x;
        wy[U] = nx.y;
        ws[U] = nx.sp;
    };
    int t = 0;
    refresh();
#pragma unroll 1
    for (; t + R <= cnt; t += R) {
        static_for<R>([&](auto Uc) { step(Uc, t + decltype(Uc)::value); });
        refresh();
    }
    static_for<R>([&](auto Uc) {
        if (t + decltype(Uc)::value < cnt) step(Uc, t + decltype(Uc)::value);
    });
}

// The step's argmin as ONE 64-bit key: high word = ~bits(delta) (delta < 0: a more negative delta has the
// larger bit pattern, so its complement is smaller; "no move" is all ones), low word = i * n + j, the
// candidate's rank in the reference's scan order (n < 65536).  The minimum key is the lexicographic
// (delta, i, j) minimum.  A warp reduces with two REDUX instructions and its lane 0 issues one
// shared-memory atomicMin -- no shuffle trees, no second reduction stage, no serial warp.
constexpr unsigned long long kNoMove = ~0ull;

__device__ __forceinline__ unsigned long long warp_min_key(float best, uint32_t bi, uint32_t bj, uint32_t n)
{
    const unsigned int hi = ~__float_as_uint(best); // best == 0.0f (no candidate) -> 0xffffffff
    const unsigned int whi = __reduce_min_sync(0xffffffffu, hi);
    const unsigned int lo = (bi != 0xffffffffu && hi == whi) ? bi * n + bj : 0xffffffffu;
    const unsigned int wlo = __reduce_min_sync(0xffffffffu, lo);
    return ((unsigned long long)whi << 32) | wlo;
}

// MAXT / MINB: launch bounds of one configuration (kCfgs).
// Per step: every warp pulls work items from a shared-memory ticket that is never reset (scan s owns
// the tickets [s * (nitems + nwarps), ...): every warp ends a scan with exactly one failed fetch),
// atomicMin of the warp keys into s_key[s & 1], ONE barrier, everyone decodes the move and applies
// it, a second barrier; the slots of scan s are re-armed for scan s + 2 behind that barrier.
template <bool FAST, bool SCREEN, int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB)
    two_opt_batch_kernel(const float2 *__restrict__ xy, uint32_t *__restrict__ tours, uint32_t n, uint32_t batch,
                         int cyclic, long long max_moves, float screen_margin, const BatchItem *__restrict__ items,
                         int nitems, BatchCounters *__restrict__ ctr)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Pt *pts = reinterpret_cast<Pt *>(smem_raw);
    __shared__ unsigned long long s_key[2];
    __shared__ unsigned int s_tour, s_item, s_shared_best[2];

    const int tid = threadIdx.x, lane = tid & 31, nthreads = blockDim.x;
    const int nwarps = nthreads >> 5;
    const uint32_t npad = n + BW + 2;
    const unsigned int per_scan = (unsigned int)(nitems + nwarps); // tickets one scan consumes

    unsigned long long my_moves = 0, my_scans = 0;
    unsigned int my_unconverged = 0;
#ifdef TL_TIMELINE
    unsigned long long ph[5] = {0, 0, 0, 0, 0};
#endif

    for (;;) {
        __syncthreads(); // previous tour fully written back; s_tour free
        if (tid == 0) s_tour = atomicAdd(&ctr->next_tour, 1u);
        __syncthreads();
        const uint32_t b = s_tour;
        if (b >= batch) break;
        uint32_t *tour = tours + (size_t)b * n;

        stage_tour<FAST>(pts, xy, tour, n, npad, cyclic, tid, nthreads);
        if (tid == 0) {
            s_item = 0;
            s_shared_best[0] = s_shared_best[1] = 0u;
            s_key[0] = s_key[1] = kNoMove;
        }
        __syncthreads();

        long long moves = 0;
        bool converged = false;
        unsigned int scan_no = 0;
#ifdef TL_TIMELINE
        unsigned long long tph = gtime_b();
#endif
        while (max_moves < 0 || moves < max_moves) {
            const unsigned int par = scan_no & 1u, base = scan_no * per_scan;
            float best = 0.0f;
            uint32_t bi = 0xffffffffu, bj = 0xffffffffu;
            float thr = SCREEN ? screen_margin : 0.0f; // best + margin

            for (;;) {
                unsigned int raw = 0;
                if (lane == 0) raw = atomicAdd(&s_item, 1u);
                int item = (int)(__shfl_sync(0xffffffffu, raw, 0) - base);
                if (item >= nitems) break;
                int k0, r0, cnt;
                load_item(items, item, lane, k0, r0, cnt);
                scan_item<FAST, SCREEN>(pts, n, cyclic, k0, r0, cnt, screen_margin, &s_shared_best[par],
                                        [&](unsigned int bits) { atomicMax(&s_shared_best[par], bits); }, best, bi, bj,
                                        thr);
            }

            TL_PH(0);
            const unsigned long long wkey = warp_min_key(best, bi, bj, n);
            if (lane == 0 && wkey != kNoMove) atomicMin(&s_key[par], wkey);
            __syncthreads();
            TL_PH(1);
            const unsigned long long key = s_key[par];
            TL_PH(2);
            my_scans += (tid == 0);
            ++scan_no;
            if (key == kNoMove) {
                converged = true;
                break;
            }
            const uint32_t rank = (uint32_t)key, mi = rank / n, mj = rank - mi * n;
            reverse_segment_inplace(EucPol<FAST>{pts}, mi, mj, nullptr, (uint32_t)tid, (uint32_t)nthreads);
            ++moves;
            __syncthreads();
            if (tid == 0) { // every thread has read s_key[par]; scan_no + 1 uses the other slots
                s_key[par] = kNoMove;
                s_shared_best[par] = 0u;
            }
            TL_PH(3);
#ifdef TL_TIMELINE
            if (tid == 0) ph[4] += 1;
#endif
        }
        my_moves += (tid == 0) ? (unsigned long long)moves : 0ull;
        my_unconverged += (tid == 0 && !converged);

        for (uint32_t q = tid; q < n; q += nthreads) tour[q] = (uint32_t)pts[q].city;
    }
    if (tid == 0) {
        if (my_moves) atomicAdd(&ctr->moves, my_moves);
        if (my_scans) atomicAdd(&ctr->scans, my_scans);
        if (my_unconverged) atomicAdd(&ctr->unconverged, my_unconverged);
#ifdef TL_TIMELINE
        for (int k = 0; k < 5; ++k) atomicAdd(&ctr->phase[k], ph[k]);
#endif
    }
}

constexpr int kMaxCluster = 8;

// A thread-block cluster per tour (see the header).  Shared state that peers touch over DSMEM:
//   rank 0's s_ticket / s_tour; every CTA's s_ckey[parity][rank] and s_shared_best[parity].
// Per step: items from rank 0's ticket; the warps' keys meet in the CTA's own s_key[parity] (shared
// memory has no native 64-bit min, and a remote one is not an option: local CAS loop), one CTA
// barrier, the CTA's key is STORED into slot [parity][rank] of every CTA, ONE cluster barrier, every
// CTA takes the minimum of the csize slots, decodes the same move and applies it to its replica.
template <bool FAST, bool SCREEN, int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB)
    two_opt_batch_cluster_kernel(const float2 *__restrict__ xy, uint32_t *__restrict__ tours, uint32_t n, uint32_t batch,
                                 int cyclic, long long max_moves, float screen_margin,
                                 const BatchItem *__restrict__ items, int nitems, BatchCounters *__restrict__ ctr)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Pt *pts = reinterpret_cast<Pt *>(smem_raw);
    __shared__ unsigned long long s_key[2];               // [scan parity]: this CTA's warps
    __shared__ unsigned long long s_ckey[2][kMaxCluster]; // [scan parity][rank]: every CTA's key of a step
    __shared__ unsigned int s_tour, s_ticket;
    __shared__ unsigned int s_shared_best[2]; // [scan parity]

    cg::cluster_group cluster = cg::this_cluster();
    const unsigned int rank = cluster.block_rank(), csize = cluster.num_blocks();
    const int tid = threadIdx.x, lane = tid & 31, nthreads = blockDim.x;
    const int nwarps = nthreads >> 5;
    const uint32_t npad = n + BW + 2;
    const unsigned int per_scan = (unsigned int)nitems + csize * (unsigned int)nwarps; // tickets one scan consumes
    unsigned int *ticket0 = cluster.map_shared_rank(&s_ticket, 0);
    const unsigned int *tour0 = cluster.map_shared_rank(&s_tour, 0);

    unsigned long long my_moves = 0, my_scans = 0;
    unsigned int my_unconverged = 0;
#ifdef TL_TIMELINE
    unsigned long long ph[5] = {0, 0, 0, 0, 0};
#endif

    for (;;) {
        cluster.sync(); // every CTA is done with the previous tour (and with rank 0's s_tour / s_ticket)
        if (rank == 0 && tid == 0) {
            s_tour = atomicAdd(&ctr->next_tour, 1u);
            s_ticket = 0u;
        }
        if (tid == 0) {
            s_shared_best[0] = s_shared_best[1] = 0u;
            s_key[0] = s_key[1] = kNoMove;
        }
        cluster.sync();
        const uint32_t b = *tour0;
        if (b >= batch) break;
        uint32_t *tour = tours + (size_t)b * n;
        stage_tour<FAST>(pts, xy, tour, n, npad, cyclic, tid, nthreads); // every CTA its own replica
        __syncthreads();

        long long moves = 0;
        bool converged = false;
        unsigned int scan_no = 0;
#ifdef TL_TIMELINE
        unsigned long long tph = gtime_b();
#endif
        while (max_moves < 0 || moves < max_moves) {
            const unsigned int par = scan_no & 1u, base = scan_no * per_scan;
            float best = 0.0f;
            uint32_t bi = 0xffffffffu, bj = 0xffffffffu;
            float thr = SCREEN ? screen_margin : 0.0f;
            // lane 0 holds the raw ticket; it is broadcast only when the item is needed, so the remote
            // atomic of the NEXT item is in flight while the current one runs
            auto fetch_raw = [&]() { return lane == 0 ? atomicAdd(ticket0, 1u) : 0u; };
            auto as_item = [&](unsigned int raw) { return (int)(__shfl_sync(0xffffffffu, raw, 0) - base); };
            auto publish = [&](unsigned int bits) {
                // a new CTA-wide best is pushed to the peers too (rare: ~log(moves) times per scan)
                if (atomicMax(&s_shared_best[par], bits) < bits)
                    for (unsigned int r = 0; r < csize; ++r)
                        if (r != rank) atomicMax(cluster.map_shared_rank(&s_shared_best[par], r), bits);
            };
            int item = as_item(fetch_raw());
            while (item < nitems) {
                const unsigned int next_raw = fetch_raw();
                int k0, r0, cnt;
                load_item(items, item, lane, k0, r0, cnt);
                scan_item<FAST, SCREEN>(pts, n, cyclic, k0, r0, cnt, screen_margin, &s_shared_best[par], publish, best,
                                        bi, bj, thr);
                item = as_item(next_raw);
            }

            TL_PH(0);
            const unsigned long long wkey = warp_min_key(best, bi, bj, n);
            if (lane == 0 && wkey != kNoMove) atomicMin(&s_key[par], wkey);
            __syncthreads();
            TL_PH(1);
            if ((unsigned int)tid < csize) *cluster.map_shared_rank(&s_ckey[par][rank], tid) = s_key[par];
            cluster.sync(); // release/acquire: every CTA's key (and every ticket fetch of this scan) has landed
            TL_PH(2);
            unsigned long long key = s_ckey[par][0];
            for (unsigned int r = 1; r < csize; ++r) key = min(key, s_ckey[par][r]);
            my_scans += (rank == 0 && tid == 0);
            ++scan_no;
            if (key == kNoMove) {
                converged = true;
                break;
            }
            const uint32_t mrank = (uint32_t)key, mi = mrank / n, mj = mrank - mi * n;
            reverse_segment_inplace(EucPol<FAST>{pts}, mi, mj, nullptr, (uint32_t)tid, (uint32_t)nthreads);
            ++moves;
            __syncthreads();
            // slot `par` is next used by scan_no + 1 (two scans on), which no CTA can start before this
            // one has passed the next cluster barrier
            if (tid == 0) {
                s_key[par] = kNoMove;
                s_shared_best[par] = 0u;
            }
            TL_PH(3);
#ifdef TL_TIMELINE
            if (tid == 0) ph[4] += 1;
#endif
        }
        if (rank == 0) {
            my_moves += (tid == 0) ? (unsigned long long)moves : 0ull;
            my_unconverged += (tid == 0 && !converged);
            for (uint32_t q = tid; q < n; q += nthreads) tour[q] = (uint32_t)pts[q].city;
        }
    }
    cluster.sync(); // no CTA leaves while a peer may still read its shared memory
#ifdef TL_TIMELINE
    if (tid == 0)
        for (int k = 0; k < 5; ++k) atomicAdd(&ctr->phase[k], ph[k]);
#endif
    if (rank == 0 && tid == 0) {
        if (my_moves) atomicAdd(&ctr->moves, my_moves);
        if (my_scans) atomicAdd(&ctr->scans, my_scans);
        if (my_unconverged) atomicAdd(&ctr->unconverged, my_unconverged);
    }
}

} // namespace

size_t two_opt_batch_smem_bytes(uint32_t n) { return (size_t)(n + BW + 2) * sizeof(Pt); }
size_t two_opt_batch_counter_bytes() { return sizeof(BatchCounters); }

namespace {

// Launch configurations (threads per tour, resident CTAs per SM).  A tour is always ONE CTA; what
// changes is how many threads work on it.  With >= ~1000 tours per GPU the smallest CTAs fill the
// machine (7 x 148 = 1036 tours in flight); when the batch is sharded over several GPUs, or the
// population is small, fewer tours are in flight and each one gets more threads, up to a whole SM,
// so that the GPU stays full (BASELINE config 5 on 8 GPUs: 128 tours per GPU).
struct BatchCfg {
    int threads, minb;
};
constexpr BatchCfg kCfgs[] = {{128, 7}, {256, 4}, {256, 3}, {512, 2}, {1024, 1}};
constexpr int kNumCfgs = (int)(sizeof(kCfgs) / sizeof(kCfgs[0]));
constexpr size_t kSmemPerSM = 200 * 1024; // shared memory the resident CTAs of one SM may use together

bool cfg_fits(int c, uint32_t n) { return two_opt_batch_smem_bytes(n) * kCfgs[c].minb <= kSmemPerSM; }

// The work items of one scan for `threads` threads working on a tour (all CTAs of a cluster together):
// ~16 (small CTAs) .. 2 (1024 threads) full-width items per warp (measured: profiles/r01n_batch_scaling.txt;
// an item costs a fixed prologue, so big CTAs on a short scan take longer items; at least 8 rows), then the
// bands' tails as quarter-warp pieces, four to an item (BatchItem above).
std::vector<BatchItem> batch_items(uint32_t n, int cyclic, int threads)
{
    const int jmax = cyclic ? (int)n - 1 : (int)n - 2;
    const int nbands = ((int)n - 3 + BW - 1) / BW; // diagonals k = 2 .. n-2 in bands of BW
    struct Piece { int k0, r0, cnt; };
    std::vector<Piece> pieces;
    long long per_warp = threads <= 128 ? 16 : threads <= 256 ? 8 : threads <= 512 ? 4 : threads <= 1024 ? 2 : 3;
    if (const char *ev = getenv("TL_BATCH_IPW")) per_warp = std::max(1, atoi(ev));
    const long long target = per_warp * (threads / 32); // items per scan to aim for
    long long full_rows = 0, all_rows = 0;
    for (int b = 0; b < nbands; ++b) all_rows += jmax - (2 + b * BW) + 1;
    // rows of a tail piece: no longer than a full-width item is going to be (many threads on a short scan)
    const int prow = (int)std::min<long long>(QD, std::max<long long>(8, (all_rows + target - 1) / target));
    for (int b = 0; b < nbands; ++b) {
        const int K0 = 2 + b * BW, H = jmax - K0 + 1; // H rows on the band's first diagonal, H - d on diagonal K0 + d
        const int Hf = std::max(0, H - (BW - 1));     // rows on which all BW diagonals are inside the triangle
        full_rows += Hf;
        for (int row0 = Hf; row0 < H; row0 += prow)
            for (int q = 0; q < 4; ++q)
                if (row0 + q * QD <= H - 1) pieces.push_back({K0 + q * QD, row0, std::min(prow, H - row0)});
    }
    const int tail_items = (int)(pieces.size() + 3) / 4;
    const long long want = std::max<long long>(1, target - tail_items);
    const int chunk = (int)std::max<long long>(8, (full_rows + want - 1) / want);
    std::vector<BatchItem> items;
    for (int b = 0; b < nbands; ++b) {
        const int K0 = 2 + b * BW, H = jmax - K0 + 1, Hf = std::max(0, H - (BW - 1));
        for (int r = 0; r < Hf; r += chunk) {
            BatchItem it{};
            for (int q = 0; q < 4; ++q) {
                it.k0[q] = K0 + q * QD;
                it.r0[q] = r;
            }
            it.cnt = std::min(chunk, Hf - r);
            items.push_back(it);
        }
    }
    for (size_t p0 = 0; p0 < pieces.size(); p0 += 4) {
        BatchItem it{};
        for (int q = 0; q < 4; ++q) {
            if (p0 + q < pieces.size()) {
                it.k0[q] = pieces[p0 + q].k0;
                it.r0[q] = pieces[p0 + q].r0;
                it.cnt = std::max(it.cnt, pieces[p0 + q].cnt);
            } else { // an empty quarter: every cell beyond the triangle (padding records, delta = +inf)
                it.k0[q] = jmax + 1;
                it.r0[q] = 0;
            }
        }
        items.push_back(it);
    }
    // longest items first: the ticket hands the short ones out last, which evens out the end of a scan
    std::stable_sort(items.begin(), items.end(), [](const BatchItem &a, const BatchItem &b) { return a.cnt > b.cnt; });
    return items;
}

using BatchKernel = void (*)(const float2 *, uint32_t *, uint32_t, uint32_t, int, long long, float, const BatchItem *, int,
                             BatchCounters *);

template <int T, int MINB>
BatchKernel pick_variant(bool fast, bool screen)
{
    if (fast && screen) return two_opt_batch_kernel<true, true, T, MINB>;
    if (fast) return two_opt_batch_kernel<true, false, T, MINB>;
    return two_opt_batch_kernel<false, false, T, MINB>;
}

template <int T, int MINB>
BatchKernel pick_cluster_variant(bool fast, bool screen)
{
    if (fast && screen) return two_opt_batch_cluster_kernel<true, true, T, MINB>;
    if (fast) return two_opt_batch_cluster_kernel<true, false, T, MINB>;
    return two_opt_batch_cluster_kernel<false, false, T, MINB>;
}

// cluster kernels exist for the configurations that fill an SM with 1024 threads: 256 x 4, 512 x 2, 1024 x 1
BatchKernel pick_cluster_kernel(int cfg, bool fast, bool screen)
{
    switch (cfg) {
    case 1: return pick_cluster_variant<kCfgs[1].threads, kCfgs[1].minb>(fast, screen);
    case 3: return pick_cluster_variant<kCfgs[3].threads, kCfgs[3].minb>(fast, screen);
    default: return pick_cluster_variant<kCfgs[4].threads, kCfgs[4].minb>(fast, screen);
    }
}

BatchKernel pick_kernel(int cfg, bool fast, bool screen)
{
    switch (cfg) {
    case 0: return pick_variant<kCfgs[0].threads, kCfgs[0].minb>(fast, screen);
    case 1: return pick_variant<kCfgs[1].threads, kCfgs[1].minb>(fast, screen);
    case 2: return pick_variant<kCfgs[2].threads, kCfgs[2].minb>(fast, screen);
    case 3: return pick_variant<kCfgs[3].threads, kCfgs[3].minb>(fast, screen);
    default: return pick_variant<kCfgs[4].threads, kCfgs[4].minb>(fast, screen);
    }
}

} // namespace

cudaError_t two_opt_batch_configure()
{
    cudaError_t e = cudaSuccess;
    for (int c = 0; c < kNumCfgs && e == cudaSuccess; ++c)
        for (int v = 0; v < 3 && e == cudaSuccess; ++v)
            e = cudaFuncSetAttribute(pick_kernel(c, v > 0, v == 2), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     kBatchMaxSmem);
    for (int c : {1, 3, 4})
        for (int v = 0; v < 3 && e == cudaSuccess; ++v)
            e = cudaFuncSetAttribute(pick_cluster_kernel(c, v > 0, v == 2), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     kBatchMaxSmem);
    return e;
}

// The first configuration (fewest threads per tour) whose CTA slots the batch fills to >= 80 %;
// a batch too small for any of them takes the largest CTAs that fit.  TL_BATCH_CFG overrides (tests).
int two_opt_batch_config(uint32_t n, uint64_t batch, int sm_count)
{
    if (const char *ev = getenv("TL_BATCH_CFG")) {
        const int c = atoi(ev);
        if (c >= 0 && c < kNumCfgs && cfg_fits(c, n)) return c;
    }
    int last = -1;
    for (int c = 0; c < kNumCfgs; ++c) {
        if (!cfg_fits(c, n)) continue;
        last = c;
        if (batch * 5 >= (uint64_t)sm_count * kCfgs[c].minb * 4) return c;
    }
    return last < 0 ? kNumCfgs - 1 : last;
}

int two_opt_batch_grid(int cfg, uint32_t n, uint64_t batch, int sm_count, bool fast, bool screen)
{
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pick_kernel(cfg, fast, screen), kCfgs[cfg].threads,
                                                  two_opt_batch_smem_bytes(n));
    if (per_sm < 1) per_sm = 1;
    const uint64_t cap = (uint64_t)sm_count * per_sm;
    return (int)(batch < cap ? batch : cap);
}

// Which engine for a batch (measured at n = 1000, profiles/r02s_batch_cluster_timing.txt; S = SMs):
//   batch > 2 S      clusters of 2 x 256 threads, 4 CTAs per SM: S * 2 tours are resident and the rest
//                    queue behind them -- the dynamic hand-out of tours beats having every tour
//                    resident on 128 threads (1024 tours: 338 vs 358 ms; 512: 180 vs 205 ms)
//   S/2 < batch <= 2 S   one CTA per tour, 512 or 1024 threads (two_opt_batch_config): a cluster's
//                    barrier and remote ticket cost ~4.5 us per step, more than a second SM saves
//                    (128 tours: 50 ms against 57-62 ms with clusters of two)
//   batch <= S/2     1024-thread CTAs, 2 / 4 / 8 per tour: the SMs that would idle halve the steps of
//                    the few tours there are (64 tours: 31 vs 50 ms; 16 tours: 17 vs 50 ms)
// Returns the cluster size (1 = the CTA-per-tour kernel) and the CTA configuration in *cfg_out.
// TL_BATCH_CLUSTER=<1|2|4|8> and TL_BATCH_CLUSTER_CFG=<1|3|4> override (tests, tuning).
int two_opt_batch_cluster_plan(uint32_t n, uint64_t batch, int sm_count, int *cfg_out)
{
    if (batch == 0) return 1;
    int cl = 1;
    *cfg_out = 4;
    if (batch > 2ull * sm_count) {
        for (int c : {1, 3})
            if (cfg_fits(c, n)) {
                *cfg_out = c;
                cl = 2;
                break;
            }
    } else if (batch * 2 <= (uint64_t)sm_count) {
        while (cl < kMaxCluster && batch * (uint64_t)(cl * 2) <= (uint64_t)sm_count) cl *= 2;
    }
    if (const char *ev = getenv("TL_BATCH_CLUSTER")) {
        const int c = atoi(ev);
        if (c == 1 || c == 2 || c == 4 || c == 8) {
            if (c > 1 && cl == 1) // forced onto a batch the plan gives to single CTAs: the smallest CTAs that fit
                for (int k : {4, 3, 1})
                    if (cfg_fits(k, n)) *cfg_out = k;
            cl = c;
        }
    }
    if (const char *ev = getenv("TL_BATCH_CLUSTER_CFG")) {
        const int c = atoi(ev);
        if ((c == 1 || c == 3 || c == 4) && cfg_fits(c, n)) *cfg_out = c;
    }
    return cl;
}

// host copy of the work-item table of one scan for configuration `cfg` and clusters of `cl` CTAs
std::vector<unsigned char> two_opt_batch_item_table(uint32_t n, int cyclic, int cfg, int cl, int *nitems)
{
    const std::vector<BatchItem> items = batch_items(n, cyclic, kCfgs[cfg].threads * cl);
    *nitems = (int)items.size();
    std::vector<unsigned char> raw(items.size() * sizeof(BatchItem));
    memcpy(raw.data(), items.data(), raw.size());
    return raw;
}

cudaError_t launch_two_opt_batch_cluster(int cfg, int cl, const float2 *xy, uint32_t *tours, uint32_t n, uint64_t batch,
                                         int cyclic, long long max_moves, float screen_margin, const void *items,
                                         int nitems, void *counters, bool fast, cudaStream_t st)
{
    const bool screen = fast && screen_margin >= 0.0f;
    const int threads = kCfgs[cfg].threads;
    BatchKernel k = pick_cluster_kernel(cfg, fast, screen);
    cudaLaunchConfig_t lc = {};
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)cl;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    lc.attrs = attr;
    lc.numAttrs = 1;
    lc.blockDim = dim3((unsigned)threads);
    lc.dynamicSmemBytes = two_opt_batch_smem_bytes(n);
    lc.stream = st;
    lc.gridDim = dim3((unsigned)cl); // for the occupancy query
    int max_clusters = 0;
    cudaError_t e = cudaOccupancyMaxActiveClusters(&max_clusters, k, &lc);
    if (e != cudaSuccess) return e;
    if (max_clusters < 1) max_clusters = 1;
    const uint64_t nclusters = batch < (uint64_t)max_clusters ? batch : (uint64_t)max_clusters;
    lc.gridDim = dim3((unsigned)(nclusters * cl));
    return cudaLaunchKernelEx(&lc, k, xy, tours, n, (uint32_t)batch, cyclic, max_moves, screen_margin,
                              reinterpret_cast<const BatchItem *>(items), nitems,
                              reinterpret_cast<BatchCounters *>(counters));
}

void launch_two_opt_batch(int cfg, const float2 *xy, uint32_t *tours, uint32_t n, uint64_t batch, int cyclic,
                          long long max_moves, float screen_margin, const void *items, int nitems, void *counters,
                          int grid, bool fast, cudaStream_t st)
{
    const bool screen = fast && screen_margin >= 0.0f;
    const int threads = kCfgs[cfg].threads;
    pick_kernel(cfg, fast, screen)<<<grid, threads, two_opt_batch_smem_bytes(n), st>>>(
        xy, tours, n, (uint32_t)batch, cyclic, max_moves, screen_margin, reinterpret_cast<const BatchItem *>(items), nitems,
        reinterpret_cast<BatchCounters *>(counters));
}

} // namespace tl
