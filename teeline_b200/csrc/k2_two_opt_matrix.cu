// k2_two_opt_matrix.cu -- K2 "Mode B" scan, matrix-backed path (f32 or int32 distances in HBM).
//
// Same move space and argmin rule as k2_two_opt.cu.  Distances come from the n x ld matrix M,
// stored in SLOT order; the tour-ordered records cs[q] = (slot, entering-edge length, city) map
// tour positions to matrix slots.  The session lays M out in tour order (slot == position) when
// it starts and re-lays it whenever the tour has fragmented, so that walking a row of the
// (i,j) triangle reads a (nearly) contiguous run of a matrix row.
//
// Walk: diagonals k = j - i again, so d(p_i+1,p_j+1) of pair (i,j) is reused as d(p_i',p_j') of
// pair (i+1,j+1): ONE matrix element is loaded per move -- each element M[a][b] of the upper
// triangle is read exactly once per scan (4 algorithmic bytes per move).  Lane l owns the
// diagonals K0 + l + 32 r, r < R, so for fixed r the 32 lanes of a warp read 32 consecutive
// columns of one matrix row: a single 128-byte request when slot == position.  The (slot, s_j)
// pairs of the columns are staged per warp in shared memory (compacted to 8 bytes) and read with
// conflict-free 64-bit LDS; the loads of row step tau+D are issued when step tau is consumed (a
// D-deep register ring, rotated by unrolling) to keep enough bytes in flight for HBM.
//
// Roofline: HBM bandwidth, 4 B per move (DESIGN.md section 4).
#include "kernels.cuh"
#include "policy.cuh"
#include "apply.cuh"

#include <type_traits>

namespace tl {

namespace {

constexpr int R = kMatR;
constexpr int BW = kMatBW;
constexpr int TI = kMatTI;
constexpr int WARPS = kMatWarps;
constexpr int ROWS_CAP = TI + 1;      // positions i0 .. i0+cnt
constexpr int COLS_CAP = TI + BW + 1; // positions i0+K0 .. i0+K0+cnt+BW
constexpr int WARP_RECS = ROWS_CAP + COLS_CAP;
constexpr int D = kMatD;              // row steps of matrix loads kept in flight per thread

#ifdef TL_TIMELINE
// Step timeline (tuning builds only, -DTL_TIMELINE): globaltimer stamps of one fused step, folded
// into running sums by the last CTA.  tl_tmark: 0 = earliest CTA past griddep_wait, 1 = earliest
// scan end, 2 = latest scan end, 3 = end of the previous step.  tl_tacc: sums (ns) of
// [gap prev end -> first start, first scan end, last scan end, tail entry, reduced, reversed, done] + count.
__device__ unsigned long long tl_tmark_par[2][4] = {{~0ull, ~0ull, 0ull, 0ull}, {~0ull, ~0ull, 0ull, 0ull}}; // by step parity
__device__ unsigned long long tl_prev_done;
#define tl_tmark tl_tmark_par[tl_par]
__device__ unsigned long long tl_tacc[8];
__device__ unsigned long long tl_tcta[3][1024]; // per CTA of the latest step: past-wait time, scan-end time, SM id
__device__ __forceinline__ unsigned long long gtime()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define TL_MARK_MIN(k) do { if (threadIdx.x == 0) { const unsigned long long t_ = gtime(); atomicMin(&tl_tmark[k], t_); \
        if (blockIdx.x < 1024) { tl_tcta[k][blockIdx.x] = t_; if (k == 0) { unsigned sm_; asm("mov.u32 %0, %%smid;" : "=r"(sm_)); tl_tcta[2][blockIdx.x] = sm_; } } } } while (0)
#define TL_MARK_MAX(k) do { if (threadIdx.x == 0) atomicMax(&tl_tmark[k], gtime()); } while (0)
#else
#define TL_MARK_MIN(k) do { } while (0)
#define TL_MARK_MAX(k) do { } while (0)
#endif

template <int N, typename F>
__device__ __forceinline__ void static_for(F &&f)
{
    if constexpr (N > 0) {
        static_for<N - 1>(f);
        f(std::integral_constant<int, N - 1>{});
    }
}

// warp argmin that also carries the record's aux word (the winning pair's d(p_i, p_j), see below)
template <typename V>
__device__ __forceinline__ void warp_argmin_2opt_aux(V &d, uint32_t &i, uint32_t &j, uint32_t &aux)
{
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const V od = __shfl_xor_sync(0xffffffffu, d, off);
        const uint32_t oi = __shfl_xor_sync(0xffffffffu, i, off);
        const uint32_t oj = __shfl_xor_sync(0xffffffffu, j, off);
        const uint32_t oa = __shfl_xor_sync(0xffffffffu, aux, off);
        if (better_2opt(od, oi, oj, d, i, j)) { d = od; i = oi; j = oj; aux = oa; }
    }
}

constexpr int kBandCap = 1024; // band table entries kept in shared memory (n up to ~260k)

__device__ __forceinline__ int find_band_m(const int32_t *band_first, int nbands, int item)
{
    int lo = 0, hi = nbands - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (band_first[mid] <= item)
            lo = mid;
        else
            hi = mid - 1;
    }
    return lo;
}

// Matrix element at byte address rowbase + 4 * col: ONE IMAD.WIDE.U32 per load (the row base is
// formed once per row step).  Streaming: every element is used once per scan, keep it out of L1.
// With PIN (L2 residency experiment, the matrix is larger than L2 but a scan re-reads the same
// elements every step): rows whose SLOT is below pin_rows carry an L2 evict_last policy, every
// other load evict_first; the policy is chosen per row (warp-uniform).
template <typename V, bool PIN>
__device__ __forceinline__ V ld_elem(uint64_t rowbase, uint32_t col, uint64_t pol)
{
    uint64_t a;
    asm("mad.wide.u32 %0, %1, 4, %2;" : "=l"(a) : "r"(col), "l"(rowbase));
    int32_t v;
    if constexpr (PIN)
        asm("ld.global.nc.L1::no_allocate.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(v) : "l"(a), "l"(pol));
    else
        asm("ld.global.nc.L1::no_allocate.b32 %0, [%1];" : "=r"(v) : "l"(a));
    return Val<V>::from_bits(v);
}

// Tail of a fused step (last CTA only), out of line so that it does not weigh on the scan loop's
// register allocation: reduce the per-CTA records, reverse the segment, update the loop state.
template <typename V>
__device__ __noinline__ void fused_apply_tail_matrix(const V *__restrict__ M, uint32_t ld, Cs *__restrict__ cs,
                                                     const Best<V> *__restrict__ blockbest, Best<V> *red,
                                                     DevState *state, unsigned int *ticket,
                                                     tl_move *__restrict__ log, uint64_t log_cap,
                                                     const ShardComm &sc)
{
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#ifdef TL_TIMELINE
    const int tl_par = 0;
    const unsigned long long t_entry = gtime();
#endif
    // (ordering: thread 0's acq_rel ticket + the caller's __syncthreads; the records are read from L2)
    StateHeader hdr{};
    if (threadIdx.x == 0) hdr = load_state_header(state); // in flight with the candidate loads
    Best<V> v{(V)0, 0xffffffffu, 0xffffffffu, 0u};
    // all of this thread's candidate loads are issued before the first compare (one round trip)
    for (int c0 = threadIdx.x; c0 < (int)gridDim.x; c0 += 4 * blockDim.x) {
        int4 raw[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int c = c0 + u * (int)blockDim.x;
            raw[u] = c < (int)gridDim.x ? __ldcg(reinterpret_cast<const int4 *>(blockbest) + c)
                                        : make_int4(0, -1, -1, 0);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const Best<V> o{Val<V>::from_bits(raw[u].x), (uint32_t)raw[u].y, (uint32_t)raw[u].z, (uint32_t)raw[u].w};
            if (better_2opt(o.delta, o.i, o.j, v.delta, v.i, v.j)) v = o;
        }
    }
    warp_argmin_2opt_aux(v.delta, v.i, v.j, v.aux);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    v = red[0];
#pragma unroll
    for (int w = 1; w < WARPS; ++w) {
        const Best<V> o = red[w];
        if (better_2opt(o.delta, o.i, o.j, v.delta, v.i, v.j)) v = o;
    }
    if (sc.world > 1) { // sharded triangle: exchange the per-rank minima over NVLink (shard_exchange.cuh)
        __shared__ Best<V> s_peer[kMaxPeers];
        __shared__ int s_fail;
        __shared__ unsigned int s_step;
        if (threadIdx.x == 0) s_step = (unsigned int)hdr.h0.y + 1u;
        __syncthreads();
        v = shard_exchange_2opt(sc, v, s_step, s_peer, &s_fail);
        if (s_fail) {
            if (threadIdx.x == 0) {
                *ticket = 0u;
                state->error = 1;
                state->done = 1;
            }
            return;
        }
    }
    const bool found = v.i != 0xffffffffu;
#ifdef TL_TIMELINE
    const unsigned long long t_reduced = gtime();
#endif
    // integer metric: the record carries d(p_i, p_j), so the reversal needs no matrix loads
    if (found)
        reverse_segment_inplace(MatPol<V>{cs, M, ld}, v.i, v.j, nullptr, threadIdx.x, blockDim.x,
                                std::is_same<V, int32_t>::value, Val<V>::from_bits((int32_t)v.aux), v.delta);
#ifdef TL_TIMELINE
    __syncthreads();
    const unsigned long long t_reversed = gtime();
#endif
    if (threadIdx.x == 0) {
        *ticket = 0u;
        finish_best_step(state, hdr, found, (float)v.delta, v.i, v.j, log, log_cap);
#ifdef TL_TIMELINE
        const unsigned long long t_done = gtime();
        const unsigned long long t0 = tl_tmark[0];
        if (tl_prev_done) tl_tacc[0] += t0 - tl_prev_done;
        tl_tacc[1] += tl_tmark[1] - t0;
        tl_tacc[2] += tl_tmark[2] - t0;
        tl_tacc[3] += t_entry - t0;
        tl_tacc[4] += t_reduced - t0;
        tl_tacc[5] += t_reversed - t0;
        tl_tacc[6] += t_done - t0;
        tl_tacc[7] += 1;
        tl_tmark[0] = ~0ull; tl_tmark[1] = ~0ull; tl_tmark[2] = 0ull; tl_prev_done = t_done;
#endif
    }
}

template <typename V, bool PIN>
__global__ void __launch_bounds__(WARPS * 32, kMatMinBlocks)
    two_opt_scan_matrix_kernel(const V *__restrict__ M, uint32_t ld, Cs *__restrict__ cs, const ScanGeom g,
                               const int32_t *__restrict__ band_first_g, Best<V> *__restrict__ blockbest,
                               DevState *state, unsigned int *ticket, tl_move *__restrict__ log,
                               uint64_t log_cap, int fuse_apply, int pin_rows, int pf_rows, const __grid_constant__ ShardComm sc)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    griddep_launch_dependents(); // PDL, as in k2_two_opt.cu
#ifdef TL_TIMELINE
    const int tl_par = 0;
#endif
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // per-warp staging, four plain 32-bit arrays (conflict-free LDS.32): matrix slot and
    // entering-edge bits of the tile's row positions and of its column positions
    int32_t *srow_slot = reinterpret_cast<int32_t *>(smem_raw) + warp * (2 * WARP_RECS);
    int32_t *srow_sp = srow_slot + ROWS_CAP;
    int32_t *scol_slot = srow_sp + ROWS_CAP;
    int32_t *scol_sp = scol_slot + COLS_CAP;
    Best<V> *red = reinterpret_cast<Best<V> *>(smem_raw + (size_t)WARPS * WARP_RECS * sizeof(int2));

    uint64_t pol_keep = 0, pol_stream = 0;
    if constexpr (PIN) {
        asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol_keep));
        asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol_stream));
    }
    const uint32_t ld4 = ld * 4u; // row pitch in bytes

    // band table (geometry only): shared-memory copy, so that looking up a work item costs no
    // global round trips
    __shared__ int32_t s_band[kBandCap];
    const int32_t *band_first = band_first_g;
    if (g.nbands + 1 <= kBandCap) {
        for (int t = threadIdx.x; t <= g.nbands; t += blockDim.x) s_band[t] = __ldg(&band_first_g[t]);
        __syncthreads();
        band_first = s_band;
    }

    V best = (V)0;
    uint32_t bi = 0xffffffffu, bj = 0xffffffffu, baux = 0u;
    // this warp's static run of work items (geometry only, so it may be looked up before the wait)
    int u_lo = g.item_begin + (blockIdx.x * WARPS + warp) * g.run;
    int u_hi = min(u_lo + g.run, g.dyn_begin);
    int t_next = 0, tf_next = 0, tl_next = 0; // band of item u_lo, first item of that band and of the next one
    if (u_lo < u_hi) {
        t_next = find_band_m(band_first, g.nbands, u_lo);
        tf_next = band_first[t_next];
        tl_next = band_first[t_next + 1];
        // L2 prefetch of the first rows of this warp's item, issued BEFORE the grid dependency
        // resolves.  Programmatic dependent launch makes this CTA resident while the previous step
        // is still running down (its CTAs finish between 30 and 38 us) and while its last CTA
        // reduces the candidates and reverses the segment -- 6 us per step during which HBM would
        // otherwise idle.  The matrix itself never changes; the tour records read here may be
        // one move stale (the apply may be rewriting them), which can only make a prefetch useless,
        // never wrong: nothing read here is used after the wait.  One lane per row, one bulk
        // prefetch of the row's ~1 KB (contiguous whenever the columns still sit in one run).
        if (pf_rows > 0) {
            const int K0p = 2 + t_next * BW;
            const int r0 = (u_lo - tf_next) * g.chunk;
            const int r1 = min(r0 + (min(u_hi, tl_next) - u_lo) * g.chunk, g.jmax - K0p + 1);
            const int rows = min(pf_rows, r1 - r0 + 1); // + the row of E
            if (lane < rows) {
                const int rs = __ldcg(&cs[r0 + lane].slot);
                const int s0 = __ldcg(&cs[r0 + K0p + lane].slot), s1 = __ldcg(&cs[r0 + K0p + lane + BW - 1].slot);
                const size_t first = (size_t)(uint32_t)rs * ld + (uint32_t)min(s0, s1);
                const size_t last = (size_t)g.n * ld; // one past the matrix
                if (rs >= 0 && rs < g.n && first + BW + 4 <= last) {
                    const uint64_t a = (reinterpret_cast<uint64_t>(M) + first * sizeof(V)) & ~(uint64_t)15;
                    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a), "r"((uint32_t)(BW * sizeof(V) + 16)) : "memory");
                }
            }
        }
    }
    griddep_wait(); // the previous step's move is applied and visible from here on
    // "done" (grid-uniform: later launches of a finished search are no-ops) is only LOADED here; the
    // branch sits behind the first tile's staging loads so that the two round trips overlap.
    // Nothing but this warp's shared-memory staging is written before it.
    const int done_flag = *reinterpret_cast<const volatile int *>(&state->done);
    TL_MARK_MIN(0);
    // the items [dyn_begin, item_end) go to whichever warp asks first; the next ticket is always
    // requested before the current item is scanned, so its latency is hidden
    const bool has_dyn = g.dyn_begin < g.item_end;
    unsigned int tk = 0;
    if (has_dyn && !done_flag && lane == 0) tk = atomicAdd(ticket + 1, 1u);
    bool first = true;

    for (;;) {
        if (u_lo >= u_hi) { // run exhausted: take the next dynamic item
            if (!has_dyn) break;
            const int item = g.dyn_begin + (int)__shfl_sync(0xffffffffu, tk, 0);
            if (item >= g.item_end) break;
            if (lane == 0) tk = atomicAdd(ticket + 1, 1u);
            u_lo = item;
            u_hi = item + 1;
            first = false;
        }
        if (!first) {
            t_next = find_band_m(band_first, g.nbands, u_lo);
            tf_next = band_first[t_next];
            tl_next = band_first[t_next + 1];
        }
        first = false;
        // as many of the run's items as lie in this band are scanned as one piece
        const int q = min(u_hi, tl_next) - u_lo;
        const int b = t_next;
        const int cidx = u_lo - tf_next; // first row chunk within the band
        u_lo += q;
        const int K0 = 2 + b * BW;
        const int H = g.jmax - K0 + 1;
        const int r_begin = cidx * g.chunk;
        const int r_end = min(r_begin + q * g.chunk, H);
        const int ntiles = (r_end - r_begin + TI - 1) / TI;
        const int tile_rows = ntiles > 0 ? (r_end - r_begin + ntiles - 1) / ntiles : 0;

        for (int i0 = r_begin; i0 < r_end; i0 += tile_rows) {
            const int cnt = min(tile_rows, r_end - i0);
            __syncwarp();
            for (int t = lane; t < cnt + 1; t += 32) {
                const Cs c = cs[i0 + t];
                srow_slot[t] = c.slot;
                srow_sp[t] = c.sp_bits;
            }
            for (int t = lane; t < cnt + BW + 1; t += 32) {
                const Cs c = cs[i0 + K0 + t];
                scol_slot[t] = c.slot;
                scol_sp[t] = c.sp_bits;
            }
            if (done_flag) return;
            __syncwarp();

            // Lane l owns the diagonals k_r = K0 + l + 32 r.  Row step tau handles the pairs
            // (i0 + tau, i0 + tau + k_r): it needs E = d(p_i, p_j), which is the element the
            // previous row step loaded as ITS d(p_i+1, p_j+1), and en = d(p_i+1, p_j+1) from
            // matrix row slot(i+1) at the columns slot(j+1) = scol_slot[tau + 1 + l + 32 r].
            // ring[] is a ring of NB = D + 1 row buffers addressed with compile-time indices
            // (the loop is unrolled NB times), so nothing is ever copied: at step tau the
            // buffer tau-1 is E, tau is en, tau+1 .. tau+D-1 are in flight, and once the step
            // is computed the loads of step tau+D are issued into the (dead) buffer of E.
            // D * R independent 4-byte loads per thread stay in flight, which is what it takes
            // to cover HBM latency at 24 warps per SM (Little: ~40 KB per SM at 6.5 TB/s).
            constexpr int NB = D + 1;
            V ring[NB][R];
            auto issue = [&](auto Bc, int t) { // loads of row step t into ring[Bc]
                constexpr int bq = decltype(Bc)::value;
                const uint32_t slotn = (uint32_t)srow_slot[t + 1];
                uint64_t rowbase;
                asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(rowbase) : "r"(slotn), "r"(ld4), "l"(M));
                uint64_t pol = 0;
                if constexpr (PIN) pol = (int)slotn < pin_rows ? pol_keep : pol_stream;
                const int32_t *cslot = scol_slot + (t + 1 + lane);
#pragma unroll
                for (int r = 0; r < R; ++r) ring[bq][r] = ld_elem<V, PIN>(rowbase, (uint32_t)cslot[32 * r], pol);
            };
            issue(std::integral_constant<int, NB - 1>{}, -1); // E of row step 0
            static_for<D>([&](auto Dc) {
                constexpr int d = decltype(Dc)::value;
                if (d < cnt) issue(Dc, d);
            });
            auto step = [&](auto Sc, int tau) {
                constexpr int s = decltype(Sc)::value;
                constexpr int e = (s + NB - 1) % NB; // buffer of E; refilled with step tau + D
                const V si = Val<V>::from_bits(srow_sp[tau + 1]); // s_i
                const int32_t *csp = scol_sp + (tau + 1 + lane);
                V dl[R];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const V sj = Val<V>::from_bits(csp[32 * r]);
                    const V cur = Val<V>::add(si, sj);
                    const V nw = Val<V>::add(ring[e][r], ring[s][r]);
                    dl[r] = Val<V>::sub(nw, cur);
                }
                V m = dl[0];
#pragma unroll
                for (int r = 1; r < R; ++r) m = Val<V>::vmin(m, dl[r]);
                if (m <= best) { // rare: a move that may beat (or tie with) this thread's best
                    const uint32_t i = (uint32_t)(i0 + tau);
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const uint32_t j = i + (uint32_t)(K0 + lane + 32 * r);
                        const bool excluded = g.cyclic && i == 0 && j == (uint32_t)(g.n - 1);
                        // full (delta, i, j) order: work items are not visited in (i, j) order
                        if (!excluded && dl[r] < (V)0 && better_2opt(dl[r], i, j, best, bi, bj)) {
                            best = dl[r];
                            bi = i;
                            bj = j;
                            baux = (uint32_t)Val<V>::bits(ring[e][r]); // d(p_i, p_j): the apply needs it
                        }
                    }
                }
                if (tau + D < cnt) issue(std::integral_constant<int, e>{}, tau + D);
                // (Tried: an in-loop L2 bulk prefetch 8-32 row steps ahead of the ring, to speed up
                // the last warps of a scan -- 10k step 40.7 -> 45.7 us, 20k 150 -> 178 us; removed.)
            };
            int t = 0;
#pragma unroll 1
            for (; t + NB <= cnt; t += NB) static_for<NB>([&](auto Sc) { step(Sc, t + decltype(Sc)::value); });
            static_for<NB>([&](auto Sc) {
                if (t + decltype(Sc)::value < cnt) step(Sc, t + decltype(Sc)::value);
            });
            // (Tried: the same prefetch issued for the NEXT step by every warp as soon as it finishes
            // its item, i.e. up to 7 us earlier -- the lines are evicted again by the rest of the
            // scan: no gain alone, 2.5 us slower together with the one before the wait.)
        }
    }

    if (done_flag) return; // warps without a work item
    warp_argmin_2opt_aux(best, bi, bj, baux);
    if (lane == 0) red[warp] = Best<V>{best, bi, bj, baux};
    __syncthreads();
    if (warp == 0) {
        Best<V> v = (lane < WARPS) ? red[lane] : Best<V>{(V)0, 0xffffffffu, 0xffffffffu, 0u};
        warp_argmin_2opt_aux(v.delta, v.i, v.j, v.aux);
        if (lane == 0) blockbest[blockIdx.x] = v;
    }
    // the last CTA to finish re-arms the dynamic work queue and, in a fused step, reduces the
    // per-CTA records and applies the move in place
    __shared__ unsigned int s_last;
    __syncthreads();
    TL_MARK_MIN(1);
    TL_MARK_MAX(2);
    if (threadIdx.x == 0) s_last = (ticket_take_acq_rel(ticket) == gridDim.x - 1) ? 1u : 0u; // thread 0 wrote blockbest
    __syncthreads();
    if (!s_last) return;
    if (threadIdx.x == 0) ticket[1] = 0u;
    if (!fuse_apply) {
        if (threadIdx.x == 0) *ticket = 0u;
        return;
    }
    fused_apply_tail_matrix<V>(M, ld, cs, blockbest, red, state, ticket, log, log_cap, sc);
}

// cs[q] = {slot q, entering edge M[slot q-1][slot q], city}; wrap copy at n when cyclic; -inf padding
template <typename V>
__global__ void __launch_bounds__(256)
    build_cs_kernel(const V *__restrict__ M, uint32_t ld, const uint32_t *__restrict__ tour, uint32_t n,
                    uint32_t npad, int cyclic, Cs *__restrict__ cs)
{
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < npad; q += gridDim.x * blockDim.x) {
        Cs c;
        c.pad = 0;
        if (q < n || (q == n && cyclic)) {
            const uint32_t slot = q == n ? 0 : q;
            const uint32_t pslot = slot == 0 ? n - 1 : slot - 1;
            c.slot = (int32_t)slot;
            c.city = (int32_t)tour[slot];
            const V e = (q == 0 && !cyclic) ? (V)0 : M[(size_t)pslot * ld + slot];
            c.sp_bits = Val<V>::bits(e);
        } else {
            c.slot = 0;
            c.city = -1;
            c.sp_bits = Val<V>::bits(Val<V>::neg_inf());
        }
        cs[q] = c;
    }
}

// slot-ordered scratch for building M in tour order
__global__ void __launch_bounds__(256)
    gather_slots_kernel(const float2 *__restrict__ xy, const uint32_t *__restrict__ tour, const Cs *__restrict__ cs,
                        uint32_t n, float2 *__restrict__ sxy, int32_t *__restrict__ slot_city)
{
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < n; q += gridDim.x * blockDim.x) {
        const uint32_t city = tour ? tour[q] : (uint32_t)cs[q].city;
        if (sxy && xy) sxy[q] = xy[city];
        if (slot_city) slot_city[q] = (int32_t)city;
    }
}

// after M has been re-laid in the current tour order: slot == position again
__global__ void __launch_bounds__(256) reset_slots_kernel(Cs *__restrict__ cs, uint32_t n, int cyclic)
{
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q <= n; q += gridDim.x * blockDim.x) {
        if (q < n)
            cs[q].slot = (int32_t)q;
        else if (cyclic)
            cs[q].slot = 0;
    }
}

} // namespace

#ifdef TL_TIMELINE
extern "C" int tl_debug_timeline(double *out8, int reset)
{
    unsigned long long h[8];
    if (cudaMemcpyFromSymbol(h, tl_tacc, sizeof h) != cudaSuccess) return 1;
    if (reset == 2) return cudaMemcpyFromSymbol(out8, tl_tcta, sizeof(unsigned long long) * 3 * 1024) != cudaSuccess; // raw u64[3][1024]
    for (int k = 0; k < 8; ++k) out8[k] = (double)h[k];
    if (reset) {
        const unsigned long long z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        const unsigned long long m[8] = {~0ull, ~0ull, 0ull, 0ull, ~0ull, ~0ull, 0ull, 0ull};
        cudaMemcpyToSymbol(tl_tacc, z, sizeof z);
        cudaMemcpyToSymbol(tl_tmark_par, m, sizeof m);
        cudaMemcpyToSymbol(tl_prev_done, z, sizeof(unsigned long long));
    }
    return 0;
}
#endif

size_t scan_matrix_smem_bytes()
{
    return (size_t)WARPS * WARP_RECS * sizeof(int2) + WARPS * sizeof(BestF);
}

cudaError_t scan_matrix_configure()
{
    const int smem = (int)scan_matrix_smem_bytes();
    cudaError_t e = cudaFuncSetAttribute(two_opt_scan_matrix_kernel<float, false>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(two_opt_scan_matrix_kernel<float, true>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(two_opt_scan_matrix_kernel<int32_t, false>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(two_opt_scan_matrix_kernel<int32_t, true>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    return e;
}

void launch_scan_matrix(const Src &src, const ScanGeom &g, const int32_t *band_first, void *blockbest,
                        DevState *state, unsigned int *ticket, tl_move *log, uint64_t log_cap, bool fuse_apply,
                        const ShardComm *shard, int grid, const MatPin &pin, cudaStream_t st)
{
    const size_t smem = scan_matrix_smem_bytes();
    ShardComm sc{};
    sc.world = 1;
    if (shard) sc = *shard;
    cudaLaunchAttribute attr[2];
    cudaLaunchConfig_t cfg = pdl_config(grid, WARPS * 32, smem, attr, st);
    if (pin.window_bytes > 0) { // driver-managed residency: persisting window over the first matrix rows
        attr[1].id = cudaLaunchAttributeAccessPolicyWindow;
        attr[1].val.accessPolicyWindow.base_ptr = const_cast<void *>(src.M);
        attr[1].val.accessPolicyWindow.num_bytes = pin.window_bytes;
        attr[1].val.accessPolicyWindow.hitRatio = pin.window_hit_ratio;
        attr[1].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        attr[1].val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        cfg.numAttrs = 2;
    }
    const int fuse = fuse_apply ? 1 : 0;
    const int pin_rows = pin.hint_rows;
    static const int pf_default = [] {
        const char *ev = getenv("TL_MAT_PREFETCH_ROWS");
        return ev ? max(0, min(32, atoi(ev))) : kMatPrefetchRows;
    }();
    const int pf_rows = pf_default;
#define TL_LAUNCH_MAT(V, PINNED, BEST)                                                                          \
    cudaLaunchKernelEx(&cfg, two_opt_scan_matrix_kernel<V, PINNED>, (const V *)src.M, src.ld, src.cs, g,        \
                       band_first, (BEST *)blockbest, state, ticket, log, (uint64_t)log_cap, fuse, pin_rows, pf_rows, sc)
    if (src.is_int()) {
        if (pin_rows > 0) TL_LAUNCH_MAT(int32_t, true, BestI); else TL_LAUNCH_MAT(int32_t, false, BestI);
    } else {
        if (pin_rows > 0) TL_LAUNCH_MAT(float, true, BestF); else TL_LAUNCH_MAT(float, false, BestF);
    }
#undef TL_LAUNCH_MAT
}

void launch_build_cs(const Src &src, const uint32_t *tour, uint32_t n, uint32_t npad, int cyclic, cudaStream_t st)
{
    const int grid = (int)((npad + 255) / 256);
    if (src.is_int())
        build_cs_kernel<int32_t><<<grid, 256, 0, st>>>((const int32_t *)src.M, src.ld, tour, n, npad, cyclic, src.cs);
    else
        build_cs_kernel<float><<<grid, 256, 0, st>>>((const float *)src.M, src.ld, tour, n, npad, cyclic, src.cs);
}

void launch_gather_slots(const float2 *xy, const uint32_t *tour, const Cs *cs, uint32_t n, float2 *sxy,
                         int32_t *slot_city, cudaStream_t st)
{
    gather_slots_kernel<<<(n + 255) / 256, 256, 0, st>>>(xy, tour, cs, n, sxy, slot_city);
}

void launch_reset_slots(const Src &src, uint32_t n, uint32_t npad, int cyclic, cudaStream_t st)
{
    (void)npad;
    reset_slots_kernel<<<(n + 256) / 256, 256, 0, st>>>(src.cs, n, cyclic);
}

} // namespace tl
