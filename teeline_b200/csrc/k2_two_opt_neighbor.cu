// k2_two_opt_neighbor.cu -- K2 candidate-list best-improvement 2-opt ("Mode N"), coordinate recompute.
//
// What it computes: Mode B's neighbourhood (0 <= i, i+2 <= j <= n-2, path[i+1..=j] reversed) and
// delta, restricted to the pairs that create an edge to one of a city's k nearest neighbours.  For
// every position i and candidate slot s, with b = K[p_i][s], j = pos[b], lo = min(i, j), hi = max(i, j):
//   (lo, hi)         the candidate edge (p_lo, p_hi) is the move's first new edge
//   (lo - 1, hi - 1) the candidate edge is its second new edge
// A generated pair counts only inside the neighbourhood.  The step's move is the argmin of
// (delta, i, j) over the generated pairs with strict '< 0' (better_2opt), as in Mode B; duplicates
// carry the same key.  With k >= n-1 every Mode B pair is generated and the moves are Mode B's.
//
// How: a grid of resident CTAs walks the n*k (position, slot) items with a grid-stride loop.  Per
// item: the record at i, the candidate, pos[b], then the records lo-1 .. hi+1; the two pairs share
// d(p_lo, p_hi), so three distances cover both.  The last CTA (acq_rel ticket) reduces the per-CTA
// records.  A short segment is reversed by that CTA; a long one is left as the pending move for the
// apply grid that every step launches (apply_two_opt_kernel, pending_only), which leaves at once when
// there is none.  The grid size cannot depend on the move: the host queues steps without reading back.
// The records, pos[] and the candidate lists (16 + 4 + 4k bytes per city) fit L2 up to about 10^6
// cities, so the scan is a chain of dependent L2 gathers.
//
// Mode NM (multi-move, TL_ALGO_TWO_OPT_NEIGHBOR_MULTI; definition in include/teeline_cuda.h): the same
// scan and G, and in step t (= DevState::scans) position q lies in block (q + o) >> bshift with
// o = (t & 1) << (bshift - 1).  Every improving pair whose i and j+1 share a block does a 64-bit atomicMin
// into that block's key: the order-preserving bits of its delta above the in-block offsets
// (i - base) << bshift | (j - base), which orders a block's pairs by (delta, i, j).  The last CTA reduces G,
// re-arms the keys while it compacts the block bests disjoint from G into a list in increasing i (a
// block-wide scan; blocks are in position order), cuts the list at the move budget, writes the log and
// ends the step.  It reverses a short G itself; the apply grid then reverses a long G cooperatively and
// each listed block move (at most 2^bshift positions) with one CTA.  These moves touch disjoint edges: a
// block move and G share at most an end position, whose entering-edge length one of them rewrites and the
// other never reads (reverse_segment_inplace reads only the coordinates of the records at i and j+1).
#include "apply.cuh"
#include "block_keys.cuh"
#include "kernels.cuh"

#include <math_constants.h>

namespace tl {

namespace {

constexpr int THREADS = kNlThreads;
constexpr int WARPS = THREADS / 32;

// an improving pair (i, j): offer it to its block when i and j+1 lie in the same block
template <typename V>
__device__ __forceinline__ void block_offer(const NlMulti &M, uint32_t off, V d, uint32_t i, uint32_t j)
{
    const uint32_t b = (i + off) >> M.bshift;
    if (b != (j + 1 + off) >> M.bshift) return;
    const uint32_t base = (b << M.bshift) - off; // wraps for block 0 at odd steps; the differences below do not
    const unsigned long long key =
        ((unsigned long long)order_bits(d) << 32) | (((i - base) << M.bshift) | (j - base));
    atomicMin(M.keys + b, key);
}

// Tail of a fused step, run by the last CTA: reduce the per-CTA records, count the step's evaluated
// pairs, then either reverse a short segment here and finish the step, or leave a long one pending.
template <class Pol>
__device__ __noinline__ void nl_tail(const Pol &P, uint32_t *pos, Best<typename Pol::V> *blockbest, DevState *state,
                                     unsigned int *ticket, tl_move *__restrict__ log, uint64_t log_cap)
{
    using V = typename Pol::V;
    __shared__ Best<V> red[WARPS];
    __shared__ unsigned long long red_cnt[WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    StateHeader hdr{};
    if (threadIdx.x == 0) hdr = load_state_header(state);
    Best<V> v{(V)0, 0xffffffffu, 0xffffffffu, 0u};
    unsigned long long cnt = 0;
    for (int c = threadIdx.x; c < (int)gridDim.x; c += blockDim.x) {
        // L2 read: the records were written by other CTAs of this launch
        const int4 raw = __ldcg(reinterpret_cast<const int4 *>(blockbest) + c);
        const Best<V> o{Val<V>::from_bits(raw.x), (uint32_t)raw.y, (uint32_t)raw.z, (uint32_t)raw.w};
        cnt += o.aux;
        if (TwoOptOrder::better(o, v)) v = o;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
    if (lane == 0) red_cnt[warp] = cnt;
    v = block_argmin<WARPS, TwoOptOrder>(v, red); // its barrier publishes red_cnt too
    cnt = 0;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) cnt += red_cnt[w];
    const bool found = v.i != 0xffffffffu;
    const bool long_seg = found && (v.j - v.i) / 2 > (uint32_t)kNlCtaSwaps;
    if (threadIdx.x == 0) {
        state->computed += cnt;
        // the pending move for this step's apply grid (none: the step is finished here)
        blockbest[gridDim.x] = long_seg ? v : Best<V>{(V)0, 0xffffffffu, 0xffffffffu, 0u};
        *ticket = 0u;
    }
    if (long_seg) return;
    if (found) reverse_segment_inplace(P, v.i, v.j, nullptr, threadIdx.x, blockDim.x, false, V(), V(), pos);
    if (threadIdx.x == 0) finish_best_step(state, hdr, found, (float)v.delta, v.i, v.j, log, log_cap);
}

// Tail of a fused Mode NM step, run by the last CTA: nl_tail's G, then the accepted block bests.
template <class Pol>
__device__ __noinline__ void nlm_tail(const Pol &P, uint32_t *pos, Best<typename Pol::V> *blockbest, DevState *state,
                                      unsigned int *ticket, tl_move *__restrict__ log, uint64_t log_cap,
                                      const NlMulti &M, uint32_t off)
{
    using V = typename Pol::V;
    __shared__ Best<V> red[WARPS];
    __shared__ unsigned long long red_cnt[WARPS];
    __shared__ unsigned long long s_moves;
    __shared__ long long s_max;
    __shared__ uint32_t s_wcnt[WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    StateHeader hdr{};
    if (threadIdx.x == 0) {
        hdr = load_state_header(state);
        s_moves = hdr.h0.x;
        s_max = hdr.h1.x;
    }
    Best<V> v{(V)0, 0xffffffffu, 0xffffffffu, 0u};
    unsigned long long cnt = 0;
    for (int c = threadIdx.x; c < (int)gridDim.x; c += blockDim.x) {
        const int4 raw = __ldcg(reinterpret_cast<const int4 *>(blockbest) + c);
        const Best<V> o{Val<V>::from_bits(raw.x), (uint32_t)raw.y, (uint32_t)raw.z, (uint32_t)raw.w};
        cnt += o.aux;
        if (TwoOptOrder::better(o, v)) v = o;
    }
#pragma unroll
    for (int off2 = 16; off2 > 0; off2 >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, off2);
    if (lane == 0) red_cnt[warp] = cnt;
    v = block_argmin<WARPS, TwoOptOrder>(v, red); // its barrier publishes red_cnt, s_moves and s_max too
    cnt = 0;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) cnt += red_cnt[w];
    const bool found = v.i != 0xffffffffu;
    const unsigned long long m = s_moves;
    // block moves this step may still apply after G (G always fits: the step runs only below the budget)
    const unsigned long long allow = s_max < 0 ? ~0ull : (unsigned long long)s_max - m - 1;
    // without G no pair improves, so no key was set
    uint32_t taken = 0;
    if (found) {
        uint2 *list = static_cast<uint2 *>(M.list);
        struct Mv {
            uint32_t i, j;
            V d;
        };
        taken = compact_block_keys<WARPS, Mv>(
            M, allow, s_wcnt,
            [&](uint32_t b, unsigned long long key, Mv &mv) {
                const uint32_t low = (uint32_t)key, base = (b << M.bshift) - off;
                mv.i = base + (low >> M.bshift);
                mv.j = base + (low & ((1u << M.bshift) - 1u));
                mv.d = from_order_bits<V>((uint32_t)(key >> 32));
                return !(mv.i == v.i && mv.j == v.j) && (mv.j < v.i || mv.i > v.j);
            },
            [&](uint32_t rank, const Mv &mv) {
                list[rank] = make_uint2(mv.i, mv.j);
                const unsigned long long e = m + 1 + rank;
                if (log && e < log_cap) log[e] = tl_move{(float)mv.d, mv.i, mv.j, 0, 0, 0};
            });
    }
    const uint32_t napply = (uint32_t)min((unsigned long long)taken, allow);
    const bool long_seg = found && (v.j - v.i) / 2 > (uint32_t)kNlCtaSwaps;
    if (threadIdx.x == 0) {
        state->computed += cnt;
        M.desc[0] = napply;
        M.desc[1] = long_seg ? v.i : 0xffffffffu;
        M.desc[2] = v.j;
        *ticket = 0u;
        state->scans = hdr.h0.y + 1;
        if (found) {
            if (log && m < log_cap) log[m] = tl_move{(float)v.delta, v.i, v.j, 0, 0, 0};
            const unsigned long long moves = m + 1 + napply;
            state->moves = moves;
            if (s_max >= 0 && (long long)moves >= s_max) state->done = 1;
        } else {
            state->done = 1;
            state->converged = 1;
        }
    }
    if (found && !long_seg) reverse_segment_inplace(P, v.i, v.j, nullptr, threadIdx.x, blockDim.x, false, V(), V(), pos);
}

// MULTI: Mode NM's fused step (block keys and nlm_tail); otherwise Mode N's scan
template <bool MULTI, class Pol>
__global__ void __launch_bounds__(THREADS, kNlMinBlocks)
    two_opt_nl_scan_kernel(Pol P, uint32_t *__restrict__ pos, const uint32_t *__restrict__ cand, uint32_t k,
                           uint32_t n, Best<typename Pol::V> *blockbest, DevState *state, unsigned int *ticket,
                           tl_move *__restrict__ log, uint64_t log_cap, int fuse_apply, NlMulti M)
{
    using V = typename Pol::V;
    using Rec = typename Pol::Rec;
    griddep_launch_dependents();
    griddep_wait(); // the previous step's move is applied and visible from here on
    // uniform across the grid: only a step's tail or apply grid writes it, after every CTA has finished
    if (*reinterpret_cast<const volatile int *>(&state->done)) return;
    // Mode NM: this step's block offset (scans is only written by a step's tail, after every CTA has read it)
    uint32_t off = 0;
    if (MULTI) off = ((uint32_t)*reinterpret_cast<const volatile unsigned long long *>(&state->scans) & 1u) << (M.bshift - 1);

    V best = (V)0;
    uint32_t bi = 0xffffffffu, bj = 0xffffffffu, cnt = 0;
    const uint64_t total = (uint64_t)n * k;
    for (uint64_t t = (uint64_t)blockIdx.x * THREADS + threadIdx.x; t < total; t += (uint64_t)gridDim.x * THREADS) {
        const uint32_t i = (uint32_t)(t / k), s = (uint32_t)(t - (uint64_t)i * k);
        const uint32_t b = __ldg(&cand[(size_t)Pol::city(P.load(i)) * k + s]);
        if (b == 0xffffffffu) continue; // padding: fewer than k other cities
        const uint32_t j = pos[b];
        const uint32_t lo = min(i, j), hi = max(i, j);
        if (hi < lo + 2) continue; // the candidate edge is a tour edge: no pair
        const bool first = hi <= n - 2, second = lo >= 1;
        if (!first && !second) continue;
        const Rec rlo = P.load(lo), rhi = P.load(hi);
        const V shared = P.dist(rlo, rhi);
        if (first) { // (lo, hi): new edges (p_lo, p_hi) and (p_lo+1, p_hi+1)
            const Rec a = P.load(lo + 1), c = P.load(hi + 1);
            const V d = Val<V>::sub(Val<V>::add(shared, P.dist(a, c)), Val<V>::add(Pol::sp(a), Pol::sp(c)));
            ++cnt;
            if (MULTI && d < (V)0) block_offer(M, off, d, lo, hi);
            if (d < (V)0 && better_2opt(d, lo, hi, best, bi, bj)) {
                best = d;
                bi = lo;
                bj = hi;
            }
        }
        if (second) { // (lo-1, hi-1): new edges (p_lo-1, p_hi-1) and (p_lo, p_hi)
            const Rec a = P.load(lo - 1), c = P.load(hi - 1);
            const V d = Val<V>::sub(Val<V>::add(P.dist(a, c), shared), Val<V>::add(Pol::sp(rlo), Pol::sp(rhi)));
            ++cnt;
            if (MULTI && d < (V)0) block_offer(M, off, d, lo - 1, hi - 1);
            if (d < (V)0 && better_2opt(d, lo - 1, hi - 1, best, bi, bj)) {
                best = d;
                bi = lo - 1;
                bj = hi - 1;
            }
        }
    }

    __shared__ Best<V> red[WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    warp_argmin_2opt(best, bi, bj);
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0) red[warp] = Best<V>{best, bi, bj, cnt};
    __syncthreads();
    if (warp == 0) {
        Best<V> v = lane < WARPS ? red[lane] : Best<V>{(V)0, 0xffffffffu, 0xffffffffu, 0u};
        const uint32_t c = __reduce_add_sync(0xffffffffu, v.aux);
        warp_argmin_2opt(v.delta, v.i, v.j);
        v.aux = c; // 2-opt records carry the CTA's evaluated-pair count in aux
        if (lane == 0) blockbest[blockIdx.x] = v;
    }
    if (!fuse_apply) return;
    __shared__ unsigned int s_last;
    __syncthreads();
    if (threadIdx.x == 0) s_last = (ticket_take_acq_rel(ticket) == gridDim.x - 1) ? 1u : 0u; // thread 0 wrote blockbest
    __syncthreads();
    if (!s_last) return;
    if (MULTI)
        nlm_tail(P, pos, blockbest, state, ticket, log, log_cap, M, off);
    else
        nl_tail(P, pos, blockbest, state, ticket, log, log_cap);
}

// Mode NM's apply grid, launched after every step's scan: desc (written by nlm_tail) names a pending long G,
// reversed by the whole grid, and the count of listed block moves, each reversed by one CTA.  The last CTA
// to finish resets desc, so a later no-op step applies nothing.
template <class Pol>
__global__ void __launch_bounds__(256)
    apply_multi_kernel(Pol P, uint32_t *pos, const uint2 *__restrict__ list, uint32_t *desc, unsigned int *ticket)
{
    using V = typename Pol::V;
    griddep_wait(); // PDL: the step's scan has finished and its writes are visible
    const uint32_t cnt = __ldcg(desc), gi = __ldcg(desc + 1), gj = __ldcg(desc + 2);
    if (cnt == 0 && gi == 0xffffffffu) return; // uniform over the grid
    if (gi != 0xffffffffu)
        reverse_segment_inplace(P, gi, gj, nullptr, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x,
                                false, V(), V(), pos);
    for (uint32_t c = blockIdx.x; c < cnt; c += gridDim.x) {
        const uint2 mv = list[c];
        reverse_segment_inplace(P, mv.x, mv.y, nullptr, threadIdx.x, blockDim.x, false, V(), V(), pos);
    }
    __syncthreads();
    if (threadIdx.x == 0 && atomicAdd(ticket, 1u) == gridDim.x - 1) { // every CTA has read desc
        *ticket = 0u;
        desc[0] = 0u;
        desc[1] = 0xffffffffu;
    }
}

// tour-ordered records (entering-edge length in the policy's metric) and pos[city] = position.
// CYCLIC (Or-opt N, which reads the closing edge): position 0 carries d(p_n-1, p_0) as its entering
// edge and position n is a copy of position 0, as launch_build_pts(..., cyclic) lays them out for K3.
template <bool CYCLIC, class Pol>
__global__ void __launch_bounds__(256)
    nl_init_kernel(Pol P, const float2 *__restrict__ xy, const uint32_t *__restrict__ tour, uint32_t n, uint32_t npad,
                   uint32_t *__restrict__ pos)
{
    using V = typename Pol::V;
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < npad; q += gridDim.x * blockDim.x) {
        if (q < n || (CYCLIC && q == n)) {
            const uint32_t c = tour[CYCLIC && q == n ? 0 : q];
            const float2 a = xy[c];
            const Pt r{a.x, a.y, (int32_t)c, 0.0f};
            P.store_id(q, r);
            if (q == 0 && !CYCLIC) {
                P.store_sp(q, (V)0);
            } else {
                const float2 b = xy[tour[CYCLIC && q == 0 ? n - 1 : q - 1]];
                P.store_sp(q, P.dist(Pt{b.x, b.y, 0, 0.0f}, r));
            }
            if (!CYCLIC || q < n) pos[c] = q;
        } else { // padding: never part of a pair
            P.store_id(q, Pt{0.0f, 0.0f, -1, 0.0f});
            P.store_sp(q, Val<V>::neg_inf());
        }
    }
}

} // namespace

void launch_nl_init(Metric metric, const float2 *xy, const uint32_t *tour, uint32_t n, uint32_t npad, bool cyclic,
                    Pt *pts, uint32_t *pos, cudaStream_t st)
{
    const int grid = (int)((npad + 255) / 256);
    with_metric(metric, [&](auto M) {
        if (cyclic)
            nl_init_kernel<true><<<grid, 256, 0, st>>>(NlPol<M>{pts}, xy, tour, n, npad, pos);
        else
            nl_init_kernel<false><<<grid, 256, 0, st>>>(NlPol<M>{pts}, xy, tour, n, npad, pos);
    });
}

void launch_nl_scan(Metric metric, Pt *pts, uint32_t *pos, const uint32_t *cand, uint32_t k, uint32_t n, void *blockbest,
                    DevState *state, unsigned int *ticket, tl_move *log, uint64_t log_cap, bool fuse_apply, int grid,
                    cudaStream_t st, const NlMulti *multi)
{
    cudaLaunchAttribute attr[1];
    const cudaLaunchConfig_t cfg = pdl_config(grid, THREADS, 0, attr, st);
    const int fuse = fuse_apply ? 1 : 0;
    const NlMulti mm = multi ? *multi : NlMulti{};
    with_metric(metric, [&](auto M) {
        using Pol = NlPol<M>;
        auto *bb = reinterpret_cast<Best<typename Pol::V> *>(blockbest);
        if (multi && fuse_apply) // a scan without its step (tl_session_scan) leaves the block keys alone
            cudaLaunchKernelEx(&cfg, two_opt_nl_scan_kernel<true, Pol>, Pol{pts}, pos, cand, k, n, bb, state, ticket, log,
                               (uint64_t)log_cap, fuse, mm);
        else
            cudaLaunchKernelEx(&cfg, two_opt_nl_scan_kernel<false, Pol>, Pol{pts}, pos, cand, k, n, bb, state, ticket,
                               log, (uint64_t)log_cap, fuse, mm);
    });
}

void launch_nlm_apply(Metric metric, Pt *pts, uint32_t *pos, const NlMulti &multi, unsigned int *ticket, int grid,
                      cudaStream_t st)
{
    cudaLaunchAttribute attr[1];
    const cudaLaunchConfig_t cfg = pdl_config(grid, 256, 0, attr, st);
    with_metric(metric, [&](auto M) {
        using Pol = NlPol<M>;
        cudaLaunchKernelEx(&cfg, apply_multi_kernel<Pol>, Pol{pts}, pos, static_cast<const uint2 *>(multi.list), multi.desc,
                           ticket);
    });
}

void launch_nl_apply(Metric metric, Pt *pts, uint32_t *pos, const void *pending, DevState *state, unsigned int *ticket,
                     tl_move *log, uint64_t log_cap, int grid, cudaStream_t st)
{
    cudaLaunchAttribute attr[1];
    const cudaLaunchConfig_t cfg = pdl_config(grid, 256, 0, attr, st);
    with_metric(metric, [&](auto M) {
        using Pol = NlPol<M>;
        cudaLaunchKernelEx(&cfg, apply_two_opt_kernel<Pol>, Pol{pts}, reinterpret_cast<const Best<typename Pol::V> *>(pending),
                           1, state, ticket, log, (uint64_t)log_cap, pos, 1);
    });
}

} // namespace tl
