// apply.cuh -- the apply step of every device-resident search on the tour-ordered records (any policy):
// 2-opt reversal, relocation of a run of positions (Or-opt, Or-opt N, 3-opt), the candidate reduction
// and the loop-state update that ends a step.
#pragma once

#include "kernels.cuh"
#include "policy.cuh"

namespace tl {

// Reverse path[mi+1..=mj] in place (swap_2opt, src/tsp/two_opt.rs:69-79) with `nthreads`
// cooperating threads, this one being `tid`.  Thread t swaps the identity fields of
// positions (mi+1+t, mj-t) and the entering-edge lengths of positions (mi+2+t, mj-t): inside
// the segment the old edge lengths are simply mirrored (the metric is bitwise symmetric); the
// two new edges are produced by thread 0.  Every field of every record is read and written by
// exactly one thread, so the update is race free without a second buffer.  If delta_out is
// non-null, thread 0 also stores (d(p_i,p_j) + d(p_i+1,p_j+1)) - (d(p_i,p_i+1) + d(p_j,p_j+1)).
// known_e1: the caller already knows e1 = d(p_i, p_j) and the move's delta (integer metric only:
// the matrix scan's winning thread held e1, and e2 = delta + (s_i + s_j) - e1 exactly), which
// saves the two dependent matrix loads -- an HBM round trip on the fused step's critical path.
// pos (nullable): city -> position map kept beside the records (candidate-list 2-opt); the thread that
// stores a position's identity also stores that city's new position.
template <class Pol>
__device__ __forceinline__ void reverse_segment_inplace(const Pol &P, uint32_t mi, uint32_t mj, float *delta_out,
                                                        uint32_t tid, uint32_t nthreads, bool known_e1 = false,
                                                        typename Pol::V e1_in = typename Pol::V(),
                                                        typename Pol::V delta_in = typename Pol::V(),
                                                        uint32_t *pos = nullptr)
{
    using V = typename Pol::V;
    using Rec = typename Pol::Rec;
    const uint32_t L = mj - mi; // segment mi+1 .. mj, L >= 2
    const uint32_t nxy = L / 2, nsp = (L - 1) / 2;
    // U swaps per thread per round: all loads of a round are issued before its first store, so a
    // round costs one memory round trip instead of U (a thread's own records never alias)
    constexpr int U = 4;
    Rec P0{}, P1{}; // the segment's outer neighbours, needed by thread 0 only: load them up front
    V sp_first = V(); // entering edge of position mi+1 (thread 0's delta needs it).  Read here and not from
                      // A[] below: position mi+1+t's edge length is rewritten by thread t-1, so a thread
                      // t > 0 must not touch that field at all (array-of-fields policies then never load it)
    if (tid == 0) {
        P0 = P.load(mi);
        P1 = P.load(mj + 1);
        sp_first = Pol::sp(P.load(mi + 1));
    }
    for (uint32_t t0 = tid; t0 < nxy; t0 += nthreads * U) {
        Rec A[U], B[U];
        V sa[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t t = t0 + u * nthreads;
            if (t < nxy) {
                A[u] = P.load(mi + 1 + t);
                B[u] = P.load(mj - t);
                if (t < nsp) sa[u] = Pol::sp(P.load(mi + 2 + t));
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t t = t0 + u * nthreads;
            if (t >= nxy) continue;
            const uint32_t a = mi + 1 + t, b = mj - t;
            if (t == 0) {
                V e1, e2;
                if (known_e1) {
                    e1 = e1_in;
                    e2 = Val<V>::sub(Val<V>::add(delta_in, Val<V>::add(sp_first, Pol::sp(P1))), e1_in);
                } else {
                    e1 = P.dist(P0, B[u]); // new edge (p_i, p_j)
                    e2 = P.dist(A[u], P1); // new edge (p_i+1, p_j+1)
                }
                if (delta_out)
                    *delta_out = (float)Val<V>::sub(Val<V>::add(e1, e2), Val<V>::add(sp_first, Pol::sp(P1)));
                P.store_sp(a, e1);
                P.store_sp(mj + 1, e2);
            }
            P.store_id(a, B[u]);
            P.store_id(b, A[u]);
            if (pos) {
                pos[B[u].city] = a;
                pos[A[u].city] = b;
            }
            if (t < nsp) { // mi+2+t <-> mj-t
                P.store_sp(a + 1, Pol::sp(B[u]));
                P.store_sp(b, sa[u]);
            }
        }
    }
}

// Loop-state update that ends a step (one thread).  The header of DevState,
// {moves, scans} and {max_moves, done, converged}, is read with two independent 16-byte loads
// (load_state_header) that the caller issues early, off the critical path.
struct StateHeader {
    ulonglong2 h0;
    longlong2 h1;
};
__device__ __forceinline__ StateHeader load_state_header(const DevState *state)
{
    StateHeader h;
    h.h0 = __ldcg(reinterpret_cast<const ulonglong2 *>(state));
    h.h1 = __ldcg(reinterpret_cast<const longlong2 *>(state) + 1);
    return h;
}
// `entry` is the move's log entry, used when found.  Returns the value of state->done after the step.
__device__ __forceinline__ int finish_step(DevState *state, const StateHeader &h, bool found, const tl_move &entry,
                                           tl_move *__restrict__ log, uint64_t log_cap)
{
    const unsigned long long m = h.h0.x;
    const long long max_moves = h.h1.x;
    state->scans = h.h0.y + 1;
    if (found) {
        if (log && m < log_cap) log[m] = entry;
        state->moves = m + 1;
        if (max_moves >= 0 && (long long)(m + 1) >= max_moves) {
            state->done = 1;
            return 1;
        }
        return 0;
    }
    state->done = 1;
    state->converged = 1;
    return 1;
}
// a 2-opt step, logged as (delta, mi, mj)
__device__ __forceinline__ int finish_best_step(DevState *state, const StateHeader &h, bool found, float delta,
                                                uint32_t mi, uint32_t mj, tl_move *__restrict__ log,
                                                uint64_t log_cap)
{
    return finish_step(state, h, found, tl_move{delta, mi, mj, 0, 0, 0}, log, log_cap);
}

// Last-CTA detection with ONE acq_rel atomic instead of fence.sc + relaxed atomic + fence.sc:
// release publishes this thread's candidate record, acquire (plus the caller's __syncthreads)
// orders the last CTA's reads of everybody else's records after it.
__device__ __forceinline__ unsigned int ticket_take_acq_rel(unsigned int *ticket)
{
    unsigned int old;
    asm volatile("atom.add.acq_rel.gpu.global.u32 %0, [%1], 1;" : "=r"(old) : "l"(ticket) : "memory");
    return old;
}

// Stand-alone apply grids: after every block has done its part of the move (caller's __syncthreads),
// the last block to finish ends the step.  Every block has read `state` by then.
__device__ __forceinline__ void grid_finish_step(unsigned int *ticket, DevState *state, bool found,
                                                 const tl_move &entry, tl_move *__restrict__ log, uint64_t log_cap)
{
    if (threadIdx.x != 0) return;
    __threadfence();
    const unsigned int tk = atomicAdd(ticket, 1u);
    if (tk == gridDim.x - 1) {
        *ticket = 0u;
        finish_step(state, load_state_header(state), found, entry, log, log_cap);
        __threadfence();
    }
}

// ---- candidate reduction ------------------------------------------------------------------------
// Argmin of Best<V> records in the order Order::better(a, b), a strict "a before b" in which the
// record {0, ~0, ~0, 0} ("no candidate") never comes before a real one.

// (delta, i, j): 2-opt's order
struct TwoOptOrder {
    template <typename V>
    static __device__ __forceinline__ bool better(const Best<V> &a, const Best<V> &b)
    {
        return better_2opt(a.delta, a.i, a.j, b.delta, b.i, b.j);
    }
};

template <class Order, typename V>
__device__ __forceinline__ void warp_argmin(Best<V> &v)
{
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        Best<V> o;
        o.delta = __shfl_xor_sync(0xffffffffu, v.delta, off);
        o.i = __shfl_xor_sync(0xffffffffu, v.i, off);
        o.j = __shfl_xor_sync(0xffffffffu, v.j, off);
        o.aux = __shfl_xor_sync(0xffffffffu, v.aux, off);
        if (Order::better(o, v)) v = o;
    }
}

// v: this thread's best record.  Every thread of the block (WARPS warps) gets the block's best.  Contains
// one __syncthreads, which also publishes shared-memory writes the caller made before the call.
template <int WARPS, class Order, typename V>
__device__ __forceinline__ Best<V> block_argmin(Best<V> v, Best<V> *sred)
{
    warp_argmin<Order>(v);
    if ((threadIdx.x & 31) == 0) sred[threadIdx.x >> 5] = v;
    __syncthreads();
    v = sred[0];
#pragma unroll
    for (int w = 1; w < WARPS; ++w)
        if (Order::better(sred[w], v)) v = sred[w];
    return v;
}

// every block reduces the candidate records cand[0 .. ncand) redundantly (at most a few hundred)
template <class Order, typename V>
__device__ __forceinline__ Best<V> block_argmin_records(const Best<V> *__restrict__ cand, int ncand, Best<V> *sred)
{
    if (ncand == 1) return cand[0]; // one pending record: nothing to reduce
    Best<V> v{(V)0, 0xffffffffu, 0xffffffffu, 0u};
    for (int c = threadIdx.x; c < ncand; c += blockDim.x) {
        const Best<V> o = cand[c];
        if (Order::better(o, v)) v = o;
    }
    return block_argmin<8, Order>(v, sred);
}

// Stand-alone apply step for Mode B (sharded sessions and the matrix path): every block
// reduces the candidate records, the grid reverses the segment, the last block to finish updates the
// loop state.
// Candidate-list 2-opt (k2_two_opt_neighbor.cu) passes its one pending long move with
// pending_only = true: no move pending means the scan already finished the step, and the grid leaves.
template <class Pol>
__global__ void __launch_bounds__(256)
    apply_two_opt_kernel(Pol P, const Best<typename Pol::V> *__restrict__ cand, int ncand, DevState *state,
                         unsigned int *ticket, tl_move *__restrict__ log, uint64_t log_cap, uint32_t *pos,
                         int pending_only)
{
    using V = typename Pol::V;
    griddep_wait(); // PDL launches only: the step's scan has finished and its writes are visible
    if (state->done) return;
    __shared__ Best<V> sred[8];
    const Best<V> v = block_argmin_records<TwoOptOrder>(cand, ncand, sred);
    const bool found = v.i != 0xffffffffu;
    if (pending_only && !found) return; // uniform over the grid
    if (found)
        reverse_segment_inplace(P, v.i, v.j, nullptr, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x,
                                false, V(), V(), pos);
    __syncthreads();
    grid_finish_step(ticket, state, found, tl_move{(float)v.delta, v.i, v.j, 0, 0, 0}, log, log_cap);
}

// ---- relocation of a run of positions -----------------------------------------------------------
// A move that gives the positions [lo, hi] new occupants and leaves every other position's city in
// place (Or-opt, Or-opt N, 3-opt) on cyclic records: position 0 carries the closing edge
// d(p_n-1, p_0) and position n is a copy of position 0.  Move supplies:
//   found, lo, hi        whether there is a move, and its span (0 <= lo <= hi <= n-1)
//   source(q)            the old position of the new occupant of q, for q in [lo, hi]
//   entry()              its log entry
//   better(a, b), of(v)  the order of its candidate records (block_argmin), and the move of a record
// Two phases with a barrier between them (block or grid), `nthreads` cooperating threads, this one
// being `tid`: first copy the new occupants of [lo, hi] to tmp ...
template <class Pol, class Move>
__device__ __forceinline__ void relocate_gather(const Pol &P, typename Pol::Rec *__restrict__ tmp, const Move &m,
                                                uint32_t tid, uint32_t nthreads)
{
    for (uint32_t q = m.lo + tid; q <= m.hi; q += nthreads) tmp[q - m.lo] = P.load(m.source(q));
}

// ... then write them back with the entering edges of lo .. hi+1 (and their pos[] entries when pos is
// non-null); thread 0 rewrites the closing edge and the wrap copy at position n when the span touches
// either end.  Every read of a relocated position goes to tmp, so the in-place writes cannot race with them.
template <class Pol, class Move>
__device__ __forceinline__ void relocate_scatter(const Pol &P, const typename Pol::Rec *__restrict__ tmp, uint32_t n,
                                                 const Move &m, uint32_t *pos, uint32_t tid, uint32_t nthreads)
{
    using Rec = typename Pol::Rec;
    // record now at position q (q in 0..n): relocated range from tmp, everything else unchanged
    auto newpt = [&](uint32_t q) -> Rec {
        const uint32_t qq = q == n ? 0u : q;
        return (qq >= m.lo && qq <= m.hi) ? tmp[qq - m.lo] : P.load(qq);
    };
    for (uint32_t q = m.lo + tid; q <= m.hi + 1; q += nthreads) {
        if (q < 1 || q > n) continue;
        Rec p = newpt(q);
        const Rec b = newpt(q - 1);
        const typename Pol::V e = P.dist(b, p);
        if (q <= m.hi) {
            Pol::set_sp(p, e);
            P.store(q, p);
            if (pos) pos[Pol::city(p)] = q;
        } else {
            P.store_sp(q, e); // hi+1: same city (or the wrap copy), new entering edge
        }
    }
    if (tid == 0 && (m.lo == 0 || m.hi >= n - 1)) {
        Rec p0 = newpt(0);
        const Rec last = newpt(n - 1);
        Pol::set_sp(p0, P.dist(last, p0));
        P.store(n, p0);
        if (m.lo == 0) {
            P.store(0, p0);
            if (pos) pos[Pol::city(p0)] = 0;
        } else {
            P.store_sp(0, Pol::sp(p0));
        }
    }
}

// The records reduction of a fused candidate-list relocation step's tail, run by the scan's last CTA of WARPS
// warps: every thread gets the best of blockbest[0 .. grid) in Move's order and the sum of the per-CTA counts of
// evaluated candidates (cnt_out).  Contains a barrier, which also publishes the caller's earlier shared writes.
template <int WARPS, class Move, typename V>
__device__ __forceinline__ Best<V> reduce_step_records(const Best<V> *blockbest, const unsigned long long *blockcnt,
                                                       unsigned long long &cnt_out)
{
    __shared__ Best<V> red[WARPS];
    __shared__ unsigned long long red_cnt[WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    Best<V> v{(V)0, 0xffffffffu, 0xffffffffu, 0u};
    unsigned long long cnt = 0;
    for (int c = threadIdx.x; c < (int)gridDim.x; c += blockDim.x) {
        // L2 reads: the records were written by other CTAs of this launch
        const int4 raw = __ldcg(reinterpret_cast<const int4 *>(blockbest) + c);
        const Best<V> o{Val<V>::from_bits(raw.x), (uint32_t)raw.y, (uint32_t)raw.z, (uint32_t)raw.w};
        cnt += __ldcg(blockcnt + c);
        if (Move::better(o, v)) v = o;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
    if (lane == 0) red_cnt[warp] = cnt;
    v = block_argmin<WARPS, Move>(v, red); // its barrier publishes red_cnt too
    cnt = 0;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) cnt += red_cnt[w];
    cnt_out = cnt;
    return v;
}

// Tail of a fused candidate-list relocation step (Or-opt N, 3-opt N), run by the scan's last CTA of
// WARPS warps: reduce the per-CTA records blockbest[0 .. grid) in Move's order, add the per-CTA counts of
// evaluated candidates to state->computed, then either relocate a span of at most kOrNlCtaSpan positions
// here through tmp and finish the step, or leave a longer one pending in blockbest[grid] for the apply
// grids (relocate_gather_kernel / relocate_scatter_kernel with pending_only).
template <int WARPS, class Move, class Pol>
__device__ __noinline__ void relocate_step_tail(const Pol &P, uint32_t n, uint32_t *pos, typename Pol::Rec *tmp,
                                                Best<typename Pol::V> *blockbest, const unsigned long long *blockcnt,
                                                DevState *state, unsigned int *ticket, tl_move *__restrict__ log,
                                                uint64_t log_cap)
{
    using V = typename Pol::V;
    StateHeader hdr{};
    if (threadIdx.x == 0) hdr = load_state_header(state);
    unsigned long long cnt;
    const Best<V> v = reduce_step_records<WARPS, Move>(blockbest, blockcnt, cnt);
    const Move m = Move::of(v);
    const bool long_span = m.found && m.hi - m.lo + 1 > (uint32_t)kOrNlCtaSpan;
    if (threadIdx.x == 0) {
        state->computed += cnt;
        // the pending move for this step's apply grids (none: the step is finished here)
        blockbest[gridDim.x] = long_span ? v : Best<V>{(V)0, 0xffffffffu, 0xffffffffu, 0u};
        *ticket = 0u;
    }
    if (long_span) return;
    if (m.found) {
        relocate_gather(P, tmp, m, threadIdx.x, blockDim.x);
        __syncthreads();
        relocate_scatter(P, tmp, n, m, pos, threadIdx.x, blockDim.x);
    }
    if (threadIdx.x == 0) finish_step(state, hdr, m.found, m.entry(), log, log_cap);
}

// The two apply grids of a relocating search, with the contract of apply_two_opt_kernel: every block
// reduces cand[0 .. ncand); with pending_only (Or-opt N's one pending record) no move means the scan
// already finished the step.  The gather grid writes nothing else, so it needs no pending_only.
template <class Pol, class Move>
__global__ void __launch_bounds__(256)
    relocate_gather_kernel(Pol P, typename Pol::Rec *__restrict__ tmp, const Best<typename Pol::V> *__restrict__ cand,
                           int ncand, const DevState *__restrict__ state)
{
    using V = typename Pol::V;
    griddep_wait(); // PDL launches only: the step's scan has finished and its writes are visible
    if (state->done) return;
    __shared__ Best<V> sred[8];
    const Move m = Move::of(block_argmin_records<Move>(cand, ncand, sred));
    if (m.found) relocate_gather(P, tmp, m, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
}

template <class Pol, class Move>
__global__ void __launch_bounds__(256)
    relocate_scatter_kernel(Pol P, const typename Pol::Rec *__restrict__ tmp, uint32_t n,
                            const Best<typename Pol::V> *__restrict__ cand, int ncand, DevState *state,
                            unsigned int *ticket, tl_move *__restrict__ log, uint64_t log_cap, uint32_t *pos,
                            int pending_only)
{
    using V = typename Pol::V;
    griddep_wait(); // PDL launches only: the gather grid has finished
    if (state->done) return;
    __shared__ Best<V> sred[8];
    const Move m = Move::of(block_argmin_records<Move>(cand, ncand, sred));
    if (pending_only && !m.found) return; // uniform over the grid
    if (m.found) relocate_scatter(P, tmp, n, m, pos, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
    __syncthreads();
    grid_finish_step(ticket, state, m.found, m.entry(), log, log_cap);
}

} // namespace tl
