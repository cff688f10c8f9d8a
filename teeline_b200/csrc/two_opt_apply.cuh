// two_opt_apply.cuh -- in-place 2-opt move on the tour-ordered records (any policy).
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

// Loop-state update after a Mode B step (one thread).  The header of DevState,
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
// Returns the value of state->done after the step.
__device__ __forceinline__ int finish_best_step(DevState *state, const StateHeader &h, bool found, float delta,
                                                uint32_t mi, uint32_t mj, tl_move *__restrict__ log,
                                                uint64_t log_cap)
{
    const unsigned long long m = h.h0.x;
    const long long max_moves = h.h1.x;
    state->scans = h.h0.y + 1;
    if (found) {
        if (log && m < log_cap) log[m] = tl_move{delta, mi, mj, 0, 0, 0};
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

// Last-CTA detection with ONE acq_rel atomic instead of fence.sc + relaxed atomic + fence.sc:
// release publishes this thread's candidate record, acquire (plus the caller's __syncthreads)
// orders the last CTA's reads of everybody else's records after it.
__device__ __forceinline__ unsigned int ticket_take_acq_rel(unsigned int *ticket)
{
    unsigned int old;
    asm volatile("atom.add.acq_rel.gpu.global.u32 %0, [%1], 1;" : "=r"(old) : "l"(ticket) : "memory");
    return old;
}

// Stand-alone apply step for Mode B (sharded sessions and the matrix path): every block
// reduces the candidate records redundantly (at most a few hundred), the grid reverses the
// segment, the last block to finish updates the loop state.
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
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    Best<V> v{(V)0, 0xffffffffu, 0xffffffffu, 0u};
    for (int c = threadIdx.x; c < ncand; c += blockDim.x) {
        const Best<V> o = cand[c];
        if (better_2opt(o.delta, o.i, o.j, v.delta, v.i, v.j)) v = o;
    }
    warp_argmin_2opt(v.delta, v.i, v.j);
    if (lane == 0) sred[warp] = v;
    __syncthreads();
    v = sred[0];
#pragma unroll
    for (int w = 1; w < 8; ++w) {
        const Best<V> o = sred[w];
        if (better_2opt(o.delta, o.i, o.j, v.delta, v.i, v.j)) v = o;
    }
    const bool found = v.i != 0xffffffffu;
    if (pending_only && !found) return; // uniform over the grid
    if (found)
        reverse_segment_inplace(P, v.i, v.j, nullptr, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x,
                                false, V(), V(), pos);
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned int tk = atomicAdd(ticket, 1u);
        if (tk == gridDim.x - 1) { // last block: everyone has read `state` by now
            *ticket = 0u;
            finish_best_step(state, load_state_header(state), found, (float)v.delta, v.i, v.j, log, log_cap);
            __threadfence();
        }
    }
}

} // namespace tl
