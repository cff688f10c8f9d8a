// k2_two_opt_ref.cu -- K2 "Mode R": the reference's first-improvement 2-opt, bit-exact.
//
// Reference loop (src/tsp/two_opt.rs:26-61):
//     while improved { improved = false;
//       for i in 0..n-3 { for j in i+2..n-1 {
//         if d(p_i,p_j) + d(p_i+1,p_j+1) < d(p_i,p_i+1) + d(p_j,p_j+1) { reverse p[i+1..=j]; improved = true } } } }
// i.e. a lexicographic cursor over (i,j) that applies a move the moment it finds one and
// keeps scanning the SAME row with the mutated path.  The comparison is between two
// separately rounded f32 sums (not a rearranged delta).
//
// GPU formulation: "find the lexicographically first improving pair at or after the cursor".
// One kernel per step (ref_step_kernel): every pair of a window of rows starting at the cursor
// is evaluated in parallel, the 64-bit key (i<<32|j) of the first improving one is minimised
// atomically, and the last CTA to finish reverses the segment in place, advances the cursor to
// (i, j+1) and resets the window; on a miss the cursor jumps past the window and the window
// grows 4x.  Everything (cursor, window, pass bookkeeping, termination) lives in DevState on
// the device; the host enqueues batches of steps and only looks at the done flag between batches.  The chain is serial by nature (every move
// changes the path the next comparison sees), so this path is latency- not throughput-bound;
// it exists for exact parity with the reference, not for the Tmove/s metric.
//
// PERSISTENT FORM (ref_persistent_kernel, coordinate problems whose tour records fit one SM's
// shared memory: n <= kRefPersistMaxN).  A step of the cursor is a few thousand pair evaluations
// followed by a serial decision, so the per-step kernel above is bound by launch + grid hand-off
// latency (about 7 us per step, 3842 steps at n = 10k).  Here ONE thread-block cluster of 16 (8)
// CTAs runs the whole chain in a single launch: every CTA holds a replica of the tour-ordered
// records in shared memory, the window's pairs are dealt to the cluster's warps, each CTA's first
// hit goes to every peer with one remote shared-memory store (DSMEM), ONE cluster barrier per
// step, and every CTA then applies the same reversal to its own replica.  Cursor, window and pass
// bookkeeping are replicated registers and go back to DevState when the launch ends (a move budget
// or a later tl_session_run resumes from there); only the window sizes differ from the per-step
// kernel's, which changes what is evaluated speculatively, never which move comes next.
#include "kernels.cuh"
#include "policy.cuh"
#include "apply.cuh"

#include <cooperative_groups.h>
#include <type_traits>

namespace tl {

namespace cg = cooperative_groups;

namespace {

constexpr unsigned long long kNoKey = ~0ull;

// One launch = one step of the cursor: find the first improving pair in the window, then the
// last CTA to finish applies it and advances the cursor (fused, like the Mode B step).
// The window [cur_i, cur_i + W) x columns is cut into UNITS of one row x 256 columns; a unit is
// one pair per thread, so a whole window is evaluated in a single parallel shot instead of a
// serial walk along the row.  Units are taken in (row, column) order by blockIdx, and a unit is
// skipped as soon as a lexicographically smaller hit is known.
template <class Pol>
__global__ void __launch_bounds__(256)
    ref_step_kernel(Pol P, uint32_t n, DevState *state, unsigned int *ticket, tl_move *__restrict__ log,
                    uint64_t log_cap)
{
    using V = typename Pol::V;
    using Rec = typename Pol::Rec;
    griddep_launch_dependents();
    griddep_wait();
    if (*reinterpret_cast<const volatile int *>(&state->done)) return;
    const uint32_t ci = (uint32_t)state->cur_i, cj = (uint32_t)state->cur_j;
    const uint32_t W = (uint32_t)state->window_rows;
    const uint32_t last_row = n - 4, last_col = n - 2;
    const uint32_t cpr = (n + 255) / 256; // column chunks per row (upper bound)
    volatile unsigned long long *gkey = &state->found_key;
    __shared__ unsigned int s_j, s_skip;
    __shared__ unsigned int s_last;

    const uint32_t rows = min(W, last_row - ci + 1);
    const uint64_t units = (uint64_t)rows * cpr;
    for (uint64_t u = blockIdx.x; u < units; u += gridDim.x) {
        const uint32_t w = (uint32_t)(u / cpr), c = (uint32_t)(u % cpr);
        const uint32_t i = ci + w;
        const uint32_t j0 = ((w == 0) ? cj : i + 2) + c * 256;
        if (j0 > last_col) continue; // block-uniform
        __syncthreads(); // the previous unit's s_j / s_skip have been consumed
        if (threadIdx.x == 0) {
            s_j = 0xffffffffu;
            // a smaller key is already known: nothing in this unit can be first
            s_skip = (*gkey < (((unsigned long long)i << 32) | j0)) ? 1u : 0u;
        }
        __syncthreads();
        if (s_skip) continue; // block-uniform
        const uint32_t j = j0 + threadIdx.x;
        if (j <= last_col) {
            const Rec pi = P.load(i), pi1 = P.load(i + 1);
            const Rec pj = P.load(j), pj1 = P.load(j + 1);
            // two separately rounded sums, compared directly (two_opt.rs:35-49)
            const V cur = Val<V>::add(Pol::sp(pi1), Pol::sp(pj1));
            const V nw = Val<V>::add(P.dist(pi, pj), P.dist(pi1, pj1));
            if (nw < cur) atomicMin(&s_j, j);
        }
        __syncthreads();
        if (threadIdx.x == 0 && s_j != 0xffffffffu)
            atomicMin(&state->found_key, ((unsigned long long)i << 32) | s_j);
    }

    // ---- fused tail: the last CTA applies the move and advances the cursor ----------------
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = (atomicAdd(ticket, 1u) == gridDim.x - 1) ? 1u : 0u;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const unsigned long long key = *gkey;
    const bool found = key != kNoKey;
    const uint32_t mi = (uint32_t)(key >> 32), mj = (uint32_t)key;
    if (found) reverse_segment_inplace(P, mi, mj, &state->last_delta, threadIdx.x, blockDim.x);
    __syncthreads();
    if (threadIdx.x == 0) {
        *ticket = 0u;
        int32_t ni, nj, nw;
        if (found) {
            const unsigned long long m = state->moves;
            if (log && m < log_cap) log[m] = tl_move{*(volatile float *)&state->last_delta, mi, mj, 0, 0, 0};
            state->moves = m + 1;
            state->improved_in_pass = 1;
            ni = (int32_t)mi;
            nj = (int32_t)mj + 1;
            if (nj > (int32_t)last_col) { ni += 1; nj = ni + 2; }
            nw = kRefWindow0;
            if (state->max_moves >= 0 && (long long)(m + 1) >= state->max_moves) state->done = 1;
        } else {
            ni = (int32_t)(ci + W);
            nj = ni + 2;
            nw = (int32_t)min(W * 4u, n);
        }
        if (ni > (int32_t)last_row) { // end of a pass over the triangle
            state->passes += 1;
            if (state->improved_in_pass) {
                state->improved_in_pass = 0;
                ni = 0;
                nj = 2;
                nw = kRefWindow0;
            } else {
                state->done = 1;
                state->converged = 1;
            }
        }
        state->cur_i = ni;
        state->cur_j = nj;
        state->window_rows = nw;
        state->found_key = kNoKey;
    }
}


// ---- persistent form ------------------------------------------------------------------------
#ifndef TL_REFP_THREADS
#define TL_REFP_THREADS 512
#endif
#ifndef TL_REFP_RB
#define TL_REFP_RB 4
#endif
#ifndef TL_REFP_ROUNDS
#define TL_REFP_ROUNDS 1 // first window after a hit: this many rounds of the cluster's warps
#endif
#ifndef TL_REFP_GROW
#define TL_REFP_GROW 4 // window growth after a miss
#endif
#ifdef TL_REFP_PROF
// tuning builds only (-DTL_REFP_PROF): cycles of rank 0 / thread 0 per phase, summed over the launch
// [0] steps, [1] hits, [2] units this warp evaluated, [3] eval cycles, [4] barrier cycles, [5] apply cycles,
// [6] whole-kernel cycles, [7] rows of all windows
__device__ unsigned long long tl_refp_prof[8];
#define REFP_CLK() clock64()
#define REFP_ADD(k, v) do { if (rank == 0 && tid == 0) tl_refp_prof[k] += (unsigned long long)(v); } while (0)
#else
#define REFP_CLK() 0ll
#define REFP_ADD(k, v) do { (void)(v); } while (0)
#endif
constexpr int kRefPThreads = TL_REFP_THREADS;
constexpr unsigned int kNoHit = 0xffffffffu;
constexpr int RB = TL_REFP_RB; // rows per unit: the 32 column records a warp loads serve RB pairs per lane
static_assert(kRefPersistMaxN <= (1 << 14), "keys are (row in window) << 14 | column");

__device__ __forceinline__ void cluster_barrier()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// Tour records in shared memory as arrays (x, y, city, entering-edge length [, matrix slot]): a warp's
// column loads and the reversal's stores touch consecutive words (conflict-free), and a load that
// needs only some fields costs only those.  Same interface as EucPol / MatPol (policy.cuh).
// Distances are recomputed in metric M.  The nint metrics belong to matrix sessions: the kernel
// recomputes the matrix entries from the coordinates (bit-equal by K1's construction) and carries
// every city's matrix slot along so that the Cs records can be restored.
template <Metric M>
struct SmemSoaPol {
    static constexpr bool kInt = metric_is_int(M);
    using V = MetricValue<M>;
    struct Rec {
        float x, y;
        int32_t city, slot;
        V sp;
    };
    float *x, *y;
    int32_t *cty, *spl, *slt;
    __device__ __forceinline__ Rec load(uint32_t q) const
    {
        return Rec{x[q], y[q], cty[q], kInt ? slt[q] : 0, Val<V>::from_bits(spl[q])};
    }
    static __device__ __forceinline__ V sp(const Rec &r) { return r.sp; }
    __device__ __forceinline__ V dist(const Rec &a, const Rec &b) const { return tl::dist<M>(a.x, a.y, b.x, b.y); }
    __device__ __forceinline__ void store_id(uint32_t q, const Rec &from) const
    {
        x[q] = from.x;
        y[q] = from.y;
        cty[q] = from.city;
        if constexpr (kInt) slt[q] = from.slot;
    }
    __device__ __forceinline__ void store_sp(uint32_t q, V v) const { spl[q] = Val<V>::bits(v); }
};

// max_steps cursor steps (or until done).  Window unit = (block of RB rows, 32 consecutive columns):
// a warp loads the 32 column records once and evaluates RB pairs per lane.
// key = (row in window) << 14 | column orders the window's pairs lexicographically; the cluster-wide
// minimum key is the reference's next move.
template <Metric M, bool SCREEN>
__global__ void __launch_bounds__(kRefPThreads, 1)
    ref_persistent_kernel(Pt *__restrict__ pts, Cs *__restrict__ cs, const float2 *__restrict__ xy, uint32_t n,
                          DevState *state, tl_move *__restrict__ log, uint64_t log_cap, uint32_t max_steps,
                          float margin)
{
    using Pol = SmemSoaPol<M>;
    using V = typename Pol::V;
    using Rec = typename Pol::Rec;
    constexpr bool kInt = Pol::kInt;
    extern __shared__ __align__(16) unsigned char ref_smem[];
    const uint32_t na = (n + 3u) & ~3u; // array pitch (words)
    const Pol P{reinterpret_cast<float *>(ref_smem), reinterpret_cast<float *>(ref_smem) + na,
                reinterpret_cast<int32_t *>(ref_smem) + 2 * (size_t)na, reinterpret_cast<int32_t *>(ref_smem) + 3 * (size_t)na,
                reinterpret_cast<int32_t *>(ref_smem) + 4 * (size_t)na};
    // [step parity]: the smallest hit key of the step known so far, CLUSTER-wide -- a warp that finds a
    // hit pushes it into every CTA's copy with a remote atomicMin (DSMEM), so every warp of the cluster
    // stops evaluating pairs behind it, and after the step's cluster barrier every copy holds the move
    __shared__ unsigned int s_min[2];
    __shared__ float s_delta;

    cg::cluster_group cluster = cg::this_cluster();
    const unsigned int rank = cluster.block_rank(), csize = cluster.num_blocks();
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t gwarp = warp * csize + rank, nwarps = (kRefPThreads / 32) * csize; // early units spread over the CTAs

    if (*reinterpret_cast<const volatile int *>(&state->done)) return; // cluster-uniform
    for (uint32_t q = tid; q < n; q += kRefPThreads) {
        if constexpr (kInt) {
            const int4 v = __ldcg(reinterpret_cast<const int4 *>(cs) + q); // Cs = {slot, sp bits, city, pad}
            const float2 c = __ldg(&xy[v.z]);
            P.x[q] = c.x;
            P.y[q] = c.y;
            P.cty[q] = v.z;
            P.spl[q] = v.y;
            P.slt[q] = v.x;
        } else {
            const float4 v = __ldcg(reinterpret_cast<const float4 *>(pts) + q); // Pt = {x, y, city, sp}
            P.x[q] = v.x;
            P.y[q] = v.y;
            P.cty[q] = __float_as_int(v.z);
            P.spl[q] = __float_as_int(v.w);
        }
    }
    if (tid == 0) s_min[0] = s_min[1] = kNoHit;
    // replicated loop state
    uint32_t ci = (uint32_t)state->cur_i, cj = (uint32_t)state->cur_j, W = (uint32_t)state->window_rows;
    int improved = state->improved_in_pass;
    unsigned long long moves = state->moves, passes = state->passes;
    const long long max_moves = state->max_moves;
    int done = 0, converged = 0;
    const uint32_t last_row = n - 4, last_col = n - 2;
    // The window right after a hit (or at the start of a pass): as many row blocks as give every warp
    // of the cluster one unit -- a step costs its synchronisation, not its pairs (1, 2 or 3 rounds and
    // growth factors 2 / 4 / 8 after a miss all end within 2 % of each other at n = 10k; one round is
    // 18 % faster at n = 1000, profiles/r03u_mode_r_persistent_soa_and_window_policy.txt).
    auto first_window = [&](uint32_t row) {
        const uint32_t chunks = (last_col - (min(row, last_row) + 2) + 1 + 31) / 32;
        return (uint32_t)RB * max(1u, min(64u, (uint32_t)TL_REFP_ROUNDS * nwarps / chunks));
    };
    if (W == (uint32_t)kRefWindow0) W = first_window(ci); // a state the per-step kernel (or session create) left
    __syncthreads();
    cluster_barrier(); // nobody pushes a hit into a peer's copy before that peer has armed it

    const long long tk0 = REFP_CLK();
    for (uint32_t step = 0; step < max_steps && !done; ++step) {
        const long long tp0 = REFP_CLK();
        const uint32_t par = step & 1u;
        // re-arm the other copy for the next step: peers push into it only after this step's barrier,
        // and this CTA's reads of it (the previous step's move) ended at that step's last __syncthreads
        if (tid == 0) s_min[par ^ 1u] = kNoHit;
        const uint32_t rows = min(W, last_row - ci + 1);
        const uint32_t cpr = (last_col - (ci + 2) + 1 + 31) / 32; // 32-column chunks of the window's longest row
        const uint32_t nblk = (rows + RB - 1) / RB;
        const uint32_t units = nblk * cpr;
        unsigned int mine = kNoHit;
        const uint32_t dq = nwarps / cpr, dr = nwarps - dq * cpr; // unit stride in (block, chunk) form
        uint32_t b = gwarp / cpr, c = gwarp - b * cpr;            // one division per step
        auto next_unit = [&]() { // (block, chunk) of the warp's next unit
            c += dr;
            b += dq;
            if (c >= cpr) { c -= cpr; b += 1; }
        };
        for (uint32_t u = gwarp; u < units; u += nwarps, next_unit()) {
            const uint32_t w0 = b * RB;
            const uint32_t i0 = ci + w0;
            const uint32_t jw = i0 + 2 + c * 32; // the warp's first column
            if (jw > last_col) continue;         // the chunk lies beyond the end of these (shorter) rows
            // every key of this and of the warp's later units is at least (first row of the block) << 14:
            // stop once a smaller hit is known (this warp's, or any in the cluster -- one read per warp)
            unsigned int known = 0;
            if (lane == 0) known = *reinterpret_cast<volatile unsigned int *>(&s_min[par]);
            known = min(mine, __shfl_sync(0xffffffffu, known, 0));
            if ((w0 << 14) > known) break;
            REFP_ADD(2, 1);
            const uint32_t j = jw + lane;
            const uint32_t nr = min((uint32_t)RB, rows - w0); // rows of this block inside the window
            // FULL: every (row, lane) of the unit is a pair of the window -- no per-pair range tests
            const bool full = nr == (uint32_t)RB && w0 != 0 && c != 0 && jw + 31 <= last_col;
            static_assert(RB <= 33, "chunk 1 starts right of every row's first column");
            const bool jin = j <= last_col;
            Rec pj{}, pj1{};
            if (jin) {
                pj = P.load(j);
                pj1 = P.load(j + 1);
            }
            Rec pi[RB + 1];
#pragma unroll
            for (int r = 0; r <= RB; ++r)
                if ((uint32_t)r <= nr) pi[r] = P.load(i0 + r); // i0 + nr <= last_row + 1
            // screened comparison: new < cur  =>  screened new < cur + margin (the margin covers the
            // screened distances' error and, for the nint metrics, the two roundings to integers)
            float spj1f = 0.f;
            if constexpr (SCREEN) spj1f = __fadd_rn((float)pj1.sp, margin);
            bool cand[RB];
            auto eval_rows = [&](auto FullC) {
                constexpr bool FULL = decltype(FullC)::value;
#pragma unroll
                for (int r = 0; r < RB; ++r) {
                    cand[r] = false;
                    // row i0 + r starts at column i + 2, the cursor's own row at cur_j
                    const uint32_t jfirst = (w0 + r == 0) ? cj : i0 + r + 2;
                    if (FULL || ((uint32_t)r < nr && jin && j >= jfirst)) {
                        if constexpr (SCREEN) { // cheap distances; anything within the error margin is re-checked exactly
                            const float nws = __fadd_rn(dist_f32_screen(pi[r].x, pi[r].y, pj.x, pj.y),
                                                        dist_f32_screen(pi[r + 1].x, pi[r + 1].y, pj1.x, pj1.y));
                            cand[r] = nws < __fadd_rn((float)pi[r + 1].sp, spj1f);
                        } else {
                            // two separately rounded sums, compared directly (two_opt.rs:35-49)
                            cand[r] = Val<V>::add(P.dist(pi[r], pj), P.dist(pi[r + 1], pj1)) < Val<V>::add(pi[r + 1].sp, pj1.sp);
                        }
                    }
                }
            };
            if (full)
                eval_rows(std::true_type{});
            else
                eval_rows(std::false_type{});
            bool any_cand = false;
#pragma unroll
            for (int r = 0; r < RB; ++r) any_cand |= cand[r];
            if (__ballot_sync(0xffffffffu, any_cand) == 0) continue; // the common case: one vote per unit
            bool hit_here = false;
#pragma unroll
            for (int r = 0; r < RB; ++r) {
                unsigned int bal = __ballot_sync(0xffffffffu, cand[r]);
                if (SCREEN && bal && !hit_here) { // warp-uniform: the exact comparison for this row's candidates
                    bool hit = false;
                    if (cand[r])
                        hit = Val<V>::add(P.dist(pi[r], pj), P.dist(pi[r + 1], pj1)) < Val<V>::add(pi[r + 1].sp, pj1.sp);
                    bal = __ballot_sync(0xffffffffu, hit);
                }
                if (bal && !hit_here) { // the block's rows in order: the first row with a hit holds its smallest key
                    hit_here = true;
                    mine = min(mine, ((w0 + r) << 14) | (jw + (uint32_t)(__ffs(bal) - 1)));
                }
            }
            if (hit_here && lane < csize) atomicMin(cluster.map_shared_rank(&s_min[par], lane), mine);
        }
        const long long tp1 = REFP_CLK();
        cluster_barrier(); // release/acquire: every hit of the step has landed in every copy
        const long long tp2 = REFP_CLK();
        const unsigned int key = s_min[par];
        const bool found = key != kNoHit;
        uint32_t ni, nj, nw_rows;
        if (found) {
            const uint32_t mi = ci + (key >> 14), mj = key & 16383u;
            reverse_segment_inplace(P, mi, mj, &s_delta, tid, kRefPThreads);
            __syncthreads();
            if (rank == 0 && tid == 0 && log && moves < log_cap) log[moves] = tl_move{s_delta, mi, mj, 0, 0, 0};
            moves += 1;
            improved = 1;
            ni = mi;
            nj = mj + 1;
            if (nj > last_col) { ni += 1; nj = ni + 2; }
            nw_rows = 0; // the first window of the new cursor, sized below
            if (max_moves >= 0 && (long long)moves >= max_moves) done = 1;
        } else {
            ni = ci + W;
            nj = ni + 2;
            nw_rows = min(W * (uint32_t)TL_REFP_GROW, n);
            __syncthreads(); // (the found branch's barrier: the steps stay symmetric)
        }
        if (ni > last_row) { // end of a pass over the triangle
            passes += 1;
            if (improved) {
                improved = 0;
                ni = 0;
                nj = 2;
                nw_rows = 0;
            } else {
                done = 1;
                converged = 1;
            }
        }
        ci = ni;
        cj = nj;
        W = nw_rows ? nw_rows : first_window(ci);
        REFP_ADD(0, 1);
        REFP_ADD(1, found ? 1 : 0);
        REFP_ADD(3, tp1 - tp0);
        REFP_ADD(4, tp2 - tp1);
        REFP_ADD(5, REFP_CLK() - tp2);
        REFP_ADD(7, rows);
    }
    REFP_ADD(6, REFP_CLK() - tk0);

    if (rank == 0) {
        for (uint32_t q = tid; q < n; q += kRefPThreads) {
            if constexpr (kInt)
                reinterpret_cast<int4 *>(cs)[q] = make_int4(P.slt[q], P.spl[q], P.cty[q], 0);
            else
                reinterpret_cast<float4 *>(pts)[q] =
                    make_float4(P.x[q], P.y[q], __int_as_float(P.cty[q]), __int_as_float(P.spl[q]));
        }
        if (tid == 0) {
            state->moves = moves;
            state->passes = passes;
            state->improved_in_pass = improved;
            state->cur_i = (int32_t)ci;
            state->cur_j = (int32_t)cj;
            state->window_rows = (int32_t)W;
            state->found_key = kNoKey;
            if (done) state->done = 1;
            if (converged) state->converged = 1;
        }
    }
    cluster_barrier(); // no CTA leaves while a peer may still push into its shared memory
}

template <class Pol>
__global__ void extract_tour_kernel(Pol P, uint32_t n, uint32_t *__restrict__ tour)
{
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < n; q += gridDim.x * blockDim.x)
        tour[q] = (uint32_t)Pol::city(P.load(q));
}

} // namespace

void launch_ref_step(const Src &src, uint32_t n, DevState *state, unsigned int *ticket, tl_move *log,
                     uint64_t log_cap, int grid, cudaStream_t st)
{
    cudaLaunchAttribute attr[1];
    const cudaLaunchConfig_t cfg = pdl_config(grid, 256, 0, attr, st);
    TL_DISPATCH_POL(src, (cudaLaunchKernelEx(&cfg, ref_step_kernel<decltype(P)>, P, n, state, ticket, log,
                                             (uint64_t)log_cap)));
}

#ifdef TL_REFP_PROF
} // namespace tl
extern "C" int tl_debug_refp(double *out8, int reset)
{
    unsigned long long h[8];
    if (cudaMemcpyFromSymbol(h, tl::tl_refp_prof, sizeof h) != cudaSuccess) return 1;
    for (int k = 0; k < 8; ++k) out8[k] = (double)h[k];
    if (reset) {
        const unsigned long long z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        cudaMemcpyToSymbol(tl::tl_refp_prof, z, sizeof z);
    }
    return 0;
}
namespace tl {
#endif

// The persistent form: one cluster of `csize` CTAs (16 needs the non-portable opt-in; 8 otherwise).
namespace {
using RefPFn = void (*)(Pt *, Cs *, const float2 *, uint32_t, DevState *, tl_move *, uint64_t, uint32_t, float);
RefPFn refp_fn(Metric metric, bool screen)
{
    return with_metric(metric, [&](auto M) -> RefPFn {
        if constexpr (M == Metric::F32_SAFE) return ref_persistent_kernel<M, false>; // no screening outside the fast-sqrt domain
        else return screen ? ref_persistent_kernel<M, true> : ref_persistent_kernel<M, false>;
    });
}
size_t refp_smem_bytes(Metric metric, uint32_t n) { return (size_t)((n + 3u) & ~3u) * (metric_is_int(metric) ? 20 : 16); }
} // namespace

// Returns the cluster size this device can run for n records, 0 if the form does not apply.
int ref_persistent_cluster_size(std::optional<Metric> metric, uint32_t n)
{
    if (!metric || n < 4 || n > (uint32_t)(metric_is_int(*metric) ? kRefPersistMaxNInt : kRefPersistMaxN)) return 0;
    static int cached_size = -1; // every instantiation has the same shape; the answer for the largest n holds for every n
    if (cached_size >= 0) return cached_size;
    const size_t smem = (size_t)kRefPersistMaxN * 16;
    static_assert((size_t)kRefPersistMaxNInt * 20 <= (size_t)kRefPersistMaxN * 16, "one shared-memory opt-in for all");
    int best = 0;
    bool ok = true;
    for (Metric m : kMetrics)
        for (int sc = 0; sc < 2; ++sc)
            ok = ok && cudaFuncSetAttribute((const void *)refp_fn(m, sc != 0), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess &&
                 cudaFuncSetAttribute((const void *)refp_fn(m, sc != 0), cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess;
    if (ok) {
        for (int cs : {16, 8, 4, 2}) {
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeClusterDimension;
            attr[0].val.clusterDim.x = (unsigned)cs;
            attr[0].val.clusterDim.y = 1;
            attr[0].val.clusterDim.z = 1;
            cudaLaunchConfig_t cfg{};
            cfg.gridDim = dim3((unsigned)cs);
            cfg.blockDim = dim3(kRefPThreads);
            cfg.dynamicSmemBytes = smem;
            cfg.attrs = attr;
            cfg.numAttrs = 1;
            int nclusters = 0;
            if (cudaOccupancyMaxActiveClusters(&nclusters, (const void *)refp_fn(Metric::NINT_GRID, true), &cfg) == cudaSuccess && nclusters >= 1) {
                best = cs;
                break;
            }
            cudaGetLastError();
        }
    }
    cudaGetLastError();
    if (const char *ev = getenv("TL_REF_CLUSTER")) { // tuning: 0 = per-step kernel, 2/4/8/16 = at most this size
        const int want = atoi(ev);
        if (want <= 0) best = 0;
        else if (want < best) best = want;
    }
    cached_size = best;
    return best;
}

// screen_margin >= 0 (fast-sqrt domain only, common.cuh: kScreenMarginScale): screened distances first;
// the nint metrics add the two roundings to integers (1.0) to it
void launch_ref_persistent(const Src &src, const float2 *xy, Metric metric, uint32_t n, DevState *state, tl_move *log,
                           uint64_t log_cap, uint32_t max_steps, int csize, float screen_margin, cudaStream_t st)
{
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)csize;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)csize);
    cfg.blockDim = dim3(kRefPThreads);
    cfg.dynamicSmemBytes = refp_smem_bytes(metric, n);
    cfg.stream = st;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const bool screen = screen_margin >= 0.0f && metric != Metric::F32_SAFE;
    const float margin = screen ? (metric_is_int(metric) ? screen_margin + 1.0009765625f : screen_margin) : -1.0f;
    cudaLaunchKernelEx(&cfg, refp_fn(metric, screen), src.pts, src.cs, xy, n, state, log, (uint64_t)log_cap, max_steps, margin);
}

void launch_apply_two_opt(const Src &src, const void *cand, int ncand, DevState *state, unsigned int *ticket,
                          tl_move *log, uint64_t log_cap, int grid, cudaStream_t st)
{
    TL_DISPATCH_POL(src, (apply_two_opt_kernel<<<grid, 256, 0, st>>>(
                             P, reinterpret_cast<const Best<typename decltype(P)::V> *>(cand), ncand, state,
                             ticket, log, log_cap, nullptr, 0)));
}

void launch_extract_tour(const Src &src, uint32_t n, uint32_t *tour, cudaStream_t st)
{
    TL_DISPATCH_POL(src, (extract_tour_kernel<<<(n + 255) / 256, 256, 0, st>>>(P, n, tour)));
}

} // namespace tl
