// k2_two_opt_cached.cu -- K2 "Mode B" with cached row minima: the same best-improvement 2-opt as
// k2_two_opt.cu / k2_two_opt_matrix.cu (same delta, same argmin rule, hence the same move sequence
// and the same local optimum, move for move), but a step re-evaluates only the pairs a move can
// have changed.
//
// After the move (I, J) -- reverse p[I+1 ..= J] -- the delta of pair (i, j), which is built from the
// edges (p_i, p_i+1) and (p_j, p_j+1), is unchanged unless one of its edges lies in [I, J]:
//   * rows i in [I, J]: the row's own edge changed (or was reversed) -> the whole row is rescanned;
//   * rows i < I: only the columns j in [I, J] changed -> those L+1 pairs are evaluated and merged
//     into the row's cached minimum -- unless that minimum sat on one of the changed columns, then
//     the row is rescanned;
//   * rows i > J: nothing changed.
// Every row keeps its minimum as ONE 64-bit key (order-preserving delta bits << 32 | j), merged with
// atomicMin; the step's move is the (delta, row, j) minimum over the rows' keys -- the reference scan
// order.  On the 10k instance the median move reverses a handful of cities and the whole search
// computes 7.6 % of the pair deltas full scans compute (5.7e9 against 7.5e10), but the work is skewed:
// most steps touch a few rows and cost their fixed latency (a launch, ~10 dependent L2 round trips:
// ~20 us), and the few moves that reverse thousands of cities rescan most rows with a row-oriented
// evaluation (two distances per pair instead of the diagonal walk's one: ~200 us for all rows at 10k
// against 35 us for a diagonal scan).  Measured (profiles/r03j_cached_timing.txt): to the local optimum
// at n = 10k 39.4 ms against 45.7 (f32 recompute) and 57 against 60 (nint matrix); n = 20k f32 127 ms
// for 2956 moves (a full scan there is ~110 us per step); from an NN start at 50k-100k the first 400
// moves are long reversals and full scans are faster (533 against 693 us per step at 50k).  It is an
// opt-in (TL_ALGO_TWO_OPT_BEST_CACHED) for searches that start near a local optimum or run long; the
// full-scan kernels remain the Tmove/s path and the default.
//
// One kernel per step (PDL between steps): every CTA takes work units of the step's description
// (written by the previous step's tail), the last CTA reduces the row keys, applies the move in
// place and writes the next description.
#include "kernels.cuh"
#include "policy.cuh"
#include "apply.cuh"

#include <cstdlib>

namespace tl {

namespace {

constexpr unsigned long long kNoKey = ~0ull;
constexpr int PC = 32;   // columns of a partial-row work unit (256 rows x PC columns, one row per thread)
constexpr int kSplitBelow = 64, kRowParts = 4; // fewer rescanned rows than this: every row in kRowParts units

template <typename V>
__device__ __forceinline__ unsigned int ord_bits(V d);
template <>
__device__ __forceinline__ unsigned int ord_bits<float>(float d)
{
    const unsigned int u = __float_as_uint(d);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u); // ascending with d
}
template <>
__device__ __forceinline__ unsigned int ord_bits<int32_t>(int32_t d)
{
    return (unsigned int)d ^ 0x80000000u;
}
template <typename V>
__device__ __forceinline__ V ord_value(unsigned int k);
template <>
__device__ __forceinline__ float ord_value<float>(unsigned int k)
{
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}
template <>
__device__ __forceinline__ int32_t ord_value<int32_t>(unsigned int k)
{
    return (int32_t)(k ^ 0x80000000u);
}

// delta of pair (i, j) from its four records, the formula of every Mode B kernel.  `sym`: take the
// two distances as d(p_j, p_i), d(p_j+1, p_i+1) -- bitwise the same value (the metric and the matrix
// are symmetric), but adjacent THREADS then read adjacent matrix columns when they sit on adjacent rows.
template <class Pol>
__device__ __forceinline__ typename Pol::V pair_delta(const Pol &P, const typename Pol::Rec &pi,
                                                      const typename Pol::Rec &pi1, const typename Pol::Rec &pj,
                                                      const typename Pol::Rec &pj1, bool sym)
{
    using V = typename Pol::V;
    const V e1 = sym ? P.dist(pj, pi) : P.dist(pi, pj);
    const V e2 = sym ? P.dist(pj1, pi1) : P.dist(pi1, pj1);
    return Val<V>::sub(Val<V>::add(e1, e2), Val<V>::add(Pol::sp(pi1), Pol::sp(pj1)));
}

template <class Pol>
__global__ void __launch_bounds__(256)
    two_opt_cached_step_kernel(Pol P0, int n, int cyclic, unsigned long long *__restrict__ rowkey, CachedDesc *desc,
                               int *__restrict__ fullrows, DevState *state, unsigned int *ticket,
                               tl_move *__restrict__ log, uint64_t log_cap)
{
    using V = typename Pol::V;
    using Rec = typename Pol::Rec;
#ifdef TL_CACHED_PLAIN
    const Pol &P = P0; // experiment: plain (L1-cached) record loads
#else
    const L2Pol<Pol> P(P0);
#endif
    griddep_launch_dependents();
    griddep_wait(); // the previous step's move is applied and its description written
    if (*reinterpret_cast<const volatile int *>(&state->done)) return;
    const int tid = threadIdx.x, lane = tid & 31;
    const int jmax = cyclic ? n - 1 : n - 2;
    const int nrows = jmax - 1; // rows 0 .. jmax-2
    const int nfull_raw = *reinterpret_cast<const volatile int *>(&desc->nfull);
    const int I = *reinterpret_cast<const volatile int *>(&desc->I), J = *reinterpret_cast<const volatile int *>(&desc->J);
    const int npart = *reinterpret_cast<const volatile int *>(&desc->npart_rows);
    // only the first `active` CTAs work on this step (a small step would otherwise pay for a thousand
    // CTAs queueing on the last-CTA ticket); the others leave at once
    const int active = *reinterpret_cast<const volatile int *>(&desc->active);
    // Every CTA reports that it has read the description (fire-and-forget).  The tail rewrites the
    // description for the next step and must not do so while a CTA of THIS grid has yet to read it: a
    // grid of 1184 CTAs is not resident at once (2 CTAs per SM for the 102-register instantiation),
    // and a CTA that starts after a short step's tail would take the next step's description for its
    // own -- work on it, take a ticket, and let the next step's tail start early (seen as a wrong move
    // or an illegal address once in ~10 runs at n = 1000 before this counter existed).
    if (tid == 0) atomicAdd(ticket + 1, 1u);
    if ((int)blockIdx.x >= active) return;
    const bool all_rows = nfull_raw < 0;
    const int nfull = all_rows ? nrows : nfull_raw;
    // a rescanned row is one work unit (a CTA walks it with the minimum in registers: one atomic per
    // row); when a step rescans only a few rows, each is cut into kRowParts units so that it does not
    // take one CTA a whole row's time
    const int parts = nfull >= kSplitBelow ? 1 : kRowParts;
    const long long units_full = (long long)nfull * parts;
    const int pcc = npart > 0 ? (J - I + PC) / PC : 0; // column chunks of the partial rows: columns I .. J
    const long long units = units_full + (long long)((npart + 255) / 256) * pcc;
    unsigned int computed = 0; // pairs evaluated by this thread in this step
    __shared__ unsigned long long s_wkey[8];

    for (long long u = blockIdx.x; u < units; u += active) {
        if (u < units_full) {
            // ---- (a part of) one row that is rescanned from scratch: columns row+2 .. jmax
            const int f = (int)(u / parts), part = (int)(u - (long long)f * parts);
            const int row = all_rows ? f : __ldcg(&fullrows[f]);
            const int ncol = jmax - (row + 2) + 1, per = (ncol + parts - 1) / parts;
            const int jb = row + 2 + part * per;
            int je = min(jmax, jb + per - 1);
            const Rec pi = P.load(row), pi1 = P.load(row + 1);
            if (cyclic && row == 0) je = min(je, n - 2); // the cyclic neighbourhood excludes (0, n-1)
            // four columns per thread and round, all eight record loads of a round issued before the first
            // delta; the running minimum is (delta, j) in two registers -- j ascends within a thread, so a
            // strict '<' keeps the lowest column of equal deltas
            V bd = (V)0;
            int bj = -1;
            for (int j0 = jb + tid; j0 <= je; j0 += 1024) {
                Rec a[4], b[4];
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    if (j0 + 256 * e <= je) {
                        a[e] = P.load(j0 + 256 * e);
                        b[e] = P.load(j0 + 256 * e + 1);
                    }
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    if (j0 + 256 * e <= je) {
                        const V d = pair_delta(P, pi, pi1, a[e], b[e], false);
                        if (d < bd) { bd = d; bj = j0 + 256 * e; }
                    }
            }
            if (jb + tid <= je) computed += (unsigned int)((je - (jb + tid)) / 256 + 1);
            const unsigned long long key = bj < 0 ? kNoKey : (((unsigned long long)ord_bits<V>(bd) << 32) | (unsigned int)bj);
            // CTA minimum of the 64-bit keys: two REDUX per warp, eight keys through shared memory
            const unsigned int hi = (unsigned int)(key >> 32);
            const unsigned int whi = __reduce_min_sync(0xffffffffu, hi);
            const unsigned int lo = hi == whi ? (unsigned int)key : 0xffffffffu;
            const unsigned int wlo = __reduce_min_sync(0xffffffffu, lo);
            __syncthreads(); // the previous unit's s_wkey has been consumed
            if (lane == 0) s_wkey[tid >> 5] = ((unsigned long long)whi << 32) | wlo;
            __syncthreads();
            if (tid == 0) {
                unsigned long long k = s_wkey[0];
#pragma unroll
                for (int w = 1; w < 8; ++w) k = min(k, s_wkey[w]);
                // atomicMin, not a store: a row that is rescanned because its minimum sat on a changed
                // column also receives the partial units' candidates (a subset of this scan's)
                if (k != kNoKey) atomicMin(&rowkey[row], k);
            }
        } else {
            // ---- rows above the reversed segment: only the columns I .. J changed; one row per thread,
            //      PC columns per unit (adjacent threads read adjacent matrix columns: pair_delta's sym)
            const long long v = u - units_full;
            const int rb = (int)(v / pcc), cc = (int)(v - (long long)rb * pcc);
            const int row = rb * 256 + tid;
            if (row < npart) {
                const Rec pi = P.load(row), pi1 = P.load(row + 1);
                const int j0 = max(row + 2, I + cc * PC);
                int j1 = min(min(J, jmax), I + cc * PC + PC - 1);
                if (cyclic && row == 0) j1 = min(j1, n - 2);
                V bd = (V)0;
                int bj = -1;
                for (int jq = j0; jq <= j1; jq += 4) {
                    Rec a[4], b[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e)
                        if (jq + e <= j1) {
                            a[e] = P.load(jq + e);
                            b[e] = P.load(jq + e + 1);
                        }
#pragma unroll
                    for (int e = 0; e < 4; ++e)
                        if (jq + e <= j1) {
                            const V d = pair_delta(P, pi, pi1, a[e], b[e], true);
                            if (d < bd) { bd = d; bj = jq + e; }
                        }
                }
                if (j1 >= j0) computed += (unsigned int)(j1 - j0 + 1);
                const unsigned long long key = bj < 0 ? kNoKey : (((unsigned long long)ord_bits<V>(bd) << 32) | (unsigned int)bj);
                if (key != kNoKey) atomicMin(&rowkey[row], key);
            }
        }
    }

    // ---- the last CTA to finish: the step's move, its application, the next step's description
    __shared__ unsigned int s_last;
    __shared__ unsigned long long s_key[8];
    __shared__ int s_row[8];
    __shared__ int s_nfull;
    __shared__ unsigned long long s_computed;
    if (tid == 0) s_computed = 0ull;
    __syncthreads();
    {   // one global atomic per CTA for the count of computed pairs
        const unsigned int wsum = __reduce_add_sync(0xffffffffu, (unsigned int)computed); // < 2^32 per warp and step
        if (lane == 0 && wsum) atomicAdd(&s_computed, (unsigned long long)wsum);
    }
    __syncthreads();
    if (tid == 0) {
        if (s_computed) atomicAdd(&state->computed, s_computed);
        s_last = (ticket_take_acq_rel(ticket) == (unsigned int)active - 1u) ? 1u : 0u;
    }
    __syncthreads();
    if (!s_last) return;
    StateHeader hdr{};
    if (tid == 0) hdr = load_state_header(state);
    // (delta, i, j) lexicographic: the keys order (delta, j) within a row, so across rows compare the
    // delta word first, then the row, and only then j
    auto better = [](unsigned long long ka, int ra, unsigned long long kb, int rb) {
        const unsigned int da = (unsigned int)(ka >> 32), db = (unsigned int)(kb >> 32);
        if (da != db) return da < db;
        if (ra != rb) return ra < rb;
        return (unsigned int)ka < (unsigned int)kb;
    };
    unsigned long long bk = kNoKey;
    int br = 0x7fffffff;
    // sixteen keys per thread in flight (eight 16-byte loads): the reduction is two or three L2 round
    // trips at n = 10 000, not nrows / 256 (the array is padded to an even count of keys, all "none")
    for (int r0 = 2 * tid; r0 < nrows; r0 += 512 * 8) {
        ulonglong2 k[8];
#pragma unroll
        for (int e = 0; e < 8; ++e)
            k[e] = r0 + 512 * e < nrows ? __ldcg(reinterpret_cast<const ulonglong2 *>(rowkey + r0 + 512 * e))
                                        : make_ulonglong2(kNoKey, kNoKey);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int r = r0 + 512 * e;
            if (k[e].x != kNoKey && better(k[e].x, r, bk, br)) { bk = k[e].x; br = r; }
            if (k[e].y != kNoKey && better(k[e].y, r + 1, bk, br)) { bk = k[e].y; br = r + 1; }
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const unsigned long long ok = __shfl_xor_sync(0xffffffffu, bk, off);
        const int orow = __shfl_xor_sync(0xffffffffu, br, off);
        if (ok != kNoKey && better(ok, orow, bk, br)) { bk = ok; br = orow; }
    }
    if (lane == 0) { s_key[tid >> 5] = bk; s_row[tid >> 5] = br; }
    __syncthreads();
    bk = s_key[0];
    br = s_row[0];
#pragma unroll
    for (int w = 1; w < 8; ++w)
        if (s_key[w] != kNoKey && better(s_key[w], s_row[w], bk, br)) { bk = s_key[w]; br = s_row[w]; }
    const bool found = bk != kNoKey;
    const int mi = br, mj = (int)(unsigned int)bk;
    if (found) {
        reverse_segment_inplace(P, (uint32_t)mi, (uint32_t)mj, nullptr, (uint32_t)tid, 256u);
        // every CTA of this grid has read the description before it is rewritten (see above)
        if (tid == 0)
            while (*reinterpret_cast<volatile unsigned int *>(ticket + 1) < gridDim.x) {}
        __syncthreads();
        // which rows the move invalidates (see the header); more than a third of the rows: rescan them all
        const int seg_rows = min(mj, nrows - 1) - mi + 1;
        if (tid == 0) s_nfull = 0;
        __syncthreads();
        if ((long long)seg_rows * 3 > nrows) {
            for (int r = tid; r < nrows; r += 256) rowkey[r] = kNoKey;
            if (tid == 0) {
                desc->nfull = -1;
                desc->npart_rows = 0;
            }
        } else {
            for (int r = mi + tid; r <= min(mj, nrows - 1); r += 256) {
                rowkey[r] = kNoKey;
                fullrows[atomicAdd(&s_nfull, 1)] = r;
            }
            for (int r0 = 2 * tid; r0 < mi; r0 += 512 * 8) {
                ulonglong2 k[8];
#pragma unroll
                for (int e = 0; e < 8; ++e)
                    k[e] = r0 + 512 * e < mi ? __ldcg(reinterpret_cast<const ulonglong2 *>(rowkey + r0 + 512 * e))
                                             : make_ulonglong2(kNoKey, kNoKey);
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const unsigned long long kk[2] = {k[e].x, k[e].y};
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int r = r0 + 512 * e + h, cj = (int)(unsigned int)kk[h];
                        if (r < mi && kk[h] != kNoKey && cj >= mi && cj <= mj) { // its minimum sat on a changed column
                            rowkey[r] = kNoKey;
                            fullrows[atomicAdd(&s_nfull, 1)] = r;
                        }
                    }
                }
            }
            __syncthreads();
            if (tid == 0) {
                desc->nfull = s_nfull;
                desc->npart_rows = mi;
            }
        }
        if (tid == 0) {
            desc->I = mi;
            desc->J = mj;
            // CTAs for the next step: one per work unit, at least 8, at most the grid
            const long long nf = desc->nfull < 0 ? nrows : desc->nfull;
            const long long nu = nf * (nf >= kSplitBelow ? 1 : kRowParts) +
                                 (long long)((desc->npart_rows + 255) / 256) * (desc->npart_rows > 0 ? (mj - mi + PC) / PC : 0);
            desc->active = (int)max(8ll, min((long long)gridDim.x, nu));
        }
    }
    __syncthreads();
    if (tid == 0) {
        if (!found) // the search ends here: nothing is rewritten, but the counter must not outlive the grid
            while (*reinterpret_cast<volatile unsigned int *>(ticket + 1) < gridDim.x) {}
        ticket[0] = 0u;
        ticket[1] = 0u;
        finish_best_step(state, hdr, found, found ? (float)ord_value<V>((unsigned int)(bk >> 32)) : 0.0f, (uint32_t)mi,
                         (uint32_t)mj, log, log_cap);
    }
}

} // namespace

void launch_two_opt_cached_step(const Src &src, uint32_t n, int cyclic, unsigned long long *rowkey, CachedDesc *desc,
                                int *fullrows, DevState *state, unsigned int *ticket, tl_move *log, uint64_t log_cap,
                                int grid, cudaStream_t st)
{
    cudaLaunchAttribute attr[1];
    cudaLaunchConfig_t cfg = pdl_config(grid, 256, 0, attr, st);
    if (getenv("TL_CACHED_NO_PDL")) cfg.numAttrs = 0; // experiment: plain stream order between steps
    TL_DISPATCH_POL(src, (cudaLaunchKernelEx(&cfg, two_opt_cached_step_kernel<decltype(P)>, P, (int)n, cyclic, rowkey, desc,
                                             fullrows, state, ticket, log, (uint64_t)log_cap)));
}

} // namespace tl
