// k6_three_opt.cu -- K6: 3-opt best-improvement scan and move application (SURVEY.md 8(f), row N2).
//
// Reference: three_opt::{find_best_move, reconnection_costs, apply_3opt}
// (src/tsp/three_opt.rs:58-131, :151-180, :182-218).  Over all triples i < j < k (skipping
// i == 0 && k == n-1), with A=p[i], B=p[i+1], C=p[j], D=p[j+1], E=p[k], F=p[(k+1)%n]:
//     orig  = (d_AB + d_CD) + d_EF
//     cost1 = (d_AC + d_BD) + d_EF      cost2 = (d_AB + d_CE) + d_DF     cost3 = (d_AC + d_BE) + d_DF
//     cost4 = (d_AD + d_BE) + d_CF      cost5 = (d_AD + d_CE) + d_BF     cost6 = (d_AE + d_BD) + d_CF
//     cost7 = (d_AE + d_CD) + d_BF
// each sum left to right in f32; per triple the FIRST minimal cost among those below orig; the
// move is accepted iff savings = orig - cost is strictly above the best so far (from 0), scanning
// i -> j -> k.  So the result is max (savings) with ties to the lowest (i, j, k); the kernel
// carries (i, j, k) in the reduction key, which makes the argmax independent of scheduling.
//
// How: a warp takes a work item (row i, 32 consecutive j) and walks k; lane l owns j = j0 + l.
//  * per (i, j): d_AC, d_BD, d_AD and the partial sums (d_AB + d_CD), (d_AC + d_BD) are hoisted;
//  * per (i, k): d_AF and d_BF do not depend on j -- they are computed once per block of 32 k
//    values (lane-parallel) and parked with the record of F in shared memory, so a row step is
//    one broadcast LDS.128 + LDS.64 per lane;  d_AE(k) = d_AF(k-1), d_BE(k) = d_BF(k-1);
//  * per (j, k): only d_CF and d_DF are new (d_CE(k) = d_CF(k-1)): 2 distances per triple;
//  * savings_max = orig - min(cost1..7) is tested against the running best; the case index is
//    only worked out in the rare slow path.
// Work items are pulled from a global ticket (row i of the triangle has ~(n-i)^2/2 triples).
//
// Roofline: FP32 issue (2 exact distances + 14 adds + min tree per triple, ~50 instructions).
#include "apply.cuh"
#include "kernels.cuh"
#include "policy.cuh"
#include "three_opt_move.cuh"

#include <math_constants.h>

namespace tl {

namespace {

constexpr int WARPS = kThreeWarps;
constexpr uint32_t kNone = 0xffffffffu;

// staged per-k entry: the record of F = p[k+1], d_EF, and the two j-independent distances
template <class Pol>
struct KEntry {
    typename Pol::Rec f;
    typename Pol::V daf, dbf;
};

template <class Pol>
__global__ void __launch_bounds__(WARPS * 32, kThreeMinBlocks)
    three_opt_scan_kernel(Pol P, uint32_t n, const int32_t *__restrict__ row_first, int item_begin, int item_end,
                          Best<typename Pol::V> *__restrict__ blockbest, const DevState *__restrict__ state,
                          unsigned int *__restrict__ work_ticket)
{
    using V = typename Pol::V;
    using Rec = typename Pol::Rec;
    __shared__ KEntry<Pol> sk[WARPS][32];
    __shared__ Best<V> red[WARPS];
    if (state->done) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    V best_s = (V)0; // savings
    uint32_t bi = kNone, bj = kNone, baux = 0;

    for (;;) {
        int item = 0;
        if (lane == 0) item = item_begin + (int)atomicAdd(work_ticket, 1u);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= item_end) break;
        // row i = largest r with row_first[r] <= item; rows i = 0 .. n-3
        int lo = 0, hi = (int)n - 3;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (__ldg(&row_first[mid]) <= item) lo = mid; else hi = mid - 1;
        }
        const uint32_t i = (uint32_t)lo;
        const uint32_t j0 = i + 1 + 32u * (uint32_t)(item - __ldg(&row_first[lo]));
        const uint32_t j = j0 + lane;
        const bool jvalid = j <= n - 2;
        const Rec ra = P.load(i), rb = P.load(i + 1);
        const Rec rc = P.load(jvalid ? j : i + 1), rd = P.load(jvalid ? j + 1 : i + 2);
        const V d_ab = Pol::sp(rb), d_cd = Pol::sp(rd);
        const V d_ac = P.dist(ra, rc), d_bd = P.dist(rb, rd), d_ad = P.dist(ra, rd);
        const V h_orig = Val<V>::add(d_ab, d_cd); // (d_AB + d_CD)
        const V h_c1 = Val<V>::add(d_ac, d_bd);   // (d_AC + d_BD)
        // carried values: d_CF of the previous step (= d_CE of this one), and the previous entry's
        // d_AF / d_BF (= d_AE / d_BE).  At k = j+1, E is D: d_CE = d_CD, d_AE = d_AD, d_BE = d_BD.
        V dcf_prev = d_cd;
        V daf_prev = (V)0, dbf_prev = (V)0;

        for (uint32_t kb = j0 + 1; kb <= n - 1; kb += 32) {
            __syncwarp();
            { // stage entries for k = kb + lane: F = p[k+1] (position n is the wrap copy of position 0)
                const uint32_t kk = min(kb + lane, n - 1);
                KEntry<Pol> e;
                e.f = P.load(kk + 1);
                e.daf = P.dist(ra, e.f);
                e.dbf = P.dist(rb, e.f);
                sk[warp][lane] = e;
            }
            if (kb == j0 + 1) { // entry "before the first": F(k-1) = p[j0+1]
                const Rec f0 = P.load(j0 + 1);
                daf_prev = P.dist(ra, f0);
                dbf_prev = P.dist(rb, f0);
            }
            __syncwarp();
            const uint32_t steps = min(32u, n - kb); // k = kb .. min(kb+31, n-1)
#pragma unroll 2
            for (uint32_t t = 0; t < steps; ++t) {
                const uint32_t k = kb + t;
                const KEntry<Pol> e = sk[warp][t]; // warp broadcast
                const V d_ef = Pol::sp(e.f);
                const V d_cf = P.dist(rc, e.f), d_df = P.dist(rd, e.f);
                const V d_ce = dcf_prev, d_ae = daf_prev, d_be = dbf_prev, d_bf = e.dbf;
                const V orig = Val<V>::add(h_orig, d_ef);
                const V c1 = Val<V>::add(h_c1, d_ef);
                const V c2 = Val<V>::add(Val<V>::add(d_ab, d_ce), d_df);
                const V c3 = Val<V>::add(Val<V>::add(d_ac, d_be), d_df);
                const V c4 = Val<V>::add(Val<V>::add(d_ad, d_be), d_cf);
                const V c5 = Val<V>::add(Val<V>::add(d_ad, d_ce), d_bf);
                const V c6 = Val<V>::add(Val<V>::add(d_ae, d_bd), d_cf);
                const V c7 = Val<V>::add(Val<V>::add(d_ae, d_cd), d_bf);
                const V m = Val<V>::vmin(Val<V>::vmin(Val<V>::vmin(c1, c2), Val<V>::vmin(c3, c4)),
                                         Val<V>::vmin(Val<V>::vmin(c5, c6), c7));
                const V s = Val<V>::sub(orig, m); // savings of the first minimal case, if any improves
                const bool active = jvalid && k > j && !(i == 0 && k == n - 1);
                if (active && s > (V)0 && s >= best_s) { // rare
                    const V cs[7] = {c1, c2, c3, c4, c5, c6, c7};
                    int ci = 0;
#pragma unroll
                    for (int q = 1; q < 7; ++q)
                        if (cs[q] < cs[ci]) ci = q; // first of equal minima (Iterator::min_by)
                    const uint32_t aux = k * 8u + (uint32_t)(ci + 1);
                    if (bi == kNone || better_three(s, i, j, aux, best_s, bi, bj, baux)) {
                        best_s = s;
                        bi = i;
                        bj = j;
                        baux = aux;
                    }
                }
                dcf_prev = d_cf;
                daf_prev = e.daf;
                dbf_prev = e.dbf;
            }
        }
    }

    // deterministic argmax: (savings desc, i, j, k asc) across lanes, warps, blocks
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const V os = __shfl_xor_sync(0xffffffffu, best_s, off);
        const uint32_t oi = __shfl_xor_sync(0xffffffffu, bi, off);
        const uint32_t oj = __shfl_xor_sync(0xffffffffu, bj, off);
        const uint32_t oa = __shfl_xor_sync(0xffffffffu, baux, off);
        if (oi != kNone && (bi == kNone || better_three(os, oi, oj, oa, best_s, bi, bj, baux))) {
            best_s = os; bi = oi; bj = oj; baux = oa;
        }
    }
    if (lane == 0) red[warp] = Best<V>{best_s, bi, bj, baux};
    __syncthreads();
    if (threadIdx.x == 0) {
        Best<V> v = red[0];
        for (int w = 1; w < WARPS; ++w) {
            const Best<V> o = red[w];
            if (o.i != kNone && (v.i == kNone || better_three(o.delta, o.i, o.j, o.aux, v.delta, v.i, v.j, v.aux))) v = o;
        }
        blockbest[blockIdx.x] = v; // delta holds the SAVINGS here; the apply step negates it
    }
}

} // namespace

void launch_three_scan(const Src &src, uint32_t n, const int32_t *row_first, int item_begin, int item_end,
                       void *blockbest, const DevState *state, unsigned int *work_ticket, int grid, cudaStream_t st)
{
    TL_DISPATCH_POL(src, (three_opt_scan_kernel<<<grid, WARPS * 32, 0, st>>>(
                             P, n, row_first, item_begin, item_end,
                             reinterpret_cast<Best<typename decltype(P)::V> *>(blockbest), state, work_ticket)));
}

void launch_three_apply(const Src &src, void *tmp, uint32_t n, const void *cand, int ncand, DevState *state,
                        unsigned int *ticket, tl_move *log, uint64_t log_cap, int grid, cudaStream_t st)
{
    TL_DISPATCH_POL(src, {
        using PolT = decltype(P);
        auto *t = reinterpret_cast<typename PolT::Rec *>(tmp);
        auto *c = reinterpret_cast<const Best<typename PolT::V> *>(cand);
        relocate_gather_kernel<PolT, ThreeMove><<<grid, 256, 0, st>>>(P, t, c, ncand, state);
        relocate_scatter_kernel<PolT, ThreeMove><<<grid, 256, 0, st>>>(P, t, n, c, ncand, state, ticket, log, log_cap,
                                                                       nullptr, 0);
    });
}

} // namespace tl
