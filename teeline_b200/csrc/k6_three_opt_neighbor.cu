// k6_three_opt_neighbor.cu -- K6 candidate-list best-improvement 3-opt ("3-opt N"), coordinate recompute.
//
// What it computes: K6's triples, costs, case choice and tie order (three_opt.rs:58-131, k6_three_opt.cu,
// oracle/algos.inc three_opt_scan_rows), restricted to the triples that the first two candidate edges of a
// sequential 3-exchange generate.  Cut edge e (0 <= e <= n-1) joins p_e and p_(e+1)%n; K6's triple
// (i, j, k), i < j < k, removes edges i, j and k.  For every position q, c = p_q:
//   1. every slot s1 with b = K[c][s1] not padding, r = pos[b];
//   2. each e2 in {(r-1) mod n, r}; t = the other endpoint of edge e2: p_(r+1)%n when e2 = r, else
//      p_(r-1)%n;
//   3. every slot s2 with b' = K[t][s2] not padding, r' = pos[b'];
//   4. each e1 in {(q-1) mod n, q} and e3 in {(r'-1) mod n, r'}: if e1, e2 and e3 are distinct, sorted
//      into i < j < k, the triple counts unless i = 0 and k = n-1 (K6's skip).
// At most 8 triples per (q, s1, s2), 8 n k^2 per step.  With A = p_i, B = p_i+1, C = p_j, D = p_j+1,
// E = p_k, F = p_(k+1)%n, orig = (d_AB + d_CD) + d_EF and cost1..cost7 are K6's left-to-right sums in
// the metric's value type; the triple's case is the first minimal cost among those below orig and its
// savings orig - cost.  A step applies the counted triple with the largest savings > 0, ties to the
// lowest (i, j, k) (better_three); duplicates carry the same key.  stats.evals counts every counted
// triple, duplicates included.  With k >= n-1 every K6 triple is generated (q = i+1, b = p_j, e2 = j,
// t = p_j+1, b' = p_k, e1 = i, e3 = k), so the moves are TL_ALGO_THREE_OPT's, move for move.
//
// How: Or-opt N's resident grid (k3_or_opt_neighbor.cu) walks the n*k (q, s1) items with a grid-stride
// loop on cyclic records (position 0 carries the closing edge, position n is the wrap copy), so every
// removed edge's length is an entering-edge field.  An item loads the records around q and r once and
// loops over e2 and s2 inside the thread.  For each edge pair the distances between their endpoints are
// computed once and shared by every chain that uses the pair: 6 per (item, e2) for the q and r edges, and
// 15 per s2 for the r' edges against both (the 3 records around q and r' give both choices of e1 and
// e3).  A chain then only sorts its three edges and picks its nine distances from those tables.
// The step tail (apply.cuh: relocate_step_tail) is Or-opt N's: the last CTA reduces the per-CTA records
// and relocates a span [i+1, k] of at most kOrNlCtaSpan positions itself; a longer one is left pending for
// the gather and scatter grids that every step launches.
#include "apply.cuh"
#include "kernels.cuh"
#include "three_opt_move.cuh"

namespace tl {

namespace {

constexpr int THREADS = kNlThreads;
constexpr int WARPS = THREADS / 32;
constexpr uint32_t kNone = 0xffffffffu;

// distances between the endpoints of two removed edges X = (x0, x1) and Y = (y0, y1): d[a][b] = d(xa, yb)
template <typename V>
struct Quad {
    V d00, d01, d10, d11;
    __device__ __forceinline__ Quad t() const { return Quad{d00, d10, d01, d11}; } // the pair seen from Y
};

template <class Pol>
__global__ void __launch_bounds__(THREADS, kNlMinBlocks)
    three_nl_scan_kernel(Pol P, uint32_t *__restrict__ pos, const uint32_t *__restrict__ cand, uint32_t k, uint32_t n,
                         Pt *tmp, Best<typename Pol::V> *blockbest, unsigned long long *blockcnt, DevState *state,
                         unsigned int *ticket, tl_move *__restrict__ log, uint64_t log_cap, int fuse_apply)
{
    using V = typename Pol::V;
    using Rec = typename Pol::Rec;
    griddep_launch_dependents();
    griddep_wait(); // the previous step's move is applied and visible from here on
    // uniform across the grid: only a step's tail or apply grid writes it, after every CTA has finished
    if (*reinterpret_cast<const volatile int *>(&state->done)) return;

    Best<V> best{(V)0, kNone, kNone, 0u};
    uint32_t cnt = 0;
    // one chain: removed edges at positions e0 (the q edge), e1 (the r edge), e2 (the r' edge) with their
    // lengths sp* and the endpoint distances of each pair (q01: edges 0 and 1, ...)
    auto chain = [&](uint32_t e0, uint32_t e1, uint32_t e2, V sp0, V sp1, V sp2, const Quad<V> &q01,
                     const Quad<V> &q02, const Quad<V> &q12) {
        if (e0 == e1 || e0 == e2 || e1 == e2) return;
        // sort into I < J < K: the pairs (I, J), (J, K), (I, K) seen from their earlier edge
        Quad<V> ij, jk, ik;
        V d_ab, d_cd, d_ef;
        uint32_t i, j, kk;
        if (e0 < e1) {
            if (e1 < e2) { // 0 1 2
                i = e0; j = e1; kk = e2; d_ab = sp0; d_cd = sp1; d_ef = sp2; ij = q01; jk = q12; ik = q02;
            } else if (e0 < e2) { // 0 2 1
                i = e0; j = e2; kk = e1; d_ab = sp0; d_cd = sp2; d_ef = sp1; ij = q02; jk = q12.t(); ik = q01;
            } else { // 2 0 1
                i = e2; j = e0; kk = e1; d_ab = sp2; d_cd = sp0; d_ef = sp1; ij = q02.t(); jk = q01; ik = q12.t();
            }
        } else {
            if (e0 < e2) { // 1 0 2
                i = e1; j = e0; kk = e2; d_ab = sp1; d_cd = sp0; d_ef = sp2; ij = q01.t(); jk = q02; ik = q12;
            } else if (e1 < e2) { // 1 2 0
                i = e1; j = e2; kk = e0; d_ab = sp1; d_cd = sp2; d_ef = sp0; ij = q12; jk = q02.t(); ik = q01.t();
            } else { // 2 1 0
                i = e2; j = e1; kk = e0; d_ab = sp2; d_cd = sp1; d_ef = sp0; ij = q12.t(); jk = q01.t(); ik = q02.t();
            }
        }
        if (i == 0 && kk == n - 1) return; // K6's skip
        ++cnt;
        // A = I0, B = I1, C = J0, D = J1, E = K0, F = K1
        const V d_ac = ij.d00, d_ad = ij.d01, d_bd = ij.d11;
        const V d_ce = jk.d00, d_cf = jk.d01, d_df = jk.d11;
        const V d_ae = ik.d00, d_be = ik.d10, d_bf = ik.d11;
        const V orig = Val<V>::add(Val<V>::add(d_ab, d_cd), d_ef);
        const V c1 = Val<V>::add(Val<V>::add(d_ac, d_bd), d_ef);
        const V c2 = Val<V>::add(Val<V>::add(d_ab, d_ce), d_df);
        const V c3 = Val<V>::add(Val<V>::add(d_ac, d_be), d_df);
        const V c4 = Val<V>::add(Val<V>::add(d_ad, d_be), d_cf);
        const V c5 = Val<V>::add(Val<V>::add(d_ad, d_ce), d_bf);
        const V c6 = Val<V>::add(Val<V>::add(d_ae, d_bd), d_cf);
        const V c7 = Val<V>::add(Val<V>::add(d_ae, d_cd), d_bf);
        const V m = Val<V>::vmin(Val<V>::vmin(Val<V>::vmin(c1, c2), Val<V>::vmin(c3, c4)),
                                 Val<V>::vmin(Val<V>::vmin(c5, c6), c7));
        const V s = Val<V>::sub(orig, m); // savings of the first minimal case, if any improves
        if (s > (V)0 && (best.i == kNone || s >= best.delta)) { // rare
            const V cs[7] = {c1, c2, c3, c4, c5, c6, c7};
            V cm = c1;
            uint32_t kase = 1;
#pragma unroll
            for (int c = 1; c < 7; ++c)
                if (cs[c] < cm) { cm = cs[c]; kase = c + 1; } // first of equal minima (Iterator::min_by)
            const Best<V> o{s, i, j, kk * 8u + kase};
            if (better_three(o, best)) best = o;
        }
    };

    const uint64_t total = (uint64_t)n * k;
    for (uint64_t it = (uint64_t)blockIdx.x * THREADS + threadIdx.x; it < total; it += (uint64_t)gridDim.x * THREADS) {
        const uint32_t q = (uint32_t)(it / k), s1 = (uint32_t)(it - (uint64_t)q * k);
        const Rec Q1 = P.load(q);
        const uint32_t b = __ldg(&cand[(size_t)Pol::city(Q1) * k + s1]);
        if (b == 0xffffffffu) continue; // padding: fewer than k other cities
        const uint32_t r = pos[b];
        // the records around q and r: edge (q-1) mod n is (Q0, Q1), edge q is (Q1, Q2); position n is the
        // wrap copy of position 0, so (p_n-1, p_0) is (Q0, Q1) at q = 0 as well
        const uint32_t qm = q == 0 ? n - 1 : q - 1, rm = r == 0 ? n - 1 : r - 1;
        const Rec Q0 = P.load(qm), Q2 = P.load(q + 1);
        const Rec X0 = P.load(rm), X1 = P.load(r), X2 = P.load(r + 1);
#pragma unroll 1
        for (int w = 0; w < 2; ++w) {
            // e2 = (r-1) mod n: edge (X0, X1), t = p_r-1; e2 = r: edge (X1, X2), t = p_r+1
            const uint32_t e1 = w ? r : rm;
            const Rec Y0 = w ? X1 : X0, Y1 = w ? X2 : X1;
            const V spy = Pol::sp(Y1);
            const uint32_t tcity = (uint32_t)Pol::city(w ? X2 : X0);
            // the q edge against the r edge, both choices of the q edge
            const V dq0y0 = P.dist(Q0, Y0), dq0y1 = P.dist(Q0, Y1), dq1y0 = P.dist(Q1, Y0);
            const V dq1y1 = P.dist(Q1, Y1), dq2y0 = P.dist(Q2, Y0), dq2y1 = P.dist(Q2, Y1);
            const Quad<V> qy[2] = {{dq0y0, dq0y1, dq1y0, dq1y1}, {dq1y0, dq1y1, dq2y0, dq2y1}};
            for (uint32_t s2 = 0; s2 < k; ++s2) {
                const uint32_t b2 = __ldg(&cand[(size_t)tcity * k + s2]);
                if (b2 == 0xffffffffu) continue;
                const uint32_t r2 = pos[b2], r2m = r2 == 0 ? n - 1 : r2 - 1;
                const Rec Z0 = P.load(r2m), Z1 = P.load(r2), Z2 = P.load(r2 + 1);
                const Rec Q[3] = {Q0, Q1, Q2}, Z[3] = {Z0, Z1, Z2};
                V dqz[3][3], dyz[2][3];
#pragma unroll
                for (int a = 0; a < 3; ++a) {
#pragma unroll
                    for (int c = 0; c < 3; ++c) dqz[a][c] = P.dist(Q[a], Z[c]);
                    if (a < 2) {
#pragma unroll
                        for (int c = 0; c < 3; ++c) dyz[a][c] = P.dist(a ? Y1 : Y0, Z[c]);
                    }
                }
                const V spq[2] = {Pol::sp(Q1), Pol::sp(Q2)}, spz[2] = {Pol::sp(Z1), Pol::sp(Z2)};
                const uint32_t eq[2] = {qm, q}, ez[2] = {r2m, r2};
#pragma unroll
                for (int a = 0; a < 2; ++a) {
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        const Quad<V> qz{dqz[a][c], dqz[a][c + 1], dqz[a + 1][c], dqz[a + 1][c + 1]};
                        const Quad<V> yz{dyz[0][c], dyz[0][c + 1], dyz[1][c], dyz[1][c + 1]};
                        chain(eq[a], e1, ez[c], spq[a], spy, spz[c], qy[a], qz, yz);
                    }
                }
            }
        }
    }

    __shared__ Best<V> red[WARPS];
    __shared__ uint32_t red_cnt[WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    warp_argmin<ThreeMove>(best);
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0) {
        red[warp] = best;
        red_cnt[warp] = cnt;
    }
    __syncthreads();
    if (warp == 0) {
        Best<V> v = lane < WARPS ? red[lane] : Best<V>{(V)0, kNone, kNone, 0u};
        warp_argmin<ThreeMove>(v);
        if (lane == 0) {
            unsigned long long c = 0;
#pragma unroll
            for (int w = 0; w < WARPS; ++w) c += red_cnt[w];
            blockbest[blockIdx.x] = v; // delta holds the SAVINGS, as in K6's records
            blockcnt[blockIdx.x] = c;
        }
    }
    if (!fuse_apply) return;
    __shared__ unsigned int s_last;
    __syncthreads();
    if (threadIdx.x == 0) s_last = (ticket_take_acq_rel(ticket) == gridDim.x - 1) ? 1u : 0u; // thread 0 wrote blockbest
    __syncthreads();
    if (!s_last) return;
    relocate_step_tail<WARPS, ThreeMove>(P, n, pos, tmp, blockbest, blockcnt, state, ticket, log, log_cap);
}

} // namespace

void launch_three_nl_scan(Metric metric, Pt *pts, uint32_t *pos, const uint32_t *cand, uint32_t k, uint32_t n, void *tmp,
                          void *blockbest, unsigned long long *blockcnt, DevState *state, unsigned int *ticket,
                          tl_move *log, uint64_t log_cap, bool fuse_apply, int grid, cudaStream_t st)
{
    cudaLaunchAttribute attr[1];
    const cudaLaunchConfig_t cfg = pdl_config(grid, THREADS, 0, attr, st);
    const int fuse = fuse_apply ? 1 : 0;
    with_metric(metric, [&](auto M) {
        using Pol = NlPol<M>;
        cudaLaunchKernelEx(&cfg, three_nl_scan_kernel<Pol>, Pol{pts}, pos, cand, k, n, reinterpret_cast<Pt *>(tmp),
                           reinterpret_cast<Best<typename Pol::V> *>(blockbest), blockcnt, state, ticket, log,
                           (uint64_t)log_cap, fuse);
    });
}

void launch_three_nl_apply(Metric metric, Pt *pts, uint32_t *pos, void *tmp, uint32_t n, const void *pending,
                           DevState *state, unsigned int *ticket, tl_move *log, uint64_t log_cap, int grid,
                           cudaStream_t st)
{
    cudaLaunchAttribute attr[1];
    const cudaLaunchConfig_t cfg = pdl_config(grid, 256, 0, attr, st);
    with_metric(metric, [&](auto M) {
        using Pol = NlPol<M>;
        const auto *pend = reinterpret_cast<const Best<typename Pol::V> *>(pending);
        cudaLaunchKernelEx(&cfg, relocate_gather_kernel<Pol, ThreeMove>, Pol{pts}, reinterpret_cast<Pt *>(tmp), pend, 1,
                           (const DevState *)state);
        cudaLaunchKernelEx(&cfg, relocate_scatter_kernel<Pol, ThreeMove>, Pol{pts}, (const Pt *)tmp, n, pend, 1, state,
                           ticket, log, (uint64_t)log_cap, pos, 1);
    });
}

} // namespace tl
