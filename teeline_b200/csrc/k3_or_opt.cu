// k3_or_opt.cu -- K3: Or-opt best-improvement scan and relocation, coordinate-recompute path.
//
// Reference: or_opt::find_best_move / apply_relocation (src/tsp/or_opt.rs:80-184).  For
// segment lengths s = 1..3, every non-wrapping segment start i and every insertion edge
// (p_j, p_j+1) outside the forbidden window {prev(i), i..i+s-1}:
//     rg  = (d(a,f) + d(l,dd)) - d(a,dd)          a = p_prev, f = p_i, l = p_i+s-1, dd = p_after
//     fwd = ((-rg + d(x,f)) + d(l,y)) - d(x,y)     x = p_j, y = p_j+1
//     rev = ((-rg + d(x,l)) + d(f,y)) - d(x,y)     (s > 1 only)
// each operation rounded to f32 in exactly this order; a candidate is accepted iff it is
// strictly below the running best, which starts at -1e-3, scanning s -> i -> j -> fwd,rev.
// So the result is the minimum of (delta, rank) with rank = (s, i, j, dir); the kernel carries
// that rank in the reduction key, which makes the argmin independent of scheduling.
//
// How: with E(q,r) = d(p_q, p_r), all five candidates of a pair (i,j) only need
// E(j,i+c) and E(j+1,i+c), c = 0..2.  A thread owns R consecutive columns j (R+1 points in
// registers) and walks down the rows; E(., i+c) of row i is E(., i+c-1) of row i+1, so one
// row step costs R+1 new distances for 5R candidates (0.225 sqrt per candidate).  The three
// live distance columns rotate through registers by unrolling 3 steps.  Row points and the
// per-row removal gains (-rg for s = 1..3, +inf when the segment is not allowed) are staged
// per warp tile with TMA bulk copies.  Forbidden (i,j) pairs only exist within 3 of the
// diagonal, so warps take a masked copy of the step there and the mask-free copy elsewhere.
//
// Roofline: FP32 issue; ~6.5 issued instructions per candidate.
#include "apply.cuh"
#include "kernels.cuh"
#include "or_opt_rank.cuh"
#include "policy.cuh"

#include <math_constants.h>

#include <type_traits>

namespace tl {

namespace {

constexpr int R = kOrR;
constexpr int CW = 32 * R;          // columns per warp
constexpr int TI = kOrTI;           // max rows per staged tile
constexpr int WARPS = kOrWarps;
constexpr int ROWPTS = TI + 3;      // positions i0 .. i0+cnt+1 (+1 slack)
constexpr uint32_t kNone = 0xffffffffu;

template <typename V>
struct __align__(16) Quad {
    V x, y, z, w;
};

template <int N, typename F>
__device__ __forceinline__ void static_for(F &&f)
{
    if constexpr (N > 0) {
        static_for<N - 1>(f);
        f(std::integral_constant<int, N - 1>{});
    }
}

// Per-row removal gains: info[i] = (-rg_1, -rg_2, -rg_3, 0); +inf disables a segment length.
template <class Pol>
__global__ void __launch_bounds__(256)
    or_rowinfo_kernel(Pol P, uint32_t n, uint32_t npad, Quad<typename Pol::V> *__restrict__ info,
                      const DevState *__restrict__ state, unsigned int *__restrict__ work_ticket)
{
    using V = typename Pol::V;
    using Rec = typename Pol::Rec;
    if (state->done) return;
    if (blockIdx.x == 0 && threadIdx.x == 0) *work_ticket = 0u; // re-arm the scan's work queue
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < npad; i += gridDim.x * blockDim.x) {
        V v[3] = {Val<V>::pos_inf(), Val<V>::pos_inf(), Val<V>::pos_inf()};
        if (i < n) {
            const uint32_t prev = i == 0 ? n - 1 : i - 1;
            const Rec a = P.load(prev);
            const V daf = Pol::sp(P.load(i)); // d(p_prev, p_i); position 0 carries the closing edge
#pragma unroll
            for (uint32_t s = 1; s <= 3; ++s) {
                if (n > s + 1 && i + s <= n) {
                    const Rec dd = P.load(i + s); // position n is the wrap copy of position 0
                    const V dldd = Pol::sp(dd);    // d(p_i+s-1, p_after)
                    const V dadd = P.dist(a, dd);
                    const V rg = Val<V>::sub(Val<V>::add(daf, dldd), dadd);
                    v[s - 1] = -rg;
                }
            }
        }
        info[i] = Quad<V>{v[0], v[1], v[2], (V)0};
    }
}

#ifdef TL_TIMELINE
// tuning builds only: per-warp start / end globaltimer stamps and item counts of the latest scan
__device__ unsigned long long tl_or_t[3][4096];
__device__ __forceinline__ unsigned long long or_gtime()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#endif

template <class Pol>
__global__ void __launch_bounds__(WARPS * 32, kOrMinBlocks)
    or_opt_scan_kernel(Pol P, const Quad<typename Pol::V> *__restrict__ info, uint32_t n, const OrOrder order,
                       Best<typename Pol::V> *__restrict__ blockbest, const DevState *__restrict__ state,
                       unsigned int *__restrict__ work_ticket)
{
    using V = typename Pol::V;
    using Rec = typename Pol::Rec;
    using Col = typename Pol::Col;
    using BestV = Best<V>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    if (state->done) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    Rec *srow = reinterpret_cast<Rec *>(smem_raw) + warp * (ROWPTS + TI);
    Quad<V> *sinfo = reinterpret_cast<Quad<V> *>(srow + ROWPTS);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + (size_t)WARPS * (ROWPTS + TI) * 16);
    uint64_t *bar = bars + warp;
    BestV *red = reinterpret_cast<BestV *>(bars + WARPS);
    if (lane == 0) mbar_init(bar, 1);
    mbar_fence_init();
    __syncthreads();
    uint32_t phase = 0;

    BestV best{Val<V>::or_threshold(), kNone, kNone, 0u}; // or_opt.rs:86: best_delta = -1e-3
#ifdef TL_TIMELINE
    const unsigned long long tl_t0 = or_gtime();
    unsigned long long tl_items = 0;
#endif

    // Work items (column block x row chunk) are pulled from a global ticket: the tiles next to the
    // diagonal run the masked step and cost about twice the others, so a static one-item-per-warp
    // split would make the whole scan wait for them.
    for (;;) {
        int tk = 0;
        if (lane == 0) tk = (int)atomicAdd(work_ticket, 1u);
        tk = __shfl_sync(0xffffffffu, tk, 0);
        if (tk >= order.total) break;
#ifdef TL_TIMELINE
        ++tl_items;
#endif
        int cb, ci;
        order.item_of_ticket(tk, cb, ci); // diagonal (masked, expensive) tiles first: kernels.cuh
        const int r_begin = ci * order.chunk;
        const int r_end = min(r_begin + order.chunk, (int)n);
        const int J0 = cb * CW;           // first column of the warp
        const int j0 = J0 + lane * R;     // first column of this lane

        // column points p_j0 .. p_j0+R and the insertion-edge lengths d(p_j, p_j+1) = sp[j+1]
        Col cc[R + 1];
        V exy[R];
#pragma unroll
        for (int c = 0; c <= R; ++c) {
            const Rec p = P.load(j0 + c);
            cc[c] = Pol::col(p);
            // columns j >= n do not exist: exy = -inf makes every candidate there +inf
            if (c > 0) exy[c - 1] = (j0 + c - 1 < (int)n) ? Pol::sp(p) : Val<V>::neg_inf();
        }

        const int ntiles = (r_end - r_begin + TI - 1) / TI;
        const int tile_rows = ntiles > 0 ? (r_end - r_begin + ntiles - 1) / ntiles : 0;
        for (int i0 = r_begin; i0 < r_end; i0 += tile_rows) {
            const int cnt = min(tile_rows, r_end - i0);
            __syncwarp();
            if (lane == 0) {
                const uint32_t rb = (uint32_t)(cnt + 2) * sizeof(Rec);
                const uint32_t ib = (uint32_t)cnt * sizeof(Quad<V>);
                mbar_expect_tx(bar, rb + ib);
                tma_load_1d(srow, P.base() + i0, rb, bar);
                tma_load_1d(sinfo, info + i0, ib, bar);
            }
            mbar_wait(bar, phase);
            phase ^= 1u;

            // A[c][.] = E(column, row i+c); three live columns rotate through A0/A1/A2
            V A[3][R + 1];
            {
                const Rec r0 = srow[0], r1 = srow[1];
#pragma unroll
                for (int c = 0; c <= R; ++c) {
                    A[0][c] = P.dist_rc(r0, cc[c]);
                    A[1][c] = P.dist_rc(r1, cc[c]);
                }
            }

            auto step = [&](auto PHc, auto MASKc, int tau) {
                constexpr int PH = decltype(PHc)::value;
                constexpr bool MASKED = decltype(MASKc)::value;
                constexpr int P0 = PH % 3, P1 = (PH + 1) % 3, P2 = (PH + 2) % 3;
                const Rec rp = srow[tau + 2];
                const Quad<V> ri = sinfo[tau];
#pragma unroll
                for (int c = 0; c <= R; ++c) A[P2][c] = P.dist_rc(rp, cc[c]);
                const int i = i0 + tau;
                // forbidden insertion edges of row i, segment length s (or_opt.rs:124): j == prev or
                // i <= j < i + s.  For i >= 1 that is j - i in [-1, s-1], i.e. (unsigned)(j - i + 1) <= s:
                // one compare per candidate on a per-row base; row 0 has prev = n - 1 instead of -1.
                const int mbase = j0 - i + 1;                         // (j - i + 1) for r = 0
                const int jwrap = i == 0 ? (int)n - 1 - j0 : -1;      // r of column n-1 in row 0, else none
                // candidate (r, k): k = 0 fwd1, 1 fwd2, 2 rev2, 3 fwd3, 4 rev3
                auto cand = [&](int r, int k) -> V {
                    const V nrg = k == 0 ? ri.x : (k <= 2 ? ri.y : ri.z);
                    const V first = (k == 2) ? A[P1][r] : (k == 4 ? A[P2][r] : A[P0][r]);
                    const V second = (k == 1) ? A[P1][r + 1] : (k == 3 ? A[P2][r + 1] : A[P0][r + 1]);
                    V d = Val<V>::sub(Val<V>::add(Val<V>::add(nrg, first), second), exy[r]);
                    if (MASKED) {
                        const unsigned s = k == 0 ? 1u : (k <= 2 ? 2u : 3u);
                        if ((unsigned)(mbase + r) <= s || r == jwrap) d = Val<V>::pos_inf();
                    }
                    return d;
                };
                V m = Val<V>::pos_inf();
#pragma unroll
                for (int r = 0; r < R; ++r) {
#pragma unroll
                    for (int k = 0; k < 5; ++k) m = Val<V>::vmin(m, cand(r, k));
                }
                if (m <= best.delta) { // rare
#pragma unroll
                    for (int r = 0; r < R; ++r) {
#pragma unroll
                        for (int k = 0; k < 5; ++k) {
                            const V d = cand(r, k);
                            const uint32_t aux = k == 0 ? 0u : (uint32_t)(k + 1); // (s-1)*2 + rev
                            const BestV o{d, (uint32_t)i, (uint32_t)(j0 + r), aux};
                            const bool take = best.i == kNone ? (d < best.delta) : better_or(o, best);
                            if (take) best = o;
                        }
                    }
                }
            };

            auto run = [&](auto MASKc) {
                int t = 0;
#pragma unroll 1
                for (; t + 3 <= cnt; t += 3)
                    static_for<3>([&](auto Uc) { step(Uc, MASKc, t + decltype(Uc)::value); });
                static_for<3>([&](auto Uc) {
                    if (t + decltype(Uc)::value < cnt) step(Uc, MASKc, t + decltype(Uc)::value);
                });
            };
            // forbidden pairs lie within 3 of the diagonal (and at (i=0, j=n-1))
            const bool near = (i0 + cnt + 2 >= J0 && i0 - 1 < J0 + CW) ||
                              (i0 == 0 && (int)n - 1 >= J0 && (int)n - 1 < J0 + CW);
            if (near)
                run(std::true_type{});
            else
                run(std::false_type{});
        }
    }

#ifdef TL_TIMELINE
    if (lane == 0 && blockIdx.x * WARPS + warp < 4096) {
        const int w = blockIdx.x * WARPS + warp;
        tl_or_t[0][w] = tl_t0;
        tl_or_t[1][w] = or_gtime();
        tl_or_t[2][w] = tl_items;
    }
#endif
    warp_argmin_or(best);
    if (lane == 0) red[warp] = best;
    __syncthreads();
    if (warp == 0) {
        BestV v = (lane < WARPS) ? red[lane] : BestV{(V)0, kNone, kNone, 0u};
        warp_argmin_or(v);
        if (lane == 0) blockbest[blockIdx.x] = v;
    }
}

} // namespace

size_t or_scan_smem_bytes()
{
    return (size_t)WARPS * (ROWPTS + TI) * 16 + WARPS * sizeof(uint64_t) + WARPS * sizeof(BestF);
}

cudaError_t or_scan_configure()
{
    const int bytes = (int)or_scan_smem_bytes();
    cudaError_t e = cudaFuncSetAttribute(or_opt_scan_kernel<EucPol<true>>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(or_opt_scan_kernel<EucPol<false>>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(or_opt_scan_kernel<MatPol<float>>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(or_opt_scan_kernel<MatPol<int32_t>>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    return e;
}

void launch_or_rowinfo(const Src &src, uint32_t n, uint32_t npad, void *info, const DevState *state,
                       unsigned int *work_ticket, cudaStream_t st)
{
    const int grid = (int)((npad + 255) / 256);
    TL_DISPATCH_POL(src, (or_rowinfo_kernel<<<grid, 256, 0, st>>>(
                             P, n, npad, reinterpret_cast<Quad<typename decltype(P)::V> *>(info), state,
                             work_ticket)));
}

void launch_or_scan(const Src &src, const void *info, uint32_t n, const OrOrder &order, void *blockbest,
                    const DevState *state, unsigned int *work_ticket, int grid, cudaStream_t st)
{
    const size_t smem = or_scan_smem_bytes();
    TL_DISPATCH_POL(src, (or_opt_scan_kernel<<<grid, WARPS * 32, smem, st>>>(
                             P, reinterpret_cast<const Quad<typename decltype(P)::V> *>(info), n, order,
                             reinterpret_cast<Best<typename decltype(P)::V> *>(blockbest), state, work_ticket)));
}

void launch_or_apply(const Src &src, void *tmp, uint32_t n, const void *cand, int ncand, DevState *state,
                     unsigned int *ticket, tl_move *log, uint64_t log_cap, int grid, cudaStream_t st)
{
    TL_DISPATCH_POL(src, {
        using PolT = decltype(P);
        auto *t = reinterpret_cast<typename PolT::Rec *>(tmp);
        auto *c = reinterpret_cast<const Best<typename PolT::V> *>(cand);
        relocate_gather_kernel<PolT, OrMove><<<grid, 256, 0, st>>>(P, t, c, ncand, state);
        relocate_scatter_kernel<PolT, OrMove><<<grid, 256, 0, st>>>(P, t, n, c, ncand, state, ticket, log, log_cap,
                                                                    nullptr, 0);
    });
}

#ifdef TL_TIMELINE
extern "C" int tl_debug_or_timeline(unsigned long long *out)
{
    return cudaMemcpyFromSymbol(out, tl_or_t, sizeof(tl_or_t)) != cudaSuccess;
}
#endif

} // namespace tl
