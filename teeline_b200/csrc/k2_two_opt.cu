// k2_two_opt.cu -- K2: best-improvement 2-opt scan ("Mode B"), coordinate-recompute path.
//
// What it computes (SURVEY.md Appendix A, "2-opt B"; neighbourhood of
// src/tsp/two_opt.rs:17,29,34): over all pairs 0 <= i, i+2 <= j <= jmax
//     delta(i,j) = (d(p_i,p_j) + d(p_i+1,p_j+1)) - (d(p_i,p_i+1) + d(p_j,p_j+1))
// each operation rounded to f32, and returns argmin with strict '<' from 0 in
// (i,j) lexicographic order (lowest (i,j) wins ties).
//
// How: the triangle is walked along DIAGONALS k = j - i.  Moving down a diagonal,
// d(p_i+1,p_j+1) of pair (i,j) is d(p_i',p_j') of pair (i+1,j+1), so every move
// costs ONE new distance (5 FP32 ops + one IEEE sqrt) plus 3 adds and a min.
// Lane l of a warp owns R consecutive diagonals K0 + l*R + r; the R+1 tour-ordered
// points it needs form a sliding window held in registers (rotated by unrolling R
// steps), so per row a lane issues two 128-bit LDS: the warp-broadcast row point
// and one new window point.  Tour-ordered points (x, y, city, entering-edge length)
// are staged per warp tile with TMA 1-D bulk copies (cp.async.bulk + mbarrier).
// The running minimum is tracked with FMNMX3 trees and a rarely taken slow path
// (improving moves are rare near a local optimum), so the hot loop carries no
// index arithmetic.
//
// Roofline: FP32 issue (no tensor cores: K=2 is not a contraction).  Algorithmic
// work 15 flop/move, ~0 bytes/move (DESIGN.md section 4).
#include "kernels.cuh"
#include "policy.cuh"
#include "apply.cuh"

#include <math_constants.h>

#include <type_traits>

namespace tl {

namespace {

constexpr int R = kScanR;
constexpr int BW = kScanBW;
constexpr int TI = kScanTI;
constexpr int WARPS = kScanWarps;
constexpr int ROWS_CAP = TI + 1;       // positions i0 .. i0+cnt
constexpr int COLS_CAP = TI + BW + 1;  // positions i0+K0 .. i0+K0+cnt+BW
constexpr int WARP_PTS = ROWS_CAP + COLS_CAP;

template <int N, typename F>
__device__ __forceinline__ void static_for(F &&f)
{
    if constexpr (N > 0) {
        static_for<N - 1>(f);
        f(std::integral_constant<int, N - 1>{});
    }
}

__device__ __forceinline__ int find_band(const int32_t *__restrict__ band_first, int nbands, int item)
{
    int lo = 0, hi = nbands - 1; // largest b with band_first[b] <= item
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(&band_first[mid]) <= item)
            lo = mid;
        else
            hi = mid - 1;
    }
    return lo;
}

// Tail of a fused step, run by the last CTA of the scan: reduce the per-CTA records, reverse the
// segment in place, update the loop state.  Kept out of line so that its registers (the batched
// reversal holds 8 records) do not weigh on the scan loop's allocation.
template <bool FAST>
__device__ __noinline__ void fused_apply_tail(Pt *__restrict__ pts, const BestF *__restrict__ blockbest, BestF *red,
                                              DevState *state, unsigned int *ticket, tl_move *__restrict__ log,
                                              uint64_t log_cap, const ShardComm &sc)
{
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // (ordering: thread 0's acq_rel ticket + the caller's __syncthreads; the records are read from L2)
    StateHeader hdr{};
    if (threadIdx.x == 0) hdr = load_state_header(state); // in flight with the candidate loads
    BestF v{0.0f, 0xffffffffu, 0xffffffffu, 0u};
    for (int c = threadIdx.x; c < (int)gridDim.x; c += blockDim.x) {
        // L2 read: the records were written by other CTAs of this launch
        const float4 raw = __ldcg(reinterpret_cast<const float4 *>(blockbest) + c);
        const BestF o{raw.x, __float_as_uint(raw.y), __float_as_uint(raw.z), __float_as_uint(raw.w)};
        if (better_2opt(o.delta, o.i, o.j, v.delta, v.i, v.j)) v = o;
    }
    warp_argmin_2opt(v.delta, v.i, v.j);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    v = red[0];
#pragma unroll
    for (int w = 1; w < WARPS; ++w) {
        const BestF o = red[w];
        if (better_2opt(o.delta, o.i, o.j, v.delta, v.i, v.j)) v = o;
    }
    if (sc.world > 1) {
        // sharded triangle: this rank's minimum goes to every peer's mailbox over NVLink and the
        // minimum over all ranks comes back, identical everywhere (shard_exchange.cuh)
        __shared__ BestF s_peer[kMaxPeers];
        __shared__ int s_fail;
        __shared__ unsigned int s_step;
        if (threadIdx.x == 0) s_step = (unsigned int)hdr.h0.y + 1u; // scans completed so far + 1
        __syncthreads();
        v = shard_exchange_2opt(sc, v, s_step, s_peer, &s_fail);
        if (s_fail) { // a peer never answered: stop the search instead of hanging the box
            if (threadIdx.x == 0) {
                *ticket = 0u;
                state->error = 1;
                state->done = 1;
            }
            return;
        }
    }
    const bool found = v.i != 0xffffffffu;
    if (found) reverse_segment_inplace(EucPol<FAST>{pts}, v.i, v.j, nullptr, threadIdx.x, blockDim.x);
    if (threadIdx.x == 0) {
        *ticket = 0u;
        finish_best_step(state, hdr, found, v.delta, v.i, v.j, log, log_cap);
    }
}

// SCREEN (FAST only): the hot loop evaluates deltas with the screening distance (no Newton step,
// 3 FP32 instructions fewer per move); a row step whose smallest screened delta is within the
// rigorous error margin of the running best is re-evaluated exactly, so every value that is
// compared, selected or returned is the exact f32 delta (common.cuh: dist_f32_screen).
template <bool FAST, bool SCREEN>
__global__ void __launch_bounds__(WARPS * 32, kScanMinBlocks)
    two_opt_scan_recompute_kernel(Pt *__restrict__ pts, const ScanGeom g,
                                  const int32_t *__restrict__ band_first, BestF *__restrict__ blockbest,
                                  DevState *state, unsigned int *ticket, tl_move *__restrict__ log,
                                  uint64_t log_cap, int fuse_apply, const __grid_constant__ ShardComm sc)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    // PDL: let the next step's launch start as soon as SMs free up; everything up to
    // griddep_wait() (barrier set-up, band look-up tables) is independent of the previous step
    griddep_launch_dependents();

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    Pt *srow = reinterpret_cast<Pt *>(smem_raw) + warp * WARP_PTS;
    Pt *scol = srow + ROWS_CAP;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + (size_t)WARPS * WARP_PTS * sizeof(Pt));
    uint64_t *bar = bars + warp;
    BestF *red = reinterpret_cast<BestF *>(bars + WARPS);

    if (lane == 0) mbar_init(bar, 1);
    mbar_fence_init();
    const int total_warps = gridDim.x * WARPS;
    const int item0 = g.item_begin + blockIdx.x * WARPS + warp;
    int t_next = 0, tf_next = 0; // table slot of this warp's first work item (geometry only)
    if (item0 < g.item_end) {
        t_next = find_band(band_first, g.nbands, item0);
        tf_next = __ldg(&band_first[t_next]);
    }
    __syncthreads();
    griddep_wait(); // the previous step's move is applied and visible from here on
    // uniform across the grid: only a fused tail writes it, after every other CTA has finished
    const int done = *reinterpret_cast<const volatile int *>(&state->done);
    if (done) return;

    uint32_t phase = 0;
    float best = 0.0f;
    uint32_t bi = 0xffffffffu, bj = 0xffffffffu;
    float thr = SCREEN ? g.screen_margin : 0.0f; // best + margin

    for (int item = item0; item < g.item_end; item += total_warps) {
        if (item != item0) {
            t_next = find_band(band_first, g.nbands, item);
            tf_next = __ldg(&band_first[t_next]);
        }
        const int b = t_next;
        const int cidx = item - tf_next; // row chunk within the band
        const int K0 = 2 + b * BW;
        const int H = g.jmax - K0 + 1; // rows 0 .. H-1 exist on the band's first diagonal
        const int r_begin = cidx * g.chunk;
        const int r_end = min(r_begin + g.chunk, H);
        const int lane_k0 = K0 + lane * R; // first diagonal of this lane

        // even tiles of at most TI rows
        const int ntiles = (r_end - r_begin + TI - 1) / TI;
        const int tile_rows = ntiles > 0 ? (r_end - r_begin + ntiles - 1) / ntiles : 0;
        for (int i0 = r_begin; i0 < r_end; i0 += tile_rows) {
            const int cnt = min(tile_rows, r_end - i0);
            __syncwarp(); // everyone is done with the previous tile's smem
            if (lane == 0) {
                const uint32_t rb = (uint32_t)(cnt + 1) * sizeof(Pt);
                const uint32_t cb = (uint32_t)(cnt + BW + 1) * sizeof(Pt);
                mbar_expect_tx(bar, rb + cb);
                tma_load_1d(srow, pts + i0, rb, bar);
                tma_load_1d(scol, pts + i0 + K0, cb, bar);
            }
            mbar_wait(bar, phase);
            phase ^= 1u;

            // carried distances E[r] = d(p_i, p_j) for j = i + lane_k0 + r, and the window of
            // points at positions j+1
            float E[R], wx[R], wy[R], ws[R];
            {
                const Pt rp0 = srow[0];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const Pt c = scol[lane * R + r];
                    E[r] = SCREEN ? dist_f32_screen(rp0.x, rp0.y, c.x, c.y) : dist_f32<FAST>(rp0.x, rp0.y, c.x, c.y);
                    const Pt w = scol[lane * R + r + 1];
                    wx[r] = w.x;
                    wy[r] = w.y;
                    ws[r] = w.sp;
                }
            }

            // One row step for compile-time window phase U (the register window is rotated by
            // unrolling R steps, so no data ever moves between registers).
            auto step = [&](auto Uc, int tau) {
                constexpr int U = decltype(Uc)::value;
                const Pt rp = srow[tau + 1];                // (x,y) of i+1 and s_i, warp broadcast
                const Pt nx = scol[tau + lane * R + R + 1]; // next window point
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
                if (m <= thr) { // rare: a move that may beat (or tie with) this thread's best
                    const uint32_t i = (uint32_t)(i0 + tau);
                    const Pt pi = srow[tau];
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const uint32_t j = i + (uint32_t)(lane_k0 + r);
                        float d = dl[r];
                        if (SCREEN) { // exact re-evaluation from the staged points
                            const Pt pj = scol[tau + lane * R + r], pj1 = scol[tau + lane * R + r + 1];
                            const float e1 = dist_f32<FAST>(pi.x, pi.y, pj.x, pj.y);
                            const float e2 = dist_f32<FAST>(rp.x, rp.y, pj1.x, pj1.y);
                            d = __fsub_rn(__fadd_rn(e1, e2), __fadd_rn(rp.sp, pj1.sp));
                        }
                        // the cyclic neighbourhood excludes (0, n-1): both edges share p_0
                        const bool excluded = g.cyclic && i == 0 && j == (uint32_t)(g.n - 1);
                        // full (delta, i, j) order: a warp that is handed several work items does
                        // not visit them in (i, j) order
                        if (d < 0.0f && !excluded && better_2opt(d, i, j, best, bi, bj)) {
                            best = d;
                            bi = i;
                            bj = j;
                            thr = SCREEN ? __fadd_rn(best, g.screen_margin) : best;
                        }
                    }
                }
                wx[U] = nx.x;
                wy[U] = nx.y;
                ws[U] = nx.sp;
            };

            int t = 0;
#pragma unroll 1
            for (; t + R <= cnt; t += R) { // full groups: straight-line code, no per-step predicate
                static_for<R>([&](auto Uc) { step(Uc, t + decltype(Uc)::value); });
            }
            // tail: fewer than R rows left; the window phase restarts at 0 after a full group
            static_for<R>([&](auto Uc) {
                if (t + decltype(Uc)::value < cnt) step(Uc, t + decltype(Uc)::value);
            });
        }
    }

    // deterministic argmin: (delta, i, j) lexicographic across lanes, warps, blocks
    warp_argmin_2opt(best, bi, bj);
    if (lane == 0) red[warp] = BestF{best, bi, bj, 0u};
    __syncthreads();
    if (warp == 0) {
        BestF v = (lane < WARPS) ? red[lane] : BestF{0.0f, 0xffffffffu, 0xffffffffu, 0u};
        warp_argmin_2opt(v.delta, v.i, v.j);
        if (lane == 0) blockbest[blockIdx.x] = v;
    }
    if (!fuse_apply) return;

    // Fused step tail (single-GPU sessions): the last CTA to finish reduces the per-CTA records,
    // reverses the segment in place and updates the loop state, saving a kernel launch per step.
    __shared__ unsigned int s_last;
    __syncthreads();
    if (threadIdx.x == 0) s_last = (ticket_take_acq_rel(ticket) == gridDim.x - 1) ? 1u : 0u; // thread 0 wrote blockbest
    __syncthreads();
    if (!s_last) return;
    fused_apply_tail<FAST>(pts, blockbest, red, state, ticket, log, log_cap, sc);
}

// tour-ordered point records from city coordinates and a tour
template <bool FAST>
__global__ void __launch_bounds__(256)
    build_pts_kernel(const float2 *__restrict__ xy, const uint32_t *__restrict__ tour, uint32_t n,
                     uint32_t npad, int cyclic, Pt *__restrict__ pts)
{
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < npad; q += gridDim.x * blockDim.x) {
        Pt p;
        if (q < n || (q == n && cyclic)) {
            const uint32_t c = tour[q == n ? 0 : q];
            const uint32_t cp = tour[q == 0 ? n - 1 : q - 1];
            const float2 a = xy[c], bprev = xy[cp];
            p.x = a.x;
            p.y = a.y;
            p.city = (int32_t)c;
            p.sp = (q == 0 && !cyclic) ? 0.0f : dist_f32<FAST>(bprev.x, bprev.y, a.x, a.y);
        } else {
            p.x = 0.0f;
            p.y = 0.0f;
            p.city = -1;
            p.sp = -CUDART_INF_F; // delta = new - (s_i + -inf) = +inf: never selected
        }
        pts[q] = p;
    }
}

} // namespace

size_t scan_recompute_smem_bytes()
{
    return (size_t)WARPS * WARP_PTS * sizeof(Pt) + WARPS * sizeof(uint64_t) + WARPS * sizeof(BestF);
}

cudaError_t scan_recompute_configure()
{
    const int bytes = (int)scan_recompute_smem_bytes();
    cudaError_t e = cudaFuncSetAttribute(two_opt_scan_recompute_kernel<true, true>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(two_opt_scan_recompute_kernel<true, false>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(two_opt_scan_recompute_kernel<false, false>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    return e;
}

void launch_scan_recompute(Pt *pts, const ScanGeom &g, const int32_t *band_first, BestF *blockbest,
                           DevState *state, unsigned int *ticket, tl_move *log, uint64_t log_cap,
                           bool fuse_apply, const ShardComm *shard, int grid, bool fast, cudaStream_t st)
{
    const size_t smem = scan_recompute_smem_bytes();
    ShardComm sc{};
    sc.world = 1;
    if (shard) sc = *shard;
    cudaLaunchAttribute attr[1];
    const cudaLaunchConfig_t cfg = pdl_config(grid, WARPS * 32, smem, attr, st);
    const int fuse = fuse_apply ? 1 : 0;
    auto kern = (fast && g.screen_margin >= 0.0f) ? two_opt_scan_recompute_kernel<true, true>
                : fast                           ? two_opt_scan_recompute_kernel<true, false>
                                                 : two_opt_scan_recompute_kernel<false, false>;
    cudaLaunchKernelEx(&cfg, kern, pts, g, band_first, blockbest, state, ticket, log, (uint64_t)log_cap, fuse, sc);
}

void launch_build_pts(const float2 *xy, const uint32_t *tour, uint32_t n, uint32_t npad, int cyclic,
                      bool fast, Pt *pts, cudaStream_t st)
{
    const int grid = (int)((npad + 255) / 256);
    if (fast)
        build_pts_kernel<true><<<grid, 256, 0, st>>>(xy, tour, n, npad, cyclic, pts);
    else
        build_pts_kernel<false><<<grid, 256, 0, st>>>(xy, tour, n, npad, cyclic, pts);
}

} // namespace tl
