// k5_knn.cu -- K5: brute-force k nearest neighbours, and the nearest-neighbour constructor.
//
// k-NN replaces DistanceMatrix::nearest for every city at once and
// lin_kernighan::build_candidates (src/tsp/distance_matrix.rs:259-297,
// src/tsp/lin_kernighan.rs:12-27; buffer rule NearestResult::add, src/tsp/mod.rs:1839-1858):
// candidates are visited in ascending position, a candidate is accepted while the buffer is
// not full or when d < d_kth, and it is inserted AFTER equal keys -- so ties resolve to the
// lower position.  One thread per query city, candidates staged through shared memory in
// tiles, the k best kept in registers with a branch-free insertion.
//
// NN tour replaces nearest_neighbor::solve (src/tsp/nearest_neighbor.rs:22-70).  With the
// buffer rule above, "first unvisited of the k nearest, else nearest unvisited" is the same
// city as "nearest unvisited, ties to the lower position" for every k, so the kernel walks a
// precomputed 32-NN list and only falls back to a block-wide argmin when all 32 are visited.
// (The reference's own fallback iterates a HashSet, so exact ties there are nondeterministic
// in the reference; see oracle/algos.inc.)
#include "kernels.cuh"

#include <algorithm>

#include <math_constants.h>

namespace tl {

namespace {

constexpr int kTile = 1024;

// Distances are compared as f32: the nint metrics' integers are exact there while distances stay
// below 2^24 (api.cu checks this for NINT problems).
template <Metric M, int K>
__global__ void __launch_bounds__(256)
    knn_kernel(const float2 *__restrict__ xy, uint32_t n, uint32_t k, uint32_t *__restrict__ out)
{
    __shared__ float2 tile[kTile];
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    const float2 pq = q < n ? xy[q] : make_float2(0.f, 0.f);
    float dk[K];
    uint32_t ik[K];
#pragma unroll
    for (int t = 0; t < K; ++t) {
        dk[t] = CUDART_INF_F;
        ik[t] = 0xffffffffu;
    }
    for (uint32_t c0 = 0; c0 < n; c0 += kTile) {
        __syncthreads();
        for (uint32_t t = threadIdx.x; t < kTile && c0 + t < n; t += blockDim.x) tile[t] = xy[c0 + t];
        __syncthreads();
        const uint32_t cnt = min((uint32_t)kTile, n - c0);
        if (q < n) {
            auto offer = [&](uint32_t c, float d) {
                if (c != q && d < dk[K - 1]) {
                    // elements <= d stay; the first slot with a larger key takes d; the rest shift
#pragma unroll
                    for (int s = K - 1; s >= 0; --s) {
                        if (dk[s] > d) {
                            if (s == 0 || dk[s > 0 ? s - 1 : 0] <= d) {
                                dk[s] = d;
                                ik[s] = c;
                            } else {
                                dk[s] = dk[s > 0 ? s - 1 : 0];
                                ik[s] = ik[s > 0 ? s - 1 : 0];
                            }
                        }
                    }
                }
            };
            // a query is one thread walking n candidates: four distances are computed before the
            // four (ordered, rarely taken) insertions so that their sqrt chains overlap
            uint32_t t = 0;
            for (; t + 4 <= cnt; t += 4) {
                float d[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const float2 pc = tile[t + u];
                    d[u] = (float)dist<M>(pq.x, pq.y, pc.x, pc.y);
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) offer(c0 + t + u, d[u]);
            }
            for (; t < cnt; ++t) {
                const float2 pc = tile[t];
                offer(c0 + t, (float)dist<M>(pq.x, pq.y, pc.x, pc.y));
            }
        }
    }
    if (q < n) {
#pragma unroll
        for (int t = 0; t < K; ++t)
            if ((uint32_t)t < k) out[(size_t)q * k + t] = ik[t];
    }
}

// explicit-matrix variant: distances from the packed triangle
template <int K>
__global__ void __launch_bounds__(256)
    knn_packed_kernel(const float *__restrict__ tri, uint32_t n, uint32_t k, uint32_t *__restrict__ out)
{
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    float dk[K];
    uint32_t ik[K];
#pragma unroll
    for (int t = 0; t < K; ++t) {
        dk[t] = CUDART_INF_F;
        ik[t] = 0xffffffffu;
    }
    for (uint32_t c = 0; c < n; ++c) {
        if (c == q) continue;
        const uint64_t hi = max(q, c), lo = min(q, c);
        const float d = __ldg(&tri[hi * (hi - 1) / 2 + lo]);
        if (d < dk[K - 1]) {
#pragma unroll
            for (int s = K - 1; s >= 0; --s) {
                if (dk[s] > d) {
                    if (s == 0 || dk[s > 0 ? s - 1 : 0] <= d) {
                        dk[s] = d;
                        ik[s] = c;
                    } else {
                        dk[s] = dk[s > 0 ? s - 1 : 0];
                        ik[s] = ik[s > 0 ? s - 1 : 0];
                    }
                }
            }
        }
    }
#pragma unroll
    for (int t = 0; t < K; ++t)
        if ((uint32_t)t < k) out[(size_t)q * k + t] = ik[t];
}

// One CTA walks the tour; visited bits live in shared memory.  The walk is a pointer chase (the next
// city is known only once the current one's list has been looked at), so its speed is the latency
// of one step.  Warp 0 walks alone while it can: the first `ks` entries of every 32-NN list are
// kept in shared memory as 16-bit positions (lane t looks at entry t: two dependent LDS and a
// ballot per step, ~100 cycles), entries ks..kk-1 are looked up in global memory only when those
// are all visited, and the other 31 warps wait at the barrier until a step needs the block-wide
// argmin (every listed neighbour visited) -- 8.3 ms -> see profiles for n = 10 000.
template <Metric M>
__global__ void __launch_bounds__(1024)
    nn_tour_kernel(const float2 *__restrict__ xy, const float *__restrict__ tri, uint32_t n,
                   const uint32_t *__restrict__ knn, uint32_t kk, uint32_t ks, uint32_t *__restrict__ tour)
{
    extern __shared__ uint32_t visited[]; // ceil(n/32) words, then n * ks uint16 list heads
    __shared__ float s_d[32];
    __shared__ uint32_t s_c[32];
    __shared__ uint32_t s_cur, s_step;
    const uint32_t words = (n + 31) / 32;
    uint16_t *heads = reinterpret_cast<uint16_t *>(visited + words);
    for (uint32_t w = threadIdx.x; w < words; w += blockDim.x) visited[w] = 0;
    for (uint32_t t = threadIdx.x; t < n * ks; t += blockDim.x) {
        const uint32_t c = knn[(size_t)(t / ks) * kk + (t % ks)];
        heads[t] = (uint16_t)c; // ks > 0 only when n <= 65535; 0xffffffff (no entry) becomes 0xffff
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        visited[0] = 1u;
        tour[0] = 0;
        s_cur = 0;
        s_step = 1;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (;;) {
        if (warp == 0) {
            uint32_t cur = s_cur, step = s_step, pick = 0xffffffffu;
            while (step < n) {
                // first unvisited entry of the sorted neighbour list (lane t looks at entry t)
                pick = 0xffffffffu;
                if (ks > 0) {
                    const uint32_t c = (uint32_t)lane < ks ? (uint32_t)heads[cur * ks + lane] : 0xffffu;
                    const bool ok = c != 0xffffu && !((visited[c >> 5] >> (c & 31)) & 1u);
                    const uint32_t m = __ballot_sync(0xffffffffu, ok);
                    if (m) pick = __shfl_sync(0xffffffffu, c, __ffs(m) - 1);
                }
                if (pick == 0xffffffffu && ks < kk) { // the rest of the list, from global memory
                    const uint32_t c = ((uint32_t)lane >= ks && (uint32_t)lane < kk) ? knn[(size_t)cur * kk + lane] : 0xffffffffu;
                    const bool ok = c != 0xffffffffu && !((visited[c >> 5] >> (c & 31)) & 1u);
                    const uint32_t m = __ballot_sync(0xffffffffu, ok);
                    if (m) pick = __shfl_sync(0xffffffffu, c, __ffs(m) - 1);
                }
                if (pick == 0xffffffffu) break; // block-wide argmin needed
                if (lane == 0) {
                    tour[step] = pick;
                    visited[pick >> 5] |= 1u << (pick & 31);
                }
                __syncwarp();
                cur = pick;
                ++step;
            }
            __syncwarp(); // every lane has read s_cur / s_step (the walk may have made no step)
            if (lane == 0) {
                s_cur = cur;
                s_step = step;
            }
        }
        __syncthreads();
        const uint32_t cur = s_cur, step = s_step;
        if (step >= n) break;
        {
            // all listed neighbours are visited: nearest unvisited, ties to the lower position
            float bd = CUDART_INF_F;
            uint32_t bc = 0xffffffffu;
            const float2 pc = tri ? make_float2(0.f, 0.f) : xy[cur];
            for (uint32_t c = threadIdx.x; c < n; c += blockDim.x) {
                if ((visited[c >> 5] >> (c & 31)) & 1u) continue;
                float d;
                if (tri) {
                    const uint64_t hi = max(cur, c), lo = min(cur, c);
                    d = __ldg(&tri[hi * (hi - 1) / 2 + lo]);
                } else {
                    const float2 p = xy[c];
                    d = (float)dist<M>(pc.x, pc.y, p.x, p.y);
                }
                if (bc == 0xffffffffu || d < bd) { bd = d; bc = c; } // c ascending within a thread
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const float od = __shfl_xor_sync(0xffffffffu, bd, off);
                const uint32_t oc = __shfl_xor_sync(0xffffffffu, bc, off);
                if (oc != 0xffffffffu && (bc == 0xffffffffu || od < bd || (od == bd && oc < bc))) { bd = od; bc = oc; }
            }
            if (lane == 0) { s_d[warp] = bd; s_c[warp] = bc; }
            __syncthreads();
            if (warp == 0) {
                bd = s_d[lane];
                bc = (lane < (int)(blockDim.x >> 5)) ? s_c[lane] : 0xffffffffu;
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) {
                    const float od = __shfl_xor_sync(0xffffffffu, bd, off);
                    const uint32_t oc = __shfl_xor_sync(0xffffffffu, bc, off);
                    if (oc != 0xffffffffu && (bc == 0xffffffffu || od < bd || (od == bd && oc < bc))) { bd = od; bc = oc; }
                }
                if (lane == 0) {
                    tour[step] = bc;
                    visited[bc >> 5] |= 1u << (bc & 31);
                    s_cur = bc;
                    s_step = step + 1;
                }
            }
            __syncthreads();
        }
    }
}

template <Metric M>
void launch_knn_k(const float2 *xy, uint32_t n, uint32_t k, uint32_t *out, cudaStream_t st)
{
    // one thread per query: a query's time is n candidates long whatever the grid, so small
    // instances get small CTAs -- more SMs busy, fewer warps sharing a scheduler
    const int threads = n >= 148u * 256u ? 256 : (n >= 148u * 128u ? 128 : 64);
    const int grid = (int)((n + threads - 1) / threads);
    if (k <= 4)
        knn_kernel<M, 4><<<grid, threads, 0, st>>>(xy, n, k, out);
    else if (k <= 8)
        knn_kernel<M, 8><<<grid, threads, 0, st>>>(xy, n, k, out);
    else if (k <= 16)
        knn_kernel<M, 16><<<grid, threads, 0, st>>>(xy, n, k, out);
    else
        knn_kernel<M, 32><<<grid, threads, 0, st>>>(xy, n, k, out);
}

} // namespace

void launch_knn(const float2 *xy, const float *tri, uint32_t n, uint32_t k, Metric metric, uint32_t *out,
                cudaStream_t st)
{
    if (tri) {
        const int grid = (int)((n + 255) / 256);
        if (k <= 4)
            knn_packed_kernel<4><<<grid, 256, 0, st>>>(tri, n, k, out);
        else if (k <= 8)
            knn_packed_kernel<8><<<grid, 256, 0, st>>>(tri, n, k, out);
        else if (k <= 16)
            knn_packed_kernel<16><<<grid, 256, 0, st>>>(tri, n, k, out);
        else
            knn_packed_kernel<32><<<grid, 256, 0, st>>>(tri, n, k, out);
    } else {
        with_metric(metric, [&](auto M) { launch_knn_k<M>(xy, n, k, out, st); });
    }
}

size_t nn_tour_smem_bytes(uint32_t n) { return (size_t)((n + 31) / 32) * 4; }

// list heads kept in shared memory beside the visited bitmap: as many entries per city as fit (at most
// 16, at least 4, else none) -- every entry kept there is one global-memory round trip saved whenever
// the nearer ones are all visited (10 entries at n = 10 000, 16 up to n = 6 300)
static uint32_t nn_tour_heads(uint32_t n, uint32_t kk)
{
    if (n > 65535) return 0;
    const size_t room = (size_t)200 * 1024 - std::min<size_t>((size_t)200 * 1024, nn_tour_smem_bytes(n));
    const uint32_t ks = (uint32_t)std::min<size_t>(std::min<uint32_t>(16u, kk), room / ((size_t)n * 2));
    return ks >= 4 ? ks : 0;
}

cudaError_t nn_tour_configure()
{
    cudaError_t e = cudaSuccess;
    for (Metric m : kMetrics)
        if (e == cudaSuccess)
            e = with_metric(m, [](auto M) { return cudaFuncSetAttribute(nn_tour_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); });
    return e;
}

void launch_nn_tour(const float2 *xy, const float *tri, uint32_t n, const uint32_t *knn, uint32_t kk,
                    Metric metric, uint32_t *tour, cudaStream_t st)
{
    const uint32_t ks = getenv("TL_NN_NO_HEADS") ? 0 : nn_tour_heads(n, kk);
    const size_t smem = nn_tour_smem_bytes(n) + (size_t)n * ks * 2;
    // EXPLICIT problems (F32_SAFE) pass tri: the kernel reads the triangle instead of recomputing
    with_metric(metric, [&](auto M) { nn_tour_kernel<M><<<1, 1024, smem, st>>>(xy, tri, n, knn, kk, ks, tour); });
}

} // namespace tl
