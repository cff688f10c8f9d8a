// k1_distance.cu -- K1: pairwise distance matrices.
//
// Replaces DistanceMatrix::build (src/tsp/distance_matrix.rs:122-153): the packed
// strict lower triangle, row `hi` = distances from city hi to cities 0..hi-1,
// idx = hi*(hi-1)/2 + lo (distance_matrix.rs:177-191).  Also builds the padded
// square, tour-ordered matrix the matrix-backed scans read.
//
// Roofline: HBM write, 4 B per pair.  A warp produces 128 consecutive packed entries per step
// with fully coalesced coordinate loads (L1/L2 hits) and stores.  The packed index is inverted
// with fp64 once per thread, then advanced incrementally.
#include "kernels.cuh"

#include <algorithm>

namespace tl {

// one matrix entry as raw bits (f32 bits or int32)
template <Metric M>
__device__ __forceinline__ uint32_t k1_dist(const float2 a, const float2 b)
{
    const MetricValue<M> d = dist<M>(a.x, a.y, b.x, b.y);
    if constexpr (metric_is_int(M))
        return (uint32_t)d;
    else
        return __float_as_uint(d);
}

__device__ __forceinline__ void packed_index_to_pair(uint64_t t, uint32_t &hi, uint32_t &lo)
{
    // largest hi with hi*(hi-1)/2 <= t
    uint64_t h = (uint64_t)((1.0 + sqrt(1.0 + 8.0 * (double)t)) * 0.5);
    while (h * (h - 1) / 2 > t) --h;
    while ((h + 1) * h / 2 <= t) ++h;
    hi = (uint32_t)h;
    lo = (uint32_t)(t - h * (h - 1) / 2);
}

// Every CTA owns one contiguous piece of the packed array (`per_cta` entries, a multiple of 1024).
// A warp produces 128 consecutive entries per step and moves 1024 entries ahead: lane l owns the
// entries T + 32 e + l, e < 4, so every coordinate load (32 lanes x 8 B = 256 contiguous bytes) and
// every store (128 contiguous bytes) is fully coalesced -- the kernel is bound by L1 wavefronts,
// and 4 consecutive entries per lane cost 8 wavefronts per 8-byte load instead of 2.  The (hi, lo)
// pair of T is found once with the closed form and then advanced incrementally (rows are longer
// than 1024 almost everywhere, so the wrap loop runs 0-1 times).
template <Metric M>
__global__ void __launch_bounds__(256) k1_packed_kernel(const float2 *__restrict__ xy, uint32_t n,
                                                        uint64_t total, uint64_t per_cta,
                                                        void *__restrict__ out)
{
    const uint64_t begin = (uint64_t)blockIdx.x * per_cta;
    const uint64_t end = min(begin + per_cta, total);
    const uint32_t lane = threadIdx.x & 31;
    uint64_t T = begin + (uint64_t)(threadIdx.x >> 5) * 128;
    if (T >= end) return;
    uint32_t hi, lo;
    packed_index_to_pair(T, hi, lo); // warp-uniform
    for (; T < end; T += 1024) {
        uint32_t *o = reinterpret_cast<uint32_t *>(out) + T;
        if (lo + 128 <= hi && T + 128 <= total) {
            // common case: the warp's 128 entries lie in one row
            const float2 ph = __ldg(&xy[hi]);
            float2 pl[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) pl[e] = __ldg(&xy[lo + 32 * e + lane]);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                // the reference evaluates cities[hi].distance(cities[lo])
                o[32 * e + lane] = k1_dist<M>(ph, pl[e]);
            }
        } else {
#pragma unroll 1
            for (int e = 0; e < 4; ++e) {
                const uint32_t k = 32 * e + lane;
                if (T + k >= total) break;
                uint32_t h = hi, l = lo + k;
                while (l >= h) {
                    l -= h;
                    ++h;
                }
                const float2 ph = __ldg(&xy[h]), pl = __ldg(&xy[l]);
                o[k] = k1_dist<M>(ph, pl);
            }
        }
        // 1024 entries ahead: row hi holds hi entries
        lo += 1024;
        while (lo >= hi) {
            lo -= hi;
            ++hi;
        }
    }
}

// Square matrix in SLOT order: M[a*ld + b] = d(slot a, slot b), a,b < n; the pad columns [n, ld)
// are zero.  sxy holds slot-ordered coordinates.  The metric is bitwise symmetric (d(a,b) == d(b,a):
// (a-b)^2 == (b-a)^2 in IEEE arithmetic, and the reference's hi.distance(lo) operand order therefore
// needs no select), so only the 64 x 64 tiles on or above the diagonal are COMPUTED: a CTA computes
// tile (bi, bj), bj >= bi -- each thread a 4 x 4 patch from 4 row and 4 column points in registers --
// stores it with 128-bit stores, and stores its transpose, staged through shared memory, as tile
// (bj, bi).  Half the arithmetic of the round-1 kernel (which was issue-bound for the nint metric:
// 141 us for the 10k x 10k int32 matrix against a 61 us write floor) for the same bytes written.
template <Metric M>
__global__ void __launch_bounds__(256) k1_square_kernel(const float2 *__restrict__ sxy, uint32_t n,
                                                        uint32_t ld, void *__restrict__ out)
{
    if (blockIdx.x < blockIdx.y) return; // the mirror tile writes this one
    __shared__ uint32_t tile[64][65];
    const uint32_t tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const uint32_t col0 = blockIdx.x * 64 + tx * 4, row0 = blockIdx.y * 64 + ty * 4;
    uint32_t *mat = reinterpret_cast<uint32_t *>(out);
    float2 c[4], r[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        c[e] = (col0 + e < n) ? __ldg(&sxy[col0 + e]) : make_float2(0.f, 0.f);
        r[e] = (row0 + e < n) ? __ldg(&sxy[row0 + e]) : make_float2(0.f, 0.f);
    }
    const bool mirror = blockIdx.x != blockIdx.y;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const uint32_t rr = row0 + a;
        uint32_t v[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const uint32_t cc = col0 + e;
            const uint32_t d = k1_dist<M>(r[a], c[e]);
            v[e] = (cc >= n || rr >= n || cc == rr) ? 0u : d;
            if (mirror) tile[ty * 4 + a][tx * 4 + e] = v[e];
        }
        if (rr < n && col0 < ld)
            *reinterpret_cast<uint4 *>(mat + (size_t)rr * ld + col0) = make_uint4(v[0], v[1], v[2], v[3]);
    }
    if (!mirror) return;
    __syncthreads();
    // transpose: this thread writes rows (blockIdx.x * 64 + ty * 4 + a) of the mirror tile, 4 columns
    // starting at blockIdx.y * 64 + tx * 4
    const uint32_t tcol0 = blockIdx.y * 64 + tx * 4;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const uint32_t trow = blockIdx.x * 64 + ty * 4 + a;
        if (trow < n && tcol0 < ld) {
            const uint32_t lr = ty * 4 + a; // local column of the computed tile
            *reinterpret_cast<uint4 *>(mat + (size_t)trow * ld + tcol0) =
                make_uint4(tile[tx * 4 + 0][lr], tile[tx * 4 + 1][lr], tile[tx * 4 + 2][lr], tile[tx * 4 + 3][lr]);
        }
    }
}

// Square slot-ordered matrix gathered from a packed city-ordered triangle
// (EXPLICIT problems): M[a][b] = tri[idx(city[a], city[b])].
__global__ void __launch_bounds__(256) k1_square_from_packed_kernel(const uint32_t *__restrict__ tri,
                                                                    const int32_t *__restrict__ slot_city,
                                                                    uint32_t n, uint32_t ld,
                                                                    uint32_t *__restrict__ out)
{
    const uint32_t col0 = (blockIdx.x * 64 + (threadIdx.x & 63)) * 4;
    const uint32_t row0 = blockIdx.y * 64 + (threadIdx.x >> 6) * 16;
    if (col0 >= ld) return;
    int32_t cc[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) cc[e] = (col0 + e < n) ? __ldg(&slot_city[col0 + e]) : -1;
    for (uint32_t r = row0; r < row0 + 16 && r < n; ++r) {
        const int32_t cr = __ldg(&slot_city[r]);
        uint32_t v[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            if (cc[e] < 0 || cc[e] == cr) {
                v[e] = 0;
            } else {
                const uint64_t hi = (uint64_t)max(cr, cc[e]), lo = (uint64_t)min(cr, cc[e]);
                v[e] = __ldg(&tri[hi * (hi - 1) / 2 + lo]);
            }
        }
        *reinterpret_cast<uint4 *>(out + (size_t)r * ld + col0) = make_uint4(v[0], v[1], v[2], v[3]);
    }
}

// ---------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------
void launch_k1_packed(const float2 *xy, uint32_t n, Metric metric, void *out, int sm_count, cudaStream_t st)
{
    const uint64_t total = (uint64_t)n * (n - 1) / 2;
    // a multiple of the SM count, at least 4 steps of 1024 entries per CTA when there is enough work
    uint64_t blocks = (uint64_t)sm_count * 16;
    uint64_t per_cta = ((total + blocks - 1) / blocks + 1023) / 1024 * 1024;
    if (per_cta < 4096) per_cta = 4096;
    blocks = (total + per_cta - 1) / per_cta;
    if (blocks == 0) blocks = 1;
    with_metric(metric, [&](auto M) { k1_packed_kernel<M><<<(unsigned)blocks, 256, 0, st>>>(xy, n, total, per_cta, out); });
}

void launch_k1_square(const float2 *sxy, uint32_t n, uint32_t ld, Metric metric, void *out, cudaStream_t st)
{
    // tiles of 64 x 64; the column blocks cover the padded width ld, the row blocks the n rows; the
    // grid is square so that every tile below the diagonal has a mirror above it
    const unsigned nb = (std::max(ld, n) + 63) / 64;
    dim3 grid(nb, nb);
    with_metric(metric, [&](auto M) { k1_square_kernel<M><<<grid, 256, 0, st>>>(sxy, n, ld, out); });
}

void launch_k1_square_from_packed(const uint32_t *tri, const int32_t *slot_city, uint32_t n,
                                  uint32_t ld, uint32_t *out, cudaStream_t st)
{
    dim3 grid((ld / 4 + 63) / 64, (n + 63) / 64);
    k1_square_from_packed_kernel<<<grid, 256, 0, st>>>(tri, slot_city, n, ld, out);
}

} // namespace tl
