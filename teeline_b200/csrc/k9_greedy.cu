// k9_greedy.cu -- K9: the greedy-edge constructor (greedy_edge::solve, src/tsp/greedy_edge.rs), exact and
// parallel, on the k-NN candidate lists.
//
// Definition (include/teeline_cuda.h, tl_greedy_tour): edge (a, b), a < b, has the key (d(a, b), a, b) with d
// the problem's metric compared as K5 compares it (f32; nint values are exact there).  The sequential greedy
// takes the edges in key order and accepts one when both endpoints have degree < 2 and lie in different
// fragments; keys never tie, so its result is one tour.
//
// State: deg[v], two adjacency slots per city, and other[v] = the far endpoint of v's fragment while v is
// free (degree < 2); a singleton is its own other.  Edge (u, v) is ELIGIBLE when both are free and
// v != other[u].  A round is two kernels:
//   best   every free city u walks its list in order and takes the first eligible entry v.  A list is
//          sorted by (d, position), which for a fixed u is the key order of the edges (u, .), so v is u's
//          minimum eligible edge among the listed ones; every unlisted city has a larger key than the last
//          listed one.  If no entry is eligible, u is EXHAUSTED and the key of its last entry is a lower
//          bound of its true minimum (no bound when the list holds every city of the set it was built on).
//   accept edge e = (u, v) is accepted when it is the best edge of both u and v and its key is below the
//          best key or bound of other[u] and of other[v] (a singleton's other is itself and is not tested).
// Why this is exact.  Call G(A) the tour the sequential greedy builds from the accepted set A, taking the
// remaining edges in key order.  Let e pass the test.  Eligibility only shrinks as edges are accepted, so
// every edge that G(A) could still accept at u, v, other[u] or other[v] has a key above key(e) (e itself
// aside): below key(e) there is none eligible now at these four cities.  Before reaching e, G(A) therefore
// changes neither the degree of u or v nor the fragments of u and v (a fragment only grows at its two free
// endpoints), so it accepts e; and no edge below key(e) touches a fragment that e changes, so G(A + e) makes
// the same choices as G(A): G(A + e) = G(A).
// Two accepted edges share none of their four cities: not u (each city has one best edge), and not
// u' = other[u], since then key(e) < key(e') < key(e) by the two tests.  A round therefore applies all of
// them at once with no write conflicts, and each stays accepted after the others (their cities' best keys
// are unchanged and bounds only rise).  The accept kernel reads other[] through a snapshot taken by the
// best kernel, so a city next to an accepted edge never tests itself against an endpoint written in the
// same round.
// Progress.  When a round accepts nothing, the host rebuilds the lists of the free cities over the free
// cities only (compacted in position order, so K5's tie order is kept; knn_kernel; indices mapped back),
// kRefreshK wide.  Every free city then has an exact minimum eligible edge (at least 3 cities are free, a
// list of >= 2 free cities holds one that is not other[u]), and the global minimum passes the test, so
// the round after a refresh accepts at least one edge.  Inputs whose edges can only be taken one by one
// (cities on a line with growing gaps) need about n rounds; stats.passes reports them.
// Stop and emit.  With two free cities left (n >= 3) the path is closed.  The tour is emitted by pointer
// jumping over the 2n directed arcs, succ(a -> b) = (b -> c) with c the other neighbour of b: one
// direction of the cycle is ranked from the arc 0 -> (lower neighbour of 0), in ceil(log2 n) + 1 rounds.
#include "kernels.cuh"

namespace tl {

namespace {

constexpr uint32_t kNone = 0xffffffffu;
constexpr uint32_t kExhausted = 0x80000000u; // best-record flag: the partner is the last listed entry
constexpr int kThreads = 256;

struct Key {
    float d;
    uint32_t lo, hi;
};
__device__ __forceinline__ bool key_less(const Key &a, const Key &b)
{
    return a.d < b.d || (a.d == b.d && (a.lo < b.lo || (a.lo == b.lo && a.hi < b.hi)));
}
__device__ __forceinline__ Key edge_key(float d, uint32_t a, uint32_t b) { return Key{d, min(a, b), max(a, b)}; }

// the best key or bound of free city c from its record; *none: no bound (list complete and exhausted)
__device__ __forceinline__ Key city_key(uint32_t c, const float *bd, const uint32_t *bv, bool *none)
{
    const uint32_t r = bv[c];
    *none = r == kNone;
    return edge_key(bd[c], c, r & ~kExhausted);
}

__global__ void __launch_bounds__(kThreads) greedy_init_kernel(uint32_t n, uint8_t *deg, uint32_t *other, GreedyState *gs)
{
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u < n) {
        deg[u] = 0;
        other[u] = u;
    }
    if (u == 0) {
        gs->status = kGreedyRun;
        gs->free = n;
        gs->round_acc = 0;
        gs->ticket = 0;
        gs->rounds = 0;
        gs->accepted = 0;
    }
}

template <Metric M>
__global__ void __launch_bounds__(kThreads)
    greedy_best_kernel(const float2 *__restrict__ xy, uint32_t n, const uint32_t *__restrict__ list, uint32_t k,
                       const uint8_t *__restrict__ deg, const uint32_t *__restrict__ other, float *__restrict__ bd,
                       uint32_t *__restrict__ bv, uint32_t *__restrict__ oth, const GreedyState *gs)
{
    if (gs->status != kGreedyRun) return;
    for (uint32_t u = blockIdx.x * blockDim.x + threadIdx.x; u < n; u += gridDim.x * blockDim.x) {
        if (deg[u] >= 2) continue;
        const uint32_t ou = other[u];
        const uint32_t *row = list + (size_t)u * k;
        uint32_t pick = kNone, last = kNone;
        bool complete = false;
        for (uint32_t t = 0; t < k; ++t) {
            const uint32_t v = row[t];
            if (v == kNone) { complete = true; break; }
            last = v;
            if (deg[v] < 2 && v != ou) { pick = v; break; }
        }
        oth[u] = ou;
        if (pick == kNone && complete) {
            bv[u] = kNone;
            continue;
        }
        const uint32_t v = pick != kNone ? pick : last;
        const float2 pu = xy[u], pv = xy[v];
        bd[u] = (float)dist<M>(pu.x, pu.y, pv.x, pv.y);
        bv[u] = pick != kNone ? v : (v | kExhausted);
    }
}

__global__ void __launch_bounds__(kThreads)
    greedy_accept_kernel(uint32_t n, uint8_t *__restrict__ deg, uint32_t *__restrict__ adj, uint32_t *__restrict__ other,
                         const float *__restrict__ bd, const uint32_t *__restrict__ bv, const uint32_t *__restrict__ oth,
                         GreedyState *gs)
{
    if (gs->status != kGreedyRun) return; // read by every block before the ticket below; only the last block writes it
    __shared__ uint32_t s_acc, s_full;
    if (threadIdx.x == 0) { s_acc = 0; s_full = 0; }
    __syncthreads();
    uint32_t acc = 0, full = 0;
    for (uint32_t u = blockIdx.x * blockDim.x + threadIdx.x; u < n; u += gridDim.x * blockDim.x) {
        // deg[u] may be raised in this kernel only when u is the larger endpoint of an accepted edge,
        // which its smaller endpoint applies: u reads either value and applies nothing
        if (deg[u] >= 2) continue;
        const uint32_t v = bv[u];
        if (v & kExhausted) continue; // also kNone
        if (bv[v] != u) continue;     // v was free when the best kernel ran, so its record is current
        const Key e = edge_key(bd[u], u, v);
        const uint32_t a = oth[u], b = oth[v];
        bool none;
        if (a != u) {
            const Key ka = city_key(a, bd, bv, &none);
            if (!none && !key_less(e, ka)) continue;
        }
        if (b != v) {
            const Key kb = city_key(b, bd, bv, &none);
            if (!none && !key_less(e, kb)) continue;
        }
        if (u > v) continue; // the smaller endpoint applies
        const uint8_t du = deg[u], dv = deg[v];
        adj[2 * (size_t)u + du] = v;
        adj[2 * (size_t)v + dv] = u;
        deg[u] = du + 1;
        deg[v] = dv + 1;
        other[a] = b;
        other[b] = a;
        ++acc;
        full += (du == 1) + (dv == 1);
    }
    if (acc) atomicAdd(&s_acc, acc);
    if (full) atomicAdd(&s_full, full);
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_acc) {
            atomicAdd(&gs->round_acc, s_acc);
            atomicAdd(&gs->accepted, (unsigned long long)s_acc);
        }
        if (s_full) atomicSub(&gs->free, s_full);
        __threadfence();
        if (atomicAdd(&gs->ticket, 1u) == gridDim.x - 1) { // last block: end the round
            __threadfence();
            const uint32_t free_now = atomicAdd(&gs->free, 0u), acc_round = atomicAdd(&gs->round_acc, 0u);
            gs->rounds += 1;
            gs->round_acc = 0;
            gs->ticket = 0;
            gs->status = free_now <= 2 ? kGreedyDone : (acc_round ? kGreedyRun : kGreedyStalled);
        }
    }
}

// ---- refresh: the free cities, compacted in position order --------------------------------------------------

constexpr int kScanThreads = 1024;

__global__ void __launch_bounds__(kScanThreads) greedy_count_kernel(uint32_t n, const uint8_t *__restrict__ deg, uint32_t *__restrict__ blockcnt)
{
    const uint32_t u = blockIdx.x * kScanThreads + threadIdx.x;
    const int c = __syncthreads_count(u < n && deg[u] < 2);
    if (threadIdx.x == 0) blockcnt[blockIdx.x] = (uint32_t)c;
}

// exclusive prefix of the block counts, in place (one thread: at most a few thousand entries)
__global__ void greedy_scan_kernel(uint32_t nb, uint32_t *blockcnt)
{
    uint32_t s = 0;
    for (uint32_t b = 0; b < nb; ++b) {
        const uint32_t c = blockcnt[b];
        blockcnt[b] = s;
        s += c;
    }
}

__global__ void __launch_bounds__(kScanThreads)
    greedy_compact_kernel(uint32_t n, const uint8_t *__restrict__ deg, const float2 *__restrict__ xy,
                          const uint32_t *__restrict__ blockoff, float2 *__restrict__ cxy, uint32_t *__restrict__ cidx)
{
    __shared__ uint32_t s_warp[kScanThreads / kWarp];
    const uint32_t u = blockIdx.x * kScanThreads + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool f = u < n && deg[u] < 2;
    const uint32_t m = __ballot_sync(0xffffffffu, f);
    if (lane == 0) s_warp[warp] = __popc(m);
    __syncthreads();
    if (warp == 0) {
        const uint32_t c = s_warp[lane];
        uint32_t incl = c;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t o = __shfl_up_sync(0xffffffffu, incl, off);
            if (lane >= off) incl += o;
        }
        s_warp[lane] = incl - c;
    }
    __syncthreads();
    if (f) {
        const uint32_t at = blockoff[blockIdx.x] + s_warp[warp] + __popc(m & ((1u << lane) - 1u));
        cxy[at] = xy[u];
        cidx[at] = u;
    }
}

// compacted k-NN rows -> the list rows of the free cities, in positions
__global__ void __launch_bounds__(kThreads)
    greedy_map_kernel(uint32_t F, uint32_t k, const uint32_t *__restrict__ cidx, const uint32_t *__restrict__ cknn,
                      uint32_t *__restrict__ list)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= F) return;
    uint32_t *row = list + (size_t)cidx[i] * k;
    for (uint32_t t = 0; t < k; ++t) {
        const uint32_t e = cknn[(size_t)i * k + t];
        row[t] = e == kNone ? kNone : cidx[e];
    }
}

// ---- emission ------------------------------------------------------------------------------------------------

// close the path: its two endpoints are the free cities, each the other's `other`
__global__ void __launch_bounds__(kThreads) greedy_close_kernel(uint32_t n, const uint8_t *__restrict__ deg, const uint32_t *__restrict__ other, uint32_t *__restrict__ adj)
{
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u < n && deg[u] < 2) adj[2 * (size_t)u + deg[u]] = other[u];
}

// arc a = 2c + s is c -> adj[a].  The arc entering the start arc 0 -> (lower neighbour of 0) becomes the
// terminal of the ranking: it points at itself with distance 0.
__global__ void __launch_bounds__(kThreads) greedy_arcs_kernel(uint32_t n, const uint32_t *__restrict__ adj, uint32_t *__restrict__ succ, uint32_t *__restrict__ dist)
{
    const uint32_t a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= 2 * n) return;
    const uint32_t c = a >> 1, b = adj[a];
    const uint32_t s = 2 * b + (adj[2 * (size_t)b] == c ? 1 : 0);
    const uint32_t start = adj[0] < adj[1] ? 0 : 1;
    succ[a] = s == start ? a : s;
    dist[a] = s == start ? 0 : 1;
}

__global__ void __launch_bounds__(kThreads)
    greedy_jump_kernel(uint32_t n2, const uint32_t *__restrict__ succ_in, const uint32_t *__restrict__ dist_in,
                       uint32_t *__restrict__ succ_out, uint32_t *__restrict__ dist_out)
{
    const uint32_t a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= n2) return;
    const uint32_t s = succ_in[a];
    succ_out[a] = succ_in[s];
    dist_out[a] = dist_in[a] + dist_in[s]; // arcs of the other direction never reach the terminal; their sums are not read
}

// every arc that has reached the terminal is `dist` arcs before it: arc number n-1-dist of the tour
__global__ void __launch_bounds__(kThreads)
    greedy_write_kernel(uint32_t n, const uint32_t *__restrict__ adj, const uint32_t *__restrict__ succ,
                        const uint32_t *__restrict__ dist, uint32_t *__restrict__ tour)
{
    const uint32_t a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a == 0) tour[0] = 0;
    if (a >= 2 * n) return;
    const uint32_t s = succ[a];
    if (succ[s] != s) return; // not on the ranked direction (its chain never ends in the terminal)
    const uint32_t at = n - 1 - dist[a];
    if (at + 1 < n) tour[at + 1] = adj[a];
}

inline int blocks(size_t work, int threads) { return (int)((work + threads - 1) / threads); }

} // namespace

void launch_greedy_init(uint32_t n, uint8_t *deg, uint32_t *other, GreedyState *gs, cudaStream_t st)
{
    greedy_init_kernel<<<blocks(n, kThreads), kThreads, 0, st>>>(n, deg, other, gs);
}

void launch_greedy_round(const float2 *xy, uint32_t n, Metric metric, const uint32_t *list, uint32_t k, GreedyBufs b,
                         int grid, cudaStream_t st)
{
    with_metric(metric, [&](auto M) {
        greedy_best_kernel<M><<<grid, kThreads, 0, st>>>(xy, n, list, k, b.deg, b.other, b.bd, b.bv, b.oth, b.state);
    });
    greedy_accept_kernel<<<grid, kThreads, 0, st>>>(n, b.deg, b.adj, b.other, b.bd, b.bv, b.oth, b.state);
}

size_t greedy_refresh_blocks(uint32_t n) { return (n + kScanThreads - 1) / kScanThreads; }

void launch_greedy_compact(const float2 *xy, uint32_t n, const uint8_t *deg, uint32_t *blockcnt, float2 *cxy,
                           uint32_t *cidx, cudaStream_t st)
{
    const uint32_t nb = (uint32_t)greedy_refresh_blocks(n);
    greedy_count_kernel<<<nb, kScanThreads, 0, st>>>(n, deg, blockcnt);
    greedy_scan_kernel<<<1, 1, 0, st>>>(nb, blockcnt);
    greedy_compact_kernel<<<nb, kScanThreads, 0, st>>>(n, deg, xy, blockcnt, cxy, cidx);
}

void launch_greedy_map(uint32_t F, uint32_t k, const uint32_t *cidx, const uint32_t *cknn, uint32_t *list, cudaStream_t st)
{
    greedy_map_kernel<<<blocks(F, kThreads), kThreads, 0, st>>>(F, k, cidx, cknn, list);
}

int launch_greedy_emit(uint32_t n, const uint8_t *deg, const uint32_t *other, uint32_t *adj, uint32_t *succ,
                       uint32_t *dist, uint32_t *tour, cudaStream_t st)
{
    // succ and dist hold two buffers of 2n entries each
    const uint32_t n2 = 2 * n;
    greedy_close_kernel<<<blocks(n, kThreads), kThreads, 0, st>>>(n, deg, other, adj);
    greedy_arcs_kernel<<<blocks(n2, kThreads), kThreads, 0, st>>>(n, adj, succ, dist);
    int rounds = 1;
    while ((1ull << (rounds - 1)) < n) ++rounds; // ceil(log2 n) + 1
    int cur = 0;
    for (int r = 0; r < rounds; ++r, cur ^= 1)
        greedy_jump_kernel<<<blocks(n2, kThreads), kThreads, 0, st>>>(n2, succ + (size_t)cur * n2, dist + (size_t)cur * n2,
                                                                     succ + (size_t)(cur ^ 1) * n2, dist + (size_t)(cur ^ 1) * n2);
    greedy_write_kernel<<<blocks(n2, kThreads), kThreads, 0, st>>>(n, adj, succ + (size_t)cur * n2, dist + (size_t)cur * n2, tour);
    return 3 + rounds;
}

} // namespace tl
