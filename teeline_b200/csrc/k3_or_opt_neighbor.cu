// k3_or_opt_neighbor.cu -- K3 candidate-list best-improvement Or-opt ("Or-opt N"), coordinate recompute.
//
// What it computes: Or-opt's move, delta, forbidden window and tie order (or_opt.rs:80-184, K3,
// oracle/algos.inc or_opt_scan_range), restricted to the moves that create an edge between a segment
// endpoint and one of its k nearest neighbours.  With f = p_i, l = p_i+s-1, a = p_prev(i),
// dd = p_(i+s)%n, x = p_j, y = p_(j+1)%n: for every position q, c = p_q, every slot t with
// b = K[c][t] not padding, and r = pos[b],
//   A  new edge (f, x), fwd   i = q,       j = r,             s = 1..3
//   B  new edge (l, y), fwd   i = q-s+1,   j = (r-1) mod n,   s = 1..3
//   C  new edge (l, x), rev   i = q-s+1,   j = r,             s = 2..3
//   D  new edge (f, y), rev   i = q,       j = (r-1) mod n,   s = 2..3
// at most 10 candidates per (position, slot).  A generated move counts only if it is a legal Or-opt
// move: n > s+1, 0 <= i, i+s <= n, j != prev(i) and j outside [i, i+s-1].  Its delta is K3's, in the
// metric's value type and in the same rounding order:
//   rg  = (d(a,f) + d(l,dd)) - d(a,dd)
//   fwd = ((-rg + d(x,f)) + d(l,y)) - d(x,y)
//   rev = ((-rg + d(x,l)) + d(f,y)) - d(x,y)
// The step applies the minimum of (delta, s, i, j, rev) over the generated moves strictly below
// Or-opt's threshold (-1e-3 f32, 0 for integer deltas): the reference's first-found rule as K3's rank
// key states it; duplicates carry the same key.  stats.evals counts the generated legal candidates,
// fwd and rev separately, duplicates included.  With k >= n-1 every legal move is generated (A
// produces every fwd move, C every rev move), so the moves are TL_ALGO_OR_OPT's, move for move.
//
// How: as Mode N (k2_two_opt_neighbor.cu), a grid of resident CTAs walks the n*k (position, slot)
// items with a grid-stride loop.  The records are cyclic (position 0 carries the closing edge, position
// n is the wrap copy), so every edge length a delta needs is an entering-edge field.  An item reads two
// short runs of records, q-3 .. q+3 and r-1 .. r+1 (plus p_n-1 when a segment starts at 0), and
// computes the candidate edge d(c, b) once for all ten moves.  The removal gains rg depend on (i, s)
// only; they are recomputed in the thread (five distances per item) rather than taken from a per-step
// row pass like K3's or_rowinfo_kernel, which would add a launch and an n x 16-byte write to every
// step (the row pass was not built and measured against this).
// The last CTA (acq_rel ticket) reduces the per-CTA records.  A relocated span [lo, hi] of at most
// kOrNlCtaSpan positions is moved by that CTA through the session's staging buffer (gather, block
// barrier, scatter); a longer one is left pending for the gather and scatter grids that every step
// launches, which leave at once when nothing is pending.  The grid size cannot depend on the move: the
// host queues steps without reading back.
#include "kernels.cuh"
#include "or_opt_rank.cuh"
#include "two_opt_apply.cuh"

namespace tl {

namespace {

constexpr int THREADS = kNlThreads;
constexpr int WARPS = THREADS / 32;
constexpr uint32_t kNone = 0xffffffffu;

// loop state and log after an Or-opt N step (one thread)
__device__ __forceinline__ void finish_or_step(DevState *state, const StateHeader &h, const OrMove &m,
                                               tl_move *__restrict__ log, uint64_t log_cap)
{
    const unsigned long long mv = h.h0.x;
    const long long max_moves = h.h1.x;
    state->scans = h.h0.y + 1;
    if (m.found) {
        if (log && mv < log_cap) log[mv] = tl_move{m.delta, m.i, m.j, (uint8_t)m.s, (uint8_t)m.rev, 0};
        state->moves = mv + 1;
        if (max_moves >= 0 && (long long)(mv + 1) >= max_moves) state->done = 1;
    } else {
        state->done = 1;
        state->converged = 1;
    }
}

// apply_relocation in two phases with a barrier between them (block or grid): first copy the new
// occupants of [lo, hi] to tmp ...
template <class Pol>
__device__ __forceinline__ void or_gather(const Pol &P, Pt *__restrict__ tmp, const OrMove &m, uint32_t tid,
                                          uint32_t nthreads)
{
    for (uint32_t q = m.lo + tid; q <= m.hi; q += nthreads) tmp[q - m.lo] = P.load(or_source(m, q));
}

// ... then write them back with the entering edges of lo .. hi+1 and their pos[] entries; thread 0 of
// the group rewrites the closing edge and the wrap copy at position n.  Every read of a relocated
// position goes to tmp, so the in-place writes cannot race with them.
template <class Pol>
__device__ __forceinline__ void or_scatter(const Pol &P, const Pt *__restrict__ tmp, uint32_t n, const OrMove &m,
                                           uint32_t *__restrict__ pos, uint32_t tid, uint32_t nthreads)
{
    using V = typename Pol::V;
    auto newpt = [&](uint32_t q) -> Pt {
        const uint32_t qq = q == n ? 0u : q;
        return (qq >= m.lo && qq <= m.hi) ? tmp[qq - m.lo] : P.load(qq);
    };
    for (uint32_t q = m.lo + tid; q <= m.hi + 1; q += nthreads) {
        if (q < 1 || q > n) continue;
        const Pt p = newpt(q), b = newpt(q - 1);
        const V e = P.dist(b, p);
        if (q <= m.hi) {
            P.store_id(q, p);
            pos[p.city] = q;
        }
        P.store_sp(q, e); // hi+1: same city (or the wrap copy), new entering edge
    }
    if (tid == 0 && (m.lo == 0 || m.hi >= n - 1)) {
        const Pt p0 = newpt(0), last = newpt(n - 1);
        const V e = P.dist(last, p0);
        if (m.lo == 0) {
            P.store_id(0, p0);
            pos[p0.city] = 0;
        }
        P.store_sp(0, e);
        P.store_id(n, p0);
        P.store_sp(n, e);
    }
}

// Tail of a fused step, run by the last CTA: reduce the per-CTA records, count the step's evaluated
// candidates, then either relocate a short span here and finish the step, or leave a long one pending.
template <class Pol>
__device__ __noinline__ void or_nl_tail(const Pol &P, uint32_t n, uint32_t *pos, Pt *tmp, Best<typename Pol::V> *blockbest,
                                        const unsigned long long *blockcnt, DevState *state, unsigned int *ticket,
                                        tl_move *__restrict__ log, uint64_t log_cap)
{
    using V = typename Pol::V;
    __shared__ Best<V> red[WARPS];
    __shared__ unsigned long long red_cnt[WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    StateHeader hdr{};
    if (threadIdx.x == 0) hdr = load_state_header(state);
    Best<V> v{(V)0, kNone, kNone, 0u};
    unsigned long long cnt = 0;
    for (int c = threadIdx.x; c < (int)gridDim.x; c += blockDim.x) {
        // L2 reads: the records were written by other CTAs of this launch
        const int4 raw = __ldcg(reinterpret_cast<const int4 *>(blockbest) + c);
        const Best<V> o{Val<V>::from_bits(raw.x), (uint32_t)raw.y, (uint32_t)raw.z, (uint32_t)raw.w};
        cnt += __ldcg(blockcnt + c);
        if (better_or(o, v)) v = o;
    }
    warp_argmin_or(v);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
    if (lane == 0) {
        red[warp] = v;
        red_cnt[warp] = cnt;
    }
    __syncthreads();
    v = red[0];
    cnt = red_cnt[0];
#pragma unroll
    for (int w = 1; w < WARPS; ++w) {
        cnt += red_cnt[w];
        if (better_or(red[w], v)) v = red[w];
    }
    const OrMove m = or_move_of(v);
    const bool long_span = m.found && m.hi - m.lo + 1 > (uint32_t)kOrNlCtaSpan;
    if (threadIdx.x == 0) {
        state->computed += cnt;
        // the pending move for this step's apply grids (none: the step is finished here)
        blockbest[gridDim.x] = long_span ? v : Best<V>{(V)0, kNone, kNone, 0u};
        *ticket = 0u;
    }
    if (long_span) return;
    if (m.found) {
        or_gather(P, tmp, m, threadIdx.x, blockDim.x);
        __syncthreads();
        or_scatter(P, tmp, n, m, pos, threadIdx.x, blockDim.x);
    }
    if (threadIdx.x == 0) finish_or_step(state, hdr, m, log, log_cap);
}

template <class Pol>
__global__ void __launch_bounds__(THREADS, kNlMinBlocks)
    or_nl_scan_kernel(Pol P, uint32_t *__restrict__ pos, const uint32_t *__restrict__ cand, uint32_t k, uint32_t n,
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
    const V thr = Val<V>::or_threshold();
    // a candidate move (i, j, s, rev) with its delta: counted if legal, kept if below the threshold and
    // better in (delta, rank)
    auto consider = [&](bool legal, V d, uint32_t i, uint32_t j, uint32_t s, uint32_t rev) {
        if (!legal) return;
        ++cnt;
        const Best<V> o{d, i, j, (s - 1) * 2 + rev};
        if (d < thr && better_or(o, best)) best = o;
    };
    // j is a legal insertion edge of the segment [i, i+s-1] (the caller checks n > s+1, 0 <= i, i+s <= n)
    auto window_ok = [&](uint32_t i, uint32_t s, uint32_t j) {
        const uint32_t prev = i == 0 ? n - 1 : i - 1;
        return j != prev && (j < i || j >= i + s);
    };
    const uint64_t total = (uint64_t)n * k;
    for (uint64_t t = (uint64_t)blockIdx.x * THREADS + threadIdx.x; t < total; t += (uint64_t)gridDim.x * THREADS) {
        const uint32_t q = (uint32_t)(t / k), slot = (uint32_t)(t - (uint64_t)q * k);
        const Rec rc = P.load(q);
        const uint32_t b = __ldg(&cand[(size_t)Pol::city(rc) * k + slot]);
        if (b == 0xffffffffu) continue; // padding: fewer than k other cities
        const uint32_t r = pos[b];
        // R[o] = record q-3+o (positions past n are padding and positions below 0 stand-ins: only read
        // for moves that are not legal); rlast = p_n-1, the a of a segment that starts at 0
        Rec R[7];
#pragma unroll
        for (int o = 0; o < 7; ++o) R[o] = o == 3 ? rc : P.load(q + o >= 3 ? q + o - 3 : q);
        const Rec rlast = q <= 2 ? P.load(n - 1) : R[0];
        const uint32_t jm = r == 0 ? n - 1 : r - 1; // j of roles B and D
        const Rec X0 = P.load(jm), X1 = P.load(r), X2 = P.load(r + 1); // p_jm, b, p_r+1 (r+1 = n: wrap copy)
        const V dcb = P.dist(rc, X1); // the candidate edge (c, b)
        // removal gain of the segment of length s whose first record is R[of]; a0: it starts at position 0
        auto neg_rg = [&](const Rec &a, const Rec &f, const Rec &dd) {
            return -Val<V>::sub(Val<V>::add(Pol::sp(f), Pol::sp(dd)), P.dist(a, dd));
        };
#pragma unroll
        for (uint32_t s = 1; s <= 3; ++s) {
            if (n <= s + 1) break;
            // segment [q, q+s-1]: roles A (fwd, j = r) and D (rev, j = jm)
            if (q + s <= n) {
                const Rec &f = R[3], &l = R[2 + s], &dd = R[3 + s];
                const V nrg = neg_rg(q == 0 ? rlast : R[2], f, dd);
                consider(window_ok(q, s, r),
                         Val<V>::sub(Val<V>::add(Val<V>::add(nrg, dcb), P.dist(l, X2)), Pol::sp(X2)), q, r, s, 0);
                if (s > 1)
                    consider(window_ok(q, s, jm),
                             Val<V>::sub(Val<V>::add(Val<V>::add(nrg, P.dist(X0, l)), dcb), Pol::sp(X1)), q, jm, s, 1);
            }
            // segment [q-s+1, q]: roles B (fwd, j = jm) and C (rev, j = r)
            if (q + 1 >= s) {
                const uint32_t i = q + 1 - s;
                const Rec &f = R[4 - s], &dd = R[4];
                const V nrg = neg_rg(i == 0 ? rlast : R[3 - s], f, dd);
                consider(window_ok(i, s, jm),
                         Val<V>::sub(Val<V>::add(Val<V>::add(nrg, P.dist(X0, f)), dcb), Pol::sp(X1)), i, jm, s, 0);
                if (s > 1)
                    consider(window_ok(i, s, r),
                             Val<V>::sub(Val<V>::add(Val<V>::add(nrg, dcb), P.dist(f, X2)), Pol::sp(X2)), i, r, s, 1);
            }
        }
    }

    __shared__ Best<V> red[WARPS];
    __shared__ uint32_t red_cnt[WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    warp_argmin_or(best);
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0) {
        red[warp] = best;
        red_cnt[warp] = cnt;
    }
    __syncthreads();
    if (warp == 0) {
        Best<V> v = lane < WARPS ? red[lane] : Best<V>{(V)0, kNone, kNone, 0u};
        warp_argmin_or(v);
        if (lane == 0) {
            unsigned long long c = 0;
#pragma unroll
            for (int w = 0; w < WARPS; ++w) c += red_cnt[w];
            blockbest[blockIdx.x] = v;
            blockcnt[blockIdx.x] = c;
        }
    }
    if (!fuse_apply) return;
    __shared__ unsigned int s_last;
    __syncthreads();
    if (threadIdx.x == 0) s_last = (ticket_take_acq_rel(ticket) == gridDim.x - 1) ? 1u : 0u; // thread 0 wrote blockbest
    __syncthreads();
    if (!s_last) return;
    or_nl_tail(P, n, pos, tmp, blockbest, blockcnt, state, ticket, log, log_cap);
}

// the apply grids of a step whose span the scan left pending: gather, then scatter and finish the step
template <class Pol>
__global__ void __launch_bounds__(256)
    or_nl_gather_kernel(Pol P, Pt *__restrict__ tmp, const Best<typename Pol::V> *__restrict__ pending,
                        const DevState *__restrict__ state)
{
    griddep_wait(); // the step's scan has finished and its writes are visible
    if (state->done) return;
    const OrMove m = or_move_of(*pending);
    if (!m.found) return; // the scan's last CTA finished the step
    or_gather(P, tmp, m, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
}

template <class Pol>
__global__ void __launch_bounds__(256)
    or_nl_scatter_kernel(Pol P, const Pt *__restrict__ tmp, uint32_t n, const Best<typename Pol::V> *__restrict__ pending,
                         uint32_t *__restrict__ pos, DevState *state, unsigned int *ticket, tl_move *__restrict__ log,
                         uint64_t log_cap)
{
    griddep_wait(); // the gather grid has finished
    if (state->done) return;
    const OrMove m = or_move_of(*pending);
    if (!m.found) return; // uniform over the grid
    or_scatter(P, tmp, n, m, pos, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned int tk = atomicAdd(ticket, 1u);
        if (tk == gridDim.x - 1) { // last block: everyone has read `state` by now
            *ticket = 0u;
            finish_or_step(state, load_state_header(state), m, log, log_cap);
            __threadfence();
        }
    }
}

cudaLaunchConfig_t pdl_config(int grid, int threads, cudaLaunchAttribute *attr, cudaStream_t st)
{
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)threads);
    cfg.stream = st;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cfg;
}

} // namespace

void launch_or_nl_scan(Metric metric, Pt *pts, uint32_t *pos, const uint32_t *cand, uint32_t k, uint32_t n, void *tmp,
                       void *blockbest, unsigned long long *blockcnt, DevState *state, unsigned int *ticket, tl_move *log,
                       uint64_t log_cap, bool fuse_apply, int grid, cudaStream_t st)
{
    cudaLaunchAttribute attr[1];
    const cudaLaunchConfig_t cfg = pdl_config(grid, THREADS, attr, st);
    const int fuse = fuse_apply ? 1 : 0;
    with_metric(metric, [&](auto M) {
        using Pol = NlPol<M>;
        cudaLaunchKernelEx(&cfg, or_nl_scan_kernel<Pol>, Pol{pts}, pos, cand, k, n, reinterpret_cast<Pt *>(tmp),
                           reinterpret_cast<Best<typename Pol::V> *>(blockbest), blockcnt, state, ticket, log,
                           (uint64_t)log_cap, fuse);
    });
}

void launch_or_nl_apply(Metric metric, Pt *pts, uint32_t *pos, void *tmp, uint32_t n, const void *pending,
                        DevState *state, unsigned int *ticket, tl_move *log, uint64_t log_cap, int grid, cudaStream_t st)
{
    cudaLaunchAttribute attr[1];
    const cudaLaunchConfig_t cfg = pdl_config(grid, 256, attr, st);
    with_metric(metric, [&](auto M) {
        using Pol = NlPol<M>;
        const auto *pend = reinterpret_cast<const Best<typename Pol::V> *>(pending);
        cudaLaunchKernelEx(&cfg, or_nl_gather_kernel<Pol>, Pol{pts}, reinterpret_cast<Pt *>(tmp), pend,
                           (const DevState *)state);
        cudaLaunchKernelEx(&cfg, or_nl_scatter_kernel<Pol>, Pol{pts}, (const Pt *)tmp, n, pend, pos, state, ticket, log,
                           (uint64_t)log_cap);
    });
}

} // namespace tl
