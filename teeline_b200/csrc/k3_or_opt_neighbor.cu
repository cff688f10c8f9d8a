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
#include "apply.cuh"
#include "kernels.cuh"
#include "or_opt_rank.cuh"

namespace tl {

namespace {

constexpr int THREADS = kNlThreads;
constexpr int WARPS = THREADS / 32;
constexpr uint32_t kNone = 0xffffffffu;

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
    relocate_step_tail<WARPS, OrMove>(P, n, pos, tmp, blockbest, blockcnt, state, ticket, log, log_cap);
}

} // namespace

void launch_or_nl_scan(Metric metric, Pt *pts, uint32_t *pos, const uint32_t *cand, uint32_t k, uint32_t n, void *tmp,
                       void *blockbest, unsigned long long *blockcnt, DevState *state, unsigned int *ticket, tl_move *log,
                       uint64_t log_cap, bool fuse_apply, int grid, cudaStream_t st)
{
    cudaLaunchAttribute attr[1];
    const cudaLaunchConfig_t cfg = pdl_config(grid, THREADS, 0, attr, st);
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
    const cudaLaunchConfig_t cfg = pdl_config(grid, 256, 0, attr, st);
    with_metric(metric, [&](auto M) {
        using Pol = NlPol<M>;
        const auto *pend = reinterpret_cast<const Best<typename Pol::V> *>(pending);
        cudaLaunchKernelEx(&cfg, relocate_gather_kernel<Pol, OrMove>, Pol{pts}, reinterpret_cast<Pt *>(tmp), pend, 1,
                           (const DevState *)state);
        cudaLaunchKernelEx(&cfg, relocate_scatter_kernel<Pol, OrMove>, Pol{pts}, (const Pt *)tmp, n, pend, 1, state,
                           ticket, log, (uint64_t)log_cap, pos, 1);
    });
}

} // namespace tl
