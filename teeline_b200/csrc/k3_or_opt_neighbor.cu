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
//
// Or-opt NM (multi-move, TL_ALGO_OR_OPT_NEIGHBOR_MULTI; definition in include/teeline_cuda.h): the same scan and
// G.  A move's hull is [a0, a1] = [min(i-1, j), max(i+s, j+1)]: every position its delta reads, and its relocated
// span is [a0+1, a1-1] with a1's entering edge rewritten.  In step t (= DevState::scans) position q lies in block
// (q + o) >> bshift with o = (t & 1) << (bshift - 1); every move below the threshold that does not wrap (i = 0,
// i+s = n or j = n-1 touch the closing edge) and whose a0 and a1 share a block does a 64-bit atomicMin into that
// block's key: the order-preserving delta bits above (s-1, i - base, j - base, rev), which orders a block's moves
// as better_or does (bshift <= 14 keeps the fields in 31 bits).  The last CTA reduces G, re-arms the keys while it
// compacts the block bests whose hull lies on either side of G's (none when G wraps) into a list in block order,
// cuts the list at the move budget, writes the log and ends the step.  It relocates a short G itself; the apply
// grids relocate a long G cooperatively and each listed block move with one CTA.  Every move is staged in tmp at
// its own positions, so the disjoint spans share the buffer.  A block move and G share at most a hull end, whose
// city neither moves and whose entering edge only one of them rewrites (the other reads that record's
// coordinates only).
#include "apply.cuh"
#include "block_keys.cuh"
#include "kernels.cuh"
#include "or_opt_rank.cuh"

namespace tl {

namespace {

constexpr int THREADS = kNlThreads;
constexpr int WARPS = THREADS / 32;
constexpr uint32_t kNone = 0xffffffffu;

// a legal move below the threshold: offer it to its block when it does not wrap and its hull lies in one block
template <typename V>
__device__ __forceinline__ void block_offer(const NlMulti &M, uint32_t off, uint32_t n, V d, uint32_t i, uint32_t j,
                                            uint32_t s, uint32_t rev)
{
    if (i == 0 || i + s == n || j == n - 1) return;
    const uint32_t a0 = min(i - 1, j), a1 = max(i + s, j + 1);
    const uint32_t b = (a0 + off) >> M.bshift;
    if (b != (a1 + off) >> M.bshift) return;
    const uint32_t base = (b << M.bshift) - off; // wraps for block 0 at odd steps; the differences below do not
    const uint32_t low =
        ((s - 1) << (2 * M.bshift + 1)) | ((i - base) << (M.bshift + 1)) | ((j - base) << 1) | rev;
    atomicMin(M.keys + b, ((unsigned long long)order_bits(d) << 32) | low);
}

// Tail of a fused Or-opt NM step, run by the last CTA: G as relocate_step_tail reduces it, then the accepted
// block bests (see the file comment).
template <class Pol>
__device__ __noinline__ void or_nlm_tail(const Pol &P, uint32_t n, uint32_t *pos, Pt *tmp,
                                         Best<typename Pol::V> *blockbest, const unsigned long long *blockcnt,
                                         DevState *state, unsigned int *ticket, tl_move *__restrict__ log,
                                         uint64_t log_cap, const NlMulti &M, uint32_t off)
{
    using V = typename Pol::V;
    __shared__ unsigned long long s_moves;
    __shared__ long long s_max;
    __shared__ uint32_t s_wcnt[WARPS];
    StateHeader hdr{};
    if (threadIdx.x == 0) {
        hdr = load_state_header(state);
        s_moves = hdr.h0.x;
        s_max = hdr.h1.x;
    }
    unsigned long long cnt;
    const Best<V> v = reduce_step_records<WARPS, OrMove>(blockbest, blockcnt, cnt); // publishes s_moves, s_max
    const OrMove g = OrMove::of(v);
    const unsigned long long m = s_moves;
    // block moves this step may still apply after G (G always fits: the step runs only below the budget)
    const unsigned long long allow = s_max < 0 ? ~0ull : (unsigned long long)s_max - m - 1;
    const bool wraps = g.i == 0 || g.i + g.s == n || g.j == n - 1; // G alone
    const uint32_t g0 = min(g.i - 1, g.j), g1 = max(g.i + g.s, g.j + 1);
    // without G no move is below the threshold, so no key was set
    uint32_t taken = 0;
    if (g.found) {
        Best<V> *list = static_cast<Best<V> *>(M.list);
        const uint32_t mask = (1u << M.bshift) - 1u;
        taken = compact_block_keys<WARPS, Best<V>>(
            M, allow, s_wcnt,
            [&](uint32_t b, unsigned long long key, Best<V> &mv) {
                const uint32_t low = (uint32_t)key, base = (b << M.bshift) - off;
                mv.delta = from_order_bits<V>((uint32_t)(key >> 32));
                mv.i = base + ((low >> (M.bshift + 1)) & mask);
                mv.j = base + ((low >> 1) & mask);
                mv.aux = ((low >> (2 * M.bshift + 1)) << 1) | (low & 1u); // (s-1)*2 + rev
                const uint32_t a0 = min(mv.i - 1, mv.j), a1 = max(mv.i + (mv.aux >> 1) + 1, mv.j + 1);
                return !wraps && (a1 <= g0 || a0 >= g1);
            },
            [&](uint32_t rank, const Best<V> &mv) {
                list[rank] = mv;
                const unsigned long long e = m + 1 + rank;
                if (log && e < log_cap) log[e] = OrMove::of(mv).entry();
            });
    }
    const uint32_t napply = (uint32_t)min((unsigned long long)taken, allow);
    const bool long_span = g.found && g.hi - g.lo + 1 > (uint32_t)kOrNlCtaSpan;
    if (threadIdx.x == 0) {
        state->computed += cnt;
        M.desc[0] = napply;
        M.desc[1] = long_span ? v.i : kNone;
        M.desc[2] = v.j;
        M.desc[3] = v.aux;
        *ticket = 0u;
        state->scans = hdr.h0.y + 1;
        if (g.found) {
            if (log && m < log_cap) log[m] = g.entry();
            const unsigned long long moves = m + 1 + napply;
            state->moves = moves;
            if (s_max >= 0 && (long long)moves >= s_max) state->done = 1;
        } else {
            state->done = 1;
            state->converged = 1;
        }
    }
    if (g.found && !long_span) {
        relocate_gather(P, tmp + g.lo, g, threadIdx.x, blockDim.x);
        __syncthreads();
        relocate_scatter(P, tmp + g.lo, n, g, pos, threadIdx.x, blockDim.x);
    }
}

// MULTI: Or-opt NM's fused step (block keys and or_nlm_tail); otherwise Or-opt N's scan
template <bool MULTI, class Pol>
__global__ void __launch_bounds__(THREADS, kNlMinBlocks)
    or_nl_scan_kernel(Pol P, uint32_t *__restrict__ pos, const uint32_t *__restrict__ cand, uint32_t k, uint32_t n,
                      Pt *tmp, Best<typename Pol::V> *blockbest, unsigned long long *blockcnt, DevState *state,
                      unsigned int *ticket, tl_move *__restrict__ log, uint64_t log_cap, int fuse_apply, NlMulti M)
{
    using V = typename Pol::V;
    using Rec = typename Pol::Rec;
    griddep_launch_dependents();
    griddep_wait(); // the previous step's move is applied and visible from here on
    // uniform across the grid: only a step's tail or apply grid writes it, after every CTA has finished
    if (*reinterpret_cast<const volatile int *>(&state->done)) return;
    // Or-opt NM: this step's block offset (scans is only written by a step's tail, after every CTA has read it)
    uint32_t off = 0;
    if (MULTI) off = ((uint32_t)*reinterpret_cast<const volatile unsigned long long *>(&state->scans) & 1u) << (M.bshift - 1);

    Best<V> best{(V)0, kNone, kNone, 0u};
    uint32_t cnt = 0;
    const V thr = Val<V>::or_threshold();
    // a candidate move (i, j, s, rev) with its delta: counted if legal, kept if below the threshold and
    // better in (delta, rank)
    auto consider = [&](bool legal, V d, uint32_t i, uint32_t j, uint32_t s, uint32_t rev) {
        if (!legal) return;
        ++cnt;
        const Best<V> o{d, i, j, (s - 1) * 2 + rev};
        if (MULTI && d < thr) block_offer(M, off, n, d, i, j, s, rev);
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
    if (MULTI)
        or_nlm_tail(P, n, pos, tmp, blockbest, blockcnt, state, ticket, log, log_cap, M, off);
    else
        relocate_step_tail<WARPS, OrMove>(P, n, pos, tmp, blockbest, blockcnt, state, ticket, log, log_cap);
}

// Or-opt NM's apply grids, launched after every step's scan.  desc (written by or_nlm_tail) names a pending long G
// and the count of listed block moves.  The gather grid stages G cooperatively and relocates each block move with
// one CTA (gather, barrier, scatter); G's positions are disjoint from every block move's, so the two run together.
// The scatter grid then writes G back, and its last CTA resets desc, so a later no-op step applies nothing.
template <class Pol>
__device__ __forceinline__ OrMove pending_g(const uint32_t *desc, uint32_t gi)
{
    return OrMove::of(Best<typename Pol::V>{(typename Pol::V)0, gi, __ldcg(desc + 2), __ldcg(desc + 3)});
}

template <class Pol>
__global__ void __launch_bounds__(256)
    or_nlm_gather_kernel(Pol P, Pt *tmp, uint32_t n, const Best<typename Pol::V> *__restrict__ list,
                         const uint32_t *desc, uint32_t *pos)
{
    griddep_wait(); // PDL: the step's scan has finished and its writes are visible
    const uint32_t cnt = __ldcg(desc), gi = __ldcg(desc + 1);
    if (cnt == 0 && gi == kNone) return; // uniform over the grid
    if (gi != kNone) {
        const OrMove g = pending_g<Pol>(desc, gi);
        relocate_gather(P, tmp + g.lo, g, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
    }
    for (uint32_t c = blockIdx.x; c < cnt; c += gridDim.x) {
        const OrMove m = OrMove::of(list[c]);
        relocate_gather(P, tmp + m.lo, m, threadIdx.x, blockDim.x);
        __syncthreads();
        relocate_scatter(P, tmp + m.lo, n, m, pos, threadIdx.x, blockDim.x);
    }
}

template <class Pol>
__global__ void __launch_bounds__(256)
    or_nlm_scatter_kernel(Pol P, const Pt *tmp, uint32_t n, uint32_t *desc, unsigned int *ticket, uint32_t *pos)
{
    griddep_wait(); // PDL: the gather grid has finished
    const uint32_t cnt = __ldcg(desc), gi = __ldcg(desc + 1);
    if (cnt == 0 && gi == kNone) return; // uniform over the grid
    if (gi != kNone) {
        const OrMove g = pending_g<Pol>(desc, gi);
        relocate_scatter(P, tmp + g.lo, n, g, pos, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
    }
    __syncthreads();
    if (threadIdx.x == 0 && atomicAdd(ticket, 1u) == gridDim.x - 1) { // every CTA has read desc
        *ticket = 0u;
        desc[0] = 0u;
        desc[1] = kNone;
    }
}

} // namespace

void launch_or_nl_scan(Metric metric, Pt *pts, uint32_t *pos, const uint32_t *cand, uint32_t k, uint32_t n, void *tmp,
                       void *blockbest, unsigned long long *blockcnt, DevState *state, unsigned int *ticket, tl_move *log,
                       uint64_t log_cap, bool fuse_apply, int grid, cudaStream_t st, const NlMulti *multi)
{
    cudaLaunchAttribute attr[1];
    const cudaLaunchConfig_t cfg = pdl_config(grid, THREADS, 0, attr, st);
    const int fuse = fuse_apply ? 1 : 0;
    const NlMulti mm = multi ? *multi : NlMulti{};
    with_metric(metric, [&](auto M) {
        using Pol = NlPol<M>;
        auto *bb = reinterpret_cast<Best<typename Pol::V> *>(blockbest);
        auto *t = reinterpret_cast<Pt *>(tmp);
        if (multi && fuse_apply) // a scan without its step (tl_session_scan) leaves the block keys alone
            cudaLaunchKernelEx(&cfg, or_nl_scan_kernel<true, Pol>, Pol{pts}, pos, cand, k, n, t, bb, blockcnt, state,
                               ticket, log, (uint64_t)log_cap, fuse, mm);
        else
            cudaLaunchKernelEx(&cfg, or_nl_scan_kernel<false, Pol>, Pol{pts}, pos, cand, k, n, t, bb, blockcnt, state,
                               ticket, log, (uint64_t)log_cap, fuse, mm);
    });
}

void launch_or_nlm_apply(Metric metric, Pt *pts, uint32_t *pos, void *tmp, uint32_t n, const NlMulti &multi,
                         unsigned int *ticket, int grid, cudaStream_t st)
{
    cudaLaunchAttribute attr[1];
    const cudaLaunchConfig_t cfg = pdl_config(grid, 256, 0, attr, st);
    with_metric(metric, [&](auto M) {
        using Pol = NlPol<M>;
        auto *t = reinterpret_cast<Pt *>(tmp);
        cudaLaunchKernelEx(&cfg, or_nlm_gather_kernel<Pol>, Pol{pts}, t, n,
                           static_cast<const Best<typename Pol::V> *>(multi.list), (const uint32_t *)multi.desc, pos);
        cudaLaunchKernelEx(&cfg, or_nlm_scatter_kernel<Pol>, Pol{pts}, (const Pt *)t, n, multi.desc, ticket, pos);
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
