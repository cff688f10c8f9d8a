/* or_opt_nl.c -- see or_opt_nl.h.  Built with -ffp-contract=off like the oracle: every f32
 * operation is rounded on its own, as in the kernels. */
#include "or_opt_nl.h"

#include <pthread.h>
#include <stdlib.h>
#include <string.h>

/* Or-opt NM's per-block best: found = 0 for a block without an in-block move below the threshold */
typedef struct {
    int found;
    tlo_move mv;
} or_block;

typedef struct {
    const tlo_problem *p;
    const int32_t *tour, *pos, *cand;
    int32_t k, q0, q1;
    int found;
    tlo_move mv;
    int64_t evals;
    /* Or-opt NM only (blk non-null): position q lies in block (q + off) / block */
    int32_t block, off;
    or_block *blk;
} or_job;

/* (delta, seg_len, i, j, reversed) lexicographic */
static int better(const tlo_move *a, const tlo_move *b)
{
    if (a->delta != b->delta) return a->delta < b->delta;
    if (a->seg_len != b->seg_len) return a->seg_len < b->seg_len;
    if (a->i != b->i) return a->i < b->i;
    if (a->j != b->j) return a->j < b->j;
    return a->reversed < b->reversed;
}

/* Or-opt's delta of (i, s, j, rev) in the problem's value type, in or_opt_scan_range's order */
static double delta_of(const tlo_problem *p, const int32_t *t, int32_t i, int32_t s, int32_t j, int rev)
{
    const int32_t n = p->n;
    const int32_t a = t[i == 0 ? n - 1 : i - 1], f = t[i], l = t[i + s - 1], dd = t[(i + s) % n];
    const int32_t x = t[j], y = t[(j + 1) % n];
    if (p->kind == TLO_PACKED_I32) {
#define DI(u, v) ((int32_t)tlo_distance(p, (u), (v)))
        const int32_t rg = (DI(a, f) + DI(l, dd)) - DI(a, dd);
        const int32_t exy = DI(x, y);
        return rev ? (double)(((-rg + DI(x, l)) + DI(f, y)) - exy) : (double)(((-rg + DI(x, f)) + DI(l, y)) - exy);
#undef DI
    }
#define DF(u, v) ((float)tlo_distance(p, (u), (v)))
    const float rg = (float)((float)(DF(a, f) + DF(l, dd)) - DF(a, dd));
    const float exy = DF(x, y);
    const float d = rev ? (float)((float)((float)(-rg + DF(x, l)) + DF(f, y)) - exy)
                        : (float)((float)((float)(-rg + DF(x, f)) + DF(l, y)) - exy);
    return (double)d;
#undef DF
}

/* the hull [a0, a1] of a move that does not wrap: every position its delta reads or its relocation writes */
static void hull(const tlo_move *m, int32_t *a0, int32_t *a1)
{
    *a0 = m->i - 1 < m->j ? m->i - 1 : m->j;
    *a1 = m->i + m->seg_len > m->j + 1 ? m->i + m->seg_len : m->j + 1;
}

/* the move touches the closing edge (p_n-1, p_0) */
static int wraps(const tlo_move *m, int32_t n)
{
    return m->i == 0 || m->i + m->seg_len == n || m->j == n - 1;
}

static void consider(or_job *jb, int32_t i, int32_t s, int32_t j, int rev)
{
    const int32_t n = jb->p->n;
    if (n <= s + 1 || i < 0 || i + s > n) return;
    const int32_t prev = i == 0 ? n - 1 : i - 1;
    if (j == prev || (j >= i && j < i + s)) return;
    jb->evals++;
    tlo_move o;
    memset(&o, 0, sizeof o);
    o.delta = delta_of(jb->p, jb->tour, i, s, j, rev);
    o.i = i;
    o.j = j;
    o.seg_len = s;
    o.reversed = rev;
    const double thr = jb->p->kind == TLO_PACKED_I32 ? 0.0 : (double)(-1e-3f); /* or_opt.rs:86 */
    if (!(o.delta < thr)) return;
    if (!jb->found || better(&o, &jb->mv)) {
        jb->found = 1;
        jb->mv = o;
    }
    if (jb->blk && !wraps(&o, n)) {
        int32_t a0, a1;
        hull(&o, &a0, &a1);
        const int32_t b = (a0 + jb->off) / jb->block;
        or_block *B = &jb->blk[b];
        if (b == (a1 + jb->off) / jb->block && (!B->found || better(&o, &B->mv))) { /* in-block move */
            B->found = 1;
            B->mv = o;
        }
    }
}

static void *or_worker(void *arg)
{
    or_job *jb = (or_job *)arg;
    const int32_t n = jb->p->n;
    for (int32_t q = jb->q0; q < jb->q1; ++q) {
        const int32_t *row = jb->cand + (size_t)jb->tour[q] * jb->k;
        for (int32_t t = 0; t < jb->k; ++t) {
            if (row[t] < 0) continue;
            const int32_t r = jb->pos[row[t]], rm = r == 0 ? n - 1 : r - 1;
            for (int32_t s = 1; s <= 3; ++s) {
                consider(jb, q, s, r, 0);          /* (f, x) */
                consider(jb, q - s + 1, s, rm, 0); /* (l, y) */
                if (s > 1) {
                    consider(jb, q - s + 1, s, r, 1); /* (l, x) */
                    consider(jb, q, s, rm, 1);        /* (f, y) */
                }
            }
        }
    }
    return NULL;
}

/* blk (nullable, nblk entries): Or-opt NM's per-block bests for blocks of `block` positions shifted by off */
static int scan_with_pos(const tlo_problem *p, const int32_t *tour, const int32_t *pos, const int32_t *cand,
                         int32_t k, int nthreads, tlo_move *mv, int64_t *evals, int32_t block, int32_t off,
                         or_block *blk, int32_t nblk)
{
    const int32_t n = p->n;
    if (nthreads < 1) nthreads = 1;
    if (nthreads > 256) nthreads = 256;
    if (n < 4 * nthreads) nthreads = 1;
    or_job jobs[256];
    pthread_t th[256];
    for (int t = 0; t < nthreads; ++t) {
        memset(&jobs[t], 0, sizeof jobs[t]);
        jobs[t].p = p; jobs[t].tour = tour; jobs[t].pos = pos; jobs[t].cand = cand; jobs[t].k = k;
        jobs[t].q0 = (int32_t)((int64_t)n * t / nthreads);
        jobs[t].q1 = (int32_t)((int64_t)n * (t + 1) / nthreads);
        jobs[t].block = block;
        jobs[t].off = off;
        jobs[t].blk = blk ? (or_block *)calloc((size_t)nblk, sizeof(or_block)) : NULL;
        if (nthreads > 1)
            pthread_create(&th[t], NULL, or_worker, &jobs[t]);
        else
            or_worker(&jobs[t]);
    }
    int found = 0;
    int64_t ev = 0;
    for (int t = 0; t < nthreads; ++t) {
        if (nthreads > 1) pthread_join(th[t], NULL);
        ev += jobs[t].evals;
        if (jobs[t].found && (!found || better(&jobs[t].mv, mv))) {
            *mv = jobs[t].mv;
            found = 1;
        }
        if (blk) { /* (delta, s, i, j, reversed) is a total order: the merge does not depend on the thread split */
            for (int32_t b = 0; b < nblk; ++b) {
                const or_block *J = &jobs[t].blk[b];
                if (J->found && (!blk[b].found || better(&J->mv, &blk[b].mv))) blk[b] = *J;
            }
            free(jobs[t].blk);
        }
    }
    if (evals) *evals = ev;
    return found;
}

int tlo_or_opt_nl_scan(const tlo_problem *p, const int32_t *tour, const int32_t *cand, int32_t k, int nthreads,
                       tlo_move *mv, int64_t *evals)
{
    int32_t *pos = (int32_t *)malloc((size_t)(p->n > 0 ? p->n : 1) * 4);
    for (int32_t q = 0; q < p->n; ++q) pos[tour[q]] = q;
    const int found = scan_with_pos(p, tour, pos, cand, k, nthreads, mv, evals, 0, 0, NULL, 0);
    free(pos);
    return found;
}

void tlo_or_opt_nl(const tlo_problem *p, int32_t *tour, const int32_t *cand, int32_t k, int64_t max_moves,
                   int nthreads, tlo_stats *st, tlo_move *log, int64_t log_cap)
{
    st->passes = st->moves = st->evals = 0;
    if (p->n < 4) return; /* or_opt.rs:31-34 */
    int32_t *pos = (int32_t *)malloc((size_t)p->n * 4);
    for (int32_t q = 0; q < p->n; ++q) pos[tour[q]] = q;
    for (;;) {
        if (max_moves >= 0 && st->moves >= max_moves) break;
        tlo_move mv;
        int64_t ev = 0;
        const int found = scan_with_pos(p, tour, pos, cand, k, nthreads, &mv, &ev, 0, 0, NULL, 0);
        st->passes++;
        st->evals += ev;
        if (!found) break;
        tlo_or_opt_apply(tour, p->n, mv.i, mv.seg_len, mv.j, mv.reversed);
        /* the relocated span: [i, j] when the segment moves towards the end, else [j+1, i+s-1] */
        const int32_t lo = mv.j >= mv.i + mv.seg_len ? mv.i : mv.j + 1;
        const int32_t hi = mv.j >= mv.i + mv.seg_len ? mv.j : mv.i + mv.seg_len - 1;
        for (int32_t q = lo; q <= hi; ++q) pos[tour[q]] = q;
        if (log && st->moves < log_cap) log[st->moves] = mv;
        st->moves++;
    }
    free(pos);
}

static void apply_logged(int32_t *tour, int32_t *pos, int32_t n, const tlo_move *mv, tlo_stats *st, tlo_move *log,
                         int64_t log_cap)
{
    tlo_or_opt_apply(tour, n, mv->i, mv->seg_len, mv->j, mv->reversed);
    const int32_t lo = mv->j >= mv->i + mv->seg_len ? mv->i : mv->j + 1;
    const int32_t hi = mv->j >= mv->i + mv->seg_len ? mv->j : mv->i + mv->seg_len - 1;
    for (int32_t q = lo; q <= hi; ++q) pos[tour[q]] = q;
    if (log && st->moves < log_cap) log[st->moves] = *mv;
    st->moves++;
}

int tlo_or_opt_nl_multi(const tlo_problem *p, int32_t *tour, const int32_t *cand, int32_t k, int32_t block,
                        int64_t step0, int64_t max_moves, int nthreads, tlo_stats *st, tlo_move *log, int64_t log_cap)
{
    st->passes = st->moves = st->evals = 0;
    const int32_t n = p->n;
    if (n < 4) return 1; /* as tlo_or_opt_nl: no scan */
    const int32_t nblk = (n + block - 1) / block + 1;
    int32_t *pos = (int32_t *)malloc((size_t)n * 4);
    or_block *blk = (or_block *)malloc((size_t)nblk * sizeof(or_block));
    for (int32_t q = 0; q < n; ++q) pos[tour[q]] = q;
    int converged = 0;
    for (int64_t t = step0;; ++t) {
        if (max_moves >= 0 && st->moves >= max_moves) break;
        const int32_t off = (int32_t)(t & 1) * (block / 2);
        memset(blk, 0, (size_t)nblk * sizeof(or_block));
        tlo_move g;
        int64_t ev = 0;
        const int found = scan_with_pos(p, tour, pos, cand, k, nthreads, &g, &ev, block, off, blk, nblk);
        st->passes++;
        st->evals += ev;
        if (!found) { converged = 1; break; }
        /* G alone when it wraps; otherwise every block best whose hull lies on either side of G's, in block order.
           All of them are read before anything is applied, so the whole step works on the start-of-step tour. */
        int32_t na = 0;
        if (!wraps(&g, n)) {
            int32_t g0, g1;
            hull(&g, &g0, &g1);
            for (int32_t b = 0; b < nblk; ++b) {
                if (!blk[b].found) continue;
                int32_t a0, a1;
                hull(&blk[b].mv, &a0, &a1);
                if (a1 <= g0 || a0 >= g1) blk[na++].mv = blk[b].mv;
            }
        }
        apply_logged(tour, pos, n, &g, st, log, log_cap);
        for (int32_t a = 0; a < na && !(max_moves >= 0 && st->moves >= max_moves); ++a)
            apply_logged(tour, pos, n, &blk[a].mv, st, log, log_cap);
    }
    free(blk);
    free(pos);
    return converged;
}
