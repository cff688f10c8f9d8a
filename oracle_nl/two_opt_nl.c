/* two_opt_nl.c -- see two_opt_nl.h.  Built with -ffp-contract=off like the oracle: every f32
 * operation is rounded on its own, as in the kernels. */
#include "two_opt_nl.h"

#include <pthread.h>
#include <stdlib.h>
#include <string.h>

/* Mode NM's per-block best: found = 0 for a block without an in-block improving pair */
typedef struct {
    int found;
    tlo_move mv;
} nl_block;

typedef struct {
    const tlo_problem *p;
    const int32_t *tour, *pos, *cand;
    int32_t k, i0, i1;
    int found;
    tlo_move mv;
    int64_t evals;
    /* Mode NM only (blk non-null): position q lies in block (q + off) / block */
    int32_t block, off;
    nl_block *blk;
} nl_job;

static int better(double d1, int32_t i1, int32_t j1, double d2, int32_t i2, int32_t j2)
{
    return d1 < d2 || (d1 == d2 && (i1 < i2 || (i1 == i2 && j1 < j2)));
}

/* Mode B's delta of pair (i, j) in the problem's value type (tlo_best_scan_rows in algos.inc) */
static double delta_of(const tlo_problem *p, const int32_t *t, int32_t i, int32_t j)
{
    const int32_t a = t[i], b = t[i + 1], c = t[j], d = t[j + 1];
    if (p->kind == TLO_PACKED_I32) {
        const int32_t dac = (int32_t)tlo_distance(p, a, c), dbd = (int32_t)tlo_distance(p, b, d);
        const int32_t dab = (int32_t)tlo_distance(p, a, b), dcd = (int32_t)tlo_distance(p, c, d);
        return (double)((dac + dbd) - (dab + dcd));
    }
    const float dac = (float)tlo_distance(p, a, c), dbd = (float)tlo_distance(p, b, d);
    const float dab = (float)tlo_distance(p, a, b), dcd = (float)tlo_distance(p, c, d);
    return (double)((float)(dac + dbd) - (float)(dab + dcd));
}

static void take(int *found, tlo_move *mv, double d, int32_t i, int32_t j)
{
    if (*found && !better(d, i, j, mv->delta, mv->i, mv->j)) return;
    *found = 1;
    memset(mv, 0, sizeof *mv);
    mv->delta = d;
    mv->i = i;
    mv->j = j;
}

static void consider(nl_job *jb, int32_t i, int32_t j)
{
    jb->evals++;
    const double d = delta_of(jb->p, jb->tour, i, j);
    if (d >= 0.0) return;
    take(&jb->found, &jb->mv, d, i, j);
    if (jb->blk) {
        const int32_t b = (i + jb->off) / jb->block;
        if (b == (j + 1 + jb->off) / jb->block) take(&jb->blk[b].found, &jb->blk[b].mv, d, i, j); /* in-block pair */
    }
}

static void *nl_worker(void *arg)
{
    nl_job *jb = (nl_job *)arg;
    const int32_t n = jb->p->n;
    for (int32_t i = jb->i0; i < jb->i1; ++i) {
        const int32_t *row = jb->cand + (size_t)jb->tour[i] * jb->k;
        for (int32_t s = 0; s < jb->k; ++s) {
            if (row[s] < 0) continue;
            const int32_t j = jb->pos[row[s]];
            const int32_t lo = i < j ? i : j, hi = i < j ? j : i;
            if (hi < lo + 2) continue;
            if (hi <= n - 2) consider(jb, lo, hi);         /* candidate edge = first new edge  */
            if (lo >= 1) consider(jb, lo - 1, hi - 1);     /* candidate edge = second new edge */
        }
    }
    return NULL;
}

/* blk (nullable, nblk entries): Mode NM's per-block bests for blocks of `block` positions shifted by off */
static int scan_with_pos(const tlo_problem *p, const int32_t *tour, const int32_t *pos, const int32_t *cand,
                         int32_t k, int nthreads, tlo_move *mv, int64_t *evals, int32_t block, int32_t off,
                         nl_block *blk, int32_t nblk)
{
    const int32_t n = p->n;
    if (nthreads < 1) nthreads = 1;
    if (nthreads > 256) nthreads = 256;
    if (n < 4 * nthreads) nthreads = 1;
    nl_job jobs[256];
    pthread_t th[256];
    for (int t = 0; t < nthreads; ++t) {
        memset(&jobs[t], 0, sizeof jobs[t]);
        jobs[t].p = p; jobs[t].tour = tour; jobs[t].pos = pos; jobs[t].cand = cand; jobs[t].k = k;
        jobs[t].i0 = (int32_t)((int64_t)n * t / nthreads);
        jobs[t].i1 = (int32_t)((int64_t)n * (t + 1) / nthreads);
        jobs[t].block = block;
        jobs[t].off = off;
        jobs[t].blk = blk ? (nl_block *)calloc((size_t)nblk, sizeof(nl_block)) : NULL;
        if (nthreads > 1)
            pthread_create(&th[t], NULL, nl_worker, &jobs[t]);
        else
            nl_worker(&jobs[t]);
    }
    int found = 0;
    int64_t ev = 0;
    for (int t = 0; t < nthreads; ++t) {
        if (nthreads > 1) pthread_join(th[t], NULL);
        ev += jobs[t].evals;
        if (jobs[t].found && (!found || better(jobs[t].mv.delta, jobs[t].mv.i, jobs[t].mv.j, mv->delta, mv->i, mv->j))) {
            *mv = jobs[t].mv;
            found = 1;
        }
        if (blk) { /* (delta, i, j) is a total order: the merge does not depend on the thread split */
            for (int32_t b = 0; b < nblk; ++b)
                if (jobs[t].blk[b].found) take(&blk[b].found, &blk[b].mv, jobs[t].blk[b].mv.delta, jobs[t].blk[b].mv.i,
                                               jobs[t].blk[b].mv.j);
            free(jobs[t].blk);
        }
    }
    if (evals) *evals = ev;
    return found;
}

int tlo_two_opt_nl_scan(const tlo_problem *p, const int32_t *tour, const int32_t *cand, int32_t k, int nthreads,
                        tlo_move *mv, int64_t *evals)
{
    int32_t *pos = (int32_t *)malloc((size_t)(p->n > 0 ? p->n : 1) * 4);
    for (int32_t q = 0; q < p->n; ++q) pos[tour[q]] = q;
    const int found = scan_with_pos(p, tour, pos, cand, k, nthreads, mv, evals, 0, 0, NULL, 0);
    free(pos);
    return found;
}

void tlo_two_opt_nl(const tlo_problem *p, int32_t *tour, const int32_t *cand, int32_t k, int64_t max_moves,
                    int nthreads, tlo_stats *st, tlo_move *log, int64_t log_cap)
{
    st->passes = st->moves = st->evals = 0;
    int32_t *pos = (int32_t *)malloc((size_t)(p->n > 0 ? p->n : 1) * 4);
    for (int32_t q = 0; q < p->n; ++q) pos[tour[q]] = q;
    for (;;) {
        if (max_moves >= 0 && st->moves >= max_moves) break;
        tlo_move mv;
        int64_t ev = 0;
        const int found = scan_with_pos(p, tour, pos, cand, k, nthreads, &mv, &ev, 0, 0, NULL, 0);
        st->passes++;
        st->evals += ev;
        if (!found) break;
        tlo_swap_2opt(tour, mv.i + 1, mv.j);
        for (int32_t q = mv.i + 1; q <= mv.j; ++q) pos[tour[q]] = q;
        if (log && st->moves < log_cap) log[st->moves] = mv;
        st->moves++;
    }
    free(pos);
}

static void apply_logged(int32_t *tour, int32_t *pos, const tlo_move *mv, tlo_stats *st, tlo_move *log, int64_t log_cap)
{
    tlo_swap_2opt(tour, mv->i + 1, mv->j);
    for (int32_t q = mv->i + 1; q <= mv->j; ++q) pos[tour[q]] = q;
    if (log && st->moves < log_cap) log[st->moves] = *mv;
    st->moves++;
}

int tlo_two_opt_nl_multi(const tlo_problem *p, int32_t *tour, const int32_t *cand, int32_t k, int32_t block,
                         int64_t step0, int64_t max_moves, int nthreads, tlo_stats *st, tlo_move *log, int64_t log_cap)
{
    st->passes = st->moves = st->evals = 0;
    const int32_t n = p->n;
    const int32_t nblk = (n + block - 1) / block + 1;
    int32_t *pos = (int32_t *)malloc((size_t)(n > 0 ? n : 1) * 4);
    nl_block *blk = (nl_block *)malloc((size_t)nblk * sizeof(nl_block));
    for (int32_t q = 0; q < n; ++q) pos[tour[q]] = q;
    int converged = 0;
    for (int64_t t = step0;; ++t) {
        if (max_moves >= 0 && st->moves >= max_moves) break;
        const int32_t off = (int32_t)(t & 1) * (block / 2);
        memset(blk, 0, (size_t)nblk * sizeof(nl_block));
        tlo_move g;
        int64_t ev = 0;
        const int found = scan_with_pos(p, tour, pos, cand, k, nthreads, &g, &ev, block, off, blk, nblk);
        st->passes++;
        st->evals += ev;
        if (!found) { converged = 1; break; }
        /* every block best disjoint from G, in increasing i (blocks are in position order); all of them
           are read before anything is applied, so the whole step works on the start-of-step tour */
        int32_t na = 0;
        for (int32_t b = 0; b < nblk; ++b) {
            if (!blk[b].found) continue;
            const tlo_move *m = &blk[b].mv;
            if (m->i == g.i && m->j == g.j) continue;
            if (m->j < g.i || m->i > g.j) blk[na++].mv = *m;
        }
        apply_logged(tour, pos, &g, st, log, log_cap);
        for (int32_t a = 0; a < na && !(max_moves >= 0 && st->moves >= max_moves); ++a)
            apply_logged(tour, pos, &blk[a].mv, st, log, log_cap);
    }
    free(blk);
    free(pos);
    return converged;
}
