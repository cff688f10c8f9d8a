/* three_opt_nl.c -- see three_opt_nl.h.  Built with -ffp-contract=off like the oracle: every f32
 * operation is rounded on its own, as in the kernels. */
#include "three_opt_nl.h"

#include <pthread.h>
#include <stdlib.h>
#include <string.h>

typedef struct {
    const tlo_problem *p;
    const int32_t *tour, *pos, *cand;
    int32_t k, q0, q1;
    int found;
    double savings;
    int32_t i, j, kk, kase;
    int64_t evals;
} three_job;

/* larger savings first, then the lowest (i, j, k) */
static int better(double s1, int32_t i1, int32_t j1, int32_t k1, double s2, int32_t i2, int32_t j2, int32_t k2)
{
    if (s1 != s2) return s1 > s2;
    if (i1 != i2) return i1 < i2;
    if (j1 != j2) return j1 < j2;
    return k1 < k2;
}

/* three_opt_scan_rows' evaluation of the triple (i, j, k): returns 1 with the savings and the case when
 * some cost is below orig */
#define THREE_EVAL(T, D)                                                                                   \
    do {                                                                                                   \
        const T d_ab = D(a, b), d_c_dt = D(c, dt), d_ac = D(a, c), d_b_dt = D(b, dt), d_a_dt = D(a, dt);    \
        const T d_ef = D(e, f), d_ce = D(c, e), d_dt_f = D(dt, f), d_be = D(b, e);                          \
        const T d_cf = D(c, f), d_bf = D(b, f), d_ae = D(a, e);                                             \
        const T orig = (T)((T)(d_ab + d_c_dt) + d_ef);                                                      \
        const T costs[7] = {                                                                                \
            (T)((T)(d_ac + d_b_dt) + d_ef),                                                                 \
            (T)((T)(d_ab + d_ce) + d_dt_f),                                                                 \
            (T)((T)(d_ac + d_be) + d_dt_f),                                                                 \
            (T)((T)(d_a_dt + d_be) + d_cf),                                                                 \
            (T)((T)(d_a_dt + d_ce) + d_bf),                                                                 \
            (T)((T)(d_ae + d_b_dt) + d_cf),                                                                 \
            (T)((T)(d_ae + d_c_dt) + d_bf),                                                                 \
        };                                                                                                  \
        int ci = -1;                                                                                        \
        for (int t = 0; t < 7; ++t)                                                                         \
            if (costs[t] < orig && (ci < 0 || costs[t] < costs[ci])) ci = t;                                \
        if (ci < 0) return 0;                                                                               \
        *savings = (double)(T)(orig - costs[ci]);                                                           \
        *kase = ci + 1;                                                                                     \
        return 1;                                                                                           \
    } while (0)

static int eval_triple(const tlo_problem *p, const int32_t *t, int32_t i, int32_t j, int32_t k, double *savings,
                       int32_t *kase)
{
    const int32_t n = p->n;
    const int32_t a = t[i], b = t[i + 1], c = t[j], dt = t[j + 1], e = t[k], f = t[(k + 1) % n];
    if (p->kind == TLO_PACKED_I32) {
#define DI(u, v) ((int32_t)tlo_distance(p, (u), (v)))
        THREE_EVAL(int32_t, DI);
#undef DI
    }
#define DF(u, v) ((float)tlo_distance(p, (u), (v)))
    THREE_EVAL(float, DF);
#undef DF
}

static void consider(three_job *jb, int32_t e1, int32_t e2, int32_t e3)
{
    const int32_t n = jb->p->n;
    if (e1 == e2 || e1 == e3 || e2 == e3) return;
    int32_t i = e1, j = e2, k = e3, x;
    if (i > j) { x = i; i = j; j = x; }
    if (j > k) { x = j; j = k; k = x; }
    if (i > j) { x = i; i = j; j = x; }
    if (i == 0 && k == n - 1) return;
    jb->evals++;
    double s;
    int32_t kase;
    if (!eval_triple(jb->p, jb->tour, i, j, k, &s, &kase)) return;
    if (!jb->found || better(s, i, j, k, jb->savings, jb->i, jb->j, jb->kk)) {
        jb->found = 1;
        jb->savings = s;
        jb->i = i;
        jb->j = j;
        jb->kk = k;
        jb->kase = kase;
    }
}

static void *three_worker(void *arg)
{
    three_job *jb = (three_job *)arg;
    const int32_t n = jb->p->n, K = jb->k;
    for (int32_t q = jb->q0; q < jb->q1; ++q) {
        const int32_t *row = jb->cand + (size_t)jb->tour[q] * K;
        const int32_t qm = q == 0 ? n - 1 : q - 1;
        for (int32_t s1 = 0; s1 < K; ++s1) {
            if (row[s1] < 0) continue;
            const int32_t r = jb->pos[row[s1]], rm = r == 0 ? n - 1 : r - 1;
            for (int w = 0; w < 2; ++w) {
                const int32_t e2 = w ? r : rm;
                const int32_t t = w ? jb->tour[(r + 1) % n] : jb->tour[rm];
                const int32_t *row2 = jb->cand + (size_t)t * K;
                for (int32_t s2 = 0; s2 < K; ++s2) {
                    if (row2[s2] < 0) continue;
                    const int32_t r2 = jb->pos[row2[s2]], r2m = r2 == 0 ? n - 1 : r2 - 1;
                    consider(jb, qm, e2, r2m);
                    consider(jb, qm, e2, r2);
                    consider(jb, q, e2, r2m);
                    consider(jb, q, e2, r2);
                }
            }
        }
    }
    return NULL;
}

static int scan_with_pos(const tlo_problem *p, const int32_t *tour, const int32_t *pos, const int32_t *cand,
                         int32_t k, int nthreads, tlo_move *mv, int32_t *k_out, int64_t *evals)
{
    const int32_t n = p->n;
    if (nthreads < 1) nthreads = 1;
    if (nthreads > 256) nthreads = 256;
    if (n < 4 * nthreads) nthreads = 1;
    three_job jobs[256];
    pthread_t th[256];
    for (int t = 0; t < nthreads; ++t) {
        memset(&jobs[t], 0, sizeof jobs[t]);
        jobs[t].p = p; jobs[t].tour = tour; jobs[t].pos = pos; jobs[t].cand = cand; jobs[t].k = k;
        jobs[t].q0 = (int32_t)((int64_t)n * t / nthreads);
        jobs[t].q1 = (int32_t)((int64_t)n * (t + 1) / nthreads);
        if (nthreads > 1)
            pthread_create(&th[t], NULL, three_worker, &jobs[t]);
        else
            three_worker(&jobs[t]);
    }
    int found = 0;
    int64_t ev = 0;
    const three_job *b = NULL;
    for (int t = 0; t < nthreads; ++t) {
        if (nthreads > 1) pthread_join(th[t], NULL);
        ev += jobs[t].evals;
        if (jobs[t].found && (!found || better(jobs[t].savings, jobs[t].i, jobs[t].j, jobs[t].kk, b->savings, b->i,
                                               b->j, b->kk))) {
            b = &jobs[t];
            found = 1;
        }
    }
    if (found) {
        memset(mv, 0, sizeof *mv);
        mv->delta = -b->savings;
        mv->i = b->i;
        mv->j = b->j;
        mv->seg_len = b->kase;
        *k_out = b->kk;
    }
    if (evals) *evals = ev;
    return found;
}

int tlo_three_opt_nl_eval(const tlo_problem *p, const int32_t *tour, int32_t i, int32_t j, int32_t k,
                          double *savings, int32_t *kase)
{
    return eval_triple(p, tour, i, j, k, savings, kase);
}

int tlo_three_opt_nl_scan(const tlo_problem *p, const int32_t *tour, const int32_t *cand, int32_t k, int nthreads,
                          tlo_move *mv, int32_t *k_out, int64_t *evals)
{
    if (evals) *evals = 0;
    if (p->n < 4) return 0;
    int32_t *pos = (int32_t *)malloc((size_t)p->n * 4);
    for (int32_t q = 0; q < p->n; ++q) pos[tour[q]] = q;
    const int found = scan_with_pos(p, tour, pos, cand, k, nthreads, mv, k_out, evals);
    free(pos);
    return found;
}

void tlo_three_opt_nl(const tlo_problem *p, int32_t *tour, const int32_t *cand, int32_t k, int64_t max_moves,
                      int nthreads, tlo_stats *st, tlo_move *log, int32_t *ks, int64_t log_cap)
{
    st->passes = st->moves = st->evals = 0;
    if (p->n < 4) return; /* three_opt.rs:25-28 */
    int32_t *pos = (int32_t *)malloc((size_t)p->n * 4);
    for (int32_t q = 0; q < p->n; ++q) pos[tour[q]] = q;
    for (;;) {
        if (max_moves >= 0 && st->moves >= max_moves) break;
        tlo_move mv;
        int32_t kk = 0;
        int64_t ev = 0;
        const int found = scan_with_pos(p, tour, pos, cand, k, nthreads, &mv, &kk, &ev);
        st->passes++;
        st->evals += ev;
        if (!found) break;
        tlo_three_opt_apply(tour, mv.i, mv.j, kk, mv.seg_len);
        for (int32_t q = mv.i + 1; q <= kk; ++q) pos[tour[q]] = q; /* the rebuilt span [i+1, k] */
        if (log && st->moves < log_cap) {
            log[st->moves] = mv;
            if (ks) ks[st->moves] = kk;
        }
        st->moves++;
    }
    free(pos);
}
