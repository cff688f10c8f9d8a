/*
 * three_opt_nl.h -- CPU ORACLE for candidate-list best-improvement 3-opt ("3-opt N",
 * TL_ALGO_THREE_OPT_NEIGHBOR; test infrastructure, NOT product code).
 *
 * A plain-C restatement of the definition in include/teeline_cuda.h (tl_problem_set_candidates) on
 * top of the pinned oracle (oracle/teeline_oracle.h), whose problem type, metric and move application
 * (tlo_three_opt_apply) it uses.  3-opt N's triples, costs, case choice and tie order are 3-opt's
 * (tlo_three_opt, algos.inc three_opt_scan_rows), restricted to the triples the candidate lists generate.
 *
 * cand: n*k cities, row c = candidates of city c (e.g. tlo_knn or the GPU's tl_knn output); entries
 * < 0 (padding) are skipped.  Cut edge e joins p_e and p_(e+1)%n.  For every position q, c = p_q, every
 * slot s1 with b = cand[c*k+s1], r = pos[b]; each e2 in {(r-1) mod n, r} with t = p_(r+1)%n when e2 = r,
 * else p_(r-1)%n; every slot s2 with b' = cand[t*k+s2], r' = pos[b']; each e1 in {(q-1) mod n, q} and
 * e3 in {(r'-1) mod n, r'}: if e1, e2, e3 are distinct, sorted into i < j < k, the triple counts unless
 * i = 0 and k = n-1.  Per triple, with A = p_i, B = p_i+1, C = p_j, D = p_j+1, E = p_k, F = p_(k+1)%n,
 * in the problem's value type (f32, or int32 for TLO_PACKED_I32) and three_opt_scan_rows' order:
 *   orig  = (d_AB + d_CD) + d_EF
 *   cost1 = (d_AC + d_BD) + d_EF   cost2 = (d_AB + d_CE) + d_DF   cost3 = (d_AC + d_BE) + d_DF
 *   cost4 = (d_AD + d_BE) + d_CF   cost5 = (d_AD + d_CE) + d_BF   cost6 = (d_AE + d_BD) + d_CF
 *   cost7 = (d_AE + d_CD) + d_BF
 * the case is the first minimal cost among those below orig, savings = orig - cost (rounded to the value
 * type).  The move is the counted triple with the largest savings > 0, ties to the lowest (i, j, k).
 * *evals counts every counted triple, duplicates included.  mv: delta = -savings, i, j, seg_len = case;
 * the third index is returned through *k_out.
 */
#ifndef THREE_OPT_NL_H
#define THREE_OPT_NL_H

#include "../oracle/teeline_oracle.h"

#ifdef __cplusplus
extern "C" {
#endif

/* The evaluation of one triple i < j < k on tour: returns 1 with its savings and case when some cost is
 * below orig, else 0. */
int tlo_three_opt_nl_eval(const tlo_problem *p, const int32_t *tour, int32_t i, int32_t j, int32_t k,
                          double *savings, int32_t *kase);
/* One scan: returns 1 and fills mv, *k_out when an improving generated triple exists. */
int tlo_three_opt_nl_scan(const tlo_problem *p, const int32_t *tour, const int32_t *cand, int32_t k,
                          int nthreads, tlo_move *mv, int32_t *k_out, int64_t *evals);
/* Scan and apply until no generated triple improves or max_moves (< 0: unlimited); st->passes = scans.
 * log[].seg_len carries the case and ks[] (nullable) the third index, as tlo_three_opt.  n < 4: returns
 * at once with the tour unchanged, as tlo_three_opt. */
void tlo_three_opt_nl(const tlo_problem *p, int32_t *tour, const int32_t *cand, int32_t k, int64_t max_moves,
                      int nthreads, tlo_stats *st, tlo_move *log, int32_t *ks, int64_t log_cap);

#ifdef __cplusplus
}
#endif
#endif
