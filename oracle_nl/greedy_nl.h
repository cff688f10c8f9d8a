/*
 * greedy_nl.h -- CPU ORACLES for the greedy-edge constructor (tl_greedy_tour; test infrastructure, NOT
 * product code).  Two independent restatements of the definition in include/teeline_cuda.h on the pinned
 * oracle's metric (tlo_dist_f32, or tlo_dist_nint compared as f32 when nint != 0):
 *
 *   edge (a, b), a < b, has the key (d(a, b), a, b); taking the edges in key order, an edge is accepted when
 *   both endpoints have degree < 2 and lie in different fragments; after n-1 edges the path's two endpoints
 *   are joined.  out[0] = 0, out[1] = the lower of city 0's two neighbours, then the cycle (n <= 3: identity).
 *
 * tlo_greedy_brute: every edge sorted by key, then union-find.  O(n^2) memory: a few thousand cities.
 * tlo_greedy_lazy:  Bentley's lazy greedy.  A heap holds, for every free city, the key of its nearest
 *   eligible city at the time it was found; eligibility only shrinks, so a popped entry that is still
 *   eligible is the global minimum, and a stale one is searched again.  The nearest eligible city comes from
 *   a uniform grid, searched ring by ring until no unsearched city can have a smaller computed distance:
 *   f32 distances are within a relative 2^-22 of the real one when every nonzero square is a normal f32,
 *   nint(d) >= d - 1/2.  Cities of degree 2 are removed from their cells.  Fast enough for 10^6 cities.
 */
#ifndef GREEDY_NL_H
#define GREEDY_NL_H

#include "../oracle/teeline_oracle.h"

#ifdef __cplusplus
extern "C" {
#endif

void tlo_greedy_brute(int32_t n, const float *x, const float *y, int nint, int32_t *out);
void tlo_greedy_lazy(int32_t n, const float *x, const float *y, int nint, int32_t *out);

#ifdef __cplusplus
}
#endif
#endif
