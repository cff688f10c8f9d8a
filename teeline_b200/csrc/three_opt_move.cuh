// three_opt_move.cuh -- 3-opt's candidate order and relocation map, shared by the full scan (K6,
// k6_three_opt.cu) and the candidate-list scan (k6_three_opt_neighbor.cu).
#pragma once

#include "common.cuh"
#include "../../include/teeline_cuda.h"

namespace tl {

// best-move record of the 3-opt scans: delta = savings, aux = k * 8 + case
template <typename V>
__device__ __forceinline__ bool better_three(V s1, uint32_t i1, uint32_t j1, uint32_t a1, V s2, uint32_t i2,
                                             uint32_t j2, uint32_t a2)
{
    // larger savings first; ties: lowest (i, j, k) -- the case is a function of the triple
    if (s1 != s2) return s1 > s2;
    if (i1 != i2) return i1 < i2;
    if (j1 != j2) return j1 < j2;
    return (a1 >> 3) < (a2 >> 3);
}
// record form; a record with i == 0xffffffff is "no candidate" and only loses
template <typename V>
__device__ __forceinline__ bool better_three(const Best<V> &a, const Best<V> &b)
{
    if (a.i == 0xffffffffu) return false;
    if (b.i == 0xffffffffu) return true;
    return better_three(a.delta, a.i, a.j, a.aux, b.delta, b.i, b.j, b.aux);
}

// ---- apply_3opt (three_opt.rs:182-218) -------------------------------------------------------------

// the move of a record, with the span [lo, hi] = [i+1, k] it rebuilds (lo >= 1, hi <= n-1): the Move of
// the relocation apply step (apply.cuh)
struct ThreeMove {
    bool found;
    float savings;
    uint32_t i, j, k, kase, lo, hi;

    template <typename V>
    static __device__ __forceinline__ ThreeMove of(const Best<V> &v)
    {
        ThreeMove m;
        m.found = v.i != 0xffffffffu;
        m.savings = (float)v.delta;
        m.i = v.i;
        m.j = v.j;
        m.k = v.aux >> 3;
        m.kase = v.aux & 7u;
        m.lo = m.i + 1;
        m.hi = m.k;
        return m;
    }
    template <typename V>
    static __device__ __forceinline__ bool better(const Best<V> &a, const Best<V> &b) { return better_three(a, b); }
    __device__ __forceinline__ uint32_t source(uint32_t q) const;
    __device__ __forceinline__ tl_move entry() const { return tl_move{-savings, i, j, (uint8_t)kase, 0, 0, k}; }
};

// new occupant of position q in [i+1, k], as an old position: the middle is rebuilt from
// seg1 = p[i+1..=j] and seg2 = p[j+1..=k] (cases 4-7 put seg2 first; odd cases reverse seg1,
// cases 2,3,6,7 reverse seg2)
__device__ __forceinline__ uint32_t three_source(const ThreeMove &m, uint32_t q)
{
    const uint32_t l1 = m.j - m.i, l2 = m.k - m.j, t = q - (m.i + 1);
    const bool first2 = m.kase >= 4;
    const bool rev1 = (m.kase & 1u) != 0;
    const bool rev2 = m.kase == 2 || m.kase == 3 || m.kase == 6 || m.kase == 7;
    const bool in_first = t < (first2 ? l2 : l1);
    const bool use2 = first2 ? in_first : !in_first;
    const uint32_t u = in_first ? t : t - (first2 ? l2 : l1);
    if (use2) return m.j + 1 + (rev2 ? l2 - 1 - u : u);
    return m.i + 1 + (rev1 ? l1 - 1 - u : u);
}

__device__ __forceinline__ uint32_t ThreeMove::source(uint32_t q) const { return three_source(*this, q); }

} // namespace tl
