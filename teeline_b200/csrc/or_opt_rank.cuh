// or_opt_rank.cuh -- Or-opt's candidate order and relocation map, shared by the full scan (K3,
// k3_or_opt.cu) and the candidate-list scan (k3_or_opt_neighbor.cu).
#pragma once

#include "common.cuh"
#include "../../include/teeline_cuda.h"

namespace tl {

// rank order of the reference scan: (seg_len, i, j, reversed) with aux = (seg_len-1)*2 + reversed
__device__ __forceinline__ bool rank_less(uint32_t i1, uint32_t j1, uint32_t a1, uint32_t i2, uint32_t j2,
                                          uint32_t a2)
{
    const uint32_t s1 = a1 >> 1, s2 = a2 >> 1;
    if (s1 != s2) return s1 < s2;
    if (i1 != i2) return i1 < i2;
    if (j1 != j2) return j1 < j2;
    return (a1 & 1u) < (a2 & 1u);
}

// (delta, rank) lexicographic; a record with i == 0xffffffff is "no candidate yet" and only loses
template <typename V>
__device__ __forceinline__ bool better_or(const Best<V> &a, const Best<V> &b)
{
    if (a.i == 0xffffffffu) return false;
    if (b.i == 0xffffffffu) return true;
    return a.delta < b.delta || (a.delta == b.delta && rank_less(a.i, a.j, a.aux, b.i, b.j, b.aux));
}

template <typename V>
__device__ __forceinline__ void warp_argmin_or(Best<V> &v)
{
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        Best<V> o;
        o.delta = __shfl_xor_sync(0xffffffffu, v.delta, off);
        o.i = __shfl_xor_sync(0xffffffffu, v.i, off);
        o.j = __shfl_xor_sync(0xffffffffu, v.j, off);
        o.aux = __shfl_xor_sync(0xffffffffu, v.aux, off);
        if (better_or(o, v)) v = o;
    }
}

// ---- relocation (apply_relocation, or_opt.rs:172-184) --------------------------------------------

// the move with its relocated span [lo, hi]: every position outside it keeps its record
// (the Move of the relocation apply step, apply.cuh)
struct OrMove {
    bool found;
    float delta;
    uint32_t i, j, s, rev, lo, hi;

    template <typename V>
    static __device__ __forceinline__ OrMove of(const Best<V> &v)
    {
        OrMove m;
        m.found = v.i != 0xffffffffu;
        m.delta = (float)v.delta;
        m.i = v.i;
        m.j = v.j;
        m.s = (v.aux >> 1) + 1;
        m.rev = v.aux & 1u;
        if (m.j >= m.i + m.s) { m.lo = m.i; m.hi = m.j; } else { m.lo = m.j + 1; m.hi = m.i + m.s - 1; }
        return m;
    }
    template <typename V>
    static __device__ __forceinline__ bool better(const Best<V> &a, const Best<V> &b) { return better_or(a, b); }
    __device__ __forceinline__ uint32_t source(uint32_t q) const;
    __device__ __forceinline__ tl_move entry() const { return tl_move{delta, i, j, (uint8_t)s, (uint8_t)rev, 0}; }
};

// new occupant of position q in [lo, hi] after the relocation, as an old position
__device__ __forceinline__ uint32_t or_source(const OrMove &m, uint32_t q)
{
    if (m.j >= m.i + m.s) { // segment moves towards the end: [i, j-s] shifts left, segment lands at j-s+1
        if (q <= m.j - m.s) return q + m.s;
        const uint32_t t = q - (m.j - m.s + 1);
        return m.i + (m.rev ? m.s - 1 - t : t);
    }
    // segment moves towards the start: lands at j+1, [j+1, i-1] shifts right by s
    if (q <= m.j + m.s) {
        const uint32_t t = q - (m.j + 1);
        return m.i + (m.rev ? m.s - 1 - t : t);
    }
    return q - m.s;
}

__device__ __forceinline__ uint32_t OrMove::source(uint32_t q) const { return or_source(*this, q); }

} // namespace tl
