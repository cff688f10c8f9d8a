// block_keys.cuh -- the per-block 64-bit keys of the multi-move candidate-list searches (Mode NM,
// k2_two_opt_neighbor.cu; Or-opt NM, k3_or_opt_neighbor.cu): order-preserving delta bits above a move's
// in-block fields, merged with atomicMin during the scan, and the last CTA's pass that compacts the
// accepted block bests into a list in block order.
#pragma once

#include "kernels.cuh"

namespace tl {

// 32 bits ordered as the delta (negative deltas only; no NaN)
__device__ __forceinline__ uint32_t order_bits(float d)
{
    const uint32_t u = __float_as_uint(d);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ uint32_t order_bits(int32_t d) { return (uint32_t)d ^ 0x80000000u; }
template <typename V>
__device__ __forceinline__ V from_order_bits(uint32_t k);
template <>
__device__ __forceinline__ float from_order_bits<float>(uint32_t k)
{
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}
template <>
__device__ __forceinline__ int32_t from_order_bits<int32_t>(uint32_t k) { return (int32_t)(k ^ 0x80000000u); }

// Run by one CTA of WARPS warps: reads and re-arms the M.nslots block keys in rounds of WARPS*32.  For a set key,
// decode(b, key, mv) fills the block's move and says whether the step accepts it; accepted moves get ranks
// 0, 1, ... in block order, and emit(rank, mv) is called for those below `allow`.  Returns the accepted count.
template <int WARPS, class Mv, class Decode, class Emit>
__device__ __forceinline__ uint32_t compact_block_keys(const NlMulti &M, unsigned long long allow, uint32_t *s_wcnt,
                                                       Decode decode, Emit emit)
{
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t taken = 0;
    for (uint32_t c0 = 0; c0 < M.nslots; c0 += WARPS * 32) {
        const uint32_t b = c0 + threadIdx.x;
        bool acc = false;
        Mv mv{};
        if (b < M.nslots) {
            const unsigned long long key = __ldcg(M.keys + b);
            if (key != ~0ull) {
                M.keys[b] = ~0ull; // re-armed for the next step
                acc = decode(b, key, mv);
            }
        }
        const uint32_t bal = __ballot_sync(0xffffffffu, acc);
        if (lane == 0) s_wcnt[warp] = __popc(bal);
        __syncthreads();
        uint32_t before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < WARPS; ++w) {
            before += w < warp ? s_wcnt[w] : 0u;
            total += s_wcnt[w];
        }
        const uint32_t rank = taken + before + __popc(bal & ((1u << lane) - 1u));
        if (acc && rank < allow) emit(rank, mv);
        taken += total;
        __syncthreads(); // s_wcnt is rewritten by the next round
    }
    return taken;
}

} // namespace tl
