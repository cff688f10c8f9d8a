// policy.cuh -- where a kernel gets distances from.
//
// Every local-search kernel is written once against a Policy:
//   EucPol<FAST> : distances recomputed from tour-ordered coordinates (16-byte Pt records)
//   MatPol<V>    : distances read from the slot-ordered n x ld matrix in HBM through the
//                  tour-ordered Cs records (slot, entering-edge length, city), V = float | int32
//   NlPol<M>     : the candidate-list searches' Pt records, distances recomputed in metric M
// EucPol and MatPol are bit-identical for EUC_2D f32 problems (SURVEY.md section 0); MatPol also serves
// EXPLICIT matrices and the TSPLIB nint metric.
#pragma once

#include "common.cuh"

namespace tl {

// CG: record loads bypass L1 (ld.global.cg).  Needed when the same records are rewritten by other
// SMs within one kernel (K2-pop: whichever worker finishes a scan applies the move), because L1 is
// not coherent across SMs.
template <bool FAST, bool CG = false>
struct EucPol {
    using V = float;
    using Rec = Pt;
    struct Col {
        float x, y;
    };
    Pt *pts;

    __device__ __forceinline__ Rec load(uint32_t q) const
    {
        if constexpr (CG) {
            const float4 v = __ldcg(reinterpret_cast<const float4 *>(pts + q));
            return Pt{v.x, v.y, __float_as_int(v.z), v.w};
        } else {
            return pts[q];
        }
    }
    __device__ __forceinline__ const Rec *base() const { return pts; }
    // the record as L2 holds it (ld.global.cg), whatever this SM's L1 still has
    __device__ __forceinline__ Rec load_l2(uint32_t q) const
    {
        const float4 v = __ldcg(reinterpret_cast<const float4 *>(pts + q));
        return Pt{v.x, v.y, __float_as_int(v.z), v.w};
    }
    static __device__ __forceinline__ Col col(const Rec &r) { return Col{r.x, r.y}; }
    static __device__ __forceinline__ V sp(const Rec &r) { return r.sp; }
    static __device__ __forceinline__ void set_sp(Rec &r, V v) { r.sp = v; }
    static __device__ __forceinline__ int32_t city(const Rec &r) { return r.city; }
    __device__ __forceinline__ V dist(const Rec &a, const Rec &b) const
    {
        return dist_f32<FAST>(a.x, a.y, b.x, b.y);
    }
    __device__ __forceinline__ V dist_rc(const Rec &a, const Col &c) const
    {
        return dist_f32<FAST>(a.x, a.y, c.x, c.y);
    }
    // everything that identifies the city at q, but not its entering-edge length
    __device__ __forceinline__ void store_id(uint32_t q, const Rec &from) const
    {
        pts[q].x = from.x;
        pts[q].y = from.y;
        pts[q].city = from.city;
    }
    __device__ __forceinline__ void store_sp(uint32_t q, V v) const { pts[q].sp = v; }
    __device__ __forceinline__ void store(uint32_t q, const Rec &r) const { pts[q] = r; }
};

template <typename VT>
struct MatPol {
    using V = VT;
    using Rec = Cs;
    struct Col {
        int32_t slot;
    };
    Cs *cs;
    const VT *M;
    uint32_t ld;

    __device__ __forceinline__ Rec load(uint32_t q) const { return cs[q]; }
    __device__ __forceinline__ const Rec *base() const { return cs; }
    __device__ __forceinline__ Rec load_l2(uint32_t q) const
    {
        const int4 v = __ldcg(reinterpret_cast<const int4 *>(cs + q));
        Cs r;
        r.slot = v.x;
        r.sp_bits = v.y;
        r.city = v.z;
        r.pad = v.w;
        return r;
    }
    static __device__ __forceinline__ Col col(const Rec &r) { return Col{r.slot}; }
    static __device__ __forceinline__ V sp(const Rec &r) { return Val<V>::from_bits(r.sp_bits); }
    static __device__ __forceinline__ void set_sp(Rec &r, V v) { r.sp_bits = Val<V>::bits(v); }
    static __device__ __forceinline__ int32_t city(const Rec &r) { return r.city; }
    __device__ __forceinline__ V dist(const Rec &a, const Rec &b) const
    {
        return __ldg(&M[(size_t)a.slot * ld + b.slot]);
    }
    __device__ __forceinline__ V dist_rc(const Rec &a, const Col &c) const
    {
        return __ldg(&M[(size_t)a.slot * ld + c.slot]);
    }
    __device__ __forceinline__ void store_id(uint32_t q, const Rec &from) const
    {
        cs[q].slot = from.slot;
        cs[q].city = from.city;
    }
    __device__ __forceinline__ void store_sp(uint32_t q, V v) const { cs[q].sp_bits = Val<V>::bits(v); }
    __device__ __forceinline__ void store(uint32_t q, const Rec &r) const { cs[q] = r; }
};

// A policy whose record loads go to L2 (ld.global.cg), whatever this SM's L1 holds.  Used by the cached
// Mode B kernel, whose steps are a few microseconds long and read the same 16-byte records from many CTAs.
template <class Pol>
struct L2Pol : Pol {
    __device__ __forceinline__ explicit L2Pol(const Pol &p) : Pol(p) {}
    __device__ __forceinline__ typename Pol::Rec load(uint32_t q) const { return Pol::load_l2(q); }
};

// NlPol<M> (candidate-list searches, k2_two_opt_neighbor.cu and k3_or_opt_neighbor.cu): Pt records with
// distances recomputed from the coordinates in metric M (the nint metrics bit-equal to
// K1's matrix entries, as in the persistent Mode R kernel); the entering-edge length is stored as the
// bits of the metric's value type.
template <Metric M>
struct NlPol {
    using V = MetricValue<M>;
    using Rec = Pt;
    Pt *pts;
    __device__ __forceinline__ Rec load(uint32_t q) const { return pts[q]; }
    static __device__ __forceinline__ V sp(const Rec &r) { return Val<V>::from_bits(__float_as_int(r.sp)); }
    static __device__ __forceinline__ int32_t city(const Rec &r) { return r.city; }
    __device__ __forceinline__ V dist(const Rec &a, const Rec &b) const { return tl::dist<M>(a.x, a.y, b.x, b.y); }
    __device__ __forceinline__ void store_id(uint32_t q, const Rec &from) const
    {
        pts[q].x = from.x;
        pts[q].y = from.y;
        pts[q].city = from.city;
    }
    __device__ __forceinline__ void store_sp(uint32_t q, V v) const { pts[q].sp = __int_as_float(Val<V>::bits(v)); }
    static __device__ __forceinline__ void set_sp(Rec &r, V v) { r.sp = __int_as_float(Val<V>::bits(v)); }
    __device__ __forceinline__ void store(uint32_t q, const Rec &r) const { pts[q] = r; }
};

} // namespace tl
