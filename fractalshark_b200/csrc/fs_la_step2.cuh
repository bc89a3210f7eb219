// fs_la_step2.cuh -- the LAv2 step of the float+exponent binary32 path (HDRx32, 32-bit iteration counts) on a record
// laid out for the step, with the comparisons done on values instead of (exponent, mantissa) pairs.
//
// What it computes: exactly GPU_LAReference::getLA + GPU_LAInfoDeep::Prepare / Evaluate + getZ (GPU_LAReference.h:271-303,
// GPU_LAInfoDeep.h:90-123, LAstep.h:157-185) on HDRFloatComplex<float> operands -- the same individually rounded binary32
// operations in the same order as fs_la_fast.cuh / fs_types.cuh, hence the same bits:
//     t     = 2*Ref + dz                      newdz = Reduce(dz * t)          unusable = cheb(newdz) >= LAThreshold
//     dz'   = newdz*ZCoeff + dc*CCoeff        z     = Ref' + dz'              rebase   = cheb(z) < cheb(dz')
// What differs from fs_la_fast.cuh (profiles/r2_lav2_view14_summary.md: after the AT cycle watch the LA walk is 64 % of
// the View 14 frame, ~150 instructions per step, the ALU pipe 71 % busy):
//   * the record (la2::Rec, 64 B = four LDG.128) carries 2*Ref's exponent, the NEXT record's Ref and the threshold next
//     to the operands they are used with; the reference-layout record needs a fifth load and two scalar ones;
//   * rebase test: z = Ref' + dz' has just been aligned, so the multiplier 2^(dz'.e - z.e) the addition applied to dz' is
//     also the factor between the two Chebyshev norms: cheb(z) < cheb(dz')  <=>  max|z.m| < max|dz'.m| * 2^(dz'.e - z.e)
//     (both sides exact or, where the product underflows, decided anyway): 4 instructions instead of two Reduce()s and a
//     lexicographic comparison;
//   * the three "exponent gap in [120, 127)" refusals are read off the multiplier fields (their sum is 128..134 exactly
//     there): 2 instructions each.
// A step that meets an exact zero, a non-finite value, a mantissa far outside [2^-60, 2^60) or such a gap is REFUSED and
// recomputed by the caller from the reference-layout record with the reference-shaped operations (la_step_as_written),
// as with fs_la_fast.cuh.  Records whose threshold mantissa is not in [1, 2) are poisoned at pack time (Ref = NaN) so
// that every step on them is refused at the first check.
#pragma once
#include "fs_types.cuh"

namespace fs {
namespace la2 {

struct alignas(16) Rec {
    float ref_re, ref_im; int32_t ref_e2; uint32_t th_lo;  // Ref with the exponent of 2*Ref; low word of th_key
    float zc_re, zc_im; int32_t zc_e; int32_t th_hi;       // ZCoeff; high word of th_key
    // th_key (signed 64 bits) = LAThreshold.e * 2^23 + the 23 fraction bits of LAThreshold.m (a mantissa in [1, 2))
    float cc_re, cc_im; int32_t cc_e; uint32_t step;      // CCoeff; StepLength
    float nx_re, nx_im; int32_t nx_e; uint32_t next;      // Ref of the following record; NextStageLAIndex
};
static_assert(sizeof(Rec) == 64, "la2::Rec");

struct Out {
    float dre, dim;  // dz' = newdz*ZCoeff + dc*CCoeff
    float zre, zim;  // z = Ref' + dz'
    int de, ze;      // (the mantissa pairs first: la_step_refused returns them through memory as aligned 8-byte pairs)
    bool unusable, rebase;
};

// clamp(127 + d, 0, 127): exponent field of 2^min(d, 0)
FS_HD int field(int d) {
#ifdef __CUDA_ARCH__
    return __viaddmin_s32_relu(d, 127, 127);
#else
    const int v = d < 0 ? d + 127 : 127;
    return v < 0 ? 0 : v;
#endif
}
FS_HD float pow2f(int f) { return u2f((uint32_t)f << 23); }
FS_HD float abs_(float x) {
#ifdef __CUDA_ARCH__
    return fabsf(x);
#else
    return __builtin_fabsf(x);
#endif
}
FS_HD float max_(float a, float b) { // operands are finite and non-negative wherever this is called
#ifdef __CUDA_ARCH__
    return fmaxf(a, b);
#else
    return a > b ? a : b;
#endif
}
// finite, non-zero and within [2^-60, 2^60)
FS_HD bool sane(float s) { return (f2u(s) - ((uint32_t)(127 - 60) << 23)) < ((uint32_t)120 << 23); }

// The record of one reference-shaped LA entry (`next_ref`: Ref of the following entry; has_next = false for the last one).
FS_HD Rec pack(HdrC<float> Ref, HdrC<float> ZCoeff, HdrC<float> CCoeff, Hdr<float> LAThreshold, uint32_t step_length,
               uint32_t next_stage, bool has_next, HdrC<float> next_ref) {
    Rec d;
    const long long th_key = (long long)LAThreshold.e * (1ll << 23) + (long long)(f2u(LAThreshold.m) & 0x007fffffu);
    d.ref_re = Ref.re; d.ref_im = Ref.im; d.ref_e2 = imax(Ref.e + 1, MIN_BIG); d.th_lo = (uint32_t)th_key;
    d.zc_re = ZCoeff.re; d.zc_im = ZCoeff.im; d.zc_e = ZCoeff.e; d.th_hi = (int32_t)(th_key >> 32);
    d.cc_re = CCoeff.re; d.cc_im = CCoeff.im; d.cc_e = CCoeff.e; d.step = step_length;
    d.nx_re = next_ref.re; d.nx_im = next_ref.im; d.nx_e = next_ref.e; d.next = next_stage;
    // refuse every step on a record without a follower or whose threshold is not a reduced positive number
    if (!has_next || !(LAThreshold.m >= 1.0f && LAThreshold.m < 2.0f)) d.ref_re = u2f(0x7fc00000u);
    return d;
}

// One step; false = refused (nothing may be used).
// The (re, im) halves of every complex operation run as one packed pair (f32x2: FMUL2 / FFMA2), each half the scalar
// operation it replaces, on the same operands in the same order.  A complex product
//     re = fma(ar, br, -(ai*bi))    im = fma(ai, br, ar*bi)
// is fma2(a, br, mul2(rot(a), bi)) with rot(a) = (-ai, ar): -(ai*bi) == (-ai)*bi bit for bit, the sign of a zero included,
// and rot() and the broadcasts of br, bi are operand modifiers, not instructions.
FS_HD bool step(const uint4 q0, const uint4 q1, const uint4 q2, const uint4 q3, float dr, float di, int de, float cr,
                float ci, int ce, Out &o) {
    const f32x2 dz = f2_make(dr, di);
    const int re2 = (int)q0.z;
    // Prepare: t = 2*Ref + dz
    const int d1 = re2 - de;
    const int fa1 = field(d1), fb1 = field(-d1);
    const float ma1 = pow2f(fa1), mb1 = pow2f(fb1);
    float tr, ti;
    f2_split(f2_fma(dz, f2_bcast(mb1), f2_mul(f2_make(u2f(q0.x), u2f(q0.y)), f2_bcast(ma1))), tr, ti);
    const int te = imax(re2, de);
    bool gap = (uint32_t)(fa1 + fb1 - 128) < 7u;
    // w = dz * t, reduced
    const f32x2 w = f2_fma(dz, f2_bcast(tr), f2_mul(f2_rot(dz), f2_bcast(ti)));
    float wr, wi;
    f2_split(w, wr, wi);
    if (!sane(abs_(wr) + abs_(wi))) return false;
    const uint32_t wb = f2u(max_(abs_(wr), abs_(wi)));
    const float sc = u2f(0x7f000000u - (wb & 0x7f800000u));
    const f32x2 n = f2_mul(w, f2_bcast(sc));
    // cheb(newdz) >= LAThreshold on (exponent, mantissa) pairs of reduced positive numbers = one signed 64-bit comparison
    // of exponent * 2^23 + mantissa field; the record carries the threshold in that form (th_key).  wb already holds the
    // larger part's own exponent field, so adding it to (de + te - 127) * 2^23 forms the key and the reduced exponent.
    const int se = de + te - 127;
    const int nwe = se + (int)(wb >> 23);
    const long long wkey = (long long)se * (1ll << 23) + (long long)wb;
    const long long tkey = (long long)(((unsigned long long)q1.w << 32) | (unsigned long long)q0.w);
    o.unusable = wkey >= tkey;
    if (o.unusable) return !gap;
    // Evaluate: dz' = newdz*ZCoeff + dc*CCoeff
    const float zr = u2f(q1.x), zi = u2f(q1.y);
    const float ccr = u2f(q2.x), cci = u2f(q2.y);
    // (newdz * ZCoeff is formed from the REDUCED newdz, as the reference does: moving 2^-k out of the product is not exact
    // when the smaller component of an un-reduced w sits in the denormal range -- found by tests/…guards[3])
    const f32x2 dc = f2_make(cr, ci);
    const f32x2 p = f2_fma(n, f2_bcast(zr), f2_mul(f2_rot(n), f2_bcast(zi)));
    const f32x2 q = f2_fma(dc, f2_bcast(ccr), f2_mul(f2_rot(dc), f2_bcast(cci)));
    const int pe = nwe + (int)q1.z, qe = ce + (int)q2.z;
    const int d2 = pe - qe;
    const int fa2 = field(d2), fb2 = field(-d2);
    const float ma2 = pow2f(fa2), mb2 = pow2f(fb2);
    const f32x2 d = f2_fma(q, f2_bcast(mb2), f2_mul(p, f2_bcast(ma2)));
    f2_split(d, o.dre, o.dim);
    o.de = imax(pe, qe);
    gap = gap || (uint32_t)(fa2 + fb2 - 128) < 7u;
    // getZ: z = Ref' + dz'
    const int ne = (int)q3.z;
    const int d3 = ne - o.de;
    const int fa3 = field(d3), fb3 = field(-d3);
    const float ma3 = pow2f(fa3), mb3 = pow2f(fb3);
    f2_split(f2_fma(d, f2_bcast(mb3), f2_mul(f2_make(u2f(q3.x), u2f(q3.y)), f2_bcast(ma3))), o.zre, o.zim);
    o.ze = imax(ne, o.de);
    gap = gap || (uint32_t)(fa3 + fb3 - 128) < 7u;
    if (gap || !sane(abs_(o.zre) + abs_(o.zim)) || !sane(abs_(o.dre) + abs_(o.dim))) return false;
    // cheb(z) < cheb(dz'): z.e - dz'.e = max(d3, 0), and mb3 = 2^-max(d3, 0) (0 once the gap is >= 127: then |z| >> |dz'|)
    o.rebase = max_(abs_(o.zre), abs_(o.zim)) < max_(abs_(o.dre), abs_(o.dim)) * mb3;
    return true;
}

} // namespace la2
} // namespace fs
