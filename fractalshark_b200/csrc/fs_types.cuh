// fs_types.cuh -- device numeric types of the per-pixel render path.
//
// Written from the behavioural contract of the reference types (SURVEY.md section 9):
//   float+exponent "HDR" scalar   <- HpSharkFloatLib/HDRFloat.h:84-1356
//   shared-exponent HDR complex   <- HpSharkFloatLib/HDRFloatComplex.h:7-696
//   plain complex                 <- HpSharkFloatLib/FloatComplex.h
//   2x32 double-float             <- HpSharkFloatLib/dblflt.cuh:68-317, CudaDblflt.h:25-282
// Differences in *how* (not *what*): every power-of-two multiplier is built with integer
// ALU ops instead of scalbnf (reference SASS: I2FP + MUFU.EX2), additions are branch-free
// selects around one FMA, and every fused multiply-add is written explicitly (the library is
// compiled with -fmad=false) so the rounding sequence is the one nvcc chose for the reference
// (SURVEY.md section 8a "Evidence from the reference's own sm_100a SASS").
#pragma once
#include <stdint.h>
#include <cuda_runtime.h>

#define FS_HD __host__ __device__ __forceinline__
#define FS_D __device__ __forceinline__

namespace fs {

// HDRFloat.h:50-58  MIN_BIG_EXPONENT = INT32_MIN >> 3
constexpr int32_t MIN_BIG = INT32_MIN >> 3;
// HDRFloat.h:122
constexpr int32_t EXP_DIFF_IGNORED = 120;

// ----------------------------------------------------------------------------------------------
// 2x32 double-float storage (dblflt.h:6-59: {head, tail}, pack(4))
// ----------------------------------------------------------------------------------------------
#pragma pack(push, 4)
struct df32 {
    float head;
    float tail;
};
#pragma pack(pop)

// ----------------------------------------------------------------------------------------------
// Wire/storage structs: byte-identical to the reference PODs that cross the boundary
// (sizes asserted against SURVEY.md section 2.2).
// ----------------------------------------------------------------------------------------------
template <class M> struct Hdr {
    M m;
    int32_t e;
};
#pragma pack(push, 4)
template <> struct Hdr<df32> {
    df32 m;
    int32_t e;
};
#pragma pack(pop)

template <class M> struct HdrC {
    M re, im;
    int32_t e;
};
#pragma pack(push, 4)
template <> struct HdrC<df32> {
    df32 re, im;
    int32_t e;
};
#pragma pack(pop)

template <class M> struct Cx {
    M re, im;
};

static_assert(sizeof(Hdr<float>) == 8 && sizeof(Hdr<double>) == 16 && sizeof(Hdr<df32>) == 12, "HDRFloat layout");
static_assert(sizeof(HdrC<float>) == 12 && sizeof(HdrC<double>) == 24 && sizeof(HdrC<df32>) == 20, "HDRFloatComplex layout");

// ----------------------------------------------------------------------------------------------
// bit helpers
// ----------------------------------------------------------------------------------------------
FS_HD uint32_t f2u(float f) {
#ifdef __CUDA_ARCH__
    return __float_as_uint(f);
#else
    union { float f; uint32_t u; } c; c.f = f; return c.u;
#endif
}
FS_HD float u2f(uint32_t u) {
#ifdef __CUDA_ARCH__
    return __uint_as_float(u);
#else
    union { float f; uint32_t u; } c; c.u = u; return c.f;
#endif
}
FS_HD uint64_t d2u(double f) {
#ifdef __CUDA_ARCH__
    return (uint64_t)__double_as_longlong(f);
#else
    union { double f; uint64_t u; } c; c.f = f; return c.u;
#endif
}
FS_HD double u2d(uint64_t u) {
#ifdef __CUDA_ARCH__
    return __longlong_as_double((long long)u);
#else
    union { double f; uint64_t u; } c; c.u = u; return c.f;
#endif
}
FS_HD int imax(int a, int b) { return a > b ? a : b; }
FS_HD int imin(int a, int b) { return a < b ? a : b; }
FS_HD int iabs(int a) { return a < 0 ? -a : a; }

// explicit single-rounding primitives (library is built with -fmad=false)
FS_HD float fma_(float a, float b, float c) {
#ifdef __CUDA_ARCH__
    return __fmaf_rn(a, b, c);
#else
    return __builtin_fmaf(a, b, c);
#endif
}
FS_HD double fma_(double a, double b, double c) {
#ifdef __CUDA_ARCH__
    return __fma_rn(a, b, c);
#else
    return __builtin_fma(a, b, c);
#endif
}

// bit-for-bit equality of numbers (cycle watches: a state that repeats exactly)
FS_HD bool bits_equal(float a, float b) { return f2u(a) == f2u(b); }
FS_HD bool bits_equal(double a, double b) { return d2u(a) == d2u(b); }
FS_HD bool bits_equal(df32 a, df32 b) { return bits_equal(a.head, b.head) && bits_equal(a.tail, b.tail); }
template <class M> FS_HD bool bits_equal(Hdr<M> a, Hdr<M> b) { return bits_equal(a.m, b.m) && a.e == b.e; }

// Cycle watch of the perturbation loops, checked at rebase events (orbit index back to 0).  A pixel inside the set
// iterates to the limit against a periodic reference orbit; at a rebase the delta (the orbit index being 0) is the whole
// state of what follows except for the comparisons with the iteration limit, and towards an attracting cycle it settles,
// in finite precision, into an exactly periodic sequence.  The watch compares the state at every rebase with one saved at
// an earlier rebase (after 1, 2, 4, 8 ... events: Brent).  On a bit-for-bit match P iterations apart the periods that
// follow repeat the one just executed -- in which nothing escaped and no step was cut short by the limit -- for as long
// as a whole period fits below the limit: a step attempted at offset o with length l passed `iter + l < n` and o + l <= P,
// so k = (n - iter - 1) / P further periods are identical.  The caller adds k * P to the iteration count and runs the
// remainder (at most P iterations) the ordinary way: the reference's count, bit for bit, without the periods between.
// Used by the BLA kernels (fs_bla.cuh; View 14: 3.1x).  Measured and not kept in the perturbation loop of the LAv2 kernels
// (fs_perturb_loop.cuh): what is left for that loop on views 5 / 14 / 19 is not periodic at its rebase events, and the watch
// cost 2 % there.
template <class Real, class IterT, int N> struct RebaseWatch {
    Real saved[N];
    IterT at;
    unsigned int events, next;
    bool have, armed;
    FS_HD RebaseWatch(bool on) : at(0), events(0), next(1), have(false), armed(on) {}
    // s = the N numbers of the state; returns the iterations to skip (0 = none)
    FS_HD IterT at_rebase(const Real (&s)[N], IterT iter, IterT n_iterations) {
        if (!armed) return 0;
        bool same = have;
        for (int k = 0; k < N; k++) same = same && bits_equal(s[k], saved[k]);
        if (same) {
            armed = false;
            const IterT P = iter - at;
            return (P != 0 && n_iterations > iter) ? ((n_iterations - iter - 1) / P) * P : (IterT)0;
        }
        if (++events == next) {
            for (int k = 0; k < N; k++) saved[k] = s[k];
            at = iter;
            next <<= 1;
            have = true;
            if (next == 0u) armed = false;
        }
        return 0;
    }
};

// Tile order of the persistent work queue: centre-out in both directions (k = 0, 1, 2, 3 ... -> mid, mid+1, mid-1,
// mid+2 ...).  Deep views are centred on the feature whose reference orbit they use, so the expensive tiles
// (interior, long orbits) sit in the middle of the frame: handing them out first leaves the cheap border tiles for
// the end of the launch, which keeps the tail of the persistent grid -- one tile's latency, ~0.3 ms on View 14 --
// off the critical path (it is what limits strong scaling once a GPU's share of the frame is ~1 ms).
FS_HD int centre_out(int k, int n) {
    const int mid = (n - 1) >> 1;
    return (k & 1) ? mid + ((k + 1) >> 1) : mid - (k >> 1);
}
// queue index -> top-left pixel of the 8x4 tile; `tiles_y` counts this shard's 4-row bands (b % shard_count == shard_index).
// (Tried and dropped: alternating expensive-first / cheap-first positions so the expensive tiles spread over the SMs
// by load -- 1.7 % faster on the whole View 14 frame, 11 % slower on an 8-way shard, where the launch lasts as long as
// its latest-started expensive tile.)
FS_HD void tile_origin(unsigned int tile, int tiles_x, int tiles_y, int shard_count, int shard_index, int &X0, int &Y0) {
    const int kx = (int)(tile % (unsigned int)tiles_x), ky = (int)(tile / (unsigned int)tiles_x);
    X0 = centre_out(kx, tiles_x) * 8;
    Y0 = (centre_out(ky, tiles_y) * shard_count + shard_index) * 4;
}

#ifdef __CUDACC__
// ---- the work queue every render kernel pulls its 8x4-pixel tiles from -----------------------------------------
// counter      tickets handed out so far (device-local, or a peer-mapped word all GPUs of a box pull from)
// yield_quota  > 0 while a progressive RenderCurrent waits for an SM slot (fs_render_current, progressive = 1, called
//              during a running render): that many CTAs leave the persistent grid at their next tile boundary, so the
//              high-priority post kernel is scheduled at once.  The reference's one-CTA-per-screen-block grid gives the
//              display stream the same chance whenever a block retires (RenderThreadPool.cpp:915-959, 1923-1948).
// grab         tickets taken per atomic (1 locally; a few over NVLink so the round trip is paid once per group)
struct TileQueue {
    unsigned int *counter;
    int *yield_quota;
    unsigned int grab;
};
struct TileCursor {
    unsigned int cur, end;
};
// One flag per CTA: set by the warp that took a retirement token, seen by the CTA's other warps at their next fetch.
static __shared__ int fs_cta_retire;
FS_D void tile_queue_begin(TileCursor &tc) {
    tc.cur = tc.end = 0;
    if (threadIdx.x == 0) fs_cta_retire = 0;
    __syncthreads();
}
// Warp-uniform: every lane gets the same ticket.  Returns false when the queue is exhausted or the CTA retires.
FS_D bool next_tile(const TileQueue &q, TileCursor &tc, unsigned int n_tiles, unsigned int &tile) {
    if (tc.cur == tc.end) {
        unsigned int base = 0xffffffffu;
        if ((threadIdx.x & 31) == 0) {
            bool retire = *(volatile int *)&fs_cta_retire != 0;
            if (!retire && q.yield_quota && *(volatile int *)q.yield_quota > 0) {
                if (atomicSub(q.yield_quota, 1) > 0) {
                    *(volatile int *)&fs_cta_retire = 1;
                    retire = true;
                } else {
                    atomicAdd(q.yield_quota, 1);
                }
            }
            if (!retire) base = atomicAdd(q.counter, q.grab);
        }
        base = __shfl_sync(0xffffffffu, base, 0);
        tc.cur = base;
        tc.end = base >= n_tiles ? base : base + q.grab; // an exhausted queue is asked again (and fails again) next time
    }
    tile = tc.cur;
    if (tile >= n_tiles) return false;
    tc.cur++;
    return true;
}
#endif

// Packed binary32 pairs (sm_100 FMUL2 / FADD2 / FFMA2): two independent IEEE operations per issued instruction,
// each lane rounded exactly like its scalar counterpart.  The host form is the two scalar operations (CPU checkers).
struct f32x2 {
    unsigned long long v; // lo = bits 0..31, hi = bits 32..63
};
FS_HD f32x2 f2_make(float lo, float hi) {
    f32x2 r;
#ifdef __CUDA_ARCH__
    asm("mov.b64 %0, {%1, %2};" : "=l"(r.v) : "f"(lo), "f"(hi));
#else
    r.v = (unsigned long long)f2u(lo) | ((unsigned long long)f2u(hi) << 32);
#endif
    return r;
}
FS_HD void f2_split(f32x2 a, float &lo, float &hi) {
#ifdef __CUDA_ARCH__
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(a.v));
#else
    lo = u2f((uint32_t)a.v);
    hi = u2f((uint32_t)(a.v >> 32));
#endif
}
FS_HD f32x2 f2_mul(f32x2 a, f32x2 b) {
#ifdef __CUDA_ARCH__
    f32x2 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
    return r;
#else
    float al, ah, bl, bh;
    f2_split(a, al, ah);
    f2_split(b, bl, bh);
    return f2_make(al * bl, ah * bh);
#endif
}
FS_HD f32x2 f2_add(f32x2 a, f32x2 b) {
#ifdef __CUDA_ARCH__
    f32x2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
    return r;
#else
    float al, ah, bl, bh;
    f2_split(a, al, ah);
    f2_split(b, bl, bh);
    return f2_make(al + bl, ah + bh);
#endif
}
FS_HD f32x2 f2_fma(f32x2 a, f32x2 b, f32x2 c) {
#ifdef __CUDA_ARCH__
    f32x2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r.v) : "l"(a.v), "l"(b.v), "l"(c.v));
    return r;
#else
    float al, ah, bl, bh, cl, ch;
    f2_split(a, al, ah);
    f2_split(b, bl, bh);
    f2_split(c, cl, ch);
    return f2_make(fma_(al, bl, cl), fma_(ah, bh, ch));
#endif
}
// (s, s): ptxas reads it as a broadcast operand (`R.F32`), no move
FS_HD f32x2 f2_bcast(float s) { return f2_make(s, s); }
// (lo, hi) -> (-hi, lo), i.e. times i.  An exact sign flip; ptxas folds it into the operand (`-R.F32x2.LO_HI.NP`).
FS_HD f32x2 f2_rot(f32x2 a) {
    float lo, hi;
    f2_split(a, lo, hi);
    return f2_make(-hi, lo);
}

// ----------------------------------------------------------------------------------------------
// Mantissa traits: 2^s multipliers and exponent-field surgery, all integer ALU.
// getMultiplier    HDRFloat.h:497-521   s<=-127 -> 0 ; s>=128 -> FLT_MAX ; else 2^s
// getMultiplierNeg HDRFloat.h:523-551   s<=-127 -> 0 ; else scalbnf(1,s)  (callers pass s<=0)
// ----------------------------------------------------------------------------------------------
template <class M> struct MT;

template <> struct MT<float> {
    static constexpr int BIAS = 127;
    FS_HD static float pow2(int s) {
        if (s <= -127) return 0.0f;
        if (s >= 128) return 3.402823466e+38f;
        return u2f((uint32_t)(s + 127) << 23);
    }
    // s <= 0 expected
    FS_HD static float pow2neg(int s) {
        return s <= -127 ? 0.0f : u2f((uint32_t)(s + 127) << 23);
    }
    FS_HD static int expfield(float m) { return (int)((f2u(m) >> 23) & 0xffu); }
    FS_HD static float with_exp0(float m) { return u2f((f2u(m) & 0x807fffffu) | 0x3f800000u); }
    FS_HD static bool is_zero(float m) { return m == 0.0f; }
    FS_HD static float zero() { return 0.0f; }
    FS_HD static float neg(float m) { return -m; }
    FS_HD static float abs(float m) { return fabsf(m); }
};

template <> struct MT<double> {
    static constexpr int BIAS = 1023;
    FS_HD static double pow2(int s) {
        if (s <= -1023) return 0.0;
        if (s >= 1024) return 1.7976931348623157e+308;
        return u2d((uint64_t)(s + 1023) << 52);
    }
    FS_HD static double pow2neg(int s) {
        return s <= -1023 ? 0.0 : u2d((uint64_t)(s + 1023) << 52);
    }
    FS_HD static int expfield(double m) { return (int)((d2u(m) >> 52) & 0x7ffull); }
    FS_HD static double with_exp0(double m) {
        return u2d((d2u(m) & 0x800FFFFFFFFFFFFFull) | 0x3FF0000000000000ull);
    }
    FS_HD static bool is_zero(double m) { return m == 0.0; }
    FS_HD static double zero() { return 0.0; }
    FS_HD static double neg(double m) { return -m; }
    FS_HD static double abs(double m) { return fabs(m); }
};

// ----------------------------------------------------------------------------------------------
// HDR scalar (M = float | double).  Value = m * 2^e.
// ----------------------------------------------------------------------------------------------
template <class M> FS_HD Hdr<M> hdr_zero() { Hdr<M> r; r.m = MT<M>::zero(); r.e = MIN_BIG; return r; }
template <class M> FS_HD Hdr<M> hdr_make(int e, M m) { Hdr<M> r; r.m = m; r.e = e; return r; }

// HDRFloat::Reduce  HDRFloat.h:414-456
template <class M> FS_HD void reduce(Hdr<M> &a) {
    if (MT<M>::is_zero(a.m)) return;
    a.e += MT<M>::expfield(a.m) - MT<M>::BIAS;
    a.m = MT<M>::with_exp0(a.m);
}
template <class M> FS_HD Hdr<M> reduced(Hdr<M> a) { reduce(a); return a; }

// HDRFloat(U number)  HDRFloat.h:295-325
template <class M> FS_HD Hdr<M> hdr_from(M x) {
    if (x == M(0)) return hdr_zero<M>();
    Hdr<M> r;
    r.e = MT<M>::expfield(x) - MT<M>::BIAS;
    r.m = MT<M>::with_exp0(x);
    return r;
}

// operator*  HDRFloat.h:829-851
template <class M> FS_HD Hdr<M> mul(Hdr<M> a, Hdr<M> b) {
    Hdr<M> r;
    r.m = a.m * b.m;
    r.e = imax(a.e + b.e, MIN_BIG);
    return r;
}
// square()  HDRFloat.h:877-884 (no clamp)
template <class M> FS_HD Hdr<M> square(Hdr<M> a) {
    Hdr<M> r;
    r.m = a.m * a.m;
    r.e = a.e * 2;
    return r;
}
// a * HDRFloat(2): mantissa * 1.0 is exact, exponent + 1 clamped (HDRFloat.h:829-868)
template <class M> FS_HD Hdr<M> mul2(Hdr<M> a) {
    a.e = imax(a.e + 1, MIN_BIG);
    return a;
}

// add_mutable / subtract_mutable  HDRFloat.h:974-1000, 1039-1065.
// Branch-free: the smaller-exponent operand is scaled by 2^-|d| (exact) and folded in with one FMA;
// |d| >= 120 drops it.  The early-return arm (d >= 120) skips the zero-mantissa exponent reset,
// exactly as the reference does.
template <class M, bool Sub> FS_HD Hdr<M> addsub(Hdr<M> a, Hdr<M> b) {
    const int d = a.e - b.e;
    const M bm = Sub ? MT<M>::neg(b.m) : b.m;
    const bool age = d >= 0;
    const int ad = iabs(d);
    const M big = age ? a.m : bm;
    const M small = age ? bm : a.m;
    const M mulv = ad >= EXP_DIFF_IGNORED ? MT<M>::zero() : MT<M>::pow2neg(-ad);
    Hdr<M> r;
    r.m = fma_(small, mulv, big);
    r.e = age ? a.e : b.e;
    if (MT<M>::is_zero(r.m) && d < EXP_DIFF_IGNORED) r.e = MIN_BIG;
    return r;
}
template <class M> FS_HD Hdr<M> add(Hdr<M> a, Hdr<M> b) { return addsub<M, false>(a, b); }
template <class M> FS_HD Hdr<M> sub(Hdr<M> a, Hdr<M> b) { return addsub<M, true>(a, b); }

// divide_mutable  HDRFloat.h:624-636
template <class M> FS_HD Hdr<M> div(Hdr<M> a, Hdr<M> b) {
    Hdr<M> r;
    r.m = a.m / b.m;
    r.e = imax(a.e - b.e, MIN_BIG);
    return r;
}

// compareToBothPositiveReduced  HDRFloat.h:1150-1167  (lexicographic on (exp, mantissa))
template <class M> FS_HD int cmp_pr(Hdr<M> a, Hdr<M> b) {
    if (a.e > b.e) return 1;
    if (a.e < b.e) return -1;
    if (a.m > b.m) return 1;
    if (a.m < b.m) return -1;
    return 0;
}
template <class M> FS_HD bool lt_pr(Hdr<M> a, Hdr<M> b) { return a.e < b.e || (a.e == b.e && a.m < b.m); }
template <class M> FS_HD bool ge_pr(Hdr<M> a, Hdr<M> b) { return !lt_pr(a, b); }
template <class M> FS_HD bool gt_pr(Hdr<M> a, Hdr<M> b) { return a.e > b.e || (a.e == b.e && a.m > b.m); }
template <class M> FS_HD bool le_pr(Hdr<M> a, Hdr<M> b) { return !gt_pr(a, b); }

// compareToBothPositiveReducedTemplate<256>() < 0  HDRFloat.h:1169-1184:
// "less" iff exp < 1, or exp == 1 and mantissa < 256  => effectively |z|^2 < 4 for reduced input.
template <class M> FS_HD bool lt_bailout(Hdr<M> a) { return a.e < 1 || (a.e == 1 && !(a.m >= M(256))); }

// ----------------------------------------------------------------------------------------------
// HDR complex with one shared exponent (M = float | double)
// ----------------------------------------------------------------------------------------------
template <class M> FS_HD HdrC<M> hc_zero() { HdrC<M> r; r.re = MT<M>::zero(); r.im = MT<M>::zero(); r.e = MIN_BIG; return r; }

// HDRFloatComplex(re, im) -> setMantexp  HDRFloatComplex.h:158-173
template <class M> FS_HD HdrC<M> hc_from(Hdr<M> re, Hdr<M> im) {
    HdrC<M> r;
    r.e = imax(re.e, im.e);
    r.re = re.m * MT<M>::pow2(re.e - r.e);
    r.im = im.m * MT<M>::pow2(im.e - r.e);
    return r;
}
template <class M> FS_HD Hdr<M> hc_re(HdrC<M> a) { return hdr_make<M>(a.e, a.re); }
template <class M> FS_HD Hdr<M> hc_im(HdrC<M> a) { return hdr_make<M>(a.e, a.im); }

// plus_mutable / sub_mutable  HDRFloatComplex.h:219-247, 384-412 (no zero-mantissa reset here)
template <class M, bool Sub> FS_HD HdrC<M> hc_addsub(HdrC<M> a, HdrC<M> b) {
    const int d = a.e - b.e;
    const M bre = Sub ? MT<M>::neg(b.re) : b.re;
    const M bim = Sub ? MT<M>::neg(b.im) : b.im;
    const bool age = d >= 0;
    const int ad = iabs(d);
    // getMultiplier(-|d|): |d| < 120 here so it is an exact power of two; >= 120 drops the operand
    const M mulv = ad >= EXP_DIFF_IGNORED ? MT<M>::zero() : MT<M>::pow2(-ad);
    HdrC<M> r;
    r.re = fma_(age ? bre : a.re, mulv, age ? a.re : bre);
    r.im = fma_(age ? bim : a.im, mulv, age ? a.im : bim);
    r.e = age ? a.e : b.e;
    return r;
}
template <class M> FS_HD HdrC<M> add(HdrC<M> a, HdrC<M> b) { return hc_addsub<M, false>(a, b); }
template <class M> FS_HD HdrC<M> sub(HdrC<M> a, HdrC<M> b) { return hc_addsub<M, true>(a, b); }

// times_mutable  HDRFloatComplex.h:267-283.  Rounding as nvcc contracted it in the reference build:
//   re = fma(ar, br, -(ai*bi))    im = fma(ai, br, (ar*bi))
template <class M> FS_HD HdrC<M> mul(HdrC<M> a, HdrC<M> b) {
    HdrC<M> r;
    const M t_re = a.im * b.im;
    const M t_im = a.re * b.im;
    r.re = fma_(a.re, b.re, MT<M>::neg(t_re));
    r.im = fma_(a.im, b.re, t_im);
    r.e = imax(a.e + b.e, MIN_BIG);
    return r;
}
// times_mutable(HDRFloat)  HDRFloatComplex.h:334-348
template <class M> FS_HD HdrC<M> mul(HdrC<M> a, Hdr<M> f) {
    HdrC<M> r;
    r.re = a.re * f.m;
    r.im = a.im * f.m;
    r.e = imax(a.e + f.e, MIN_BIG);
    return r;
}
// Reduce  HDRFloatComplex.h:473-527
template <class M> FS_HD void reduce(HdrC<M> &a) {
    if (MT<M>::is_zero(a.re) && MT<M>::is_zero(a.im)) return;
    const int k = imax(MT<M>::expfield(a.re), MT<M>::expfield(a.im)) - MT<M>::BIAS;
    const M mulv = MT<M>::pow2(-k);
    a.re = a.re * mulv;
    a.im = a.im * mulv;
    a.e += k;
}
// chebychevNorm  HDRFloatComplex.h:691-695: both parts share the exponent, so the lexicographic max
// degenerates to the larger |mantissa| (ties/NaN resolve to the imaginary part as in the reference).
template <class M> FS_HD Hdr<M> cheb(HdrC<M> a) {
    const M ar = MT<M>::abs(a.re), ai = MT<M>::abs(a.im);
    return hdr_make<M>(a.e, ar > ai ? ar : ai);
}
// norm_squared  HDRFloatComplex.h:544-548  (nvcc: fma(re, re, im*im))
template <class M> FS_HD Hdr<M> norm2(HdrC<M> a) {
    return hdr_make<M>(a.e << 1, fma_(a.re, a.re, a.im * a.im));
}

// ----------------------------------------------------------------------------------------------
// Plain complex (FloatComplex.h): same contraction pattern as above.
// ----------------------------------------------------------------------------------------------
template <class M> FS_HD Cx<M> add(Cx<M> a, Cx<M> b) { Cx<M> r; r.re = a.re + b.re; r.im = a.im + b.im; return r; }
template <class M> FS_HD Cx<M> mul(Cx<M> a, Cx<M> b) {
    Cx<M> r;
    const M t_re = a.im * b.im;
    const M t_im = a.re * b.im;
    r.re = fma_(a.re, b.re, -t_re);
    r.im = fma_(a.im, b.re, t_im);
    return r;
}
template <class M> FS_HD Cx<M> mul(Cx<M> a, M f) { Cx<M> r; r.re = a.re * f; r.im = a.im * f; return r; }
template <class M> FS_HD void reduce(Cx<M> &) {}
template <class M> FS_HD M cheb(Cx<M> a) {
    const M ar = a.re < 0 ? -a.re : a.re, ai = a.im < 0 ? -a.im : a.im;
    return ar > ai ? ar : ai;
}
template <class M> FS_HD M norm2(Cx<M> a) { return fma_(a.re, a.re, a.im * a.im); }

} // namespace fs
