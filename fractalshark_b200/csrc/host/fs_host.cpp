// fs_host.cpp -- host-side INPUT generation for the render path (libfshost.so): view coordinates,
// the high-precision reference orbit and the LAv2 table, produced in the reference's wire layouts so
// they can be handed to libfsgpu.so (or to the reference GPURenderer) unchanged.
//
// These are the callers' data formats either side of the hot path (SURVEY.md section 8f rows 1 and 4):
//   coordinates  Fractal.cpp:1789-1844, 2831-2840 ; PointZoomBBConverter.cpp:271-312, 388-397
//   orbit (ST)   RefOrbitCalc.cpp:415-647 ; PerturbationResults.cpp:812-868
//   LA table     LAReference.cpp:28-207, 774-1074 ; LAInfoDeep.h:109-502 ; LAParameters.h:66-72
// The reference builds these on the host with GMP + un-fused IEEE arithmetic (x86-64 baseline has no
// FMA), so everything here is plain C++ compiled without -mfma; nothing in this file runs on the GPU.
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include <memory>
#include <atomic>
#include <chrono>
#include <stdio.h>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <unistd.h>

#include "../fs_types.cuh"
#include "fs_gmp_min.h"

using namespace fs;

namespace {

// --------------------------------------------------------------------------------------------
// host numeric policies (un-fused)
// --------------------------------------------------------------------------------------------
template <class M> Hdr<M> h_from_mant(M mant) { // explicit HDRFloat(T mant): exp 0, Reduce (HDRFloat.h:206-212)
    Hdr<M> r; r.m = mant; r.e = 0; reduce(r); return r;
}
template <class M> Hdr<M> h_from_int(int v) { return hdr_from<M>((M)v); } // HDRFloat(U number) (HDRFloat.h:295-325)
template <class M> Hdr<M> h_mul_scalar(Hdr<M> a, M s) { return mul(a, h_from_mant<M>(s)); } // HDRFloat.h:853-868
template <class M> Hdr<M> h_min_pr(Hdr<M> a, Hdr<M> b) { return cmp_pr(a, b) < 0 ? a : b; }

template <class M> HdrC<M> hc_mul_unfused(HdrC<M> a, HdrC<M> b) { // HDRFloatComplex.h:267-283 on the host
    HdrC<M> r;
    r.re = (a.re * b.re) - (a.im * b.im);
    r.im = (a.re * b.im) + (a.im * b.re);
    r.e = imax(a.e + b.e, MIN_BIG);
    return r;
}
template <class M> Hdr<M> hc_norm2_unfused(HdrC<M> a) { return hdr_make<M>(a.e << 1, a.re * a.re + a.im * a.im); }
// plus_mutable(HDRFloat real)  HDRFloatComplex.h:350-382
template <class M> HdrC<M> hc_add_real(HdrC<M> a, Hdr<M> real) {
    const int d = a.e - real.e;
    if (d >= EXP_DIFF_IGNORED) return a;
    if (d >= 0) {
        a.re = a.re + real.m * MT<M>::pow2(-d);
    } else if (d > -EXP_DIFF_IGNORED) {
        const M mulv = MT<M>::pow2(d);
        a.e = real.e;
        a.re = a.re * mulv + real.m;
        a.im = a.im * mulv;
    } else {
        a.e = real.e;
        a.re = real.m;
        a.im = M(0);
    }
    return a;
}
// reciprocal  HDRFloatComplex.h:556-561
template <class M> HdrC<M> hc_recip(HdrC<M> a) {
    const M t = M(1.0f) / (a.re * a.re + a.im * a.im);
    HdrC<M> r;
    r.re = a.re * t;
    r.im = -a.im * t;
    r.e = imax(-a.e, MIN_BIG);
    return r;
}

template <class M> struct HostHdr {
    using Mant = M;
    using Real = Hdr<M>;
    using Cplx = HdrC<M>;
    static constexpr bool kHdr = true;
    static Real r_int(int v) { return h_from_int<M>(v); }
    static Real r_scale(Real a, float s) { return h_mul_scalar<M>(a, (M)s); }
    using Scale = Real; // r_scale's factor as the HDRFloat it is converted to (HDRFloat.h:853-868), made once
    static Scale r_scale_pre(float s) { return h_from_mant<M>((M)s); }
    static Real r_scale_by(Real a, Scale s) { return mul(a, s); }
    static Real r_mul(Real a, Real b) { return mul(a, b); }
    static Real r_div(Real a, Real b) { return div(a, b); }
    static Real r_min(Real a, Real b) { return h_min_pr(a, b); }
    static int r_cmp(Real a, Real b) { return cmp_pr(a, b); }
    static void r_reduce(Real &a) { reduce(a); }
    static bool r_is_zero(Real a) { return a.m == M(0); }
    static Cplx c_one() { Cplx c; c.re = M(1); c.im = M(0); c.e = 0; return c; }
    static Cplx c_zero() { return hc_zero<M>(); }
    static Cplx c_mul(Cplx a, Cplx b) { return hc_mul_unfused(a, b); }
    static Cplx c_mul2(Cplx a) { return mul(a, hdr_make<M>(1, M(1))); }
    static Cplx c_add(Cplx a, Cplx b) { return add(a, b); }
    static Cplx c_add_one(Cplx a) { return hc_add_real(a, h_from_int<M>(1)); }
    static void c_reduce(Cplx &a) { reduce(a); }
    static Real c_cheb(Cplx a) { return cheb(a); }
    static Real c_norm2(Cplx a) { return hc_norm2_unfused(a); }
    static Cplx c_recip(Cplx a) { return hc_recip(a); }
    static bool c_is_zero(Cplx a) { return a.re == M(0) && a.im == M(0); }
    static Real at_lim(bool small_exp) {
        Real lim = hdr_make<M>(32, M(1));
        if (sizeof(M) == 8 && !small_exp) lim.e = 256; // LAInfoDeep.h:477-485
        reduce(lim);
        return lim;
    }
    static Real at_factor() { return hdr_from<M>((M)4294967296.0); } // ATInfo() ctor: HDRFloat(0x1.0p32)
    static Real at_four() { return h_from_mant<M>(M(4.0f)); }
    static Real r_square_reduced(Real a) { Real r = square(a); reduce(r); return r; }
};

template <class M> struct HostPlain {
    using Mant = M;
    using Real = M;
    using Cplx = Cx<M>;
    static constexpr bool kHdr = false;
    static Real r_int(int v) { return (M)v; }
    static Real r_scale(Real a, float s) { return a * (M)s; }
    using Scale = M;
    static Scale r_scale_pre(float s) { return (M)s; }
    static Real r_scale_by(Real a, Scale s) { return a * s; }
    static Real r_mul(Real a, Real b) { return a * b; }
    static Real r_div(Real a, Real b) { return a / b; }
    static Real r_min(Real a, Real b) { return std::min(a, b); }
    static int r_cmp(Real a, Real b) { return a > b ? 1 : (a < b ? -1 : 0); }
    static void r_reduce(Real &) {}
    static bool r_is_zero(Real a) { return a == M(0); }
    static Cplx c_one() { Cplx c; c.re = M(1); c.im = M(0); return c; }
    static Cplx c_zero() { Cplx c; c.re = M(0); c.im = M(0); return c; }
    static Cplx c_mul(Cplx a, Cplx b) {
        Cplx r;
        r.re = (a.re * b.re) - (a.im * b.im);
        r.im = (a.re * b.im) + (a.im * b.re);
        return r;
    }
    static Cplx c_mul2(Cplx a) { a.re *= M(2); a.im *= M(2); return a; }
    static Cplx c_add(Cplx a, Cplx b) { a.re += b.re; a.im += b.im; return a; }
    static Cplx c_add_one(Cplx a) { a.re += M(1); return a; }
    static void c_reduce(Cplx &) {}
    static Real c_cheb(Cplx a) { const M x = fabs(a.re), y = fabs(a.im); return x > y ? x : y; }
    static Real c_norm2(Cplx a) { return a.re * a.re + a.im * a.im; }
    static Cplx c_recip(Cplx a) {
        const M t = M(1) / (a.re * a.re + a.im * a.im);
        Cplx r; r.re = a.re * t; r.im = -a.im * t; return r;
    }
    static bool c_is_zero(Cplx a) { return a.re == M(0) && a.im == M(0); }
    static Real at_lim(bool) { return (M)4294967296.0f; }
    static Real at_factor() { return (M)4294967296.0; }
    static Real at_four() { return M(4); }
    static Real r_square_reduced(Real a) { return a * a; }
};

// reference wire structs (same declarations as in fs_capi.cu; sizes asserted there)
template <class N, class IterT> struct WireLA {
    typename N::Cplx Ref, ZCoeff, CCoeff;
    typename N::Real LAThreshold, LAThresholdC, MinMag;
    IterT StepLength, NextStageLAIndex;
};
template <class N, class IterT> struct WireAT {
    IterT StepLength;
    typename N::Real ThresholdC, SqrEscapeRadius;
    typename N::Cplx RefC, ZCoeff, CCoeff, InvZCoeff, CCoeffSqrInvZCoeff, CCoeffInvZCoeff;
    typename N::Real CCoeffNormSqr, RefCNormSqr, factor;
};
template <class IterT> struct WireStage { IterT LAIndex, MacroItCount; };

// LAParameters defaults (LAParameters.h:66-72): method 1, 2^-24, 2^-24, 2^-6, 2^-3, 2^-10, 2^-10
struct LaParams {
    float la_scale = ldexpf(1.f, -24), lac_scale = ldexpf(1.f, -24);
    float stage0_thr2 = ldexpf(1.f, -6), thr2 = ldexpf(1.f, -3);
};

// --------------------------------------------------------------------------------------------
// View
// --------------------------------------------------------------------------------------------
struct Mpf {
    fs_mpf_t v;
    explicit Mpf(unsigned long prec) { fs_mpf_init2(v, prec); }
    Mpf(const Mpf &o) { fs_mpf_init2(v, (unsigned long)o.v->_mp_prec * 64); fs_mpf_set(v, o.v); }
    Mpf &operator=(const Mpf &o) { fs_mpf_set(v, o.v); return *this; }
    ~Mpf() { fs_mpf_clear(v); }
};

} // namespace

struct fsh_view {
    unsigned long prec;
    Mpf minX, minY, maxX, maxY, cx, cy;
    uint32_t w, h, aa;
    explicit fsh_view(unsigned long p) : prec(p), minX(p), minY(p), maxX(p), maxY(p), cx(p), cy(p), w(0), h(0), aa(1) {}
};

struct fsh_orbit {
    int numeric = 0;
    int pextras = 0;                  // 0 Disable, 1 Bad, 2 SimpleCompression
    uint64_t uncompressed_count = 0;  // SimpleCompression: GetCountOrbitEntries(); `count` is then the compressed size
    std::shared_ptr<fsh_orbit> plain; // SimpleCompression: the host-side replay of this orbit (RuntimeDecompressor view)
    std::shared_ptr<fsh_orbit> base; // 2x32 types: the double / HDR-double orbit they were converted from
    std::vector<unsigned char> data;
    uint64_t count = 0, period = 0;
    size_t elem_bytes = 0;
    unsigned char max_radius[16] = {0}; // Real, reduced
    unsigned char x_low[16] = {0}, y_low[16] = {0};
};

struct fsh_blas {
    std::vector<std::vector<unsigned char>> levels;
    std::vector<uint64_t> counts;
    std::vector<const void *> ptrs;
    size_t elem_bytes = 0;
    int32_t lm2 = 0;
};

struct fsh_la {
    std::vector<unsigned char> las, stages, at;
    void *las_own = nullptr; // the builder's own record array, taken over as is (no copy); nullptr: `las` holds the records
    uint64_t num_las = 0, num_stages = 0, stage_count = 0;
    int use_at = 0, is_valid = 0;
    fsh_la() = default;
    fsh_la(const fsh_la &) = delete;
    fsh_la &operator=(const fsh_la &) = delete;
    ~fsh_la() { free(las_own); }
};

namespace {

// HDRFloat(mpf_t)  HDRFloat.h:366-389: mpf_get_d_2exp truncates, then the mantissa is cast to M
template <class M> Hdr<M> hdr_from_mpf(const fs_mpf_struct *f) {
    if (fs_mpf_sgn(f) == 0) return hdr_zero<M>();
    long e = 0;
    const double d = fs_mpf_get_d_2exp(&e, f);
    Hdr<M> r;
    r.m = (M)d;
    r.e = (int32_t)e;
    return r;
}

template <class N> struct FromMpf;
template <class M> struct FromMpf<HostHdr<M>> {
    static Hdr<M> raw(const fs_mpf_struct *f) { return hdr_from_mpf<M>(f); }
    static Hdr<M> coord(const fs_mpf_struct *f) { Hdr<M> r = hdr_from_mpf<M>(f); reduce(r); return r; } // FillCoord
};
template <class M> struct FromMpf<HostPlain<M>> {
    static M raw(const fs_mpf_struct *f) { return (M)fs_mpf_get_d(f); }
    static M coord(const fs_mpf_struct *f) { return (M)fs_mpf_get_d(f); }
};

// orbit element writers: x Left-order, y Right-order for HDR (GPU_ReferenceIter.h:119-125)
template <class N> struct ElemIO;
template <class M> struct ElemIO<HostPlain<M>> {
    static constexpr size_t kBytes = 2 * sizeof(M);
    static void put(unsigned char *p, M x, M y) { memcpy(p, &x, sizeof(M)); memcpy(p + sizeof(M), &y, sizeof(M)); }
    static void get(const unsigned char *p, M &x, M &y) { memcpy(&x, p, sizeof(M)); memcpy(&y, p + sizeof(M), sizeof(M)); }
};
template <> struct ElemIO<HostHdr<float>> {
    static constexpr size_t kBytes = 16;
    static void put(unsigned char *p, Hdr<float> x, Hdr<float> y) {
        memcpy(p, &x.m, 4); memcpy(p + 4, &x.e, 4); memcpy(p + 8, &y.e, 4); memcpy(p + 12, &y.m, 4);
    }
    static void get(const unsigned char *p, Hdr<float> &x, Hdr<float> &y) {
        memcpy(&x.m, p, 4); memcpy(&x.e, p + 4, 4); memcpy(&y.e, p + 8, 4); memcpy(&y.m, p + 12, 4);
    }
};
template <> struct ElemIO<HostHdr<double>> {
    static constexpr size_t kBytes = 32;
    static void put(unsigned char *p, Hdr<double> x, Hdr<double> y) {
        memset(p, 0, 32);
        memcpy(p, &x.m, 8); memcpy(p + 8, &x.e, 4); memcpy(p + 16, &y.e, 4); memcpy(p + 24, &y.m, 8);
    }
    static void get(const unsigned char *p, Hdr<double> &x, Hdr<double> &y) {
        memcpy(&x.m, p, 8); memcpy(&x.e, p + 8, 4); memcpy(&y.e, p + 16, 4); memcpy(&y.m, p + 24, 8);
    }
};

// --------------------------------------------------------------------------------------------
// Reference orbit, single-threaded GMP loop (RefOrbitCalc.cpp:447-623).
// Periodicity test |z| < 2 * MaxRadius * |dz/dc| is evaluated in (double mantissa, int exponent)
// arithmetic here; it decides only where the orbit stops.
// --------------------------------------------------------------------------------------------
struct XD { // extended double
    double m; long e;
};
XD xd_norm(double m, long e) {
    if (m == 0) return {0, -(1L << 40)};
    int k; m = frexp(m, &k);
    return {m, e + k};
}
XD xd_mul(XD a, XD b) { return xd_norm(a.m * b.m, a.e + b.e); }
XD xd_add(XD a, XD b) {
    if (a.m == 0) return b;
    if (b.m == 0) return a;
    if (a.e < b.e) std::swap(a, b);
    const long d = a.e - b.e;
    if (d > 200) return a;
    return xd_norm(a.m + ldexp(b.m, (int)-d), a.e);
}
XD xd_neg(XD a) { a.m = -a.m; return a; }
bool xd_lt_abs(XD a, XD b) { // |a| < |b|
    if (b.m == 0) return false;
    if (a.m == 0) return true;
    if (a.e != b.e) return a.e < b.e;
    return fabs(a.m) < fabs(b.m);
}
XD xd_absmax(XD a, XD b) { return xd_lt_abs(a, b) ? XD{fabs(b.m), b.e} : XD{fabs(a.m), a.e}; }
XD xd_from_mpf(const fs_mpf_struct *f) {
    if (fs_mpf_sgn(f) == 0) return {0, -(1L << 40)};
    long e; const double d = fs_mpf_get_d_2exp(&e, f);
    return {d, e};
}

// One product per iteration on a thread of its own (the three-thread form of the reference's producer,
// RefOrbitCalc.cpp:1532-2157: x*x, y*y and 2x*y of one iteration side by side).  mpf_mul is deterministic and the operands
// are only read, so the orbit is the one the single-threaded loop gives, bit for bit.  Worth it once a product costs
// microseconds: View 14 runs at 22,095 bits, 14 us per product.
struct MulThread {
    fs_mpf_struct *dst = nullptr;
    const fs_mpf_struct *a = nullptr, *b = nullptr;
    std::atomic<uint64_t> req{0}, ack{0};
    uint64_t n = 0;
    bool stop = false;
    std::thread th;
    static void relax(int &spins) {
#if defined(__x86_64__) || defined(__i386__)
        if (spins < 4096) { spins++; __builtin_ia32_pause(); return; }
#endif
        std::this_thread::yield();
    }
    void start() {
        th = std::thread([this] {
            uint64_t seen = 0;
            for (;;) {
                int spins = 0;
                uint64_t r;
                while ((r = req.load(std::memory_order_acquire)) == seen) relax(spins);
                seen = r;
                if (stop) return;
                fs_mpf_mul(dst, a, b);
                ack.store(seen, std::memory_order_release);
            }
        });
    }
    void post() { req.store(++n, std::memory_order_release); }
    void wait() {
        int spins = 0;
        while (ack.load(std::memory_order_acquire) != n) relax(spins);
    }
    ~MulThread() {
        if (th.joinable()) {
            stop = true;
            req.store(++n, std::memory_order_release);
            th.join();
        }
    }
};

template <class N> void compute_orbit(const fsh_view *v, fsh_orbit *o, uint64_t max_iters, bool periodicity) {
    using IO = ElemIO<N>;
    const unsigned long prec = v->prec;
    Mpf zx(prec), zy(prec), zx2(prec), t1(prec), t2(prec), t3(prec), delta(prec);
    // FS_ORBIT_THREADS=1: the single-threaded loop whatever the precision
    const char *ot = getenv("FS_ORBIT_THREADS");
    const bool three_threads = prec >= 4096 && std::thread::hardware_concurrency() >= 3 && !(ot && atoi(ot) == 1);
    MulThread mul_yy, mul_xy;
    if (three_threads) {
        mul_yy.dst = t2.v; mul_yy.a = zy.v; mul_yy.b = zy.v;
        mul_xy.dst = t3.v; mul_xy.a = zx2.v; mul_xy.b = zy.v;
        mul_yy.start();
        mul_xy.start();
    }
    o->elem_bytes = IO::kBytes;
    o->data.clear();
    o->data.reserve((size_t)std::min<uint64_t>(max_iters + 2, 1u << 22) * IO::kBytes);
    auto push = [&](typename N::Real x, typename N::Real y) {
        const size_t off = o->data.size();
        o->data.resize(off + IO::kBytes);
        IO::put(o->data.data() + off, x, y);
        o->count++;
    };
    // MaxRadius = T{maxY - minY} / T{2.0f}, reduced (PerturbationResults.cpp:823-857)
    fs_mpf_sub(delta.v, v->maxY.v, v->minY.v);
    {
        typename N::Real rad = FromMpf<N>::raw(delta.v);
        rad = N::r_div(rad, N::kHdr ? N::r_int(2) : N::r_int(2));
        N::r_reduce(rad);
        memcpy(o->max_radius, &rad, sizeof(rad));
        typename N::Real xl = FromMpf<N>::raw(v->cx.v), yl = FromMpf<N>::raw(v->cy.v);
        memcpy(o->x_low, &xl, sizeof(xl));
        memcpy(o->y_low, &yl, sizeof(yl));
    }
    const XD max_radius = xd_mul(xd_from_mpf(delta.v), XD{0.5, 0});
    // entry 0 is the zero element (PerturbationResults.cpp:861-868)
    if constexpr (N::kHdr) {
        const typename N::Real zr = hdr_zero<typename N::Mant>();
        push(zr, zr);
    } else {
        push(typename N::Real{}, typename N::Real{});
    }
    fs_mpf_set(zx.v, v->cx.v);
    fs_mpf_set(zy.v, v->cy.v);
    const double cxd = fs_mpf_get_d(v->cx.v), cyd = fs_mpf_get_d(v->cy.v);
    XD dzdcX{0.5, 1}, dzdcY{0, -(1L << 40)};
    o->period = 0;
    for (uint64_t i = 0; i < max_iters; i++) {
        fs_mpf_mul_2exp(zx2.v, zx.v, 1);
        if (three_threads) { // y*y and 2x*y start now; this thread stores the element, tests the period and squares x
            mul_yy.post();
            mul_xy.post();
        }
        push(FromMpf<N>::raw(zx.v), FromMpf<N>::raw(zy.v));
        if (periodicity) {
            const XD zxd = xd_from_mpf(zx.v), zyd = xd_from_mpf(zy.v);
            const XD n2 = xd_absmax(zxd, zyd);
            const XD r0 = xd_absmax(dzdcX, dzdcY);
            const XD n3 = xd_mul(xd_mul(max_radius, r0), XD{0.5, 2});
            if (xd_lt_abs(n2, n3)) {
                o->period = o->count;
                if (three_threads) { mul_yy.wait(); mul_xy.wait(); }
                break;
            }
            const XD ox = dzdcX;
            dzdcX = xd_add(xd_mul(XD{0.5, 2}, xd_add(xd_mul(zxd, dzdcX), xd_neg(xd_mul(zyd, dzdcY)))), XD{0.5, 1});
            dzdcY = xd_mul(XD{0.5, 2}, xd_add(xd_mul(zxd, dzdcY), xd_mul(zyd, ox)));
        }
        const double zxd0 = fs_mpf_get_d(zx.v), zyd0 = fs_mpf_get_d(zy.v);
        fs_mpf_mul(t1.v, zx.v, zx.v);
        if (three_threads) {
            mul_yy.wait();
            mul_xy.wait();
            fs_mpf_sub(zx.v, t1.v, t2.v);
            fs_mpf_add(zx.v, zx.v, v->cx.v);
            fs_mpf_add(zy.v, t3.v, v->cy.v);
        } else {
            fs_mpf_mul(t2.v, zy.v, zy.v);
            fs_mpf_sub(zx.v, t1.v, t2.v);
            fs_mpf_add(zx.v, zx.v, v->cx.v);
            fs_mpf_mul(zy.v, zx2.v, zy.v);
            fs_mpf_add(zy.v, zy.v, v->cy.v);
        }
        const double tx = zxd0 + cxd, ty = zyd0 + cyd;
        if (tx * tx + ty * ty > 256.0) break;
    }
}

// --------------------------------------------------------------------------------------------
// LA table construction (single-thread routine of the reference)
// --------------------------------------------------------------------------------------------
// A small persistent pool for the record-parallel phase of the table builders: threads are created once per process
// (FS_HOST_THREADS, default min(hardware threads, 16)), a job is a function of an index range, the caller works too.
class HostPool {
  public:
    static HostPool &get() { static HostPool p; return p; }
    size_t threads() const { return workers.size() + 1; }
    // min_grain: indices per claim at least; heavy items (a record of an upper LA stage is a chain of tens of composites)
    // want a small one, and are worth the threads from a few dozen items on
    void run(size_t n, const std::function<void(size_t, size_t)> &fn, size_t min_grain = 64) {
        if (n == 0) return;
        if (!have_workers() || n < 8 * min_grain) { fn(0, n); return; }
        dispatch(n, std::max<size_t>(min_grain, n / (threads() * 8)), fn);
    }
    // n tasks, one index each, claimed in index order; a task may wait for a task with a smaller index (which some thread
    // has claimed before and runs to completion), never for a larger one.  Without workers they run one after the other.
    void run_tasks(size_t n, const std::function<void(size_t, size_t)> &fn) {
        if (n == 0) return;
        if (!have_workers()) { for (size_t k = 0; k < n; k++) fn(k, k + 1); return; }
        dispatch(n, 1, fn);
    }

  private:
    // a forked child has the pool object but none of its threads: it works alone
    bool have_workers() const { return !workers.empty() && getpid() == owner; }
    void dispatch(size_t n, size_t g, const std::function<void(size_t, size_t)> &fn) {
        std::lock_guard<std::mutex> one_job(job_mu); // callers on different threads take turns (jobs never nest)
        {
            std::lock_guard<std::mutex> lk(mu);
            job = &fn;
            total = n;
            grain = g;
            next.store(0);
            pending = workers.size();
            left.store(pending, std::memory_order_relaxed);
            generation++;
            posted.store(generation, std::memory_order_release);
        }
        wake.notify_all();
        work();
        // the caller spins as well: the jobs of one build are tens of microseconds long
        for (int spin = 0; spin < kSpin; spin++) {
            if (left.load(std::memory_order_acquire) == 0) break;
            cpu_relax(spin);
        }
        std::unique_lock<std::mutex> lk(mu);
        done.wait(lk, [&] { return pending == 0; });
        job = nullptr;
    }
    // a few hundred pauses, then yields: with fewer cores than threads the thread being waited for gets the core
    static void cpu_relax(int spin) {
#if defined(__x86_64__) || defined(__i386__)
        if (spin < 256) { __builtin_ia32_pause(); return; }
#endif
        std::this_thread::yield();
    }
    static constexpr int kSpin = 1500;
    HostPool() {
        size_t want = std::thread::hardware_concurrency();
        if (const char *e = getenv("FS_HOST_THREADS")) want = (size_t)atoi(e);
        want = std::min<size_t>(std::max<size_t>(want, 1), 16);
        owner = getpid();
        for (size_t t = 1; t < want; t++) workers.emplace_back([this] { loop(); });
    }
    ~HostPool() {
        if (getpid() != owner) {
            for (auto &t : workers) t.detach();
            return;
        }
        {
            std::lock_guard<std::mutex> lk(mu);
            stop = true;
            generation++;
        }
        wake.notify_all();
        for (auto &t : workers) t.join();
    }
    void work() {
        for (;;) {
            const size_t lo = next.fetch_add(grain);
            if (lo >= total) break;
            (*job)(lo, std::min(total, lo + grain));
        }
    }
    void loop() {
        size_t seen = 0;
        for (;;) {
            // the jobs of one table build follow each other within microseconds: look for the next one for a while before
            // going to sleep on the condition variable (a wake-up through the futex costs more than most of these jobs)
            for (int spin = 0; spin < kSpin; spin++) {
                if (posted.load(std::memory_order_acquire) != seen) break;
                cpu_relax(spin);
            }
            {
                std::unique_lock<std::mutex> lk(mu);
                wake.wait(lk, [&] { return generation != seen; });
                seen = generation;
                if (stop) return;
            }
            work();
            left.fetch_sub(1, std::memory_order_release);
            std::lock_guard<std::mutex> lk(mu);
            if (--pending == 0) done.notify_one();
        }
    }
    std::vector<std::thread> workers;
    pid_t owner = 0;
    std::mutex mu, job_mu;
    std::condition_variable wake, done;
    const std::function<void(size_t, size_t)> *job = nullptr;
    std::atomic<size_t> next{0}, posted{0}, left{0};
    size_t total = 0, grain = 1, pending = 0, generation = 0;
    bool stop = false;
};
template <class F> void parallel_for(size_t n, F &&fn, size_t min_grain = 64) { HostPool::get().run(n, std::function<void(size_t, size_t)>(fn), min_grain); }

// Array of trivially copyable records in uninitialised storage (no value-initialisation pass over megabytes that are about
// to be overwritten), which can hand its allocation to the object that outlives the builder.
template <class T> struct RawVec {
    T *p = nullptr;
    size_t n = 0, cap = 0;
    RawVec() = default;
    RawVec(const RawVec &) = delete;
    RawVec &operator=(const RawVec &) = delete;
    ~RawVec() { free(p); }
    size_t size() const { return n; }
    bool empty() const { return n == 0; }
    T *data() { return p; }
    const T *data() const { return p; }
    T &operator[](size_t i) { return p[i]; }
    const T &operator[](size_t i) const { return p[i]; }
    void reserve(size_t c) {
        if (c <= cap) return;
        T *q = static_cast<T *>(malloc(c * sizeof(T)));
        if (!q) throw std::bad_alloc();
        if (n) memcpy(static_cast<void *>(q), p, n * sizeof(T));
        free(p);
        p = q;
        cap = c;
    }
    void push_back(const T &v) {
        if (n == cap) reserve(cap ? cap * 2 : 64);
        p[n++] = v;
    }
    void pop_back() { n--; }
    void clear() { n = 0; }
    void resize_uninit(size_t c) { reserve(c); n = c; }
    T *release() { T *q = p; p = nullptr; n = cap = 0; return q; }
};

template <class N, class IterT> struct LaBuilder {
    using Real = typename N::Real;
    using Cplx = typename N::Cplx;
    using LA = WireLA<N, IterT>;
    using AT = WireAT<N, IterT>;
    static constexpr int lowBound = 64;     // LAReference.h:56
    int periodDivisor = 2; // LAReference.cpp:17-19: 2, or 8 when the orbit is compressed (SimpleCompression)
    static constexpr int MaxLAStages = 1024;

    const fsh_orbit *orbit;
    bool small_exp = false; // UseSmallExponents: true when the table is destined for a 2x32 type (RefOrbitCalc.cpp:2329-2346)
    LaParams P;
    RawVec<LA> las;
    std::vector<WireStage<IterT>> stages;
    AT at;
    bool use_at = false, is_valid = false;
    IterT stage_count = 0;

    Cplx orbit_at(uint64_t i) const { // PerturbationResults::GetComplex<SubType>
        Real x, y;
        ElemIO<N>::get(orbit->data.data() + i * ElemIO<N>::kBytes, x, y);
        if constexpr (N::kHdr) return hc_from<typename N::Mant>(x, y);
        else { Cplx c; c.re = x; c.im = y; return c; }
    }

    static LA la_blank() { LA l; memset(&l, 0, sizeof(l)); if constexpr (N::kHdr) {
            l.Ref = N::c_zero(); l.ZCoeff = N::c_zero(); l.CCoeff = N::c_zero();
            l.LAThreshold.e = MIN_BIG; l.LAThresholdC.e = MIN_BIG; l.MinMag.e = MIN_BIG; }
        return l; }
    LA la_new(Cplx z) const { // LAInfoDeep(la_parameters, z)  LAInfoDeep.h:109-133
        LA l = la_blank();
        l.Ref = z;
        l.ZCoeff = N::c_one();
        l.CCoeff = N::c_one();
        l.LAThreshold = N::r_int(1);
        l.LAThresholdC = N::r_int(1);
        l.MinMag = N::r_int(4);
        return l;
    }
    // Step  LAInfoDeep.h:185-259 ; returns "period detected"
    bool la_step(const LA &a, LA &out, Cplx z) const {
        const Real mz = N::c_cheb(z), mZ = N::c_cheb(a.ZCoeff), mC = N::c_cheb(a.CCoeff);
        out.MinMag = N::r_min(mz, a.MinMag);
        Real t1 = N::r_scale(N::r_div(mz, mZ), P.la_scale);
        N::r_reduce(t1);
        Real t2 = N::r_scale(N::r_div(mz, mC), P.lac_scale);
        N::r_reduce(t2);
        out.LAThreshold = N::r_min(a.LAThreshold, t1);
        out.LAThresholdC = N::r_min(a.LAThresholdC, t2);
        const Cplx z2 = N::c_mul2(z);
        Cplx oz = N::c_mul(z2, a.ZCoeff);
        N::c_reduce(oz);
        Cplx oc = N::c_add_one(N::c_mul(z2, a.CCoeff));
        N::c_reduce(oc);
        out.ZCoeff = oz;
        out.CCoeff = oc;
        out.Ref = a.Ref;
        return N::r_cmp(out.MinMag, N::r_scale(a.MinMag, P.stage0_thr2)) < 0;
    }
    LA la_step(const LA &a, Cplx z) const { LA r = la_blank(); la_step(a, r, z); return r; }
    bool la_detect(const LA &a, Cplx z) const { // DetectPeriod  LAInfoDeep.h:135-157 (method 1)
        return N::r_cmp(N::c_cheb(z), N::r_scale(a.MinMag, P.thr2)) < 0;
    }
    // Composite  LAInfoDeep.h:294-381
    bool la_comp(const LA &a, LA &out, const LA &b) const {
        const Cplx z = b.Ref;
        const Real mz = N::c_cheb(z);
        Real mZ = N::c_cheb(a.ZCoeff), mC = N::c_cheb(a.CCoeff);
        Real t1 = N::r_scale(N::r_div(mz, mZ), P.la_scale);
        N::r_reduce(t1);
        Real t2 = N::r_scale(N::r_div(mz, mC), P.lac_scale);
        N::r_reduce(t2);
        Real oT = N::r_min(a.LAThreshold, t1), oTC = N::r_min(a.LAThresholdC, t2);
        const Cplx z2 = N::c_mul2(z);
        Cplx oz = N::c_mul(z2, a.ZCoeff);
        N::c_reduce(oz);
        Cplx oc = N::c_mul(z2, a.CCoeff);
        N::c_reduce(oc);
        mZ = N::c_cheb(oz);
        mC = N::c_cheb(oc);
        t1 = N::r_div(b.LAThreshold, mZ);
        N::r_reduce(t1);
        t2 = N::r_div(b.LAThreshold, mC);
        N::r_reduce(t2);
        oT = N::r_min(oT, t1);
        oTC = N::r_min(oTC, t2);
        oz = N::c_mul(oz, b.ZCoeff);
        N::c_reduce(oz);
        oc = N::c_add(N::c_mul(oc, b.ZCoeff), b.CCoeff);
        N::c_reduce(oc);
        out.LAThreshold = oT;
        out.LAThresholdC = oTC;
        out.ZCoeff = oz;
        out.CCoeff = oc;
        out.Ref = a.Ref;
        const Real temp = N::r_min(mz, a.MinMag);
        out.MinMag = N::r_min(temp, b.MinMag);
        return N::r_cmp(temp, N::r_scale(a.MinMag, P.thr2)) < 0;
    }
    LA la_comp(const LA &a, const LA &b) const { LA r = la_blank(); la_comp(a, r, b); return r; }

    // ---- two-phase construction -------------------------------------------------------------------------------------
    // Which orbit elements (stage 0) or previous-stage records (higher stages) end up in which record is decided by the
    // MinMag chain alone: Step / Composite report "period detected" from min(|z|, MinMag) and DetectPeriod from |z| and
    // MinMag (LAInfoDeep.h:135-157, 185-259, 294-381) -- ZCoeff, CCoeff and the thresholds never steer the walk.  So a
    // stage runs in two phases: phase 1 walks CreateLAFromOrbit / CreateNewLAStage exactly as written, carrying only
    // {Ref, MinMag} and noting for every record pushed where it starts and how many elements it absorbs (a run of
    // consecutive indices); phase 2 builds each record from its note -- the same Step / Composite calls on the same
    // operands in the same order, hence the same bytes (tests/test_table_construction.py compares them with the
    // reference's own builder) -- on all host threads at once, the records being independent of each other.
    struct Note { uint32_t kind; IterT first, count; }; // kind 0: LAInfoDeep(orbit[first]); 1: copy of previous-stage record
                                                        // `first`; 2: LAInfoDeep(0); 3: already complete
    // what phase 1 carries for the record under construction (the walk's `LA`), and what it leaves behind for phase 2
    struct LAx { Real MinMag; Note n; IterT StepLength, NextStageLAIndex; Real chebRef; }; // chebRef: pipelined walks only
    std::vector<Note> notes; // notes of the records of the stage under construction
    std::vector<Real> chebs; // Chebyshev norm of every orbit element: all that phase 1 of stage 0 reads
    size_t stage_begin = 0;  // index of that stage's first record in `las`
    typename N::Scale thr_stage0, thr_detect; // the two period-detection factors, converted once

    LAx x_new_zero() const { return LAx{N::r_int(4), Note{2, 0, 0}, 0, 0, N::c_cheb(N::c_zero())}; } // LAInfoDeep(z): MinMag = 4 (LAInfoDeep.h:109-133)
    LAx x_new_at(IterT i) const { return LAx{N::r_int(4), Note{0, i, 0}, 0, 0, chebs[i]}; }
    LAx x_copy_prev(IterT prev_idx, IterT j) const { return LAx{las[prev_idx + j].MinMag, Note{1, j, 0}, 0, 0, Real{}}; }
    // Step  LAInfoDeep.h:185-259, the MinMag part: one more orbit element (always a.n.first + a.n.count + 1)
    bool x_step(const LAx &a, LAx &out, IterT i) const {
        out.n = Note{a.n.kind, a.n.first, a.n.count + 1};
        out.chebRef = a.chebRef;
        out.MinMag = N::r_min(chebs[i], a.MinMag);
        return N::r_cmp(out.MinMag, N::r_scale_by(a.MinMag, thr_stage0)) < 0;
    }
    LAx x_step(const LAx &a, IterT i) const { LAx r = a; x_step(a, r, i); return r; }
    bool x_detect(const LAx &a, Real cheb_z) const { // DetectPeriod  LAInfoDeep.h:135-157 (method 1)
        return N::r_cmp(cheb_z, N::r_scale_by(a.MinMag, thr_detect)) < 0;
    }
    // Composite  LAInfoDeep.h:294-381, the MinMag part: one more previous-stage record, consecutive as well
    bool x_comp(const LAx &a, LAx &out, const LA &b) const {
        out.n = Note{a.n.kind, a.n.first, a.n.count + 1};
        out.chebRef = a.chebRef;
        const Real temp = N::r_min(N::c_cheb(b.Ref), a.MinMag);
        out.MinMag = N::r_min(temp, b.MinMag);
        return N::r_cmp(temp, N::r_scale_by(a.MinMag, thr_detect)) < 0;
    }
    LAx x_comp(const LAx &a, const LA &b) const { LAx r = a; x_comp(a, r, b); return r; }
    void x_push(const LAx &a) {
        LA l = la_blank();
        l.StepLength = a.StepLength; l.NextStageLAIndex = a.NextStageLAIndex;
        las.push_back(l);
        notes.push_back(a.n);
    }
    void x_push_done(const LA &a) { las.push_back(a); notes.push_back(Note{3, 0, 0}); }
    void x_pop() { las.pop_back(); notes.pop_back(); }
    // phase 2 of the stage whose records are las[stage_begin ...]; prev_idx = first record of the previous stage
    void fill_stage(IterT prev_idx) {
        const size_t n = notes.size();
        auto job = [&](size_t lo, size_t hi) {
            for (size_t k = lo; k < hi; k++) {
                const Note nt = notes[k];
                if (nt.kind == 3) continue;
                LA &dst = las[stage_begin + k];
                LA l;
                if (nt.kind == 1) l = las[(size_t)prev_idx + nt.first];
                else l = la_new(nt.kind == 2 ? N::c_zero() : orbit_at(nt.first));
                for (IterT c = 1; c <= nt.count; c++) {
                    LA nl = la_blank();
                    if (nt.kind == 1) la_comp(l, nl, las[(size_t)prev_idx + nt.first + c]);
                    else la_step(l, nl, orbit_at((nt.kind == 2 ? (IterT)0 : nt.first) + c));
                    l = nl;
                }
                l.StepLength = dst.StepLength;
                l.NextStageLAIndex = dst.NextStageLAIndex;
                dst = l;
            }
        };
        parallel_for(n, job);
        notes.clear();
    }

    IterT nth_root_period(double maxRef, double ratio) const {
        const double nth = round(log2(maxRef) / periodDivisor);
        return (IterT)round(pow(ratio, 1.0 / nth));
    }

    // CreateLAFromOrbit  LAReference.cpp:28-207
    bool stage0(IterT maxRef) {
        notes.clear();
        stage_begin = las.size();
        las.reserve((size_t)maxRef + 4); // the walk holds references into `las` across push_back
        thr_stage0 = N::r_scale_pre(P.stage0_thr2);
        thr_detect = N::r_scale_pre(P.thr2);
        chebs.resize((size_t)maxRef + 1);
        parallel_for(chebs.size(), [&](size_t lo, size_t hi) { for (size_t k = lo; k < hi; k++) chebs[k] = N::c_cheb(orbit_at(k)); });
        const auto t0 = std::chrono::steady_clock::now();
        const bool ok = stage0_walk(maxRef);
        const auto t1 = std::chrono::steady_clock::now();
        fill_stage(0);
        if (getenv("FS_LA_TIMING")) fprintf(stderr, "stage 0: walk %.3f ms, fill %.3f ms, %zu records\n", std::chrono::duration<double, std::milli>(t1 - t0).count(), std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t1).count(), las.size() - stage_begin);
        return ok;
    }
    bool stage0_walk(IterT maxRef) {
        is_valid = false;
        stages.assign(MaxLAStages, WireStage<IterT>{0, 0});
        use_at = false;
        stage_count = 0;
        stages[0].LAIndex = 0;
        IterT Period = 0;
        // isZCoeffZero() of the first step needs the coefficient itself
        if (N::c_is_zero(la_step(la_new(N::c_zero()), orbit_at(1)).ZCoeff)) return false;
        LAx la = x_step(x_new_zero(), 1);
        IterT nextIdx = 0;
        IterT i;
        for (i = 2; i < maxRef; i++) {
            LAx nl;
            if (!x_step(la, nl, i)) { la = nl; continue; }
            Period = i;
            la.StepLength = Period; la.NextStageLAIndex = nextIdx;
            x_push(la);
            nextIdx = i;
            if (i + 1 < maxRef) { la = x_step(x_new_at(i), i + 1); i += 2; }
            else { la = x_new_at(i); i += 1; }
            break;
        }
        stage_count = 1;
        IterT PeriodBegin = Period, PeriodEnd = PeriodBegin + Period;
        if (Period == 0) {
            if (maxRef > (IterT)lowBound) {
                la = x_step(x_new_at(0), 1);
                nextIdx = 0;
                i = 2;
                Period = nth_root_period((double)maxRef, (double)maxRef);
                PeriodBegin = 0;
                PeriodEnd = Period;
            } else {
                la.StepLength = maxRef; la.NextStageLAIndex = nextIdx;
                x_push(la);
                x_push_done(la_new(orbit_at(maxRef)));
                stages[0].MacroItCount = 1;
                return false;
            }
        } else if (Period > (IterT)lowBound) {
            x_pop();
            la = x_step(x_new_at(0), 1);
            nextIdx = 0;
            i = 2;
            Period = nth_root_period((double)maxRef, (double)maxRef);
            PeriodBegin = 0;
            PeriodEnd = Period;
        }
        for (; i < maxRef; i++) {
            LAx nl;
            const bool det = x_step(la, nl, i);
            if (!det && i < PeriodEnd) { la = nl; continue; }
            la.StepLength = i - PeriodBegin; la.NextStageLAIndex = nextIdx;
            x_push(la);
            nextIdx = i;
            PeriodBegin = i;
            PeriodEnd = PeriodBegin + Period;
            const IterT ip1 = i + 1;
            const bool detected = x_detect(nl, chebs[ip1]);
            if (detected || ip1 >= maxRef) {
                la = x_new_at(i);
            } else {
                la = x_step(x_new_at(i), ip1);
                i++;
            }
        }
        la.StepLength = i - PeriodBegin; la.NextStageLAIndex = nextIdx;
        x_push(la);
        stages[0].MacroItCount = (IterT)las.size();
        LA la2 = la_new(orbit_at(maxRef));
        la2.StepLength = 0; la2.NextStageLAIndex = 0;
        x_push_done(la2);
        return true;
    }

    // CreateNewLAStage  LAReference.cpp:774-968
    bool next_stage(IterT maxRef) {
        if (stage_count >= (IterT)MaxLAStages) return false;
        notes.clear();
        stage_begin = las.size();
        las.reserve(las.size() + (size_t)stages[stage_count - 1].MacroItCount + 4); // references into `las` stay valid
        const IterT prev_idx = stages[stage_count - 1].LAIndex;
        const auto t0 = std::chrono::steady_clock::now();
        const bool ok = next_stage_walk(maxRef);
        const auto t1 = std::chrono::steady_clock::now();
        fill_stage(prev_idx);
        if (getenv("FS_LA_TIMING")) fprintf(stderr, "stage %d: walk %.3f ms, fill %.3f ms, %zu records\n", (int)stage_count - 1, std::chrono::duration<double, std::milli>(t1 - t0).count(), std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t1).count(), las.size() - stage_begin);
        return ok;
    }
    bool next_stage_walk(IterT maxRef) {
        const IterT PrevStage = stage_count - 1, CurrentStage = stage_count;
        const IterT PrevIdx = stages[PrevStage].LAIndex;
        const IterT PrevCount = stages[PrevStage].MacroItCount;
        const LA PrevLA = las[PrevIdx];
        const LA PrevLAp1 = las[PrevIdx + 1];
        IterT Period = 0;
        stages[CurrentStage].LAIndex = (IterT)las.size();
        LAx la = x_comp(x_copy_prev(PrevIdx, 0), PrevLAp1);
        IterT nextIdx = 0;
        IterT i = PrevLA.StepLength + PrevLAp1.StepLength;
        IterT j;
        for (j = 2; j < PrevCount; j++) {
            LAx nl;
            const LA &Pj = las[PrevIdx + j];
            const bool det = x_comp(la, nl, Pj);
            if (det) {
                if (N::r_is_zero(Pj.LAThreshold)) break;
                Period = i;
                la.StepLength = Period; la.NextStageLAIndex = nextIdx;
                x_push(la);
                nextIdx = j;
                const LA &Pjp1 = las[PrevIdx + j + 1];
                if (x_detect(nl, N::c_cheb(Pjp1.Ref)) || j + 1 >= PrevCount) {
                    la = x_copy_prev(PrevIdx, j);
                    i += Pj.StepLength;
                    j++;
                } else {
                    la = x_comp(x_copy_prev(PrevIdx, j), Pjp1);
                    i += Pj.StepLength + Pjp1.StepLength;
                    j += 2;
                }
                break;
            }
            la = nl;
            i += las[PrevIdx + j].StepLength;
        }
        stage_count++;
        IterT PeriodBegin = Period, PeriodEnd = PeriodBegin + Period;
        if (Period == 0) {
            if (maxRef > PrevLA.StepLength * (IterT)lowBound) {
                la = x_comp(x_copy_prev(PrevIdx, 0), PrevLAp1);
                i = PrevLA.StepLength + PrevLAp1.StepLength;
                nextIdx = 0;
                j = 2;
                const double Ratio = (double)maxRef / (double)PrevLA.StepLength;
                Period = PrevLA.StepLength * nth_root_period((double)maxRef, Ratio);
                PeriodBegin = 0;
                PeriodEnd = Period;
            } else {
                la.StepLength = maxRef; la.NextStageLAIndex = nextIdx;
                x_push(la);
                LA la2 = la_new(orbit_at(maxRef));
                la2.StepLength = 0; la2.NextStageLAIndex = 0;
                x_push_done(la2);
                stages[CurrentStage].MacroItCount = 1;
                return false;
            }
        } else if (Period > PrevLA.StepLength * (IterT)lowBound) {
            x_pop();
            la = x_comp(x_copy_prev(PrevIdx, 0), PrevLAp1);
            i = PrevLA.StepLength + PrevLAp1.StepLength;
            nextIdx = 0;
            j = 2;
            const double Ratio = (double)Period / (double)PrevLA.StepLength;
            Period = PrevLA.StepLength * nth_root_period((double)maxRef, Ratio);
            PeriodBegin = 0;
            PeriodEnd = Period;
        }
        for (; j < PrevCount; j++) {
            LAx nl;
            const LA &Pj = las[PrevIdx + j];
            const bool det = x_comp(la, nl, Pj);
            if (det || i >= PeriodEnd) {
                la.StepLength = i - PeriodBegin; la.NextStageLAIndex = nextIdx;
                x_push(la);
                nextIdx = j;
                PeriodBegin = i;
                PeriodEnd = PeriodBegin + Period;
                const LA &Pjp1 = las[PrevIdx + j + 1];
                if (x_detect(nl, N::c_cheb(Pjp1.Ref)) || j + 1 >= PrevCount) {
                    la = x_copy_prev(PrevIdx, j);
                } else {
                    la = x_comp(x_copy_prev(PrevIdx, j), Pjp1);
                    i += las[PrevIdx + j].StepLength;
                    j++;
                }
            } else {
                la = nl;
            }
            i += las[PrevIdx + j].StepLength;
        }
        la.StepLength = i - PeriodBegin; la.NextStageLAIndex = nextIdx;
        x_push(la);
        stages[CurrentStage].MacroItCount = (IterT)las.size() - stages[CurrentStage].LAIndex;
        LA la2 = la_new(orbit_at(maxRef));
        la2.StepLength = 0; la2.NextStageLAIndex = 0;
        x_push_done(la2);
        return true;
    }


    // ---- pipelined construction -------------------------------------------------------------------------------------
    // The walk of stage k + 1 reads three things of a stage-k record: |Ref| (Chebyshev norm), MinMag and StepLength -- all
    // of them products of stage k's own walk -- plus, once per stage, "is LAThreshold of this record zero"
    // (LAReference.cpp:829-833), which only the fill knows.  So the walks of all stages run at the same time, each one or
    // two records behind the walk below it (one thread per stage, records handed over through a published count), on
    // slim records {MinMag, |Ref|, StepLength, NextStage, note}; the one LAThreshold question is answered "not zero" on
    // the spot and checked when the fills are done (zero: the table is rebuilt by the stage-after-stage path above).
    // Stage 0's records are filled by the remaining threads while its walk is still going.  Same walk, same notes, same
    // fill calls as the two-phase form: same bytes (tests/test_table_construction.py runs both against the reference).
    struct Slim { Real MinMag, chebRef; IterT StepLength, NextStage; Note n; };
    static constexpr size_t kMaxPipelinedStages = 12;
    // (the words other threads poll sit on cache lines of their own: a store to a line that a dozen cores are reading costs
    // the storing core a coherence round trip each time -- with one line for everything and a publish per record the
    // pipelined build took 6 ms where the stage-after-stage one takes 2)
    struct alignas(64) Walk {
        alignas(64) std::atomic<size_t> pub{0}; // rec[0 .. pub) are final (regular records: a further record follows each)
        alignas(64) std::atomic<int> follow{0}; // 0 undecided, 1 a next stage follows this one, 2 this is the last stage
        std::atomic<int> done{0};               // 1: rec[0 .. count] complete (count regular records and the closing one)
        alignas(64) std::atomic<size_t> fill_next{0}; // first record no thread has claimed for filling yet
        alignas(64) Slim *rec = nullptr;
        LA *out = nullptr;                    // where this stage's filled records go
        std::atomic<uint32_t> *stamp = nullptr;
        size_t count = 0, n_rec = 0; // MacroItCount; records in rec[] (count regular ones and the closing one)
        size_t cap = 0;              // room in rec[] / out[]
        bool overflowed = false;     // the stage has more records than room was set aside for: the build is redone stage after stage
        long long spec = -1;         // previous-stage record whose LAThreshold the walk took to be non-zero
        bool ran = false, ok = false;
        double t_begin = 0, t_end = 0; // FS_LA_TIMING: the walk's start and end, ms after the build's start
    };
    // The walks' record arrays live as long as the process: a fresh 4 MB allocation per stage and build is a page fault per
    // 4 KB written (0.5 ms of a 1 ms walk on the 16-core box, more than the walk's arithmetic).  One build at a time.
    static constexpr size_t kFillChunk = 16; // records per fill claim
    struct Scratch {
        std::mutex mu;
        Slim *rec[kMaxPipelinedStages] = {};
        LA *out[kMaxPipelinedStages] = {};                      // filled records of stages 1 ... (stage 0 goes straight to `las`)
        std::atomic<uint32_t> *stamp[kMaxPipelinedStages] = {}; // per fill chunk: the number of the build that completed it
        size_t cap[kMaxPipelinedStages] = {};
        uint32_t build_no = 0;
        void get(size_t k, size_t n) {
            if (cap[k] >= n) return;
            free(rec[k]);
            free(out[k]);
            free(stamp[k]);
            cap[k] = 0;
            rec[k] = static_cast<Slim *>(malloc(n * sizeof(Slim)));
            out[k] = k == 0 ? nullptr : static_cast<LA *>(malloc(n * sizeof(LA)));
            stamp[k] = static_cast<std::atomic<uint32_t> *>(calloc(n / kFillChunk + 2, sizeof(std::atomic<uint32_t>)));
            if (!rec[k] || (k != 0 && !out[k]) || !stamp[k]) throw std::bad_alloc();
            cap[k] = n;
        }
        ~Scratch() { for (size_t k = 0; k < kMaxPipelinedStages; k++) { free(rec[k]); free(out[k]); free(stamp[k]); } }
    };
    static Scratch &scratch() { static Scratch s; return s; }
    // waiting for another thread's progress: a few pauses, then yields (with fewer cores than threads the thread being
    // waited for must get the core)
    struct Backoff {
        int n = 0;
        void operator()() {
#if defined(__x86_64__) || defined(__i386__)
            if (n < 64) { n++; __builtin_ia32_pause(); return; }
#endif
            std::this_thread::yield();
        }
    };
    // the walk of the stage above P, as a reader of P's records
    struct Reader {
        const Walk &P;
        size_t seen = 0; // last value of P.pub this thread has loaded
        // may previous-stage index j be evaluated (reads records j and j + 1)?  false: j >= P.count
        bool have(size_t j) {
            if (seen >= j + 2) return true;
            Backoff relax;
            for (;;) {
                seen = P.pub.load(std::memory_order_acquire);
                if (seen >= j + 2) return true;
                if (P.done.load(std::memory_order_acquire)) { seen = P.pub.load(std::memory_order_acquire); return j < P.count; }
                relax();
            }
        }
        // j + 1 >= PrevCount, for a j that `have` has admitted
        bool is_last(size_t j) const {
            if (seen >= j + 2) return false;
            return j + 1 >= P.count; // admitted without the published count reaching it: P is done
        }
    };
    struct Emit {
        Walk &w;
        size_t n = 0;
        size_t batch = 1, told = 0; // records per publish
        void push(const LAx &a) {
            if (n + 2 > w.cap) { w.overflowed = true; return; } // (room for the closing record stays)
            w.rec[n++] = Slim{a.MinMag, a.chebRef, a.StepLength, a.NextStageLAIndex, a.n};
        }
        void pop() { if (n) n--; }
        void publish() {
            if (n - told < batch) return;
            told = n;
            w.pub.store(n, std::memory_order_release);
        }
        void close(Real cheb_last, bool ok) { // the closing record LAInfoDeep(orbit[maxRef]) with StepLength 0
            w.count = n;
            w.rec[n] = Slim{N::r_int(4), cheb_last, 0, 0, Note{3, 0, 0}};
            w.n_rec = n + 1;
            w.ok = ok;
            w.pub.store(n, std::memory_order_release);
            w.done.store(1, std::memory_order_release);
        }
    };
    LAx xs_copy(const Walk &Pv, IterT j) const { return LAx{Pv.rec[j].MinMag, Note{1, j, 0}, 0, 0, Pv.rec[j].chebRef}; }
    bool xs_comp(const LAx &a, LAx &out, const Slim &b) const { // x_comp on a slim record
        out.n = Note{a.n.kind, a.n.first, a.n.count + 1};
        out.chebRef = a.chebRef;
        const Real temp = N::r_min(b.chebRef, a.MinMag);
        out.MinMag = N::r_min(temp, b.MinMag);
        return N::r_cmp(temp, N::r_scale_by(a.MinMag, thr_detect)) < 0;
    }
    LAx xs_comp(const LAx &a, const Slim &b) const { LAx r = a; xs_comp(a, r, b); return r; }

    // stage0_walk on slim records
    void p_stage0(Walk &W, IterT maxRef) {
        W.ran = true;
        Emit E{W};
        E.batch = 128; // a publish is a store to a line a dozen threads poll: rarely
        IterT Period = 0;
        if (N::c_is_zero(la_step(la_new(N::c_zero()), orbit_at(1)).ZCoeff)) {
            W.follow.store(2, std::memory_order_release);
            W.count = 0;
            W.ok = false;
            W.done.store(1, std::memory_order_release);
            return;
        }
        LAx la = x_step(x_new_zero(), 1);
        IterT nextIdx = 0;
        IterT i;
        for (i = 2; i < maxRef; i++) {
            LAx nl;
            if (!x_step(la, nl, i)) { la = nl; continue; }
            Period = i;
            la.StepLength = Period; la.NextStageLAIndex = nextIdx;
            E.push(la);
            nextIdx = i;
            if (i + 1 < maxRef) { la = x_step(x_new_at(i), i + 1); i += 2; }
            else { la = x_new_at(i); i += 1; }
            break;
        }
        IterT PeriodBegin = Period, PeriodEnd = PeriodBegin + Period;
        if (Period == 0) {
            if (maxRef > (IterT)lowBound) {
                la = x_step(x_new_at(0), 1);
                nextIdx = 0;
                i = 2;
                Period = nth_root_period((double)maxRef, (double)maxRef);
                PeriodBegin = 0;
                PeriodEnd = Period;
            } else {
                la.StepLength = maxRef; la.NextStageLAIndex = nextIdx;
                E.push(la);
                W.follow.store(2, std::memory_order_release);
                E.close(chebs[maxRef], false); // MacroItCount 1: this record and the closing one
                return;
            }
        } else if (Period > (IterT)lowBound) {
            E.pop();
            la = x_step(x_new_at(0), 1);
            nextIdx = 0;
            i = 2;
            Period = nth_root_period((double)maxRef, (double)maxRef);
            PeriodBegin = 0;
            PeriodEnd = Period;
        }
        W.follow.store(1, std::memory_order_release); // nothing pushed from here on is taken back
        // x_step(la, nl, i) for every element, written so that an element which neither lowers MinMag nor ends the period
        // costs one comparison: the right-hand side of the period test, MinMag * threshold, and the test's outcome for an
        // unchanged MinMag stand until MinMag changes.  Same comparisons on the same values, hence the same decisions.
        const Real four = N::r_int(4); // LAInfoDeep(z): MinMag = 4
        Real T = N::r_scale_by(la.MinMag, thr_stage0);
        bool self_det = N::r_cmp(la.MinMag, T) < 0;
        for (; i < maxRef; i++) {
            const Real c = chebs[i];
            const bool lower = N::r_cmp(c, la.MinMag) < 0; // r_min(c, MinMag): c if it compares less, MinMag otherwise
            const bool det = lower ? N::r_cmp(c, T) < 0 : self_det;
            if (!det && i < PeriodEnd) {
                la.n.count++;
                if (lower) {
                    la.MinMag = c;
                    T = N::r_scale_by(c, thr_stage0);
                    self_det = N::r_cmp(c, T) < 0;
                }
                continue;
            }
            LAx nl = la; // the record with this element, which only the look-ahead below reads
            nl.n.count++;
            if (lower) nl.MinMag = c;
            la.StepLength = i - PeriodBegin; la.NextStageLAIndex = nextIdx;
            E.push(la);
            E.publish();
            nextIdx = i;
            PeriodBegin = i;
            PeriodEnd = PeriodBegin + Period;
            const IterT ip1 = i + 1;
            const bool detected = x_detect(nl, chebs[ip1]);
            if (detected || ip1 >= maxRef) {
                la = x_new_at(i);
            } else {
                // x_step(x_new_at(i), ip1), whose period test nobody reads
                la = LAx{N::r_min(chebs[ip1], four), Note{0, i, 1}, 0, 0, chebs[i]};
                i++;
            }
            T = N::r_scale_by(la.MinMag, thr_stage0);
            self_det = N::r_cmp(la.MinMag, T) < 0;
        }
        la.StepLength = i - PeriodBegin; la.NextStageLAIndex = nextIdx;
        E.push(la);
        E.close(chebs[maxRef], true);
    }

    // next_stage_walk on slim records; Pv = the stage below, possibly still being walked
    void p_next(const Walk &Pv, Walk &W, IterT maxRef, bool may_follow) {
        W.ran = true;
        Emit E{W};
        E.batch = 4;
        Reader R{Pv};
        R.have(0); // records 0 and 1 (a stage that is followed has at least one regular record and its closing one)
        const Slim PrevLA = Pv.rec[0], PrevLAp1 = Pv.rec[1];
        IterT Period = 0;
        LAx la = xs_comp(xs_copy(Pv, 0), PrevLAp1);
        IterT nextIdx = 0;
        IterT i = PrevLA.StepLength + PrevLAp1.StepLength;
        IterT j;
        for (j = 2; R.have(j); j++) {
            LAx nl;
            const Slim &Pj = Pv.rec[j];
            const bool det = xs_comp(la, nl, Pj);
            if (det) {
                W.spec = (long long)j; // `if (Pj.LAThreshold == 0) break;` -- taken to be non-zero, checked after the fills
                Period = i;
                la.StepLength = Period; la.NextStageLAIndex = nextIdx;
                E.push(la);
                nextIdx = j;
                const Slim &Pjp1 = Pv.rec[j + 1];
                if (x_detect(nl, Pjp1.chebRef) || R.is_last(j)) {
                    la = xs_copy(Pv, j);
                    i += Pj.StepLength;
                    j++;
                } else {
                    la = xs_comp(xs_copy(Pv, j), Pjp1);
                    i += Pj.StepLength + Pjp1.StepLength;
                    j += 2;
                }
                break;
            }
            la = nl;
            i += Pj.StepLength;
        }
        IterT PeriodBegin = Period, PeriodEnd = PeriodBegin + Period;
        if (Period == 0) {
            if (maxRef > PrevLA.StepLength * (IterT)lowBound) {
                la = xs_comp(xs_copy(Pv, 0), PrevLAp1);
                i = PrevLA.StepLength + PrevLAp1.StepLength;
                nextIdx = 0;
                j = 2;
                const double Ratio = (double)maxRef / (double)PrevLA.StepLength;
                Period = PrevLA.StepLength * nth_root_period((double)maxRef, Ratio);
                PeriodBegin = 0;
                PeriodEnd = Period;
            } else {
                la.StepLength = maxRef; la.NextStageLAIndex = nextIdx;
                E.push(la);
                W.follow.store(2, std::memory_order_release);
                E.close(chebs[maxRef], false);
                return;
            }
        } else if (Period > PrevLA.StepLength * (IterT)lowBound) {
            E.pop();
            la = xs_comp(xs_copy(Pv, 0), PrevLAp1);
            i = PrevLA.StepLength + PrevLAp1.StepLength;
            nextIdx = 0;
            j = 2;
            const double Ratio = (double)Period / (double)PrevLA.StepLength;
            Period = PrevLA.StepLength * nth_root_period((double)maxRef, Ratio);
            PeriodBegin = 0;
            PeriodEnd = Period;
        }
        W.follow.store(may_follow ? 1 : 2, std::memory_order_release);
        for (; R.have(j); j++) {
            LAx nl;
            const Slim &Pj = Pv.rec[j];
            const bool det = xs_comp(la, nl, Pj);
            if (det || i >= PeriodEnd) {
                la.StepLength = i - PeriodBegin; la.NextStageLAIndex = nextIdx;
                E.push(la);
                E.publish();
                nextIdx = j;
                PeriodBegin = i;
                PeriodEnd = PeriodBegin + Period;
                const Slim &Pjp1 = Pv.rec[j + 1];
                if (x_detect(nl, Pjp1.chebRef) || R.is_last(j)) {
                    la = xs_copy(Pv, j);
                } else {
                    la = xs_comp(xs_copy(Pv, j), Pjp1);
                    i += Pv.rec[j].StepLength;
                    j++;
                }
            } else {
                la = nl;
            }
            i += Pv.rec[j].StepLength;
        }
        la.StepLength = i - PeriodBegin; la.NextStageLAIndex = nextIdx;
        E.push(la);
        E.close(chebs[maxRef], true);
    }

    // one record from its note (phase 2 of the two-phase form, for one record); prev = the previous stage's first record
    void fill_one(LA &dst, const Slim &r, const LA *prev, IterT maxRef) const {
        const Note nt = r.n;
        LA l;
        if (nt.kind == 3) l = la_new(orbit_at(maxRef));
        else if (nt.kind == 1) l = prev[nt.first];
        else l = la_new(nt.kind == 2 ? N::c_zero() : orbit_at(nt.first));
        for (IterT c = 1; c <= nt.count; c++) {
            LA nl = la_blank();
            if (nt.kind == 1) la_comp(l, nl, prev[(size_t)nt.first + c]);
            else la_step(l, nl, orbit_at((nt.kind == 2 ? (IterT)0 : nt.first) + c));
            l = nl;
        }
        l.StepLength = r.StepLength;
        l.NextStageLAIndex = r.NextStage;
        dst = l;
    }

    // false: not applicable here (more stages than walkers) or the LAThreshold assumption failed -- build stage after stage
    bool build_pipelined(IterT maxRef) {
        thr_stage0 = N::r_scale_pre(P.stage0_thr2);
        thr_detect = N::r_scale_pre(P.thr2);
        chebs.resize((size_t)maxRef + 1);
        parallel_for(chebs.size(), [&](size_t lo, size_t hi) { for (size_t k = lo; k < hi; k++) chebs[k] = N::c_cheb(orbit_at(k)); });
        const auto t0 = std::chrono::steady_clock::now();
        std::unique_ptr<Walk[]> W(new Walk[kMaxPipelinedStages]);
        const size_t cap = (size_t)maxRef + 4; // no stage has more records than the orbit has elements
        Scratch &scr = scratch();
        std::lock_guard<std::mutex> one_build(scr.mu);
        const uint32_t build_no = ++scr.build_no == 0 ? ++scr.build_no : scr.build_no;
        las.clear();
        las.reserve(cap + cap / 2);
        for (size_t k = 0; k < kMaxPipelinedStages; k++) {
            // a stage is a fraction of the one below it (View 14: 31,219 / 1,827 / 782 / 14 / 2 records); should one outgrow
            // half of it, the walk notes it and the table is built stage after stage instead
            size_t cap_k = (cap >> std::min<size_t>(k, 20)) + 1024;
            if (k > 0 && getenv("FS_LA_TEST_SMALL_STAGES")) cap_k = std::min<size_t>(cap_k, 64); // test hook: forces the overflow path
            scr.get(k, cap_k);
            W[k].cap = cap_k;
            W[k].rec = scr.rec[k];
            W[k].out = k == 0 ? las.data() : scr.out[k]; // stage 0's place in `las` is its beginning whatever follows
            W[k].stamp = scr.stamp[k];
        }
        std::atomic<bool> overflow{false};
        std::atomic<int> walks_done{0}; // set by the walk of the last stage (the walks below it have ended before)
        // Filling runs behind the walks, on every thread that is not walking: records are claimed in chunks, stage 0 first.
        // A record of stage k > 0 is a chain of composites over filled records of stage k - 1; whoever fills it makes sure
        // those are complete, by filling lower stages itself while it waits (so the wait always ends: stage 0 waits for
        // nothing).  try_fill(k): fill one chunk of stage k if one can be claimed; false: none right now.
        std::function<bool(size_t)> try_fill = [&](size_t k) -> bool {
            Walk &S = W[k];
            for (;;) {
                size_t a = S.fill_next.load(std::memory_order_relaxed);
                const bool ended = S.done.load(std::memory_order_acquire) != 0;
                const size_t avail = ended ? S.n_rec : S.pub.load(std::memory_order_acquire);
                if (a >= avail) return false;
                size_t b = a + kFillChunk;
                if (b > avail) {
                    if (!ended) return false; // chunks stay aligned: a partial one only at the stage's end
                    b = avail;
                }
                if (!S.fill_next.compare_exchange_weak(a, a + kFillChunk, std::memory_order_relaxed)) continue;
                const LA *prev = k == 0 ? nullptr : W[k - 1].out;
                for (size_t r = a; r < b; r++) {
                    const Note nt = S.rec[r].n;
                    if (nt.kind == 1) {
                        const std::atomic<uint32_t> *st = W[k - 1].stamp;
                        for (size_t c = (size_t)nt.first / kFillChunk; c <= ((size_t)nt.first + nt.count) / kFillChunk; c++) {
                            Backoff relax;
                            while (st[c].load(std::memory_order_acquire) != build_no) {
                                bool helped = false;
                                for (size_t below = 0; below < k && !helped; below++) helped = try_fill(below);
                                if (!helped) relax();
                            }
                        }
                    }
                    fill_one(S.out[r], S.rec[r], prev, maxRef);
                }
                S.stamp[a / kFillChunk].store(build_no, std::memory_order_release);
                return true;
            }
        };
        auto try_any = [&]() -> bool {
            for (size_t k = 0; k < kMaxPipelinedStages; k++)
                if (try_fill(k)) return true; // (a stage that does not exist never has anything published)
            return false;
        };
        auto task = [&](size_t k, size_t) {
            Backoff relax;
            auto now = [&] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); };
            if (k == 0) {
                W[0].t_begin = now();
                p_stage0(W[0], maxRef);
                W[0].t_end = now();
                if (W[0].follow.load() == 2) walks_done.store(1, std::memory_order_release);
            } else if (k < kMaxPipelinedStages) {
                Walk &Pv = W[k - 1];
                // whether this stage exists is known once the stage below is past its first period; until then, help
                while (Pv.follow.load(std::memory_order_acquire) == 0) {
                    if (!try_any()) relax();
                }
                if (Pv.follow.load(std::memory_order_acquire) == 1) {
                    const bool may_follow = k + 1 < (size_t)MaxLAStages;
                    W[k].t_begin = now();
                    p_next(Pv, W[k], maxRef, may_follow);
                    W[k].t_end = now();
                    if (W[k].follow.load() == 2) walks_done.store(1, std::memory_order_release);
                    else if (k + 1 == kMaxPipelinedStages) { overflow.store(true); walks_done.store(1, std::memory_order_release); }
                } else {
                    W[k].follow.store(2, std::memory_order_release);
                }
            }
            // Only a task behind the walkers' may wait for the walks to end: tasks are claimed in order, so by then every
            // walker has been claimed and runs (or has run) on some thread.  A walker that waited here with fewer threads
            // than stages would wait for a walk nobody has started.
            if (k >= kMaxPipelinedStages) {
                while (!walks_done.load(std::memory_order_acquire)) {
                    if (!try_any()) relax();
                }
            }
            while (try_any()) {}
        };
        HostPool::get().run_tasks(kMaxPipelinedStages + HostPool::get().threads(), task);
        const auto t1 = std::chrono::steady_clock::now();
        if (overflow.load()) return false;
        for (size_t k = 0; k < kMaxPipelinedStages; k++)
            if (W[k].overflowed) return false;
        stages.assign(MaxLAStages, WireStage<IterT>{0, 0});
        use_at = false;
        is_valid = false;
        walk_ok = W[0].ok;
        if (W[0].n_rec == 0) { // the first step's ZCoeff is zero: no table at all (stage0_walk's first return)
            las.clear();
            stage_count = 0;
            return true;
        }
        // the stages one behind the other: stage 0 is in place, the others come from their own arrays
        size_t n_stages = 0, total = 0;
        while (n_stages < kMaxPipelinedStages && W[n_stages].ran) { total += W[n_stages].n_rec; n_stages++; }
        las.resize_uninit(W[0].n_rec);
        las.resize_uninit(total);
        size_t off = 0;
        for (size_t k = 0; k < n_stages; k++) {
            const Walk &S = W[k];
            stages[k].LAIndex = (IterT)off;
            stages[k].MacroItCount = (IterT)S.count;
            if (k > 0) {
                if (S.spec >= 0 && N::r_is_zero(W[k - 1].out[(size_t)S.spec].LAThreshold)) return false;
                memcpy(static_cast<void *>(las.data() + off), S.out, S.n_rec * sizeof(LA));
            }
            off += S.n_rec;
        }
        stage_count = (IterT)n_stages;
        if (getenv("FS_LA_TIMING")) {
            fprintf(stderr, "pipelined: walks and fills %.3f ms, layout %.3f ms, %zu stages, %zu records;",
                    std::chrono::duration<double, std::milli>(t1 - t0).count(),
                    std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t1).count(), n_stages, total);
            for (size_t k = 0; k < n_stages; k++) fprintf(stderr, " walk %zu: %.3f-%.3f ms (%zu)", k, W[k].t_begin, W[k].t_end, W[k].n_rec);
            fprintf(stderr, "\n");
        }
        return true;
    }
    bool walk_ok = false; // stage 0's walk returned true (a table with an AT block and is_valid follow)

    // LAInfoDeep::CreateAT  LAInfoDeep.h:456-502 ; ATInfo::Usable  ATInfo.h:92-106
    void create_at(const LA &a, const LA &next, bool small_exp) {
        at.ZCoeff = a.ZCoeff;
        at.CCoeff = N::c_mul(a.ZCoeff, a.CCoeff);
        N::c_reduce(at.CCoeff);
        at.InvZCoeff = N::c_recip(a.ZCoeff);
        N::c_reduce(at.InvZCoeff);
        at.CCoeffSqrInvZCoeff = N::c_mul(N::c_mul(at.CCoeff, at.CCoeff), at.InvZCoeff);
        N::c_reduce(at.CCoeffSqrInvZCoeff);
        at.CCoeffInvZCoeff = N::c_mul(at.CCoeff, at.InvZCoeff);
        N::c_reduce(at.CCoeffInvZCoeff);
        at.RefC = N::c_mul(next.Ref, a.ZCoeff);
        N::c_reduce(at.RefC);
        at.CCoeffNormSqr = N::c_norm2(at.CCoeff);
        N::r_reduce(at.CCoeffNormSqr);
        at.RefCNormSqr = N::c_norm2(at.RefC);
        N::r_reduce(at.RefCNormSqr);
        const Real lim = N::at_lim(small_exp);
        at.SqrEscapeRadius = N::r_min(N::r_mul(N::c_norm2(a.ZCoeff), a.LAThreshold), lim);
        N::r_reduce(at.SqrEscapeRadius);
        at.ThresholdC = N::r_min(a.LAThresholdC, N::r_div(lim, N::c_cheb(at.CCoeff)));
    }
    bool at_usable(Real sqr_radius) const {
        Real result = N::r_mul(N::r_mul(at.CCoeffNormSqr, sqr_radius), at.factor);
        N::r_reduce(result);
        return N::r_cmp(result, at.RefCNormSqr) > 0 && N::r_cmp(at.SqrEscapeRadius, N::at_four()) > 0;
    }

    // GenerateApproximationData  LAReference.cpp:971-1017 ; CreateATFromLA :1050-1074
    void build() {
        memset(&at, 0, sizeof(at));
        at.factor = N::at_factor();
        const IterT maxRef = (IterT)orbit->count - 1;
        if (maxRef == 0) { is_valid = false; return; }
        // FS_LA_PIPELINE=0: the stage-after-stage (two-phase) form only
        const char *pe = getenv("FS_LA_PIPELINE");
        const bool pipeline_off = pe && atoi(pe) == 0;
        bool ok;
        bool pipelined = false;
        if (!pipeline_off) {
            try {
                pipelined = build_pipelined(maxRef);
            } catch (const std::bad_alloc &) {
                pipelined = false; // no room for the walks' arrays: the stage-after-stage form needs a fraction of it
            }
        }
        if (pipelined) {
            ok = walk_ok;
        } else {
            las.clear();
            ok = stage0(maxRef);
            if (ok) while (next_stage(maxRef)) {}
        }
        if (ok) {
            Real radius;
            memcpy(&radius, orbit->max_radius, sizeof(radius));
            const Real sqr_radius = N::r_square_reduced(radius);
            use_at = false;
            for (IterT s = stage_count; s > 0;) {
                s--;
                const IterT idx = stages[s].LAIndex;
                create_at(las[idx], las[idx + 1], small_exp);
                at.StepLength = las[idx].StepLength;
                if (at.StepLength > 0 && at_usable(sqr_radius)) { use_at = true; break; }
            }
            is_valid = true;
        }
        // Trim(): stages keep MaxLAStages entries in the reference only until trimmed to the used count
        stages.resize(std::max<size_t>((size_t)stage_count, 1));
    }
};

// --------------------------------------------------------------------------------------------
// 2x32 types: orbit, LA table and AT are computed in double / HDR-double and converted element-wise
// (RefOrbitCalc.cpp:2490-2516, PerturbationResults.cpp:241-348, DoubleTo2x32Converter HDRFloat.h:1739-1762).
// --------------------------------------------------------------------------------------------
// MattDblflt(double)  dblflt.h:38-52: split + two-sum renormalisation
df32 h_df_from_double(double d) {
    const float a = (float)d;
    const float b = (float)(d - (double)a);
    df32 z;
    z.head = a + b;
    float t1 = z.head - a;
    float t2 = z.head - t1;
    t1 = b - t1;
    t2 = a - t2;
    z.tail = t1 + t2;
    return z;
}
df32 to_df(double v) { return h_df_from_double(v); }
Hdr<df32> to_df(Hdr<double> v) { Hdr<df32> r; r.m = h_df_from_double(v.m); r.e = v.e; return r; }            // HDRFloat(const HDRFloat<SrcT>&)
Cx<df32> to_df(Cx<double> v) { Cx<df32> r; r.re = h_df_from_double(v.re); r.im = h_df_from_double(v.im); return r; }
HdrC<df32> to_df(HdrC<double> v) { HdrC<df32> r; r.re = h_df_from_double(v.re); r.im = h_df_from_double(v.im); r.e = v.e; return r; }

struct HostDf { using Real = df32; using Cplx = Cx<df32>; };          // T = CudaDblflt<MattDblflt>
struct HostHdrDf { using Real = Hdr<df32>; using Cplx = HdrC<df32>; }; // T = HDRFloat<CudaDblflt<MattDblflt>>
static_assert(sizeof(WireLA<HostDf, uint32_t>) == 80 && sizeof(WireLA<HostDf, uint64_t>) == 88, "LAInfoDeep 2x32");
static_assert(sizeof(WireLA<HostHdrDf, uint32_t>) == 104 && sizeof(WireLA<HostHdrDf, uint64_t>) == 112, "LAInfoDeep HDRx2x32");
static_assert(sizeof(WireAT<HostDf, uint32_t>) == 140 && sizeof(WireAT<HostHdrDf, uint64_t>) == 192, "ATInfo 2x32");

template <class ND, class NS, class IterT> WireLA<ND, IterT> convert_la_rec(const WireLA<NS, IterT> &s) {
    WireLA<ND, IterT> d;
    memset(&d, 0, sizeof(d));
    d.Ref = to_df(s.Ref); d.ZCoeff = to_df(s.ZCoeff); d.CCoeff = to_df(s.CCoeff);
    d.LAThreshold = to_df(s.LAThreshold); d.LAThresholdC = to_df(s.LAThresholdC); d.MinMag = to_df(s.MinMag);
    d.StepLength = s.StepLength; d.NextStageLAIndex = s.NextStageLAIndex;
    return d;
}
template <class ND, class NS, class IterT> WireAT<ND, IterT> convert_at(const WireAT<NS, IterT> &s) {
    WireAT<ND, IterT> d;
    memset(&d, 0, sizeof(d));
    d.StepLength = s.StepLength;
    d.ThresholdC = to_df(s.ThresholdC); d.SqrEscapeRadius = to_df(s.SqrEscapeRadius);
    d.RefC = to_df(s.RefC); d.ZCoeff = to_df(s.ZCoeff); d.CCoeff = to_df(s.CCoeff); d.InvZCoeff = to_df(s.InvZCoeff);
    d.CCoeffSqrInvZCoeff = to_df(s.CCoeffSqrInvZCoeff); d.CCoeffInvZCoeff = to_df(s.CCoeffInvZCoeff);
    d.CCoeffNormSqr = to_df(s.CCoeffNormSqr); d.RefCNormSqr = to_df(s.RefCNormSqr); d.factor = to_df(s.factor);
    return d;
}

// LA table for a 2x32 target: built on the double-typed base orbit with UseSmallExponents, then converted.
template <class NS, class ND, class IterT> fsh_la *build_la_2x32(const fsh_orbit *base, int period_divisor = 2) {
    LaBuilder<NS, IterT> b;
    b.orbit = base;
    b.periodDivisor = period_divisor;
    b.small_exp = true;
    b.build();
    fsh_la *r = new fsh_la();
    std::vector<WireLA<ND, IterT>> out(b.las.size());
    for (size_t i = 0; i < b.las.size(); i++) out[i] = convert_la_rec<ND, NS, IterT>(b.las[i]);
    r->las.resize(out.size() * sizeof(WireLA<ND, IterT>));
    if (!out.empty()) memcpy(r->las.data(), out.data(), r->las.size());
    r->stages.resize(b.stages.size() * sizeof(b.stages[0]));
    memcpy(r->stages.data(), b.stages.data(), r->stages.size());
    const WireAT<ND, IterT> at = convert_at<ND, NS, IterT>(b.at);
    r->at.resize(sizeof(at));
    memcpy(r->at.data(), &at, sizeof(at));
    r->num_las = b.las.size();
    r->num_stages = b.stages.size();
    r->stage_count = b.stage_count;
    r->use_at = b.use_at;
    r->is_valid = b.is_valid;
    return r;
}

// ---- SimpleCompression ---------------------------------------------------------------------------------------
// One replay step in the low type, host flavour (no contraction: each operator rounds once):
//   zx' = zx*zx - zy*zy + OrbitXLow ; zy' = T{2}*zx_old*zy + OrbitYLow, both HdrReduce'd
template <class N> struct RcHost;
template <class M> struct RcHost<HostPlain<M>> {
    static void step(M &zx, M &zy, M X, M Y) {
        const M a = zx * zx, b = zy * zy, o = zx;
        zx = (a - b) + X;
        zy = ((M(2) * o) * zy) + Y;
    }
    // err = (|z - it|^2) * 10^exp >= |it|^2
    static bool drifted(M zx, M zy, M ix, M iy, M scale) {
        const M ex = zx - ix, ey = zy - iy;
        const M norm = ix * ix + iy * iy;
        const M err = (ex * ex + ey * ey) * scale;
        return err >= norm;
    }
    static M scale(int e) { return (M)pow(10, e); }
};
template <class M> struct RcHost<HostHdr<M>> {
    using R = Hdr<M>;
    static void step(R &zx, R &zy, R X, R Y) {
        const R o = zx;
        zx = add(sub(mul(zx, zx), mul(zy, zy)), X);
        reduce(zx);
        zy = add(mul(mul(hdr_make<M>(1, M(1)), o), zy), Y);
        reduce(zy);
    }
    static bool drifted(R zx, R zy, R ix, R iy, R scale) {
        const R ex = sub(zx, ix), ey = sub(zy, iy);
        R norm = add(mul(ix, ix), mul(iy, iy));
        reduce(norm);
        R err = mul(add(mul(ex, ex), mul(ey, ey)), scale);
        reduce(err);
        return cmp_pr(err, norm) >= 0;
    }
    static R scale(int e) { return hdr_from<M>((M)pow(10, e)); } // static_cast<T>(std::pow(10, exp)): HDRFloat(double)
};

template <class N> fsh_orbit *compress_orbit(const fsh_orbit *src, int32_t error_exp) {
    using Real = typename N::Real;
    using IO = ElemIO<N>;
    using RC = RcHost<N>;
    fsh_orbit *o = new fsh_orbit();
    o->numeric = src->numeric;
    o->pextras = 2;
    o->period = src->period;
    o->elem_bytes = 8 + IO::kBytes;
    o->uncompressed_count = src->count;
    memcpy(o->max_radius, src->max_radius, sizeof(o->max_radius));
    memcpy(o->x_low, src->x_low, sizeof(o->x_low));
    memcpy(o->y_low, src->y_low, sizeof(o->y_low));
    Real X, Y;
    memcpy(&X, src->x_low, sizeof(Real));
    memcpy(&Y, src->y_low, sizeof(Real));
    auto plain = std::make_shared<fsh_orbit>();
    plain->numeric = src->numeric;
    plain->count = src->count;
    plain->period = src->period;
    plain->elem_bytes = IO::kBytes;
    plain->data.assign((size_t)src->count * IO::kBytes, 0);
    memcpy(plain->max_radius, src->max_radius, sizeof(o->max_radius));
    memcpy(plain->x_low, src->x_low, sizeof(o->x_low));
    memcpy(plain->y_low, src->y_low, sizeof(o->y_low));
    auto push = [&](uint64_t index, Real x, Real y) {
        const size_t off = o->data.size();
        o->data.resize(off + o->elem_bytes, 0);
        const uint64_t raw = index & 0x7FFFFFFFFFFFFFFFull; // CompressionIndex : 63, Rebase : 1 (= 0)
        memcpy(o->data.data() + off, &raw, 8);
        IO::put(o->data.data() + off + 8, x, y);
        o->count++;
    };
    const Real scale = RC::scale(error_exp);
    // entry 0 is the zero element pushed by InitResults (PerturbationResults.cpp:861-863); the compressor's
    // running value starts at (OrbitXLow, OrbitYLow), the replay of entry 0 (:2336)
    Real ix, iy;
    IO::get(src->data.data(), ix, iy);
    push(0, ix, iy);
    IO::put(plain->data.data(), ix, iy);
    Real zx = X, zy = Y;
    for (uint64_t i = 1; i < src->count; i++) {
        IO::get(src->data.data() + i * IO::kBytes, ix, iy);
        if (RC::drifted(zx, zy, ix, iy, scale)) {
            push(i, ix, iy);
            zx = ix;
            zy = iy;
        }
        IO::put(plain->data.data() + i * IO::kBytes, zx, zy); // value the decompressor reproduces at index i
        RC::step(zx, zy, X, Y);
    }
    o->plain = plain;
    return o;
}

// Orbit for a 2x32 target from its double-typed base (CopyFullOrbitVector, PerturbationResults.cpp:241-290)
void convert_orbit_2x32(const std::shared_ptr<fsh_orbit> &base, fsh_orbit *o, bool hdr) {
    o->base = base;
    o->count = base->count;
    o->period = base->period;
    o->elem_bytes = hdr ? 24 : 16;
    o->data.resize((size_t)o->count * o->elem_bytes);
    for (uint64_t i = 0; i < o->count; i++) {
        unsigned char *p = o->data.data() + i * o->elem_bytes;
        if (hdr) {
            Hdr<double> x, y;
            ElemIO<HostHdr<double>>::get(base->data.data() + i * base->elem_bytes, x, y);
            const Hdr<df32> cx = to_df(x), cy = to_df(y);
            memcpy(p, &cx.m, 8); memcpy(p + 8, &cx.e, 4); memcpy(p + 12, &cy.e, 4); memcpy(p + 16, &cy.m, 8);
        } else {
            double x, y;
            ElemIO<HostPlain<double>>::get(base->data.data() + i * base->elem_bytes, x, y);
            const df32 cx = to_df(x), cy = to_df(y);
            memcpy(p, &cx, 8); memcpy(p + 8, &cy, 8);
        }
    }
    auto conv3 = [&](const unsigned char *src, unsigned char *dst) {
        if (hdr) { Hdr<double> v; memcpy(&v, src, sizeof(v)); const Hdr<df32> c = to_df(v); memcpy(dst, &c, sizeof(c)); }
        else { double v; memcpy(&v, src, sizeof(v)); const df32 c = to_df(v); memcpy(dst, &c, sizeof(c)); }
    };
    conv3(base->max_radius, o->max_radius);
    conv3(base->x_low, o->x_low);
    conv3(base->y_low, o->y_low);
}

template <class N, class IterT> fsh_la *build_la(const fsh_orbit *o, int period_divisor = 2) {
    LaBuilder<N, IterT> b;
    b.orbit = o;
    b.periodDivisor = period_divisor;
    b.build();
    fsh_la *r = new fsh_la();
    r->num_las = b.las.size();
    r->las_own = b.las.release(); // the builder's array, as is
    r->stages.resize(b.stages.size() * sizeof(b.stages[0]));
    memcpy(r->stages.data(), b.stages.data(), r->stages.size());
    r->at.resize(sizeof(b.at));
    memcpy(r->at.data(), &b.at, sizeof(b.at));
    r->num_stages = b.stages.size();
    r->stage_count = b.stage_count;
    r->use_at = b.use_at;
    r->is_valid = b.is_valid;
    return r;
}

// --------------------------------------------------------------------------------------------
// BLA table construction (BLAS::Init  BLAS.cpp:212-254; leaves :74-92; merge :25-47 + BLA.cuh:61-88;
// level fill :96-143; pairwise merge upwards :145-210).  Level l, entry i covers orbit steps
// [i*2^l + 1, (i+1)*2^l]; levels 0 and 1 are never stored (m_FirstLevel = 2).
// --------------------------------------------------------------------------------------------
template <class N> struct WireBLA { // BLA.h:7-14
    typename N::Real r2, Ax, Ay, Bx, By;
    int32_t l;
};
static_assert(sizeof(WireBLA<HostHdr<float>>) == 44 && sizeof(WireBLA<HostHdr<double>>) == 88, "BLA<HDRFloat>");
static_assert(sizeof(WireBLA<HostPlain<double>>) == 48 && sizeof(WireBLA<HostPlain<float>>) == 24, "BLA<plain>");

template <class N> struct BlaOps;
template <class M> struct BlaOps<HostHdr<M>> {
    using Real = Hdr<M>;
    static Real mul_(Real a, Real b) { return mul(a, b); }
    static Real add_(Real a, Real b) { return add(a, b); }
    static Real sub_(Real a, Real b) { return sub(a, b); }
    static Real div_(Real a, Real b) { return div(a, b); }
    static void red(Real &a) { reduce(a); }
    static Real one() { return h_from_int<M>(1); }
    static Real zero() { return hdr_zero<M>(); }
    static Real eps() { return div(h_from_int<M>(1), h_from_mant<M>((M)(1L << 23))); } // T(1) / T{1L << BLA_BITS}
    // HdrSqrt  HDRFloat.h:1358-1383 (result not reduced)
    static Real sqrt_(Real a) {
        const bool odd = (a.e & 1) != 0;
        Real r;
        r.e = odd ? (a.e - 1) / 2 : a.e / 2;
        r.m = (M)::sqrt(odd ? M(2) * a.m : a.m);
        return r;
    }
    // HDRFloat::compareTo  HDRFloat.h:1207-1247
    static int compare_to(Real a, Real b) {
        if (a.m == 0 && b.m == 0) return 0;
        if (a.m > 0) {
            if (b.m <= 0) return 1;
            if (a.e > b.e) return 1;
            if (a.e < b.e) return -1;
            return a.m > b.m ? 1 : (a.m < b.m ? -1 : 0);
        }
        if (b.m > 0) return -1;
        if (a.e > b.e) return -1;
        if (a.e < b.e) return 1;
        return a.m > b.m ? 1 : (a.m < b.m ? -1 : 0);
    }
    static Real max_reduced(Real a, Real b) { return compare_to(a, b) > 0 ? a : b; }       // HdrMaxReduced :1477-1494
    static Real min_pos_reduced(Real a, Real b) { return cmp_pr(a, b) < 0 ? a : b; }       // HdrMinPositiveReduced :1518-1535
    // 2 * orbit point as (RealA, ImagA): HDRFloatComplex{x, y}.getRe() * 2 (BLAS.cpp:76-78, HDRFloatComplex.h:158-173)
    static void leaf_a(Real x, Real y, Real &ra, Real &ia) {
        const HdrC<M> c = hc_from<M>(x, y);
        ra = mul(hc_re(c), h_from_mant<M>(M(2)));
        ia = mul(hc_im(c), h_from_mant<M>(M(2)));
    }
};
template <class M> struct BlaOps<HostPlain<M>> {
    using Real = M;
    static Real mul_(Real a, Real b) { return a * b; }
    static Real add_(Real a, Real b) { return a + b; }
    static Real sub_(Real a, Real b) { return a - b; }
    static Real div_(Real a, Real b) { return a / b; }
    static void red(Real &) {}
    static Real one() { return M(1); }
    static Real zero() { return M(0); }
    static Real eps() { return M(1) / M(1L << 23); }
    static Real sqrt_(Real a) { return (M)::sqrt(a); }
    static Real max_reduced(Real a, Real b) { return a > b ? a : b; }
    static Real min_pos_reduced(Real a, Real b) { return a < b ? a : b; }
    static void leaf_a(Real x, Real y, Real &ra, Real &ia) { ra = x * 2; ia = y * 2; }
};

template <class N> struct BlaBuilder {
    using O = BlaOps<N>;
    using Real = typename N::Real;
    using Rec = WireBLA<N>;
    const fsh_orbit *orbit = nullptr;
    Real bla_size{};
    std::vector<size_t> per_level;
    std::vector<std::vector<Rec>> B;
    int32_t lm2 = 0;

    Rec one_step(size_t m) const { // CreateOneStep  BLAS.cpp:74-92
        Real x, y, ra, ia;
        ElemIO<N>::get(orbit->data.data() + m * orbit->elem_bytes, x, y);
        O::leaf_a(x, y, ra, ia);
        const Real mA = O::sqrt_(O::add_(O::mul_(ra, ra), O::mul_(ia, ia)));
        const Real r = O::mul_(mA, O::eps());
        Rec b;
        memset(&b, 0, sizeof(b));
        b.r2 = O::mul_(r, r);
        b.Ax = ra; b.Ay = ia; b.Bx = O::one(); b.By = O::zero(); b.l = 1;
        return b;
    }
    static Real hypot_(Real x, Real y) { // hypotA / hypotB  BLA.cuh:40-56
        Real r = O::sqrt_(O::add_(O::mul_(x, x), O::mul_(y, y)));
        O::red(r);
        return r;
    }
    Rec merge(const Rec &x, const Rec &y) const { // MergeTwoBlas  BLAS.cpp:25-47
        Rec b;
        memset(&b, 0, sizeof(b));
        b.l = x.l + y.l;
        // getNewA: A = y.A * x.A   BLA.cuh:66-75
        b.Ax = O::sub_(O::mul_(y.Ax, x.Ax), O::mul_(y.Ay, x.Ay)); O::red(b.Ax);
        b.Ay = O::add_(O::mul_(y.Ax, x.Ay), O::mul_(y.Ay, x.Ax)); O::red(b.Ay);
        // getNewB: B = y.A * x.B + y.B   BLA.cuh:78-88
        b.Bx = O::add_(O::sub_(O::mul_(y.Ax, x.Bx), O::mul_(y.Ay, x.By)), y.Bx); O::red(b.Bx);
        b.By = O::add_(O::add_(O::mul_(y.Ax, x.By), O::mul_(y.Ay, x.Bx)), y.By); O::red(b.By);
        const Real xA = hypot_(x.Ax, x.Ay), xB = hypot_(x.Bx, x.By);
        Real tempR = O::div_(O::sub_(O::sqrt_(y.r2), O::mul_(xB, bla_size)), xA);
        O::red(tempR);
        const Real r = O::min_pos_reduced(O::sqrt_(x.r2), O::max_reduced(O::zero(), tempR));
        b.r2 = O::mul_(r, r);
        return b;
    }
    Rec l_step(size_t level, size_t m) const { // CreateLStep  BLAS.cpp:49-72
        if (level == 0) return one_step(m);
        const size_t m2 = m << 1, mx = m2 - 1, my = m2;
        if (my <= per_level[level - 1]) return merge(l_step(level - 1, mx), l_step(level - 1, my));
        return l_step(level - 1, mx);
    }
    void build() { // Init  BLAS.cpp:212-254
        constexpr size_t kFirst = 2;
        size_t m = (size_t)orbit->count - 1;
        if (orbit->count == 0 || m == 0) return;
        for (; m > 1; m = (m + 1) >> 1) per_level.push_back(m);
        per_level.push_back(m);
        B.resize(per_level.size());
        lm2 = (int32_t)per_level.size() - 2;
        if (lm2 < 0) lm2 = 0;
        if (kFirst >= per_level.size()) return;
        for (size_t l = kFirst; l < B.size(); l++) B[l].resize(per_level[l]);
        // every record of a level depends on the level below only: record-parallel on the host pool (same calls, same bytes)
        parallel_for(per_level[kFirst], [&](size_t lo, size_t hi) { for (size_t i = lo + 1; i < hi + 1; i++) B[kFirst][i - 1] = l_step(kFirst, i); });
        // Merge  BLAS.cpp:160-210
        size_t src = kFirst;
        const size_t max_level = per_level.size() - 1;
        for (size_t n_src = per_level[src]; src < max_level && n_src > 1; src++) {
            const size_t n_dst = per_level[src + 1];
            parallel_for(n_dst, [&](size_t lo, size_t hi) {
                for (size_t i = lo; i < hi; i++) {
                    const size_t mx = i << 1, my = mx + 1;
                    B[src + 1][i] = my < n_src ? merge(B[src][mx], B[src][my]) : B[src][mx];
                }
            });
            n_src = n_dst;
        }
    }
};

template <class N> fsh_blas *build_blas(const fsh_orbit *o) {
    BlaBuilder<N> b;
    b.orbit = o;
    memcpy(&b.bla_size, o->max_radius, sizeof(b.bla_size));
    b.build();
    fsh_blas *r = new fsh_blas();
    r->elem_bytes = sizeof(WireBLA<N>);
    r->lm2 = b.lm2;
    r->levels.resize(b.B.size());
    for (size_t l = 0; l < b.B.size(); l++) {
        r->levels[l].resize(b.B[l].size() * sizeof(WireBLA<N>));
        if (!b.B[l].empty()) memcpy(r->levels[l].data(), b.B[l].data(), r->levels[l].size());
        r->counts.push_back(b.B[l].size());
        r->ptrs.push_back(b.B[l].empty() ? nullptr : r->levels[l].data());
    }
    return r;
}

unsigned long pick_precision(const char *a, const char *b) {
    const size_t n = std::max(strlen(a), strlen(b));
    const unsigned long bits = (unsigned long)(n * 3.3219281) + 64;
    return bits < 256 ? 256 : bits;
}

template <class N> void fill_coord(const fs_mpf_struct *f, void *dst) {
    if (!dst) return;
    const typename N::Real v = FromMpf<N>::coord(f);
    memcpy(dst, &v, sizeof(v));
}

} // namespace

extern "C" {

// numeric tags as in include/fs_gpu.h
enum { NUM_F32 = 0, NUM_F64 = 1, NUM_2X32 = 2, NUM_HDR32 = 3, NUM_HDR64 = 4, NUM_HDR2X32 = 5, NUM_2X64 = 6, NUM_4X32 = 7,
       NUM_4X64 = 8, NUM_2X32_DIRECT = 0x102 /* MattDblflt as FillCoord builds it for Gpu2x32 */ };

fsh_view *fsh_view_create(const char *minX, const char *minY, const char *maxX, const char *maxY, uint32_t scrn_w,
                          uint32_t scrn_h, uint32_t antialiasing, int32_t square_aspect) {
    const unsigned long prec = std::max(pick_precision(minX, maxX), pick_precision(minY, maxY));
    fsh_view *v = new fsh_view(prec);
    if (fs_mpf_set_str(v->minX.v, minX, 10) || fs_mpf_set_str(v->minY.v, minY, 10) ||
        fs_mpf_set_str(v->maxX.v, maxX, 10) || fs_mpf_set_str(v->maxY.v, maxY, 10)) {
        delete v;
        return nullptr;
    }
    v->w = scrn_w; v->h = scrn_h; v->aa = antialiasing ? antialiasing : 1;
    if (square_aspect && scrn_w && scrn_h) { // PointZoomBBConverter::SquareAspectRatio :271-312
        Mpf ratio(prec), mwidth(prec), height(prec), tmp(prec), w(prec), h(prec);
        fs_mpf_set_ui(w.v, scrn_w);
        fs_mpf_set_ui(h.v, scrn_h);
        fs_mpf_div(ratio.v, w.v, h.v);
        fs_mpf_sub(mwidth.v, v->maxX.v, v->minX.v);
        fs_mpf_div(mwidth.v, mwidth.v, ratio.v);
        fs_mpf_sub(height.v, v->maxY.v, v->minY.v);
        const int c = fs_mpf_cmp(height.v, mwidth.v);
        if (c > 0) {
            fs_mpf_sub(tmp.v, height.v, mwidth.v);
            fs_mpf_mul(tmp.v, ratio.v, tmp.v);
            fs_mpf_div_ui(tmp.v, tmp.v, 2);
            fs_mpf_sub(v->minX.v, v->minX.v, tmp.v);
            fs_mpf_add(v->maxX.v, v->maxX.v, tmp.v);
        } else if (c < 0) {
            fs_mpf_sub(tmp.v, mwidth.v, height.v);
            fs_mpf_div_ui(tmp.v, tmp.v, 2);
            fs_mpf_sub(v->minY.v, v->minY.v, tmp.v);
            fs_mpf_add(v->maxY.v, v->maxY.v, tmp.v);
        }
    }
    // reference point = view centre
    fs_mpf_add(v->cx.v, v->minX.v, v->maxX.v);
    fs_mpf_div_ui(v->cx.v, v->cx.v, 2);
    fs_mpf_add(v->cy.v, v->minY.v, v->maxY.v);
    fs_mpf_div_ui(v->cy.v, v->cy.v, 2);
    return v;
}

// A frame of a zoom sequence around v's centre: the same cx, cy, precision and size, bounds = centre -/+ v's half-extents
// times `scale` (a decimal string; > 1 zooms out).  The offsets are formed at extra precision, so scale "1" gives v's
// bounds bit for bit and scale "2" exactly twice its extents.  Frames of one sequence share v's reference orbit.
fsh_view *fsh_view_zoom(const fsh_view *v, const char *scale) {
    const unsigned long prec = v->prec, wide = v->prec + 128;
    Mpf s(wide), d(wide), t(wide);
    if (fs_mpf_set_str(s.v, scale, 10) || fs_mpf_sgn(s.v) <= 0) return nullptr;
    fsh_view *z = new fsh_view(prec);
    z->w = v->w; z->h = v->h; z->aa = v->aa;
    fs_mpf_set(z->cx.v, v->cx.v);
    fs_mpf_set(z->cy.v, v->cy.v);
    auto side = [&](Mpf &dst, const Mpf &bound, const Mpf &centre) { // dst = centre + (bound - centre) * scale
        fs_mpf_sub(d.v, bound.v, centre.v);
        fs_mpf_mul(t.v, d.v, s.v);
        fs_mpf_add(t.v, centre.v, t.v);
        fs_mpf_set(dst.v, t.v);
    };
    side(z->minX, v->minX, v->cx);
    side(z->maxX, v->maxX, v->cx);
    side(z->minY, v->minY, v->cy);
    side(z->maxY, v->maxY, v->cy);
    return z;
}

void fsh_view_destroy(fsh_view *v) { delete v; }
uint32_t fsh_view_precision_bits(const fsh_view *v) { return (uint32_t)v->prec; }

// FillGpuCoords + centre deltas (Fractal.cpp:1830-1844, 2831-2840). Any output may be NULL.
int32_t fsh_view_coords(const fsh_view *v, int32_t numeric, void *cx, void *cy, void *dx, void *dy, void *center_x,
                        void *center_y) {
    const unsigned long prec = v->prec;
    Mpf ddx(prec), ddy(prec), cenx(prec), ceny(prec), div(prec);
    fs_mpf_sub(ddx.v, v->maxX.v, v->minX.v);
    fs_mpf_set_ui(div.v, (unsigned long)v->w * v->aa);
    fs_mpf_div(ddx.v, ddx.v, div.v);
    fs_mpf_sub(ddy.v, v->maxY.v, v->minY.v);
    fs_mpf_set_ui(div.v, (unsigned long)v->h * v->aa);
    fs_mpf_div(ddy.v, ddy.v, div.v);
    fs_mpf_sub(cenx.v, v->cx.v, v->minX.v);
    fs_mpf_sub(ceny.v, v->cy.v, v->maxY.v);
#define FSH_FILL(N)                                                                                                    \
    fill_coord<N>(v->minX.v, cx); fill_coord<N>(v->minY.v, cy); fill_coord<N>(ddx.v, dx); fill_coord<N>(ddy.v, dy);   \
    fill_coord<N>(cenx.v, center_x); fill_coord<N>(ceny.v, center_y); return 0;
    // FillCoord for the 2x32 types (Fractal.cpp:1813-1826): CudaDblflt(double(src)); HDRFloat<CudaDblflt>(src)
    // splits the mpf mantissa into head/tail without renormalising and does NOT reduce
    auto fill_df = [&](const fs_mpf_struct *f, void *dst, bool hdr) {
        if (!dst) return;
        if (!hdr) {
            const df32 v = h_df_from_double(fs_mpf_get_d(f));
            memcpy(dst, &v, sizeof(v));
        } else {
            Hdr<df32> v;
            if (fs_mpf_sgn(f) == 0) { v.m.head = 0; v.m.tail = 0; v.e = MIN_BIG; }
            else {
                long e = 0;
                const double m = fs_mpf_get_d_2exp(&e, f);
                v.m.head = (float)m;
                v.m.tail = (float)(m - (double)v.m.head);
                v.e = (int32_t)e;
            }
            memcpy(dst, &v, sizeof(v));
        }
    };
    // FillCoord for the direct kernels' split types (Fractal.cpp:1752-1779, 1805-1810): limb k is the
    // conversion of what is left after subtracting limbs 0..k-1 in full precision
    auto fill_split = [&](const fs_mpf_struct *f, void *dst, int limbs, bool as_float) {
        if (!dst) return;
        Mpf rest(prec), limb(prec);
        fs_mpf_set(rest.v, f);
        for (int k = 0; k < limbs; k++) {
            double d = fs_mpf_get_d(rest.v);
            if (as_float) {
                const float fl = (float)d;
                memcpy(static_cast<char *>(dst) + 4 * k, &fl, 4);
                d = (double)fl;
            } else {
                memcpy(static_cast<char *>(dst) + 8 * k, &d, 8);
            }
            fs_mpf_set_d(limb.v, d);
            fs_mpf_sub(rest.v, rest.v, limb.v);
        }
    };
    if (numeric == NUM_2X32_DIRECT || numeric == NUM_2X64 || numeric == NUM_4X32 || numeric == NUM_4X64) {
        const int limbs = (numeric == NUM_4X32 || numeric == NUM_4X64) ? 4 : 2;
        const bool fl = numeric == NUM_2X32_DIRECT || numeric == NUM_4X32;
        fill_split(v->minX.v, cx, limbs, fl); fill_split(v->minY.v, cy, limbs, fl);
        fill_split(ddx.v, dx, limbs, fl); fill_split(ddy.v, dy, limbs, fl);
        fill_split(cenx.v, center_x, limbs, fl); fill_split(ceny.v, center_y, limbs, fl);
        return 0;
    }
    switch (numeric) {
    case NUM_F32: FSH_FILL(HostPlain<float>)
    case NUM_F64: FSH_FILL(HostPlain<double>)
    case NUM_HDR32: FSH_FILL(HostHdr<float>)
    case NUM_HDR64: FSH_FILL(HostHdr<double>)
    case NUM_2X32:
    case NUM_HDR2X32: {
        const bool hdr = numeric == NUM_HDR2X32;
        fill_df(v->minX.v, cx, hdr); fill_df(v->minY.v, cy, hdr); fill_df(ddx.v, dx, hdr); fill_df(ddy.v, dy, hdr);
        fill_df(cenx.v, center_x, hdr); fill_df(ceny.v, center_y, hdr);
        return 0;
    }
    default: return -1;
    }
#undef FSH_FILL
}

fsh_orbit *fsh_orbit_compute(const fsh_view *v, int32_t numeric, uint64_t max_iterations, int32_t periodicity) {
    fsh_orbit *o = new fsh_orbit();
    o->numeric = numeric;
    switch (numeric) {
    case NUM_F32: compute_orbit<HostPlain<float>>(v, o, max_iterations, periodicity != 0); break;
    case NUM_F64: compute_orbit<HostPlain<double>>(v, o, max_iterations, periodicity != 0); break;
    case NUM_HDR32: compute_orbit<HostHdr<float>>(v, o, max_iterations, periodicity != 0); break;
    case NUM_HDR64: compute_orbit<HostHdr<double>>(v, o, max_iterations, periodicity != 0); break;
    case NUM_2X32:
    case NUM_HDR2X32: {
        auto base = std::make_shared<fsh_orbit>();
        base->numeric = numeric == NUM_2X32 ? NUM_F64 : NUM_HDR64;
        if (numeric == NUM_2X32) compute_orbit<HostPlain<double>>(v, base.get(), max_iterations, periodicity != 0);
        else compute_orbit<HostHdr<double>>(v, base.get(), max_iterations, periodicity != 0);
        convert_orbit_2x32(base, o, numeric == NUM_HDR2X32);
        break;
    }
    default: delete o; return nullptr;
    }
    return o;
}
// Orbit with the `Bad` prefix (PerturbExtras::Bad, GPU_ReferenceIter.h:10-21) for the scaled kernel.
//   to_float == 0: same T as `src` (double or HDRFloat<float>), record = {u32 bad, u32 pad, x, y}; the flag is the
//                  underflow test of RefOrbitCalc.cpp:550-562 (|zx| <= FLT_MIN or |zy| <= FLT_MIN or
//                  (zx^2 + zy^2) * 1e-7 <= FLT_MIN), false for entry 0 and for the last entry (:625-627)
//   to_float == 1: the binary32 copy made by CopyUsefulPerturbationResults / CopyFullOrbitVector
//                  (RefOrbitCalc.cpp:2585-2620, PerturbationResults.cpp:258-264): x, y cast to float, flag copied
fsh_orbit *fsh_orbit_with_bad(const fsh_orbit *src, int32_t to_float) {
    if (src->numeric != NUM_F64 && src->numeric != NUM_HDR32) return nullptr;
    fsh_orbit *o = new fsh_orbit();
    o->numeric = to_float ? NUM_F32 : src->numeric;
    o->count = src->count;
    o->period = src->period;
    o->elem_bytes = to_float ? 16 : 24;
    o->data.assign((size_t)o->count * o->elem_bytes, 0);
    memcpy(o->max_radius, src->max_radius, sizeof(o->max_radius));
    memcpy(o->x_low, src->x_low, sizeof(o->x_low));
    memcpy(o->y_low, src->y_low, sizeof(o->y_low));
    const double small = 1.1754944e-38;
    for (uint64_t i = 0; i < src->count; i++) {
        const unsigned char *p = src->data.data() + i * src->elem_bytes;
        unsigned char *q = o->data.data() + i * o->elem_bytes;
        double xv, yv;
        float xf, yf;
        if (src->numeric == NUM_F64) {
            memcpy(&xv, p, 8); memcpy(&yv, p + 8, 8);
            xf = (float)xv; yf = (float)yv;
        } else {
            Hdr<float> x, y;
            ElemIO<HostHdr<float>>::get(p, x, y);
            xv = ldexp((double)x.m, x.e < -2000 ? -2000 : x.e);
            yv = ldexp((double)y.m, y.e < -2000 ? -2000 : y.e);
            // (float)HDRFloat<float>: mantissa * getMultiplier(exp)  HDRFloat.h:497-557
            auto mult = [](int e) { return e <= -127 ? 0.0f : (e >= 128 ? 3.402823466e+38f : ldexpf(1.0f, e)); };
            xf = x.m * mult(x.e); yf = y.m * mult(y.e);
        }
        uint32_t bad = 0;
        if (i != 0 && i + 1 != src->count)
            bad = (fabs(xv) <= small || fabs(yv) <= small || (xv * xv + yv * yv) * 0.0000001 <= small) ? 1u : 0u;
        memcpy(q, &bad, 4);
        if (to_float) { memcpy(q + 8, &xf, 4); memcpy(q + 12, &yf, 4); }
        else memcpy(q + 8, p, 16);
    }
    return o;
}
// SimpleCompression (RefOrbitCompressor, PerturbationResults.cpp:2334-2381): waypoints {CompressionIndex, x, y}
// wherever replaying z <- z^2 + c in the low type drifts by more than 10^-error_exp relative; the orbit between
// waypoints is recomputed by the consumer.  Returns the compressed orbit (GPUReferenceIter<T, SimpleCompression>[],
// 8-byte index prefix); `plain` holds the host replay (RuntimeDecompressor, PerturbationResultsHelpers.h:34-197),
// which is what the LA table is built from.  2x32 targets compress their double-typed base and convert the
// waypoints (CopyFullOrbitVector, PerturbationResults.cpp:264-267).
fsh_orbit *fsh_orbit_compress(const fsh_orbit *src, int32_t error_exp) {
    if (src->pextras != 0) return nullptr;
    switch (src->numeric) {
    case NUM_F32: return compress_orbit<HostPlain<float>>(src, error_exp);
    case NUM_F64: return compress_orbit<HostPlain<double>>(src, error_exp);
    case NUM_HDR32: return compress_orbit<HostHdr<float>>(src, error_exp);
    case NUM_HDR64: return compress_orbit<HostHdr<double>>(src, error_exp);
    case NUM_2X32:
    case NUM_HDR2X32: {
        const bool hdr = src->numeric == NUM_HDR2X32;
        std::shared_ptr<fsh_orbit> cb(hdr ? compress_orbit<HostHdr<double>>(src->base.get(), error_exp)
                                          : compress_orbit<HostPlain<double>>(src->base.get(), error_exp));
        fsh_orbit *o = new fsh_orbit();
        o->numeric = src->numeric;
        o->pextras = 2;
        o->count = cb->count;
        o->uncompressed_count = cb->uncompressed_count;
        o->period = cb->period;
        o->elem_bytes = 8 + (hdr ? 24 : 16);
        o->data.assign((size_t)o->count * o->elem_bytes, 0);
        for (uint64_t i = 0; i < cb->count; i++) {
            const unsigned char *p = cb->data.data() + i * cb->elem_bytes;
            unsigned char *q = o->data.data() + i * o->elem_bytes;
            memcpy(q, p, 8);
            if (hdr) {
                Hdr<double> x, y;
                ElemIO<HostHdr<double>>::get(p + 8, x, y);
                const Hdr<df32> cx = to_df(x), cy = to_df(y);
                memcpy(q + 8, &cx.m, 8); memcpy(q + 16, &cx.e, 4); memcpy(q + 20, &cy.e, 4); memcpy(q + 24, &cy.m, 8);
            } else {
                double x, y;
                ElemIO<HostPlain<double>>::get(p + 8, x, y);
                const df32 cx = to_df(x), cy = to_df(y);
                memcpy(q + 8, &cx, 8); memcpy(q + 16, &cy, 8);
            }
        }
        memcpy(o->max_radius, src->max_radius, sizeof(o->max_radius));
        memcpy(o->x_low, src->x_low, sizeof(o->x_low));
        memcpy(o->y_low, src->y_low, sizeof(o->y_low));
        // the table is built on the double-typed replay and converted (build_la_2x32 reads plain->base)
        o->plain = std::make_shared<fsh_orbit>();
        o->plain->numeric = src->numeric;
        o->plain->base = cb->plain;
        return o;
    }
    default: return nullptr;
    }
}
uint64_t fsh_orbit_uncompressed_count(const fsh_orbit *o) { return o->pextras == 2 ? o->uncompressed_count : o->count; }
// host replay of a compressed orbit in the Disable layout (what RuntimeDecompressor hands to the host code)
const void *fsh_orbit_replay_data(const fsh_orbit *o) {
    if (o->pextras != 2 || !o->plain || o->plain->data.empty()) return nullptr;
    return o->plain->data.data();
}
void fsh_orbit_destroy(fsh_orbit *o) { delete o; }
const void *fsh_orbit_data(const fsh_orbit *o) { return o->data.data(); }
uint64_t fsh_orbit_count(const fsh_orbit *o) { return o->count; }
uint64_t fsh_orbit_period(const fsh_orbit *o) { return o->period; }
uint64_t fsh_orbit_elem_bytes(const fsh_orbit *o) { return o->elem_bytes; }
const void *fsh_orbit_x_low(const fsh_orbit *o) { return o->x_low; }
const void *fsh_orbit_y_low(const fsh_orbit *o) { return o->y_low; }
const void *fsh_orbit_max_radius(const fsh_orbit *o) { return o->max_radius; }

static fsh_la *la_build_unguarded(const fsh_orbit *o, uint32_t iter_bytes);
fsh_la *fsh_la_build(const fsh_orbit *o, uint32_t iter_bytes) {
    try { // nothing is thrown across the C boundary: out of memory reads as "no table"
        return la_build_unguarded(o, iter_bytes);
    } catch (const std::exception &) {
        return nullptr;
    }
}
static fsh_la *la_build_unguarded(const fsh_orbit *o, uint32_t iter_bytes) {
    const bool u64 = iter_bytes == 8;
    // compressed orbit: the table is built from what the host-side RuntimeDecompressor replays
    // (LAReference.cpp reads the orbit through GetComplex), with the coarser period divisor
    const int pd = o->pextras == 2 ? 8 : 2;
    if (o->pextras == 2) o = o->plain.get();
    switch (o->numeric) {
    case NUM_F32: return u64 ? build_la<HostPlain<float>, uint64_t>(o, pd) : build_la<HostPlain<float>, uint32_t>(o, pd);
    case NUM_F64: return u64 ? build_la<HostPlain<double>, uint64_t>(o, pd) : build_la<HostPlain<double>, uint32_t>(o, pd);
    case NUM_HDR32: return u64 ? build_la<HostHdr<float>, uint64_t>(o, pd) : build_la<HostHdr<float>, uint32_t>(o, pd);
    case NUM_HDR64: return u64 ? build_la<HostHdr<double>, uint64_t>(o, pd) : build_la<HostHdr<double>, uint32_t>(o, pd);
    case NUM_2X32:
        return u64 ? build_la_2x32<HostPlain<double>, HostDf, uint64_t>(o->base.get(), pd)
                   : build_la_2x32<HostPlain<double>, HostDf, uint32_t>(o->base.get(), pd);
    case NUM_HDR2X32:
        return u64 ? build_la_2x32<HostHdr<double>, HostHdrDf, uint64_t>(o->base.get(), pd)
                   : build_la_2x32<HostHdr<double>, HostHdrDf, uint32_t>(o->base.get(), pd);
    default: return nullptr;
    }
}
void fsh_la_destroy(fsh_la *l) { delete l; }
const void *fsh_la_las(const fsh_la *l) { return l->las_own ? l->las_own : l->las.data(); }
uint64_t fsh_la_num_las(const fsh_la *l) { return l->num_las; }
const void *fsh_la_stages(const fsh_la *l) { return l->stages.data(); }
uint64_t fsh_la_num_stages(const fsh_la *l) { return l->num_stages; }
const void *fsh_la_at(const fsh_la *l) { return l->at.data(); }
uint64_t fsh_la_at_bytes(const fsh_la *l) { return l->at.size(); }
uint64_t fsh_la_stage_count(const fsh_la *l) { return l->stage_count; }
int32_t fsh_la_use_at(const fsh_la *l) { return l->use_at; }
int32_t fsh_la_is_valid(const fsh_la *l) { return l->is_valid; }

// BLAS<IterType, T>::Init(GetCountOrbitEntries(), GetMaxRadius())  Fractal.cpp:2739-2740
fsh_blas *fsh_blas_build(const fsh_orbit *o) {
    switch (o->numeric) {
    case NUM_F32: return build_blas<HostPlain<float>>(o);
    case NUM_F64: return build_blas<HostPlain<double>>(o);
    case NUM_HDR32: return build_blas<HostHdr<float>>(o);
    case NUM_HDR64: return build_blas<HostHdr<double>>(o);
    default: return nullptr;
    }
}
void fsh_blas_destroy(fsh_blas *b) { delete b; }
uint32_t fsh_blas_num_levels(const fsh_blas *b) { return (uint32_t)b->levels.size(); } // m_B.size() (= m_L)
int32_t fsh_blas_lm2(const fsh_blas *b) { return b->lm2; }
uint64_t fsh_blas_elem_bytes(const fsh_blas *b) { return b->elem_bytes; }
const void *const *fsh_blas_levels(const fsh_blas *b) { return b->ptrs.data(); }
const uint64_t *fsh_blas_level_counts(const fsh_blas *b) { return b->counts.data(); }

} // extern "C"
