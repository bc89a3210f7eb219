// fs_num.cuh -- numeric policies: one uniform vocabulary (Real, Cplx, r_*/c_* ops) over the six
// arithmetic variants of the render path so each kernel is written once.
//   NumPlain<float>, NumPlain<double>           <- T = float / double         (LAKernel.cuh:46-55)
//   NumHdr<float>,  NumHdr<double>              <- T = HDRFloat<float|double>
// The 2x32 variants (Num2x32, NumHdr2x32) live in fs_df32.cuh and plug into the same vocabulary.
#pragma once
#include "fs_types.cuh"

namespace fs {

// ---- plain scalars share the HDR vocabulary -------------------------------------------------
FS_HD float add(float a, float b) { return a + b; }
FS_HD double add(double a, double b) { return a + b; }
FS_HD float sub(float a, float b) { return a - b; }
FS_HD double sub(double a, double b) { return a - b; }
FS_HD float mul(float a, float b) { return a * b; }
FS_HD double mul(double a, double b) { return a * b; }
FS_HD void reduce(float &) {}
FS_HD void reduce(double &) {}
FS_HD bool lt_pr(float a, float b) { return a < b; }
FS_HD bool lt_pr(double a, double b) { return a < b; }
FS_HD bool ge_pr(float a, float b) { return a >= b; }
FS_HD bool ge_pr(double a, double b) { return a >= b; }
FS_HD bool gt_pr(float a, float b) { return a > b; }
FS_HD bool gt_pr(double a, double b) { return a > b; }
FS_HD bool le_pr(float a, float b) { return a <= b; }
FS_HD bool le_pr(double a, double b) { return a <= b; }
// HdrCompareToBothPositiveReducedLT<T,256>  HDRFloat.h:1562-1586 : plain types use a true "< 256"
FS_HD bool lt_bailout(float a) { return a < 256.0f; }
FS_HD bool lt_bailout(double a) { return a < 256.0; }

template <class M> struct NumPlain {
    using Mant = M;
    using Real = M;
    using Cplx = Cx<M>;
    static constexpr bool kHdr = false;
    static constexpr bool kDf = false;
    FS_HD static Real zero() { return M(0); }
    FS_HD static Real from_int(int x) { return (M)x; }
    FS_HD static Real neg(Real a) { return -a; }
    FS_HD static Cplx c_make(Real re, Real im) { Cplx c; c.re = re; c.im = im; return c; }
    FS_HD static Cplx c_zero() { Cplx c; c.re = M(0); c.im = M(0); return c; }
    FS_HD static Real c_re(Cplx c) { return c.re; }
    FS_HD static Real c_im(Cplx c) { return c.im; }
    // Ref * HDRFloat(2)
    FS_HD static Cplx c_mul2(Cplx c) { return mul(c, M(2)); }

    // One perturbation step, rounding sequence of the reference build (SURVEY.md section 8a):
    //   sy = fma(Zy,2,dy)  sx = fma(Zx,2,dx)  ny = fma(sx,dy,sy*dx)  nx = fma(sx,dx,-(sy*dy))
    //   dy' = dcy + ny     dx' = dcx + nx
    FS_HD static void perturb(Real &dx, Real &dy, Real zx, Real zy, Real dcx, Real dcy) {
        const M sy = fma_(zy, M(2), dy);
        const M sx = fma_(zx, M(2), dx);
        const M t1 = sy * dx;
        const M t2 = sy * dy;
        const M ny = fma_(sx, dy, t1);
        const M nx = fma_(sx, dx, -t2);
        dy = dcy + ny;
        dx = dcx + nx;
    }
    // |z|^2 = fma(x, x, y*y)
    FS_HD static Real norm2(Real x, Real y) { return fma_(x, x, y * y); }
    // pixel deltas `dx * T(X) - centerX` / `-dy * T(Y) - centerY` (LAKernel.cuh:41-42, BLAKernels.cuh:61-62):
    // nvcc contracts them for the plain types (reference SASS: DFMA X, dx, -centerX ; DFMA Y, -dy, -centerY)
    FS_HD static Real delta_x(Real dx, int X, Real centerX) { return fma_((M)X, dx, -centerX); }
    FS_HD static Real delta_y(Real dy, int Y, Real centerY) { return fma_((M)Y, -dy, -centerY); }
};

template <class M> struct NumHdr {
    using Mant = M;
    using Real = Hdr<M>;
    using Cplx = HdrC<M>;
    static constexpr bool kHdr = true;
    static constexpr bool kDf = false;
    FS_HD static Real zero() { return hdr_zero<M>(); }
    // T(X): HDRFloat(int) converts through the mantissa type (HDRFloat.h:295-325)
    FS_HD static Real from_int(int x) { return hdr_from<M>((M)x); }
    FS_HD static Real neg(Real a) { a.m = -a.m; return a; }
    FS_HD static Cplx c_make(Real re, Real im) { return hc_from<M>(re, im); }
    FS_HD static Cplx c_zero() { return hc_zero<M>(); }
    FS_HD static Real c_re(Cplx c) { return hc_re(c); }
    FS_HD static Real c_im(Cplx c) { return hc_im(c); }
    FS_HD static Cplx c_mul2(Cplx c) { return mul(c, hdr_make<M>(1, M(1))); }

    // custom_perturb2  HDRFloat.h:725-794 : products aligned with exact 2^-|diff| (0 once
    // |diff| >= 127 / 1023, no 120-gap shortcut), two FMAs per component, then Reduce.
    // The reference calls the single-precision `__fmaf_rn` for every mantissa type, so with a double mantissa
    // its operands are rounded to binary32 first (reference SASS: DMUL products, F2F.F32.F64, FFMA): the
    // HDRx64 perturbation step carries binary32 precision.  Reproduced, not fixed.
    FS_HD static M fmaf_as_ref(M a, M b, M c) {
        if constexpr (sizeof(M) == 8) return (M)fma_((float)a, (float)b, (float)c);
        else return fma_(a, b, c);
    }
    template <bool Minus>
    FS_HD static Real fused3(M p1, int e1, M p2, int e2, Real c) {
        const int diff = e1 - e2;
        const int maxe = imax(e1, e2);
        const M mulv = MT<M>::pow2neg(-iabs(diff));
        const M q2 = Minus ? MT<M>::neg(p2) : p2;
        const bool ge = diff >= 0;
        const M sum = fmaf_as_ref(ge ? q2 : p1, mulv, ge ? p1 : q2);
        const int diff2 = maxe - c.e;
        const M mul2v = MT<M>::pow2neg(-iabs(diff2));
        const bool ge2 = diff2 >= 0;
        Real r;
        r.e = imax(maxe, c.e);
        r.m = fmaf_as_ref(ge2 ? c.m : sum, mul2v, ge2 ? sum : c.m);
        reduce(r);
        return r;
    }
    FS_HD static void perturb(Real &dx, Real &dy, Real zx, Real zy, Real dcx, Real dcy) {
        const Real s1 = add(mul2(zy), dy); // tempSum1 = 2*Zy + dy   LAKernel.cuh:144-150
        const Real s2 = add(mul2(zx), dx); // tempSum2 = 2*Zx + dx
        const Real nx = fused3<true>(dx.m * s2.m, dx.e + s2.e, dy.m * s1.m, dy.e + s1.e, dcx);
        const Real ny = fused3<false>(dx.m * s1.m, dx.e + s1.e, dy.m * s2.m, dy.e + s2.e, dcy);
        dx = nx;
        dy = ny;
    }
    // HdrReduce(x.square() + y.square())  LAKernel.cuh:206-208
    FS_HD static Real norm2(Real x, Real y) { return reduced(add(square(x), square(y))); }
    // pixel deltas (LAKernel.cuh:41-42): HDR operators, not reduced
    FS_HD static Real delta_x(Real dx, int X, Real centerX) { return sub(mul(dx, from_int(X)), centerX); }
    FS_HD static Real delta_y(Real dy, int Y, Real centerY) { return sub(mul(neg(dy), from_int(Y)), centerY); }
};

// Per-step self-test of a perturbation policy (fs_selftest_numeric_op 80-85, host: lockstep_numeric_op 80-83): one
// record of 8 cells of 16 bytes, each cell one Real in its in-memory layout.  In: dx, dy, zx, zy, dcx, dcy,
// {int32 X, int32 Y}.  Out: perturb(dx, dy, zx, zy, dcx, dcy) in cells 0-1, norm2(dx, dy) in 2,
// delta_x(zx, X, dcx) in 3, delta_y(zy, Y, dcy) in 4, add(zx, dx) in 5.  tests/test_exact_perturb.py holds each
// result to the bound of tests/exact_perturb.py.  (Num2x32 / NumHdr2x32 are device-only.)
constexpr int kPerturbRecordBytes = 128;
template <class Num> FS_HD void perturb_selftest(const unsigned char *in, unsigned char *out) {
    using Real = typename Num::Real;
    static_assert(sizeof(Real) <= 16, "one cell per number");
    Real v[6], r[6];
    for (int k = 0; k < 6; k++) memcpy(&v[k], in + 16 * k, sizeof(Real));
    int32_t xy[2];
    memcpy(xy, in + 96, sizeof(xy));
    r[0] = v[0];
    r[1] = v[1];
    Num::perturb(r[0], r[1], v[2], v[3], v[4], v[5]);
    r[2] = Num::norm2(v[0], v[1]);
    r[3] = Num::delta_x(v[2], xy[0], v[4]);
    r[4] = Num::delta_y(v[3], xy[1], v[5]);
    r[5] = add(v[2], v[0]);
    for (int k = 0; k < kPerturbRecordBytes; k++) out[k] = 0;
    for (int k = 0; k < 6; k++) memcpy(out + 16 * k, &r[k], sizeof(Real));
}

} // namespace fs
