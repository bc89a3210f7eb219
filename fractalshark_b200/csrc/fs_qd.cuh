// fs_qd.cuh -- extended-precision scalars for the direct kernels Gpu2x64, Gpu4x32 and Gpu4x64.
//
//   dd64      double-double {head, tail}: the NVIDIA double-double routines the reference ships as
//             HpSharkFloatLib/dbldbl.cuh:86-203 (error-free sum after Knuth, add/sub after Thall, FMA products).
//             Every operation there is an individually rounded intrinsic, so the value of each routine is
//             fixed by its operation sequence, reproduced here (same operand order).
//   Quad<F>   four-limb expansion (x most significant) after Hida/Li/Bailey's QD library as ported to CUDA by
//             Lu/He/Luo, the form the reference vendors in FractalSharkLib/QuadDouble/{inline,gqd_basic}.cuh and
//             FractalSharkLib/QuadFloat/{inline,gqf_basic}.cuh: sloppy add (gqd_basic.cuh:177-225), sloppy
//             multiply (:300-344), sqr (:351-393), scalar multiply (:267-292), renormalisation (:31-123),
//             comparisons (:501-533).  The double flavour keeps the zero shortcuts of two_sum / quick_two_sum
//             and the branching renormalisation; the float flavour is the branch-free variant of gqf_basic.cuh.
//             Products are split with one FMA (p = a*b, e = fma(a, b, -p)) -- exact -- where the reference
//             uses a Dekker split written with plain operators that its build leaves to the compiler's
//             contraction; the two agree to the last limb's rounding (~2^-200 / ~2^-90 relative), far below
//             what moves an escape count (tests/test_gpu_parity.py compares whole frames with the reference
//             kernels; tests/test_exact_escape.py holds every operation to its error bound against exact
//             rationals and the kernels' counts to exact arithmetic).
#pragma once
#include "fs_types.cuh"

namespace fs {

// ---- double-double -------------------------------------------------------------------------------------------
// device only (__dadd_rn); QuadOps below is host-callable as well (oracle/lockstep_check.cpp builds it with g++)
#ifdef __CUDACC__
struct dd64 {
    double head, tail;
};
FS_D dd64 dd_two_sum(double a, double b) { // add_double_to_dbldbl  dbldbl.cuh:86-96
    dd64 z;
    z.head = __dadd_rn(a, b);
    double t1 = __dadd_rn(z.head, -a);
    double t2 = __dadd_rn(z.head, -t1);
    t1 = __dadd_rn(b, -t1);
    t2 = __dadd_rn(a, -t2);
    z.tail = __dadd_rn(t1, t2);
    return z;
}
template <bool Sub> FS_D dd64 dd_addsub(dd64 a, dd64 b) { // add_dbldbl / sub_dbldbl  dbldbl.cuh:121-162
    const double bh = Sub ? -b.head : b.head, bt = Sub ? -b.tail : b.tail;
    double t1 = __dadd_rn(a.head, bh);
    double t2 = __dadd_rn(t1, -a.head);
    double t3 = __dadd_rn(__dadd_rn(a.head, __dadd_rn(t2, -t1)), __dadd_rn(bh, -t2));
    double t4 = __dadd_rn(a.tail, bt);
    t2 = __dadd_rn(t4, -a.tail);
    const double t5 = __dadd_rn(__dadd_rn(a.tail, __dadd_rn(t2, -t4)), __dadd_rn(bt, -t2));
    t3 = __dadd_rn(t3, t4);
    t4 = __dadd_rn(t1, t3);
    t3 = __dadd_rn(__dadd_rn(t1, -t4), t3);
    t3 = __dadd_rn(t3, t5);
    dd64 z;
    z.head = __dadd_rn(t4, t3);
    z.tail = __dadd_rn(__dadd_rn(t4, -z.head), t3);
    return z;
}
FS_D dd64 dd_add(dd64 a, dd64 b) { return dd_addsub<false>(a, b); }
FS_D dd64 dd_sub(dd64 a, dd64 b) { return dd_addsub<true>(a, b); }
FS_D dd64 dd_mul(dd64 a, dd64 b) { // mul_dbldbl  dbldbl.cuh:169-180 (sqr_dbldbl :182-192 is the same sequence)
    const double th = __dmul_rn(a.head, b.head);
    double tt = __fma_rn(a.head, b.head, -th);
    tt = __fma_rn(a.tail, b.tail, tt);
    tt = __fma_rn(a.head, b.tail, tt);
    tt = __fma_rn(a.tail, b.head, tt);
    dd64 z;
    z.head = __dadd_rn(th, tt);
    z.tail = __dadd_rn(__dadd_rn(th, -z.head), tt);
    return z;
}
#endif

// ---- four-limb expansions --------------------------------------------------------------------------------------
template <class F> struct Quad {
    F x, y, z, w;
};
template <class F> struct QuadOps {
    static constexpr bool kBranchy = sizeof(F) == 8; // QuadDouble keeps the zero shortcuts, QuadFloat dropped them
    using Q = Quad<F>;

    FS_HD static Q make(F x, F y, F z, F w) { Q q; q.x = x; q.y = y; q.z = z; q.w = w; return q; }
    // fl(a+b), err; |a| >= |b|
    FS_HD static F quick_two_sum(F a, F b, F &err) {
        if (kBranchy && b == F(0)) { err = F(0); return a + b; }
        const F s = a + b;
        err = b - (s - a);
        return s;
    }
    FS_HD static F two_sum(F a, F b, F &err) {
        if (kBranchy && (a == F(0) || b == F(0))) { err = F(0); return a + b; }
        const F s = a + b;
        const F bb = s - a;
        err = (a - (s - bb)) + (b - bb);
        return s;
    }
    FS_HD static F two_prod(F a, F b, F &err) {
        const F p = a * b;
        err = fma_(a, b, -p);
        return p;
    }
    FS_HD static void three_sum(F &a, F &b, F &c) {
        F t1, t2, t3;
        t1 = two_sum(a, b, t2);
        a = two_sum(c, t1, t3);
        b = two_sum(t2, t3, c);
    }
    FS_HD static void three_sum2(F &a, F &b, F &c) {
        F t1, t2, t3;
        t1 = two_sum(a, b, t2);
        a = two_sum(c, t1, t3);
        b = t2 + t3;
    }
    // five limbs -> four
    FS_HD static void renorm(F &c0, F &c1, F &c2, F &c3, F &c4) {
        F s0, s1, s2 = F(0), s3 = F(0);
        s0 = quick_two_sum(c3, c4, c4);
        s0 = quick_two_sum(c2, s0, c3);
        s0 = quick_two_sum(c1, s0, c2);
        c0 = quick_two_sum(c0, s0, c1);
        s0 = quick_two_sum(c0, c1, s1);
        if (!kBranchy) {
            s1 = quick_two_sum(s1, c2, s2);
            s2 = quick_two_sum(s2, c3, s3);
            s3 += c4;
        } else if (s1 != F(0)) {
            s1 = quick_two_sum(s1, c2, s2);
            if (s2 != F(0)) {
                s2 = quick_two_sum(s2, c3, s3);
                if (s3 != F(0)) s3 += c4;
                else s2 += c4;
            } else {
                s1 = quick_two_sum(s1, c3, s2);
                if (s2 != F(0)) s2 = quick_two_sum(s2, c4, s3);
                else s1 = quick_two_sum(s1, c4, s2);
            }
        } else {
            s0 = quick_two_sum(s0, c2, s1);
            if (s1 != F(0)) {
                s1 = quick_two_sum(s1, c3, s2);
                if (s2 != F(0)) s2 = quick_two_sum(s2, c4, s3);
                else s1 = quick_two_sum(s1, c4, s2);
            } else {
                s0 = quick_two_sum(s0, c3, s1);
                if (s1 != F(0)) s1 = quick_two_sum(s1, c4, s2);
                else s0 = quick_two_sum(s0, c4, s1);
            }
        }
        c0 = s0; c1 = s1; c2 = s2; c3 = s3;
    }
    FS_HD static Q neg(Q a) { return make(-a.x, -a.y, -a.z, -a.w); }
    // sloppy_add  gqd_basic.cuh:177-225
    FS_HD static Q add(Q a, Q b) {
        F s0 = a.x + b.x, s1 = a.y + b.y, s2 = a.z + b.z, s3 = a.w + b.w;
        const F v0 = s0 - a.x, v1 = s1 - a.y, v2 = s2 - a.z, v3 = s3 - a.w;
        F u0 = s0 - v0, u1 = s1 - v1, u2 = s2 - v2, u3 = s3 - v3;
        const F w0 = a.x - u0, w1 = a.y - u1, w2 = a.z - u2, w3 = a.w - u3;
        u0 = b.x - v0; u1 = b.y - v1; u2 = b.z - v2; u3 = b.w - v3;
        F t0 = w0 + u0, t1 = w1 + u1, t2 = w2 + u2;
        const F t3 = w3 + u3;
        s1 = two_sum(s1, t0, t0);
        three_sum(s2, t0, t1);
        three_sum2(s3, t0, t2);
        t0 = t0 + t1 + t3;
        renorm(s0, s1, s2, s3, t0);
        return make(s0, s1, s2, s3);
    }
    FS_HD static Q sub(Q a, Q b) { return add(a, neg(b)); }
    FS_HD static Q mul_pwr2(Q a, F b) { return make(a.x * b, a.y * b, a.z * b, a.w * b); }
    // quad * scalar  gqd_basic.cuh:267-292
    FS_HD static Q mul(Q a, F b) {
        F p0, p1, p2, p3, q0, q1, q2, s0, s1, s2, s3, s4;
        p0 = two_prod(a.x, b, q0);
        p1 = two_prod(a.y, b, q1);
        p2 = two_prod(a.z, b, q2);
        p3 = a.w * b;
        s0 = p0;
        s1 = two_sum(q0, p1, s2);
        three_sum(s2, q1, p2);
        three_sum2(q1, q2, p3);
        s3 = q1;
        s4 = q2 + p2;
        renorm(s0, s1, s2, s3, s4);
        return make(s0, s1, s2, s3);
    }
    // sloppy_mul  gqd_basic.cuh:300-344
    FS_HD static Q mul(Q a, Q b) {
        F p0, p1, p2, p3, p4, p5, q0, q1, q2, q3, q4, q5, t0, t1, s0, s1, s2;
        p0 = two_prod(a.x, b.x, q0);
        p1 = two_prod(a.x, b.y, q1);
        p2 = two_prod(a.y, b.x, q2);
        p3 = two_prod(a.x, b.z, q3);
        p4 = two_prod(a.y, b.y, q4);
        p5 = two_prod(a.z, b.x, q5);
        three_sum(p1, p2, q0);
        three_sum(p2, q1, q2);
        three_sum(p3, p4, p5);
        s0 = two_sum(p2, p3, t0);
        s1 = two_sum(q1, p4, t1);
        s2 = q2 + p5;
        s1 = two_sum(s1, t0, t0);
        s2 += (t0 + t1);
        s1 = s1 + (a.x * b.w + a.y * b.z + a.z * b.y + a.w * b.x + q0 + q3 + q4 + q5);
        renorm(p0, p1, s0, s1, s2);
        return make(p0, p1, s0, s1);
    }
    // sqr  gqd_basic.cuh:351-393
    FS_HD static Q sqr(Q a) {
        F p0, p1, p2, p3, p4, p5, q0, q1, q2, q3, s0, s1, t0, t1;
        p0 = two_prod(a.x, a.x, q0);
        p1 = two_prod(F(2) * a.x, a.y, q1);
        p2 = two_prod(F(2) * a.x, a.z, q2);
        p3 = two_prod(a.y, a.y, q3);
        p1 = two_sum(q0, p1, q0);
        q0 = two_sum(q0, q1, q1);
        p2 = two_sum(p2, p3, p3);
        s0 = two_sum(q0, p2, t0);
        s1 = two_sum(q1, p3, t1);
        s1 = two_sum(s1, t0, t0);
        t0 += t1;
        s1 = quick_two_sum(s1, t0, t0);
        p2 = quick_two_sum(s0, s1, t1);
        p3 = quick_two_sum(t1, t0, q0);
        p4 = F(2) * a.x * a.w;
        p5 = F(2) * a.y * a.z;
        p4 = two_sum(p4, p5, p5);
        q2 = two_sum(q2, q3, q3);
        t0 = two_sum(p4, q2, t1);
        t1 = t1 + p5 + q3;
        p3 = two_sum(p3, t0, p4);
        p4 = p4 + q0 + t1;
        renorm(p0, p1, p2, p3, p4);
        return make(p0, p1, p2, p3);
    }
    FS_HD static bool le(Q a, Q b) { // operator<=(quad, quad)  gqd_basic.cuh:514-519
        return a.x < b.x || (a.x == b.x && (a.y < b.y || (a.y == b.y && (a.z < b.z || (a.z == b.z && a.w <= b.w)))));
    }
    FS_HD static bool le(Q a, F b) { return a.x < b || (a.x == b && a.y <= F(0)); } // operator<=(quad, scalar) :531-533
};

// The Quad<F> operations by number, for the per-operation self-test (fs_selftest_numeric_op 60-67 / 70-77) and its
// host build: 0 add, 1 sub, 2 mul(q, q), 3 mul(q, b.x), 4 sqr(a), 5 mul_pwr2(a, b.x), 6 le(a, b), 7 le(a, b.x);
// the comparisons return {1 or 0, 0, 0, 0}.
template <class F> FS_HD Quad<F> quad_selftest_op(uint32_t k, Quad<F> a, Quad<F> b) {
    using O = QuadOps<F>;
    switch (k) {
    case 0: return O::add(a, b);
    case 1: return O::sub(a, b);
    case 2: return O::mul(a, b);
    case 3: return O::mul(a, b.x);
    case 4: return O::sqr(a);
    case 5: return O::mul_pwr2(a, b.x);
    case 6: return O::make(O::le(a, b) ? F(1) : F(0), 0, 0, 0);
    default: return O::make(O::le(a, b.x) ? F(1) : F(0), 0, 0, 0);
    }
}

// The escape-time loop of the four-limb direct kernels (mandel_4x_float / mandel_4x_double, LowPrecisionKernels.cuh:5-144)
// for the kernel's own pixel (X, Y), Y already flipped.  One iteration per bailout test, non-strict bailout on the
// rounded quad sum, no n_iterations - (P-1).  The float flavour builds x0 with quad * quad and compares with a quad 4,
// the double flavour with quad * scalar and a scalar 4, as the reference does.  Host-callable: oracle/lockstep_check.cpp
// runs this very loop on the CPU.
template <class F, class IterT>
FS_HD IterT quad_escape_count(Quad<F> cx, Quad<F> cy, Quad<F> dx, Quad<F> dy, int X, int Y, IterT n_iterations) {
    using O = QuadOps<F>;
    using Q = Quad<F>;
    Q x0, y0;
    if constexpr (sizeof(F) == 4) {
        y0 = O::add(cy, O::mul(dy, O::make((F)Y, 0, 0, 0)));
        x0 = O::add(cx, O::mul(dx, O::make((F)X, 0, 0, 0)));
    } else {
        y0 = O::add(cy, O::mul(dy, (F)Y));
        x0 = O::add(cx, O::mul(dx, (F)X));
    }
    Q x = O::make(0, 0, 0, 0), y = x;
    Q zr, zi;
    if constexpr (sizeof(F) == 4) { zr = O::sqr(x); zi = O::sqr(y); }
    else { zr = O::mul(x, x); zi = O::mul(y, y); }
    IterT iter = 0;
    for (;;) {
        bool in;
        if constexpr (sizeof(F) == 4) in = O::le(O::add(zr, zi), O::make(4.0f, 0, 0, 0));
        else in = O::le(O::add(zr, zi), 4.0);
        if (!(in && iter < n_iterations)) break;
        y = O::mul(x, y);
        if constexpr (sizeof(F) == 4) y = O::mul_pwr2(y, 2.0f);
        else y = O::mul(y, 2.0);
        y = O::add(y, y0);
        x = O::add(O::sub(zr, zi), x0);
        if constexpr (sizeof(F) == 4) { zr = O::sqr(x); zi = O::sqr(y); }
        else { zr = O::mul(x, x); zi = O::mul(y, y); }
        iter++;
    }
    return iter;
}

} // namespace fs
