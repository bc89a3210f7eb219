// fs_scaled_loop.cuh -- HDRx32 perturbation steps evaluated in plain binary32 on a per-pixel scaled delta.
//
// What it computes: exactly the float+exponent step of LAKernel.cuh:130-236 / HDRFloat.h:725-794 (the same
// sequence of individually rounded operations), hence bit-identical iteration counts.
//
// Why it can be done in plain floats: every HDRFloat<float> operation rounds a 24-bit mantissa and keeps the
// exponent in a separate integer, i.e. it is binary32 arithmetic with an unbounded exponent.  A power-of-two
// rescaling commutes with every rounding as long as no intermediate leaves the normal binary32 range, so with
//     d = w * 2^k   (w = (wx, wy) plain floats, k one integer per pixel, c' = c * 2^-k)
// the step   S = 2Z + d ; w' = (wx*Sx - wy*Sy + c'x , wx*Sy + wy*Sx + c'y)   is 2 FFMA + 4 FMUL + 4 FADD with
// no exponent work at all (the float+exponent form needs ~140 instructions for the same 20 roundings, see
// profiles/r1_lav2_v2_summary.md).  The escape test |Z'+d'|^2 < 4 and the rebase test |Z'+d'|^2 < |d'|^2 cannot
// fire while |d'| is small against Z'; one precomputed threshold per orbit element (`th`) decides that with
// one FMNMX + FMUL + FSETP, and only steps past the threshold evaluate the two tests (exactly, also in plain
// floats).
//
// Validity is checked, not assumed: a chunk of kChunk steps runs speculatively from a saved state and commits
// only if every intermediate provably stayed in range (components of w within [2^-6, 2^95], orbit elements
// flagged eligible when the table is built, c' either exactly representable or provably below half an ulp of
// every sum it is added to).  Otherwise the chunk is discarded and the pixel takes one float+exponent step
// (fs_perturb_loop.cuh, hdr32fast::step) before trying again.  Exact zeros, which the reference treats with
// non-canonical exponents (HDRFloat.h:974-1000 vs :725-794), always go to that path.
//
// The arithmetic in this header is FS_HD so tests/lockstep_check.cpp can run it on the CPU in lockstep with
// the oracle's float+exponent restatement (every step compared by value).
#pragma once
#include <math.h>
#include "fs_types.cuh"

namespace fs {
namespace scaled {

// One entry per reference-orbit element n:
//   ax, ay  2*Z_n as plain floats
//   th      > 0: largest |d|_inf (true scale) for which a step ARRIVING at Z_n can neither escape nor rebase
//           (regular element, both components in [2^-20, 2));  otherwise a class code that always fails the
//           threshold test and sends the arriving step to the exact tests:
//             kThExact (0)   regular element where the tests must always run (last element, |Z_n| close to 2)
//             kThZero  (-1)  Z_n = 0: the step starting here needs d itself inside the normal range (k >= -100)
//             kThTiny  (-2)  a component in [2^-77, 2^-20), |Z_n|_inf < 1: needs 2^k exact (k >= -126) or d negligible
//             NaN            never touched by the plain-float step (one component zero, out of range, ...)
//   idx     the element's own index n (bit pattern), so a chunk reads its position off the last element it loaded
struct alignas(16) FastElem {
    float ax, ay, th;
    uint32_t idx;
};
constexpr float kThExact = 0.0f, kThZero = -1.0f, kThTiny = -2.0f;

#ifndef FS_PO_CHUNK
#define FS_PO_CHUNK 16
#endif
constexpr int kChunk = FS_PO_CHUNK; // speculative steps per commit
constexpr int kNorm = 16;         // (re)normalisation puts |w|_inf into [2^16, 2^17)
constexpr float kLo = 0x1p-6f;    // every component of every committed w must be >= kLo ...
constexpr float kLoWarn = 0x1p0f; // ... and a chunk that came this close re-centres w before the next one
constexpr float kHi = 0x1p40f;    // |w|_inf < kHi at every chunk boundary (< 2^95 inside a chunk: <= x10 per step)
constexpr float kTestScale = 0x1p-40f; // the rebase test squares w * 2^-40 (keeps (2^95)^2 inside binary32; a square
                                       // that underflows is > 2^20 below the other side, the decision is unaffected)
constexpr int kCMaxExp = 30;      // c' must be below 2^31
constexpr int kCDropExp = -110;   // c' below 2^-109 is dropped: any sum it could change is rejected by kLo anyway
constexpr int kDeepK = -126;      // the exact escape/rebase tests need 2^k and 2^-k representable
constexpr int kNegligibleK = -200; // below this, d is < 2^-25 of every eligible non-zero orbit component (>= 2^-77)
constexpr int kZeroKmin = -100;
constexpr int kMinZExp = -20, kTinyZExp = -77;
constexpr uint64_t kMaxElems = 0xffffffffull; // idx is 32 bits; longer orbits keep the float+exponent loop

FS_HD float pow2i(int e) { return u2f((uint32_t)(e + 127) << 23); } // exact 2^e, e in [-126, 127]
FS_HD int fexp(float f) { return (int)((f2u(f) >> 23) & 0xffu) - 127; }
FS_HD bool is_nan(float f) { return f != f; }

// Table entry from one HDRx32 orbit element {x.m, x.e, y.e, y.m} (GPU_ReferenceIter.h:119-125).
FS_HD FastElem make_fast_elem(float xm, int xe, float ym, int ye, uint64_t n, bool last) {
    FastElem e;
    e.ax = 0.0f; e.ay = 0.0f; e.th = kThZero; e.idx = (uint32_t)n;
    const bool zero = xm == 0.0f && ym == 0.0f;
    if (!zero) {
        const float axm = fabsf(xm), aym = fabsf(ym);
        const bool nrm = axm >= 0.25f && axm < 4.0f && aym >= 0.25f && aym < 4.0f;
        const int vx = xe + fexp(xm), vy = ye + fexp(ym); // floor(log2 |component|)
        const bool ok = nrm && vx >= kTinyZExp && vy >= kTinyZExp && vx <= 0 && vy <= 0;
        if (!ok) {
            e.th = u2f(0x7fc00000u);
        } else {
            // 2*Z exactly: |m| in [0.25,4), exponent in [-77,0]  =>  two exact scalings
            e.ax = (xm * pow2i(xe + 1 + 60)) * pow2i(-60);
            e.ay = (ym * pow2i(ye + 1 + 60)) * pow2i(-60);
            if (vx < kMinZExp || vy < kMinZExp) {
                // |Z|_inf < 1 keeps |Z|^2 < 2: with d negligible such an element cannot escape
                e.th = (vx >= 0 || vy >= 0) ? u2f(0x7fc00000u) : kThTiny;
            } else {
                const double a = 0.5 * fabs((double)e.ax), b = 0.5 * fabs((double)e.ay);
                const double margin = 1.0 - 0x1p-18;
                // no rebase while |d|_2 < |Z|_2 / 2, and |d|_2 <= sqrt(2) |d|_inf
                const double th_rebase = sqrt(a * a + b * b) * 0.35355339059327373 * margin;
                // no escape while (a+g)^2 + (b+g)^2 < 4 with g = |d|_inf
                const double s = a + b, q = a * a + b * b, lim = 4.0 * margin;
                const double disc = s * s - 2.0 * (q - lim);
                double g = disc > 0.0 ? 0.5 * (sqrt(disc) - s) * margin : 0.0;
                if (!(g > 0.0)) g = 0.0;
                e.th = (float)(th_rebase < g ? th_rebase : g); // kThExact when g == 0
                if (last) e.th = kThExact; // arriving at the last element always rebases (LAKernel.cuh:214)
            }
        }
    }
    return e;
}

FS_HD FastElem load_elem_at(const FastElem *p, int off) {
#ifdef __CUDA_ARCH__
    const uint4 v = __ldg(reinterpret_cast<const uint4 *>(p) + off);
    FastElem e;
    e.ax = __uint_as_float(v.x); e.ay = __uint_as_float(v.y); e.th = __uint_as_float(v.z); e.idx = v.w;
    return e;
#else
    return p[off];
#endif
}

// c = (cX, cY) of the pixel with reduced mantissas: sign|mantissa bits and value exponent per component
// (a zero component gets an exponent far below every drop threshold).
struct CRed {
    uint32_t xb, yb;
    int xe, ye;
};
FS_HD CRed reduce_c(Hdr<float> cX, Hdr<float> cY) {
    CRed c;
    c.xb = f2u(cX.m) & 0x807fffffu; c.xe = cX.m != 0.0f ? cX.e + fexp(cX.m) : -(1 << 30);
    c.yb = f2u(cY.m) & 0x807fffffu; c.ye = cY.m != 0.0f ? cY.e + fexp(cY.m) : -(1 << 30);
    return c;
}

// Per-pixel state of the scaled form  d = w * 2^k  at orbit element E.
struct Lane {
    float wx, wy;
    float ax, ay;   // 2*Z of the element the next step starts from
    int k;
    float sk;       // 2^k      (0 when not representable: d is then negligible against every eligible Z)
    float sk2;      // 2^(k+1)
    float ik;       // 2^-k     (clamped to 2^126: only makes the threshold test more conservative)
    float ccx, ccy; // c * 2^-k (0 when dropped)
};

FS_HD bool scale_ok(int k, const CRed &c) { return k <= 0 && c.xe - k <= kCMaxExp && c.ye - k <= kCMaxExp; }
FS_HD void set_scale(Lane &L, int k, const CRed &c) {
    const int ex = c.xe - k, ey = c.ye - k;
    L.k = k;
    L.sk = k >= -126 ? pow2i(k) : 0.0f;
    L.sk2 = k >= -127 ? pow2i(k + 1) : 0.0f;
    L.ik = pow2i(imin(-k, 126));
    L.ccx = ex >= kCDropExp ? u2f(c.xb | ((uint32_t)(ex + 127) << 23)) : 0.0f;
    L.ccy = ey >= kCDropExp ? u2f(c.yb | ((uint32_t)(ey + 127) << 23)) : 0.0f;
}
// May a step start from an element of class `th` at scale exponent k?
FS_HD bool elem_allows(float th, int k) {
    if (th >= 0.0f) return true;                                            // regular
    if (th == kThZero) return k >= kZeroKmin;
    if (th == kThTiny) return k >= kDeepK || k <= kNegligibleK;
    return false;                                                           // NaN
}

// Try to express the float+exponent state (dX, dY) at orbit index n in scaled form.
template <class IterT>
FS_HD bool enter(const FastElem *tab, const CRed &c, float dxm, int dxe, float dym, int dye, IterT n, IterT iter,
                 IterT n_iterations, Lane &L) {
    if (!(fabsf(dxm) >= 0x1p-60f && fabsf(dym) >= 0x1p-60f)) return false; // zero, NaN or far from normalised
    if ((uint64_t)(n_iterations - iter) < (uint64_t)kChunk) return false;
    const int vx = dxe + fexp(dxm), vy = dye + fexp(dym);
    const int k = imax(vx, vy) - kNorm;
    if (imin(vx, vy) - k < -5 || !scale_ok(k, c)) return false;
    const FastElem E0 = load_elem_at(tab + n, 0);
    if (!elem_allows(E0.th, k)) return false;
    set_scale(L, k, c);
    L.ax = E0.ax; L.ay = E0.ay;
    // mantissas are floats in (2^-60, 4) and the values land in [2^-5, 2^17): one exact scaling each
    L.wx = dxm * pow2i(dxe - k);
    L.wy = dym * pow2i(dye - k);
    return true;
}

// Re-centre w on 2^kNorm without leaving the scaled form (exact: a power-of-two shift of w, k and c').
// Returns false (state untouched) when the shifted state would violate an entry condition.
template <class IterT> FS_HD bool renorm(const FastElem *tab, Lane &L, const CRed &c, IterT n) {
    const float m = fmaxf(fabsf(L.wx), fabsf(L.wy)), mn = fminf(fabsf(L.wx), fabsf(L.wy));
    const int e = fexp(m) - kNorm;
    const int k = L.k + e;
    // min component >= 2^-5 after the shift  <=>  its exponent >= e - 5
    if (e > 100 || e < -100 || !(fexp(mn) >= e - 5) || !scale_ok(k, c)) return false;
    if (!elem_allows(load_elem_at(tab + n, 0).th, k)) return false;
    const float f = pow2i(-e);
    L.wx *= f; L.wy *= f;
    set_scale(L, k, c);
    return true;
}

// Back to float+exponent form (reduced mantissas; components are non-zero by construction).
FS_HD void leave(const Lane &L, float &dxm, int &dxe, float &dym, int &dye) {
    dxm = u2f((f2u(L.wx) & 0x807fffffu) | 0x3f800000u); dxe = L.k + fexp(L.wx);
    dym = u2f((f2u(L.wy) & 0x807fffffu) | 0x3f800000u); dye = L.k + fexp(L.wy);
}

enum Mode : int { kDone = 0, kFast = 1, kSlow = 2, kTry = 3 };

// One fast-mode round of one pixel: a speculative chunk of up to kChunk straight-line steps from (w, element n).
// The first step whose result passes the threshold of the element it arrives at ends the chunk and gets the
// exact escape / rebase tests (LAKernel.cuh:196-226), one shared copy of that code.  A chunk commits only if
// every component of every intermediate w stayed >= kLo; otherwise the state is restored and the pixel takes a
// float+exponent step.  Returns the pixel's next mode; whenever that is kSlow, (dxm, dxe, dym, dye) hold the
// committed state in float+exponent form.  n is the orbit index (RefIteration) in either form.
template <class IterT, bool Count>
FS_HD Mode fast_round(const FastElem *tab, IterT last, IterT n_iterations, const CRed &c, Lane &L, IterT &n, IterT &iter,
                      float &dxm, int &dxe, float &dym, int &dye, unsigned long long &steps) {
    const float wx0 = L.wx, wy0 = L.wy;
    const FastElem *p = tab + n; // step u arrives at p[u + 1]
    float wx = wx0, wy = wy0, ax = L.ax, ay = L.ay, th = 0.0f, lo = 0x1p100f;
    uint32_t idx = 0;
    bool trig = false;
#pragma unroll
    for (int u = 0; u < kChunk; u++) {
        const FastElem En = load_elem_at(p, u + 1);
        // (a packed form of these ten operations -- FFMA2, 2 FMUL2, FFMA2, FADD2, 11 instead of 17 instructions per
        // step -- was measured bit-exact and no faster, 27.50 vs 27.65 ms on View 5: the packed instructions occupy
        // the FP32 datapath for two passes each, and that datapath, not instruction issue, is what the step fills)
        const float Sx = fma_(wx, L.sk, ax), Sy = fma_(wy, L.sk, ay); // 2Z + d
        const float pa = wx * Sx, pb = wy * Sy, pc = wx * Sy, pd = wy * Sx;
        const float sumX = pa - pb, sumY = pc + pd;
        wx = sumX + L.ccx;
        wy = sumY + L.ccy;
        ax = En.ax; ay = En.ay; th = En.th; idx = En.idx;
        const float m = fmaxf(fabsf(wx), fabsf(wy));
        lo = fminf(fminf(fabsf(wx), fabsf(wy)), lo);
        if (!(m < th * L.ik)) { trig = true; break; }
    }
    const IterT n0 = n;
    const int cnt = (int)(idx - (uint32_t)n0); // steps executed (the last one possibly still needing the exact tests)
    IterT n1 = n0 + (IterT)cnt;
    bool ok = lo >= kLo, done = false, recentre = false;
    if (trig && ok) {
        if (!elem_allows(th, L.k)) {
            ok = false;
        } else if (L.k < kDeepK) {
            // d is negligible against Z' (both components in [2^-77, 1)): no escape, no rebase by norm;
            // everything else at this depth takes the float+exponent step
            if (L.k > kNegligibleK || th != kThTiny || n1 >= last) ok = false;
        } else {
            const float tx = fma_(wx, L.sk2, ax), ty = fma_(wy, L.sk2, ay); // 2*(Z' + d')
            const float tx2 = tx * tx, ty2 = ty * ty;
            const float n2 = tx2 + ty2;
            if (!(n2 < 16.0f)) {
                done = true;
            } else {
                const float hik = 0.5f * L.ik;
                const float Tx = fma_(ax, hik, wx), Ty = fma_(ay, hik, wy); // (Z' + d') * 2^-k
                const float Txs = Tx * kTestScale, Tys = Ty * kTestScale, dxs = wx * kTestScale, dys = wy * kTestScale;
                const float Tx2 = Txs * Txs, Ty2 = Tys * Tys, dx2 = dxs * dxs, dy2 = dys * dys;
                const float N2 = Tx2 + Ty2, D2 = dx2 + dy2;
                if (N2 < D2 || n1 >= last) {
                    // rebase: the next step runs on Z_0.  T itself is exact once its components are >= kLo; a T the
                    // next chunk may not start from at this scale (|T| >= kHi, or Z_0 not allowed at k) is committed
                    // and re-centred below instead of sending the whole chunk back to the float+exponent step
                    const FastElem E0 = load_elem_at(tab, 0);
                    const float Tlo = fminf(fabsf(Tx), fabsf(Ty));
                    ok = Tlo >= kLo;
                    recentre = !(elem_allows(E0.th, L.k) && fmaxf(fabsf(Tx), fabsf(Ty)) < kHi);
                    wx = Tx; wy = Ty; ax = E0.ax; ay = E0.ay;
                    lo = fminf(Tlo, lo);
                    n1 = 0;
                }
            }
        }
    }
    if (!ok) {
        // discard the chunk (L still holds the state at its start)
        leave(L, dxm, dxe, dym, dye);
        return kSlow;
    }
    if (done) {
        iter += (IterT)(cnt - 1);
        if (Count) steps += (unsigned long long)cnt;
        return kDone;
    }
    iter += (IterT)cnt;
    if (Count) steps += (unsigned long long)cnt;
    n = n1;
    L.wx = wx; L.wy = wy; L.ax = ax; L.ay = ay;
    const bool budget = (uint64_t)(n_iterations - iter) >= (uint64_t)kChunk;
    if (budget && !recentre && fmaxf(fabsf(wx), fabsf(wy)) < kHi && lo >= kLoWarn) return kFast;
    if (budget && renorm<IterT>(tab, L, c, n)) return kFast;
    leave(L, dxm, dxe, dym, dye);
    return kSlow;
}

} // namespace scaled
} // namespace fs
