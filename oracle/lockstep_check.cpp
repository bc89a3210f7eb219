// lockstep_check.cpp -- TEST INFRASTRUCTURE ONLY (built into oracle/liblockstep.so, loaded by tests/).
//
// Runs the product's scaled plain-float perturbation chunks (fractalshark_b200/csrc/fs_scaled_loop.cuh, the
// FS_HD arithmetic the CUDA kernel executes) on the CPU, in lockstep with the oracle's float+exponent
// restatement of LAKernel.cuh:130-236 (oracle_cpu.cpp: perturb_step).  After every committed chunk the two
// states are compared BY VALUE (reduced mantissa + exponent of both delta components, orbit index, iteration
// count); rejected chunks and everything the scaled form refuses go through the oracle step, exactly like the
// kernel falls back to its float+exponent step.  x86 binary32 with -ffp-contract=off and explicit fmaf is the
// same IEEE arithmetic the GPU executes (no FTZ on either side), so a clean run here is evidence for the
// bit-exactness argument in the header of fs_scaled_loop.cuh on every step it touched.
#include "oracle_cpu.cpp"

#include <mutex>
#include <cstdio>
#include <cstdlib>

#include "../fractalshark_b200/csrc/fs_scaled_loop.cuh"
#include "../fractalshark_b200/csrc/fs_at_fast.cuh"
#include "../fractalshark_b200/csrc/fs_la_fast.cuh"
#include "../fractalshark_b200/csrc/fs_la_step2.cuh"
#include "../fractalshark_b200/csrc/fs_num.cuh"
#include "../fractalshark_b200/csrc/fs_qd.cuh"

namespace {

struct LockStats {
    uint64_t fast_steps = 0, slow_steps = 0, chunks_ok = 0, chunks_rejected = 0, entries_refused = 0, mismatches = 0,
             finished_fast = 0;
};

template <class IterT>
IterT lockstep_pixel(const Lav2Job<IterT> &J, const fs::scaled::FastElem *tab, int X, int Y, LockStats &st) {
    using namespace fs::scaled;
    uint64_t steps = 0;
    PerturbState<IterT> S; // the oracle shadow (float+exponent form)
    lav2_prologue(J, X, Y, steps, S);
    if (!(J.mode == 1 || J.mode == 2)) return S.iter;
    const IterT last = J.orbit_count - 1;
    const CRed c = reduce_c(fs::Hdr<float>{S.cX.mantissa, S.cX.exp}, fs::Hdr<float>{S.cY.mantissa, S.cY.exp});
    // same per-lane control flow as PerturbLoop<NumHdr<float>>::run in fs_perturb_loop.cuh
    Lane L;
    Mode mode = kTry;
    PerturbState<IterT> F = S; // what the scaled path believes
    for (unsigned round = 0;; ++round) {
        if (mode == kTry) {
            F = S;
            const bool in = enter<IterT>(tab, c, F.dX.mantissa, F.dX.exp, F.dY.mantissa, F.dY.exp, F.RefIteration, F.iter,
                                         J.n_iterations, L);
            if (!in) st.entries_refused++;
            mode = in ? kFast : kSlow;
        }
        if (mode == kFast) {
            unsigned long long fsteps = 0;
            const IterT iter_before = F.iter;
            mode = fast_round<IterT, true>(tab, last, J.n_iterations, c, L, F.RefIteration, F.iter, F.dX.mantissa, F.dX.exp,
                                           F.dY.mantissa, F.dY.exp, fsteps);
            st.fast_steps += fsteps;
            bool alive = true;
            for (unsigned long long i = 0; i < fsteps && alive; i++) alive = perturb_step(J, S);
            if (mode == kDone) {
                st.finished_fast++;
                if (alive || S.iter != F.iter) st.mismatches++;
                return F.iter;
            }
            if (!alive) { st.mismatches++; return S.iter; }
            if (fsteps) st.chunks_ok++; else if (F.iter == iter_before && mode == kSlow) st.chunks_rejected++;
            // compare by value: the scaled state (w * 2^k) against the shadow
            float fxm, fym; int fxe, fye;
            leave(L, fxm, fxe, fym, fye);
            HF ax = S.dX, ay = S.dY;
            Reduce(ax); Reduce(ay);
            if (!(ax.mantissa == fxm && ax.exp == fxe && ay.mantissa == fym && ay.exp == fye &&
                  S.RefIteration == F.RefIteration && S.iter == F.iter))
                st.mismatches++;
            if (mode == kSlow) { S.dX = F.dX; S.dY = F.dY; } // continue from the scaled path's representation
        } else {
            st.slow_steps++;
            if (!perturb_step(J, S)) return S.iter;
            mode = kTry;
        }
    }
}

// AT shortcut: the product's mantissa recurrence (fs_at_fast.cuh) against the oracle's float+exponent loop
// (oracle_cpu.cpp lav2_prologue, ATInfo.h:155-188), pass by pass: same escape decision at every pass, same mantissas
// bit for bit, exponent equal to c's after the first pass.
struct AtStats {
    uint64_t pixels = 0, refused = 0, passes = 0, mismatches = 0, escaped = 0, mono = 0;
};
template <class IterT> void lockstep_at_pixel(const Lav2Job<IterT> &J, int X, int Y, uint64_t max_passes, AtStats &st) {
    const HF DeltaReal = sub(mul(J.dx, hf_from_number((float)X)), J.centerX);
    const HF negdy{-J.dy.mantissa, J.dy.exp};
    const HF DeltaImaginary = sub(mul(negdy, hf_from_number((float)Y)), J.centerY);
    const HC DeltaSub0 = hc_from(DeltaReal, DeltaImaginary);
    if (!(J.is_valid && J.use_at && cmpPR(cheb(DeltaSub0), J.at->ThresholdC) <= 0)) return;
    const ATInfoF<IterT> &AT = *J.at;
    uint64_t n_pass = J.n_iterations / AT.StepLength;
    if (n_pass > max_passes) n_pass = max_passes;
    HC c = add(mul(DeltaSub0, AT.CCoeff), AT.RefC);
    Reduce(c);
    st.pixels++;
    const fs::atfast::Plan<float> plan = fs::atfast::plan<float>(fs::HdrC<float>{c.re, c.im, c.exp},
                                                                 fs::Hdr<float>{AT.SqrEscapeRadius.mantissa, AT.SqrEscapeRadius.exp},
                                                                 n_pass > 0);
    if (!plan.ok) { st.refused++; return; }
    if (plan.mono) st.mono++;
    HC z = hc_zero();
    float re = 0.0f, im = 0.0f;
    for (uint64_t i = 0; i < n_pass; i++) {
        const float rr = z.re * z.re, ii = z.im * z.im;
        HF nsq{rr + ii, z.exp << 1};
        Reduce(nsq);
        const bool esc_o = cmpPR(nsq, AT.SqrEscapeRadius) > 0;
        const bool esc_f = fs::atfast::escaped(fs::atfast::norm(re, im), plan.thr);
        if (esc_o != esc_f) { st.mismatches++; return; }
        if (esc_o) {
            st.escaped++;
            // the lean chunk test of lav2_at relies on this: with plan.mono an escaped |z|^2 stays escaped (or turns
            // inf/NaN) on every later pass, so the last pass of a 16-pass chunk still shows it
            if (plan.mono)
                for (int k = 0; k < 16; k++) {
                    fs::atfast::advance(re, im, plan.s, c.re, c.im);
                    if (!fs::atfast::escaped(fs::atfast::norm(re, im), plan.thr)) { st.mismatches++; return; }
                }
            return;
        }
        const int32_t e2 = z.exp + z.exp;
        HC z2{rr - ii, fmaf(z.re, z.im, z.re * z.im), e2 < MIN_BIG_EXPONENT ? MIN_BIG_EXPONENT : e2};
        z = add(z2, c);
        fs::atfast::advance(re, im, plan.s, c.re, c.im);
        st.passes++;
        if (bits(z.re) != bits(re) || bits(z.im) != bits(im) || z.exp != plan.E) { st.mismatches++; return; }
    }
}

// LA steps: the product's select-free step (fs_la_fast.cuh) evaluated on the inputs of every step the oracle attempts;
// whatever it accepts must agree bit for bit (decision, new delta, z, rebase-by-norm), whatever it refuses is counted.
struct LaStats {
    uint64_t steps = 0, refused = 0, mismatches = 0, unusable = 0;
    uint64_t refused2 = 0, mismatches2 = 0; // the same for the step on step-shaped records (fs_la_step2.cuh)
};
// la2::step on the record la2::pack builds from a reference-shaped entry, against what the oracle computed for that step
template <class Rec>
int la2_check(const Rec &r, const HC &next_ref, const HC &dz, const HC &dc, bool unusable, const HC &ndz, const HC &z, bool by_norm) {
    const fs::la2::Rec rec = fs::la2::pack(fs::HdrC<float>{r.Ref.re, r.Ref.im, r.Ref.exp}, fs::HdrC<float>{r.ZCoeff.re, r.ZCoeff.im, r.ZCoeff.exp},
                                           fs::HdrC<float>{r.CCoeff.re, r.CCoeff.im, r.CCoeff.exp},
                                           fs::Hdr<float>{r.LAThreshold.mantissa, r.LAThreshold.exp}, (uint32_t)r.StepLength,
                                           (uint32_t)r.NextStageLAIndex, true, fs::HdrC<float>{next_ref.re, next_ref.im, next_ref.exp});
    uint4 q[4];
    memcpy(q, &rec, sizeof(rec));
    fs::la2::Out o;
    if (!fs::la2::step(q[0], q[1], q[2], q[3], dz.re, dz.im, dz.exp, dc.re, dc.im, dc.exp, o)) return 1; // refused
    if (o.unusable != unusable) return 2;
    if (unusable) return 0;
    // bit for bit, except the SIGN of an exact zero: where the reference's addition drops an operand (gap >= 120) it
    // returns the other one untouched (HDRFloatComplex.h:219-247), the product adds `dropped * 0` to it, which turns a -0
    // component into +0.  No operation of the path can tell the two apart (no division, IEEE comparisons, |x| in the norms).
    auto same = [](float a, float b) { return bits(a) == bits(b) || (a == 0.0f && b == 0.0f); };
    if (!same(o.dre, ndz.re) || !same(o.dim, ndz.im) || o.de != ndz.exp || !same(o.zre, z.re) || !same(o.zim, z.im) ||
        o.ze != z.exp || o.rebase != by_norm)
        return 2;
    return 0;
}
struct LaObserver {
    LaStats &st;
    template <class Rec>
    void la_step(const Rec &r, const HC &next_ref, const HC &dz, const HC &dc, bool unusable, bool, const HC &ndz, const HC &z,
                 bool by_norm) {
        fs::lafast::StepOut o;
        st.steps++;
        if (unusable) st.unusable++;
        {
            const int rc2 = la2_check(r, next_ref, dz, dc, unusable, ndz, z, by_norm);
            if (rc2 == 1) st.refused2++;
            if (rc2 == 2) st.mismatches2++;
        }
        const bool ok = fs::lafast::step(r.Ref.re, r.Ref.im, r.Ref.exp, r.ZCoeff.re, r.ZCoeff.im, r.ZCoeff.exp, r.CCoeff.re,
                                         r.CCoeff.im, r.CCoeff.exp, r.LAThreshold.mantissa, r.LAThreshold.exp, next_ref.re,
                                         next_ref.im, next_ref.exp, dz.re, dz.im, dz.exp, dc.re, dc.im, dc.exp, o);
        if (!ok) { st.refused++; return; }
        if (o.unusable != unusable) { st.mismatches++; return; }
        if (unusable) return;
        if (bits(o.dz.re) != bits(ndz.re) || bits(o.dz.im) != bits(ndz.im) || o.dz.e != ndz.exp || bits(o.z.re) != bits(z.re) ||
            bits(o.z.im) != bits(z.im) || o.z.e != z.exp || o.rebase != by_norm)
            st.mismatches++;
    }
};

} // namespace

extern "C" {

// Identity behind the 6-rounding AT pass (fs_at_fast.cuh `advance`): fma(a, b, RN(a*b)) == 2*RN(a*b) for binary32 and
// binary64, checked on `count` pseudo-random operand pairs whose exponents are drawn to cover normal, denormal-product,
// overflow and binade-edge cases (operands with few mantissa bits make exact ties frequent).  Returns the mismatches.
uint64_t lockstep_twice_product_identity(uint64_t count, uint64_t seed) {
    uint64_t bad = 0, x = seed * 0x9E3779B97F4A7C15ull + 1;
    auto next = [&]() { x ^= x << 13; x ^= x >> 7; x ^= x << 17; return x; };
    for (uint64_t i = 0; i < count; i++) {
        const uint64_t r = next(), q = next();
        // binary32: exponent fields chosen so products land anywhere from deep underflow to overflow
        uint32_t ma = (uint32_t)(r & 0x7fffffu), mb = (uint32_t)((r >> 23) & 0x7fffffu);
        if (q & 1) ma &= 0x7ff000u;       // short mantissas: exact halfway cases in the denormal range
        if (q & 2) mb &= 0x7e0000u;
        const uint32_t ea = (uint32_t)((q >> 8) % 255u), eb = (q & 4) ? (uint32_t)((254u + 22u - ea + (q >> 20) % 9u) % 255u)
                                                                      : (uint32_t)((q >> 16) % 255u);
        float a, b;
        const uint32_t ba = ((uint32_t)(r >> 63) << 31) | (ea << 23) | ma, bb = ((uint32_t)((r >> 62) & 1) << 31) | (eb << 23) | mb;
        memcpy(&a, &ba, 4); memcpy(&b, &bb, 4);
        const float p = a * b;
        const float t = __builtin_fmaf(a, b, p), u = p + p;
        if (bits(t) != bits(u) && !(t != t && u != u)) bad++;
        // binary64
        const uint64_t da = (r & 0x800fffffffffffffull) | ((uint64_t)((q >> 24) % 2047u) << 52);
        const uint64_t db = (next() & 0x800fffffffffffffull & ((q & 8) ? 0xffffffff00000000ull : ~0ull)) |
                            ((uint64_t)((q & 16) ? (2046u + 51u - (q >> 24) % 2047u + (q >> 40) % 9u) % 2047u : (q >> 36) % 2047u) << 52);
        double A, B;
        memcpy(&A, &da, 8); memcpy(&B, &db, 8);
        const double P = A * B;
        const double T = __builtin_fma(A, B, P), U = P + P;
        uint64_t tb, ub;
        memcpy(&tb, &T, 8); memcpy(&ub, &U, 8);
        if (tb != ub && !(T != T && U != U)) bad++;
    }
    return bad;
}


// The plan lav2_at makes for one pixel: c = (re, im) x 2^ce (reduced), R = rm x 2^re_.  out[0] = ok (mantissa recurrence
// applies), out[1] = mono (lean chunk test applies), out[2] = E; thr_out = the pre-scaled escape threshold.
void lockstep_at_plan(float cre, float cim, int ce, float rm, int re_, int *out, float *thr_out) {
    const fs::atfast::Plan<float> p = fs::atfast::plan<float>(fs::HdrC<float>{cre, cim, ce}, fs::Hdr<float>{rm, re_}, true);
    out[0] = p.ok; out[1] = p.mono; out[2] = p.E;
    *thr_out = p.thr;
}

// With a lean plan: iterate z <- z^2 + c from z = (zre, zim) x 2^E for `passes` passes and report the first pass whose
// entering |z|^2 is over the threshold (-1: none) and whether every later pass also reads as escaped.
int lockstep_at_growth(float cre, float cim, int ce, float rm, int re_, float zre, float zim, int passes, int *stays) {
    const fs::atfast::Plan<float> p = fs::atfast::plan<float>(fs::HdrC<float>{cre, cim, ce}, fs::Hdr<float>{rm, re_}, true);
    int first = -1;
    *stays = 1;
    for (int i = 0; i < passes; i++) {
        const bool esc = fs::atfast::escaped(fs::atfast::norm(zre, zim), p.thr);
        if (esc && first < 0) first = i;
        if (!esc && first >= 0) *stays = 0;
        fs::atfast::advance(zre, zim, p.s, cre, cim);
    }
    return first;
}

// stats[6]: pixels that take the AT shortcut, pixels the fast form refused, passes compared, mismatches, pixels escaped,
// pixels whose plan allows the lean (last-pass-only) chunk test
uint64_t lockstep_at(const void *at, int use_at, int is_valid, int w, int h, const void *dx, const void *dy,
                     const void *cenx, const void *ceny, uint64_t n_iter, uint64_t max_passes, int col_step, int row_step,
                     uint64_t *stats) {
    using IterT = uint32_t;
    Lav2Job<IterT> J;
    memset((void *)&J, 0, sizeof(J));
    J.mode = 1;
    J.at = (const ATInfoF<IterT> *)at;
    J.use_at = use_at && at;
    J.is_valid = is_valid;
    J.width = w; J.height = h;
    memcpy(&J.dx, dx, 8); memcpy(&J.dy, dy, 8); memcpy(&J.centerX, cenx, 8); memcpy(&J.centerY, ceny, 8);
    J.n_iterations = (IterT)n_iter;
    AtStats st;
    for (int y = 0; y < h; y += (row_step < 1 ? 1 : row_step))
        for (int x = 0; x < w; x += (col_step < 1 ? 1 : col_step)) lockstep_at_pixel(J, x, y, max_passes, st);
    stats[0] = st.pixels; stats[1] = st.refused; stats[2] = st.passes; stats[3] = st.mismatches; stats[4] = st.escaped; stats[5] = st.mono;
    return st.mismatches;
}

// The cycle watch of the chunked AT loop (fs_at_fast.cuh CycleWatch, the code the kernel runs) against the loop that
// executes every pass: for every sampled pixel that takes the AT shortcut with an accepted plan, both must end with the same
// pass count and the same (re, im), bit for bit.  The chunk structure is the kernel's: 16 passes per escape test, a chunk
// with an escaped pass is replayed pass by pass, the watch is consulted after every clean chunk.
// stats[5]: pixels compared, pixels whose cycle was found, passes executed with the watch, passes executed without, mismatches
uint64_t lockstep_at_cycle(const void *at, int use_at, int is_valid, int w, int h, const void *dx, const void *dy,
                           const void *cenx, const void *ceny, uint64_t n_iter, int col_step, int row_step, uint64_t *stats) {
    using IterT = uint32_t;
    Lav2Job<IterT> J;
    memset((void *)&J, 0, sizeof(J));
    J.at = (const ATInfoF<IterT> *)at;
    J.use_at = use_at && at;
    J.is_valid = is_valid;
    memcpy(&J.dx, dx, 8); memcpy(&J.dy, dy, 8); memcpy(&J.centerX, cenx, 8); memcpy(&J.centerY, ceny, 8);
    uint64_t pixels = 0, found = 0, with = 0, without = 0, mism = 0;
    if (!(J.is_valid && J.use_at)) { stats[0] = stats[1] = stats[2] = stats[3] = stats[4] = 0; return 0; }
    const ATInfoF<IterT> &AT = *J.at;
    const IterT at_max = (IterT)(n_iter / AT.StepLength);
    constexpr int K = fs::kWatchChunk;
    for (int y = 0; y < h; y += (row_step < 1 ? 1 : row_step))
        for (int x = 0; x < w; x += (col_step < 1 ? 1 : col_step)) {
            const HF DeltaReal = sub(mul(J.dx, hf_from_number((float)x)), J.centerX);
            const HF negdy{-J.dy.mantissa, J.dy.exp};
            const HF DeltaImaginary = sub(mul(negdy, hf_from_number((float)y)), J.centerY);
            const HC d0 = hc_from(DeltaReal, DeltaImaginary);
            if (cmpPR(cheb(d0), AT.ThresholdC) > 0) continue;
            HC c = add(mul(d0, AT.CCoeff), AT.RefC);
            Reduce(c);
            const fs::atfast::Plan<float> plan = fs::atfast::plan<float>(fs::HdrC<float>{c.re, c.im, c.exp},
                                                                        fs::Hdr<float>{AT.SqrEscapeRadius.mantissa, AT.SqrEscapeRadius.exp}, at_max > 0);
            if (!plan.ok) continue;
            pixels++;
            // every pass
            float re0 = 0.0f, im0 = 0.0f;
            IterT i0 = 0;
            for (; i0 < at_max; i0++) {
                if (fs::atfast::escaped(fs::atfast::norm(re0, im0), plan.thr)) break;
                fs::atfast::advance(re0, im0, plan.s, c.re, c.im);
            }
            without += i0;
            // chunked, with the watch
            float re = 0.0f, im = 0.0f;
            IterT i = 0, skipped = 0;
            fs::CycleWatch<float, IterT> watch(re, im, i);
            while (at_max - i >= (IterT)K) {
                const float sre = re, sim = im;
                bool esc = false;
                for (int u = 0; u < K; u++) {
                    if (fs::atfast::escaped(fs::atfast::norm(re, im), plan.thr)) { esc = true; break; }
                    fs::atfast::advance(re, im, plan.s, c.re, c.im);
                }
                if (esc) { re = sre; im = sim; break; }
                i += (IterT)K;
                watch.after_chunk(re, im, i, at_max, skipped);
            }
            for (; i < at_max; i++) {
                if (fs::atfast::escaped(fs::atfast::norm(re, im), plan.thr)) break;
                fs::atfast::advance(re, im, plan.s, c.re, c.im);
            }
            with += i - skipped;
            if (!watch.armed) found++;
            if (i != i0 || bits(re) != bits(re0) || bits(im) != bits(im0)) mism++;
        }
    stats[0] = pixels; stats[1] = found; stats[2] = with; stats[3] = without; stats[4] = mism;
    return mism;
}

// Returns the number of lockstep mismatches (0 = every committed chunk matched the oracle by value).
// stats[7]: fast steps, slow steps, chunks committed, chunks rejected, entries refused, mismatches, pixels finished in a chunk
uint64_t lockstep_render_lav2(int mode, const void *orbit, uint64_t count, const void *las, const void *stages,
                              const void *at, uint64_t stage_count, int use_at, int is_valid, int w, int h,
                              const void *dx, const void *dy, const void *cenx, const void *ceny, uint64_t n_iter,
                              void *out, int col_step, int row_step, int threads, uint64_t *stats) {
    using IterT = uint32_t;
    Lav2Job<IterT> J;
    J.mode = mode;
    J.orbit = (const OrbitElemF *)orbit;
    J.orbit_count = (IterT)count;
    J.las = (const LAInfoDeepF<IterT> *)las;
    J.stages = (const LAStageInfo<IterT> *)stages;
    J.at = (const ATInfoF<IterT> *)at;
    J.la_stage_count = (IterT)stage_count;
    J.use_at = use_at && at;
    J.is_valid = is_valid && las;
    J.width = w; J.height = h; J.pitch = (w + 15) / 16 * 16;
    memcpy(&J.dx, dx, 8); memcpy(&J.dy, dy, 8); memcpy(&J.centerX, cenx, 8); memcpy(&J.centerY, ceny, 8);
    J.n_iterations = (IterT)n_iter;
    J.out = (IterT *)out;
    std::vector<fs::scaled::FastElem> tab(count);
    for (uint64_t n = 0; n < count; n++)
        tab[n] = fs::scaled::make_fast_elem(J.orbit[n].xm, J.orbit[n].xe, J.orbit[n].ym, J.orbit[n].ye, n, n + 1 >= count);
    std::mutex mu;
    LockStats total;
    if (col_step < 1) col_step = 1;
    parallel_rows(0, h, threads, [&](int y) {
        LockStats st;
        for (int x = 0; x < w; x += col_step) J.out[(size_t)y * J.pitch + x] = lockstep_pixel(J, tab.data(), x, y, st);
        std::lock_guard<std::mutex> g(mu);
        total.fast_steps += st.fast_steps; total.slow_steps += st.slow_steps; total.chunks_ok += st.chunks_ok;
        total.chunks_rejected += st.chunks_rejected; total.entries_refused += st.entries_refused;
        total.mismatches += st.mismatches; total.finished_fast += st.finished_fast;
    }, row_step);
    if (stats) {
        stats[0] = total.fast_steps; stats[1] = total.slow_steps; stats[2] = total.chunks_ok; stats[3] = total.chunks_rejected;
        stats[4] = total.entries_refused; stats[5] = total.mismatches; stats[6] = total.finished_fast;
    }
    return total.mismatches;
}


// LA-step lockstep over a pixel sub-grid (HDRx32, AT + LA prologue only).  out[0..3] = steps, refused, mismatches, unusable.
void lockstep_la(const void *las, const void *stages, const void *at, uint64_t la_stage_count, int use_at, int is_valid, int w,
                 int h, const void *dx, const void *dy, const void *cx, const void *cy, uint64_t n_iterations, int iter_bytes,
                 int col_step, int row_step, uint64_t *out) {
    LaStats st;
    auto run = [&](auto it) {
        using IterT = decltype(it);
        Lav2Job<IterT> J{};
        J.mode = 3;
        J.orbit = nullptr;
        J.orbit_count = 0;
        J.las = (const LAInfoDeepF<IterT> *)las;
        J.stages = (const LAStageInfo<IterT> *)stages;
        J.at = (const ATInfoF<IterT> *)at;
        J.la_stage_count = (IterT)la_stage_count;
        J.use_at = use_at && at;
        J.is_valid = is_valid && las;
        J.width = w; J.height = h; J.pitch = w;
        memcpy(&J.dx, dx, 8); memcpy(&J.dy, dy, 8); memcpy(&J.centerX, cx, 8); memcpy(&J.centerY, cy, 8);
        J.n_iterations = (IterT)n_iterations;
        LaObserver obs{st};
        for (int y = 0; y < h; y += row_step)
            for (int x = 0; x < w; x += col_step) {
                uint64_t steps = 0;
                PerturbState<IterT> S;
                lav2_prologue(J, x, y, steps, S, &obs);
            }
    };
    if (iter_bytes == 8) run(uint64_t{}); else run(uint32_t{});
    out[0] = st.steps; out[1] = st.refused; out[2] = st.mismatches; out[3] = st.unusable;
    out[4] = st.refused2; out[5] = st.mismatches2;
}

// The LA step on step-shaped records (fs_la_step2.cuh) against the reference-shaped operations on synthetic inputs aimed
// at its guards: exponent gaps of the three aligned additions spread over [-140, 140] (the reference drops an operand at
// |gap| >= 120, the select-free form at 127), exact zeros in every operand, mantissas far from [1, 2) (un-reduced deltas,
// near-total cancellation in dz * (2 Ref + dz) and in the sums), thresholds one ulp either side of cheb(newdz), records
// whose threshold is not reduced.  Whatever la2::step accepts must agree bit for bit with the oracle's step.
// out[0..3] = cases, accepted, refused, mismatches.
void lockstep_la2_fuzz(uint64_t count, uint64_t seed, uint64_t *out) {
    uint64_t s = seed * 0x9E3779B97F4A7C15ull + 0x632BE59BD9B4E019ull;
    auto next = [&]() { s ^= s << 13; s ^= s >> 7; s ^= s << 17; return s; };
    auto pick_mant = [&]() -> float {
        const uint64_t r = next();
        const unsigned kind = (unsigned)(r & 15u);
        float m;
        const uint32_t frac = (uint32_t)(r >> 20) & 0x007fffffu;
        if (kind == 0) m = 0.0f;                                                         // exact zero
        else if (kind == 1) m = fbits(((uint32_t)(127 - 1 - (unsigned)((r >> 8) % 126u)) << 23) | frac); // tiny: down to 2^-126
        else if (kind == 2) m = fbits(((uint32_t)(127 + 1 + (unsigned)((r >> 8) & 7u)) << 23) | frac);  // un-reduced, up to 2^8
        else if (kind == 3) m = fbits(0x3f800000u | ((r >> 50) & 1u ? 0x007fffffu : 0u));               // 1.0 or 2 - ulp
        else m = fbits(0x3f800000u | frac);                                                             // reduced [1, 2)
        return (r >> 63) ? -m : m;
    };
    uint64_t accepted = 0, refused = 0, mismatches = 0;
    for (uint64_t n = 0; n < count; n++) {
        LAInfoDeepF<uint32_t> r{};
        const int base = (int)(next() % 4001) - 2000;
        auto gap = [&]() -> int { const uint64_t q = next(); return (q & 7u) == 0 ? (int)((q >> 8) % 281) - 140 : (int)((q >> 8) % 61) - 30; };
        HC dz{pick_mant(), pick_mant(), base};
        r.Ref = HC{pick_mant(), pick_mant(), base + gap()};
        r.ZCoeff = HC{pick_mant(), pick_mant(), (int)(next() % 2001) - 1000};
        r.CCoeff = HC{pick_mant(), pick_mant(), (int)(next() % 2001) - 1000};
        // dc chosen so that dc * CCoeff lands within `gap` of newdz * ZCoeff (exponents: ~2 base + ZCoeff.e)
        HC dc{pick_mant(), pick_mant(), 2 * base + r.ZCoeff.exp - r.CCoeff.exp + gap()};
        HC next_ref{pick_mant(), pick_mant(), 2 * base + r.ZCoeff.exp + gap()};
        r.StepLength = 1;
        r.NextStageLAIndex = 0;
        // the oracle's step (oracle_cpu.cpp lav2_prologue, LAKernel.cuh:91-127)
        HC newdz = mul(dz, add(mul(r.Ref, HF{1.0f, 1}), dz));
        Reduce(newdz);
        HF cn = cheb(newdz);
        // threshold: mostly around cheb(newdz) (equal, one ulp below / above, an exponent apart), sometimes anything
        const uint64_t q = next();
        HF th = cn;
        switch ((unsigned)(q & 7u)) {
        case 0: break;
        case 1: th.mantissa = fbits(bits(th.mantissa) + 1u); break;
        case 2: th.mantissa = fbits(bits(th.mantissa) - 1u); break;
        case 3: th.exp += 1; break;
        case 4: th.exp -= 1; break;
        case 5: th = HF{pick_mant(), cn.exp}; break; // possibly not reduced / zero / negative: the record must be refused
        default: th = HF{fbits(0x3f800000u | ((uint32_t)(q >> 20) & 0x007fffffu)), cn.exp + (int)((q >> 8) % 5) - 2}; break;
        }
        if (!(th.mantissa >= 1.0f && th.mantissa < 2.0f) && (q & 7u) != 5) th.mantissa = 1.0f;
        r.LAThreshold = th;
        const bool unusable = cmpPR(cn, r.LAThreshold) >= 0;
        HC ndz = dz, z = dz;
        bool by_norm = false;
        if (!unusable) {
            ndz = add(mul(newdz, r.ZCoeff), mul(dc, r.CCoeff));
            z = add(next_ref, ndz);
            HF n0 = cheb(z), nN = cheb(ndz);
            Reduce(n0);
            Reduce(nN);
            by_norm = cmpPR(n0, nN) < 0;
        }
        const int rc = la2_check(r, next_ref, dz, dc, unusable, ndz, z, by_norm);
        if (rc == 0) accepted++;
        else if (rc == 1) refused++;
        else {
            if (getenv("FS_FUZZ_VERBOSE") && mismatches < 12) {
                fprintf(stderr, "mismatch: dz=(%a,%a,%d) Ref=(%a,%a,%d) ZC=(%a,%a,%d) CC=(%a,%a,%d) dc=(%a,%a,%d) nref=(%a,%a,%d) th=(%a,%d)\n",
                        dz.re, dz.im, dz.exp, r.Ref.re, r.Ref.im, r.Ref.exp, r.ZCoeff.re, r.ZCoeff.im, r.ZCoeff.exp, r.CCoeff.re, r.CCoeff.im,
                        r.CCoeff.exp, dc.re, dc.im, dc.exp, next_ref.re, next_ref.im, next_ref.exp, th.mantissa, th.exp);
                fprintf(stderr, "   oracle: newdz=(%a,%a,%d) unusable=%d ndz=(%a,%a,%d) z=(%a,%a,%d) by_norm=%d\n", newdz.re, newdz.im, newdz.exp,
                        (int)unusable, ndz.re, ndz.im, ndz.exp, z.re, z.im, z.exp, (int)by_norm);
                const fs::la2::Rec rec = fs::la2::pack(fs::HdrC<float>{r.Ref.re, r.Ref.im, r.Ref.exp}, fs::HdrC<float>{r.ZCoeff.re, r.ZCoeff.im, r.ZCoeff.exp},
                                                       fs::HdrC<float>{r.CCoeff.re, r.CCoeff.im, r.CCoeff.exp}, fs::Hdr<float>{th.mantissa, th.exp}, 1, 0, true,
                                                       fs::HdrC<float>{next_ref.re, next_ref.im, next_ref.exp});
                uint4 qq[4];
                memcpy(qq, &rec, sizeof(rec));
                fs::la2::Out o;
                const bool ok = fs::la2::step(qq[0], qq[1], qq[2], qq[3], dz.re, dz.im, dz.exp, dc.re, dc.im, dc.exp, o);
                fprintf(stderr, "   la2:    ok=%d unusable=%d ndz=(%a,%a,%d) z=(%a,%a,%d) rebase=%d\n", (int)ok, (int)o.unusable, o.dre, o.dim, o.de,
                        o.zre, o.zim, o.ze, (int)o.rebase);
            }
            mismatches++;
        }
    }
    out[0] = count; out[1] = accepted; out[2] = refused; out[3] = mismatches;
}


// The host build of the product's HDRFloat<float> / HDRFloatComplex<float> operations (fs_types.cuh, FS_HD) on operand arrays:
// the CPU pre-image of fs_selftest_numeric_op, so that the per-operation vectors of the GPU suite can be checked against
// orc_numeric_op without a GPU as well (tests/test_oracle_and_host.py).  Ops as in include/fs_gpu.h; -1: not a host op.
int lockstep_numeric_op(uint32_t op, const void *a_, const void *b_, void *out_, uint64_t n) {
    struct Hf { float m; int32_t e; };
    struct Hc { float re, im; int32_t e; };
    const Hf *fa = (const Hf *)a_, *fb = (const Hf *)b_; Hf *fo = (Hf *)out_;
    const Hc *ca = (const Hc *)a_, *cb = (const Hc *)b_; Hc *co = (Hc *)out_;
    auto hf = [](Hf v) { return fs::hdr_make<float>(v.e, v.m); };
    auto hc = [](Hc v) { fs::HdrC<float> c; c.re = v.re; c.im = v.im; c.e = v.e; return c; };
    for (uint64_t i = 0; i < n; i++) {
        fs::Hdr<float> r; fs::HdrC<float> c;
        switch (op) {
        case 0: r = fs::add(hf(fa[i]), hf(fb[i])); fo[i] = Hf{r.m, r.e}; break;
        case 1: r = fs::sub(hf(fa[i]), hf(fb[i])); fo[i] = Hf{r.m, r.e}; break;
        case 2: r = fs::mul(hf(fa[i]), hf(fb[i])); fo[i] = Hf{r.m, r.e}; break;
        case 3: r = fs::square(hf(fa[i])); fo[i] = Hf{r.m, r.e}; break;
        case 4: r = hf(fa[i]); fs::reduce(r); fo[i] = Hf{r.m, r.e}; break;
        case 5: r = fs::div(hf(fa[i]), hf(fb[i])); fo[i] = Hf{r.m, r.e}; break;
        case 6: fo[i] = Hf{0.0f, fs::cmp_pr(hf(fa[i]), hf(fb[i]))}; break;
        case 10: c = fs::add(hc(ca[i]), hc(cb[i])); co[i] = Hc{c.re, c.im, c.e}; break;
        case 11: c = fs::mul(hc(ca[i]), hc(cb[i])); co[i] = Hc{c.re, c.im, c.e}; break;
        case 12: c = hc(ca[i]); fs::reduce(c); co[i] = Hc{c.re, c.im, c.e}; break;
        case 13: r = fs::cheb(hc(ca[i])); co[i] = Hc{r.m, 0.0f, r.e}; break;
        case 14: c = fs::mul(hc(ca[i]), fs::hdr_make<float>(cb[i].e, cb[i].re)); co[i] = Hc{c.re, c.im, c.e}; break;
        case 50: case 51: case 52: case 53: case 54: case 55: case 56: {
            struct Wire { double m; int32_t e; int32_t pad; };
            const Wire wa = ((const Wire *)a_)[i], wb = ((const Wire *)b_)[i];
            const fs::Hdr<double> x = fs::hdr_make<double>(wa.e, wa.m), y = fs::hdr_make<double>(wb.e, wb.m);
            fs::Hdr<double> q = fs::hdr_make<double>(0, 0.0);
            switch (op) {
            case 50: q = fs::add(x, y); break;
            case 51: q = fs::sub(x, y); break;
            case 52: q = fs::mul(x, y); break;
            case 53: q = fs::square(x); break;
            case 54: q = x; fs::reduce(q); break;
            case 55: q = fs::div(x, y); break;
            default: q = fs::hdr_make<double>(fs::cmp_pr(x, y), 0.0); break;
            }
            ((Wire *)out_)[i] = Wire{q.m, q.e, 0};
            break;
        }
        case 80: case 81: case 82: case 83: { // perturbation policies (fs_num.cuh perturb_selftest), 128-byte records
            const unsigned char *in = (const unsigned char *)a_ + (size_t)fs::kPerturbRecordBytes * i;
            unsigned char *o = (unsigned char *)out_ + (size_t)fs::kPerturbRecordBytes * i;
            if (op == 80) fs::perturb_selftest<fs::NumPlain<float>>(in, o);
            else if (op == 81) fs::perturb_selftest<fs::NumPlain<double>>(in, o);
            else if (op == 82) fs::perturb_selftest<fs::NumHdr<float>>(in, o);
            else fs::perturb_selftest<fs::NumHdr<double>>(in, o);
            break;
        }
        case 40: {
            fs::Hdr<float> dx = hf(fa[3 * i]), dy = hf(fa[3 * i + 1]);
            fs::NumHdr<float>::perturb(dx, dy, hf(fa[3 * i + 2]), hf(fb[3 * i]), hf(fb[3 * i + 1]), hf(fb[3 * i + 2]));
            fo[3 * i] = Hf{dx.m, dx.e}; fo[3 * i + 1] = Hf{dy.m, dy.e}; fo[3 * i + 2] = Hf{0.0f, 0};
            break;
        }
        default: return -1;
        }
    }
    return 0;
}

// The host build of the Quad<F> operations (fs_qd.cuh quad_selftest_op): the CPU pre-image of fs_selftest_numeric_op
// 60-67 (Quad<double>, 32-byte elements) and 70-77 (Quad<float>, 16-byte elements).  -1: not a Quad op.
int lockstep_quad_op(uint32_t op, const void *a_, const void *b_, void *out_, uint64_t n) {
    if (op >= 60 && op <= 67) {
        const fs::Quad<double> *a = (const fs::Quad<double> *)a_, *b = (const fs::Quad<double> *)b_;
        for (uint64_t i = 0; i < n; i++) ((fs::Quad<double> *)out_)[i] = fs::quad_selftest_op<double>(op - 60, a[i], b[i]);
        return 0;
    }
    if (op >= 70 && op <= 77) {
        const fs::Quad<float> *a = (const fs::Quad<float> *)a_, *b = (const fs::Quad<float> *)b_;
        for (uint64_t i = 0; i < n; i++) ((fs::Quad<float> *)out_)[i] = fs::quad_selftest_op<float>(op - 70, a[i], b[i]);
        return 0;
    }
    return -1;
}

// The escape-time loop of Gpu4x32 (limb_bytes 4) / Gpu4x64 (limb_bytes 8) -- fs_qd.cuh quad_escape_count, the code the
// kernels run -- for `n` pixels given by their kernel coordinates (X[i], Y[i]) (Y already flipped).  out[i] = count.
// Returns 0, or -1 for an unknown limb size.
int lockstep_quad_pixels(int limb_bytes, int iter_bytes, const void *cx, const void *cy, const void *dx, const void *dy,
                         uint64_t n_iterations, const int32_t *X, const int32_t *Y, uint64_t n, uint64_t *out, int threads) {
    auto run = [&](auto limb, auto it) {
        using F = decltype(limb);
        using IterT = decltype(it);
        fs::Quad<F> c[4];
        memcpy(&c[0], cx, sizeof(c[0])); memcpy(&c[1], cy, sizeof(c[0]));
        memcpy(&c[2], dx, sizeof(c[0])); memcpy(&c[3], dy, sizeof(c[0]));
        parallel_rows(0, (int)n, threads, [&](int i) {
            out[i] = (uint64_t)fs::quad_escape_count<F, IterT>(c[0], c[1], c[2], c[3], X[i], Y[i], (IterT)n_iterations);
        });
    };
    if (limb_bytes == 4) { if (iter_bytes == 8) run(0.0f, uint64_t{}); else run(0.0f, uint32_t{}); return 0; }
    if (limb_bytes == 8) { if (iter_bytes == 8) run(0.0, uint64_t{}); else run(0.0, uint32_t{}); return 0; }
    return -1;
}

} // extern "C"
