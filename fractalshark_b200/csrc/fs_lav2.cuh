// fs_lav2.cuh -- the perturbation + LAv2 render kernel (row a1/a2/a3 of SURVEY.md section 8).
//
// Algorithm (what): FractalSharkGpuLib/LAKernel.cuh:3-315 -- AT shortcut, multi-stage LA skipping,
// then plain perturbation with rebasing; table access per FractalSharkLib/GPU_LAReference.h:241-303,
// GPU_LAInfoDeep.h:90-123, HpSharkFloatLib/ATInfo.h:155-188, FractalSharkGpuLib/Perturb.cuh:146-232.
//
// Execution (how, B200-first): a persistent grid of warps (SM count x resident warps) pulls 8x4-pixel
// tiles from an atomic queue, so escape-count divergence costs at most one warp-tile, never a wave
// tail; LA records and orbit elements are repacked to 16-byte-aligned records and fetched with
// 128-bit loads; all exponent alignment is integer ALU work (no MUFU).  The reference launches one
// 16x8 CTA per screen block with 32-bit field loads and scalbnf-based alignment.
// Round 2: the AT shortcut stops executing passes once a pixel's state repeats exactly (CycleWatch in fs_at_fast.cuh,
// StateWatch below: interior pixels, 97 % of the AT passes of View 14), and the HDRx32 / 32-bit LA walk runs on
// step-shaped 64-byte records fetched with two 256-bit loads (fs_la_step2.cuh, lav2_stages_v2).
#pragma once
#include "fs_num.cuh"
#include "fs_df32.cuh"
#include <type_traits>
#include "fs_perturb_loop.cuh"
#include "fs_at_fast.cuh"
#include "fs_la_fast.cuh"
#include "fs_la_step2.cuh"

#ifndef FS_AT_PACKED
#define FS_AT_PACKED 1
#endif
#ifndef FS_AT_LEAN
#define FS_AT_LEAN 1
#endif
#ifndef FS_AT_CHUNK
#define FS_AT_CHUNK 16
#endif
#ifndef FS_AT_CYCLE
// Cycle detection in the AT shortcut (1 = on): see lav2_at.
#define FS_AT_CYCLE 1
#endif
#ifndef FS_LA_STEP2
// HDRx32 with 32-bit iteration counts: 1 (default) = the LA walk on step-shaped records (fs_la_step2.cuh), 0 = the
// generic walk below on reference-shaped records.  Both bit-exact (GPU parity suite).
#define FS_LA_STEP2 1
#endif
#ifndef FS_AT_WATCH_EVERY_PASS
// 1: the cycle watch compares the state with the saved one after every pass (finds a period P as soon as P passes have
// run since the save), 0: after every chunk of FS_AT_CHUNK passes (finds it once P * 16 / gcd(P, 16) have).
#define FS_AT_WATCH_EVERY_PASS 0
#endif
#ifndef FS_LA2_LDG256
#define FS_LA2_LDG256 1
#endif
#ifndef FS_LA2_PREFETCH
#define FS_LA2_PREFETCH 0
#endif
#ifndef FS_LA_FAST
// HDRx32: 1 = flattened LA walk with the select-free step of fs_la_fast.cuh, 0 (default) = the nested walk on the
// reference-shaped operations.  Both are bit-exact (GPU parity suite; oracle/lockstep_check.cpp for the step).  Measured
// on View 14, 3840x2160: 7.37 ms flattened vs 7.08 ms nested -- the step is ~137 SASS instructions either way (the
// nested form's selects cost what the flattened form's guards and second scaling multiply cost), so the build keeps
// the nested walk; the flattened one is the per-lane state machine a lane-level refill would start from.
#define FS_LA_FAST 0
#endif
// resident CTAs per SM the compiler must allow for lav2_kernel; undefined = plain __launch_bounds__(256) (HDRx32: 60
// registers, 4 CTAs; an explicit 1 lets ptxas take 70 registers = 3 CTAs: View 5 29.0 vs 27.7 ms).
// Measured: 5 (48 registers, 32 B spilled) View 14 7.13 vs 7.29 ms but View 5 28.8 vs 27.7 ms and an 8-way shard 1.17
// vs 1.08 ms; 6 (40 registers) worse everywhere.
#ifdef FS_LAV2_MIN_CTAS
#define FS_LAV2_BOUNDS(Num) __launch_bounds__(256, FS_LAV2_MIN_CTAS)
#else
// HDRx32 is held to 64 registers (4 CTAs of 256 threads per SM; with the flattened LA walk, FS_LA_FAST, ptxas would
// otherwise take 71 and lose a quarter of the resident warps); the other numeric types keep the compiler's own choice.
#define FS_LAV2_BOUNDS(Num) __launch_bounds__(256, (Num::kHdr && !Num::kDf && sizeof(typename Num::Mant) == 4) ? 4 : 0)
#endif

namespace fs {

#ifdef FS_TILE_TIMING
// development build only: per-tile {start (globaltimer ns), duration (SM cycles)} of the last lav2_kernel launch, and
// per-launch-thread executed AT passes (indexed by a running counter: order is irrelevant for the histogram)
__device__ unsigned long long *fs_tile_times;
__device__ unsigned int *fs_at_passes;
__device__ unsigned int fs_at_passes_n;
#endif

enum class Lav2Mode : int { Full = 1, PO = 2, LAO = 3 }; // RenderAlgorithm.h:12-17

// ---- device-side table records (our own layout; filled by the upload code in fs_capi.cu) ------
template <class Num, class IterT> struct alignas(16) LaRec {
    typename Num::Cplx Ref;
    typename Num::Cplx ZCoeff;
    typename Num::Cplx CCoeff;
    typename Num::Real LAThreshold;
    typename Num::Real LAThresholdC;
    IterT StepLength;
    IterT NextStageLAIndex;
};

template <class IterT> struct StageRec {
    IterT LAIndex;
    IterT MacroItCount;
};

template <class Num, class IterT> struct AtDev {
    IterT StepLength;
    typename Num::Real ThresholdC;
    typename Num::Real SqrEscapeRadius;
    typename Num::Cplx RefC;
    typename Num::Cplx CCoeff;
    typename Num::Cplx InvZCoeff;
};

// One frame of a zoom batch (fs_render_perturb_lav2_frames): what differs between frames that share the orbit and tables.
template <class Num, class IterT> struct Lav2Frame {
    typename Num::Real dx, dy, centerX, centerY;
    IterT *out; // this frame's iteration buffer, same padded layout as Lav2Args::out
};

template <class Num, class IterT> struct Lav2Args {
    IterT *out;              // iteration buffer, row pitch = roundup16(width)
    const void *orbit;       // reference-layout orbit elements (GPU_ReferenceIter.h:119-125)
    const void *orbit_fast;  // HDRx32 only: per-element table of fs_scaled_loop.cuh (nullptr = not built)
    IterT orbit_count;       // uncompressed entries
    const LaRec<Num, IterT> *las;
    const StageRec<IterT> *stages;
    AtDev<Num, IterT> at;
    IterT la_stage_count;
    int la_valid;
    int use_at;
    int width, height, pitch;
    int shard_count, shard_index; // 4-row tile bands are dealt round-robin to shards (multi-GPU)
    typename Num::Real dx, dy, centerX, centerY;
    IterT n_iterations;
    TileQueue queue;
    unsigned long long *step_counter; // optional: executed perturbation/LA/AT steps (bench roofline)
    float4 *at_state;                 // HDRx32 two-launch form: per-pixel AT result {dz.re, dz.im, dz.e}; iter sits in `out`
    const void *las2;                 // HDRx32 / 32-bit counts: la2::Rec[] (fs_la_step2.cuh), nullptr = not built
    const void *stages2;              // ... and la2 stage records {LAIndex, MacroItCount, LAThresholdC.m, LAThresholdC.e}
    const unsigned int *order;        // optional: queue position -> tile ticket (lav2_probe_kernel: expensive tiles first)
    int at_cycle;                     // 1: cycle detection in the AT shortcut (CycleWatch), 0: every pass is executed
    IterT *sink;                      // optional mapped host copy of `out` (fs_set_result_sink): finished pixels stream out over PCIe
    const Lav2Frame<Num, IterT> *frames; // Lav2Layout::Frames: n_frames records; dx, dy, centerX, centerY, out unused
    unsigned int n_frames;
    // Lav2Layout::ExpMap: height radii and width directions (expmap_dc); dx, dy, centerX, centerY unused
    const typename Num::Real *exp_radius, *exp_dir_x, *exp_dir_y;
};

// How lav2_kernel maps pixels to dc and where it stores them.  Rect: one frame, dc = delta_x / delta_y of the linear map
// (fs_render_perturb_lav2).  Frames: a zoom batch of linear maps (fs_render_perturb_lav2_frames).  ExpMap: one frame of an
// exponential map, dc = expmap_dc of its tables (fs_render_perturb_lav2_expmap); otherwise the Rect code.
enum class Lav2Layout : int { Rect = 0, Frames = 1, ExpMap = 2 };

// How a launch treats the AT shortcut.  Fused = one launch does everything (the reference's structure).  On deep views
// the AT loop is most of the frame and perfectly regular (every interior pixel runs n/StepLength passes) while what
// follows it is short and divergent; run back to back inside one warp-tile they serialise (the tile lasts AT + the
// slowest lane's LA/perturbation tail), which is what bounds a launch once a GPU's share of the frame is small.
// AtOnly / AfterAt split the frame into two launches over the same tile queue: the first leaves {dz, iter} per pixel
// (16 B + the iteration cell), the second picks them up.  Same arithmetic, same results.  Measured on View 14 the
// split is SLOWER (9.7 vs 8.5 ms; 8-way shard 2.03 vs 1.30 ms): each launch pays its own ramp and drain, which is
// what dominates at that grain, so Fused stays the default (fs_set_split_at is an A/B switch).
enum class AtPhase : int { Fused = 0, AtOnly = 1, AfterAt = 2 };

// 16-byte vector loads of an aligned record (one LDG.128 per 16 bytes instead of one load per field)
template <class T> FS_D T ldg_rec(const T *p) {
    static_assert(sizeof(T) % 16 == 0, "record size");
    union U {
        T t;
        uint4 v[sizeof(T) / 16];
        FS_D U() {}
    } u;
    const uint4 *q = reinterpret_cast<const uint4 *>(p);
#pragma unroll
    for (int i = 0; i < (int)(sizeof(T) / 16); i++) u.v[i] = __ldg(q + i);
    return u.t;
}

// ---- orbit element fetch ----------------------------------------------------------------------
template <class Num> struct OrbitIO;

template <> struct OrbitIO<NumPlain<float>> {
    static constexpr int kBytes = 8;
    FS_D static void load(const void *base, uint64_t i, float &x, float &y) {
        const float2 v = __ldg(reinterpret_cast<const float2 *>(base) + i);
        x = v.x; y = v.y;
    }
};
template <> struct OrbitIO<NumPlain<double>> {
    static constexpr int kBytes = 16;
    FS_D static void load(const void *base, uint64_t i, double &x, double &y) {
        const double2 v = __ldg(reinterpret_cast<const double2 *>(base) + i);
        x = v.x; y = v.y;
    }
};
// HDRx32 element = {x.mant, x.exp, y.exp, y.mant}: x Left-order, y Right-order. One LDG.128.
template <> struct OrbitIO<NumHdr<float>> {
    static constexpr int kBytes = 16;
    FS_D static void load(const void *base, uint64_t i, Hdr<float> &x, Hdr<float> &y) {
        const uint4 v = __ldg(reinterpret_cast<const uint4 *>(base) + i);
        x.m = __uint_as_float(v.x); x.e = (int)v.y;
        y.e = (int)v.z; y.m = __uint_as_float(v.w);
    }
};
// HDR-double element (32 B) = {x.mant f64, x.exp, pad | y.exp, pad, y.mant f64}. Two LDG.128.
template <> struct OrbitIO<NumHdr<double>> {
    static constexpr int kBytes = 32;
    FS_D static void load(const void *base, uint64_t i, Hdr<double> &x, Hdr<double> &y) {
        const uint4 *p = reinterpret_cast<const uint4 *>(base) + 2 * i;
        const uint4 a = __ldg(p), b = __ldg(p + 1);
        x.m = __hiloint2double((int)a.y, (int)a.x); x.e = (int)a.z;
        y.e = (int)b.x; y.m = __hiloint2double((int)b.w, (int)b.z);
    }
};

// 2x32 element (16 B) = {x.head, x.tail, y.head, y.tail}. One LDG.128.
template <> struct OrbitIO<Num2x32> {
    static constexpr int kBytes = 16;
    FS_D static void load(const void *base, uint64_t i, df32 &x, df32 &y) {
        const float4 v = __ldg(reinterpret_cast<const float4 *>(base) + i);
        x.head = v.x; x.tail = v.y; y.head = v.z; y.tail = v.w;
    }
};
// HDRx2x32 element (24 B) = {x.head, x.tail, x.exp | y.exp, y.head, y.tail}: x Left-order, y Right-order. Three LDG.64.
template <> struct OrbitIO<NumHdr2x32> {
    static constexpr int kBytes = 24;
    FS_D static void load(const void *base, uint64_t i, Hdr<df32> &x, Hdr<df32> &y) {
        const uint2 *p = reinterpret_cast<const uint2 *>(base) + 3 * i;
        const uint2 a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + 2);
        x.m.head = __uint_as_float(a.x); x.m.tail = __uint_as_float(a.y); x.e = (int)b.x;
        y.e = (int)b.y; y.m.head = __uint_as_float(c.x); y.m.tail = __uint_as_float(c.y);
    }
};

// ---- small vocabulary shims so the kernel reads the same for plain and HDR numbers ------------
template <class Num> FS_D bool c_is_ge(typename Num::Real a, typename Num::Real b) { return ge_pr(a, b); }

// ---- cycle detection in the AT shortcut -----------------------------------------------------------------------------
// PerformAT (ATInfo.h:155-188) iterates z <- z*z + c until |z|^2 passes the escape radius or n / StepLength passes are
// done.  For a pixel inside the set the second case is the rule, and the passes are a deterministic map F of two binary32
// (binary64) numbers: in AT coordinates the pixel's orbit falls towards an attracting cycle and, in finite precision,
// reaches an exactly periodic sequence of states after a few hundred passes (View 14: the interior pixels run 18,402
// passes each in the reference).  Once the state after a chunk equals, bit for bit, a state saved at an earlier chunk
// boundary P passes before, every later state is known: no pass of the cycle escaped (each was tested), so none ever
// will, and  z after `at_max` passes = F^((at_max - i) mod P) (z).  The watch below saves a state at chunk counts 1, 2, 4,
// 8 ... (Brent's schedule) and compares after every chunk; on a hit it advances the pass counter by the largest multiple
// of P that fits and lets the loop finish the remainder (< P passes) the ordinary way.  Same z, same pass count, hence the
// same iteration buffer as the reference, bit for bit; what changes is the number of executed passes.
// (CycleWatch itself lives in fs_at_fast.cuh so that oracle/lockstep_check.cpp can run it on the CPU.)

// The same watch for the general loop (any numeric type): the state is the whole complex number, exponent included.
FS_D bool same_bits(float a, float b) { return __float_as_uint(a) == __float_as_uint(b); }
FS_D bool same_bits(double a, double b) { return __double_as_longlong(a) == __double_as_longlong(b); }
FS_D bool same_bits(df32 a, df32 b) { return same_bits(a.head, b.head) && same_bits(a.tail, b.tail); }
template <class M> FS_D bool same_state(Cx<M> a, Cx<M> b) { return same_bits(a.re, b.re) && same_bits(a.im, b.im); }
template <class M> FS_D bool same_state(HdrC<M> a, HdrC<M> b) { return same_bits(a.re, b.re) && same_bits(a.im, b.im) && a.e == b.e; }
template <class Cplx, class IterT> struct StateWatch {
    Cplx saved;
    IterT at, next;
    bool armed;
    FS_D StateWatch(Cplx z, IterT i) : saved(z), at(i), next(i + (IterT)FS_AT_CHUNK), armed(true) {}
    // called with `i` = passes completed, a multiple of FS_AT_CHUNK
    FS_D void after_chunk(Cplx z, IterT &i, IterT at_max, IterT &skipped) {
        if (!armed) return;
        if (same_state(z, saved)) {
            const IterT P = i - at;
            skipped = ((at_max - i) / P) * P;
            i += skipped;
            armed = false;
        } else if (i == next) {
            saved = z;
            next = i + (i - at) * 2;
            at = i;
        }
    }
};

// ---- AT shortcut of one pixel (LAKernel.cuh:66-89, ATInfo.h:128-188) -----------------------------------------------
template <class Num, class IterT, bool Count>
FS_D void lav2_at(const Lav2Args<Num, IterT> &A, const typename Num::Cplx dc, typename Num::Cplx &dz, IterT &iter,
                  unsigned long long &steps_at) {
    using Real = typename Num::Real;
    using Cplx = typename Num::Cplx;
    if (A.la_valid && A.use_at && le_pr(cheb(dc), A.at.ThresholdC)) {
        const IterT at_max = A.n_iterations / A.at.StepLength;
        Cplx c = add(mul(dc, A.at.CCoeff), A.at.RefC);
        reduce(c);
        Cplx z = Num::c_zero();
        IterT i = 0;
        IterT at_skipped = 0; // passes the cycle watch accounted for without executing them
        bool at_done = false;
        if constexpr (Num::kHdr && !Num::kDf) {
            // Fast form of the loop below for the float+exponent types (binary32 and binary64 mantissas): the
            // recurrence on the mantissas with the exponent pinned to c's (fs_at_fast.cuh has the argument and the
            // scalar form that oracle/lockstep_check.cpp runs against the oracle).  7 instructions per pass instead
            // of 38 (HDRx32); on View 14 this loop was 83 % of the frame.
            using M = typename Num::Mant;
            const atfast::Plan<M> plan = atfast::plan<M>(c, A.at.SqrEscapeRadius, at_max > 0);
            if (plan.ok) {
                const M s = plan.s, thr = plan.thr;
                const int E = plan.E;
                M re = M(0), im = M(0);
                // sixteen passes per escape test; if a pass of the chunk escaped, the chunk is replayed pass by pass
                // from its saved start to stop at the exact pass.  Which pass values decide "some pass escaped":
                //  * lean form (plan.mono: R > 4 and |c| <= R/4): once |z|^2 > R, |z'| >= |z|^2 - |c| > 3R/4 > 1.5 sqrt(R),
                //    so |z|^2 stays above R (by a factor > 2.25 per pass, or turns inf/NaN) -- the value entering
                //    the LAST pass of the chunk tells whether any earlier one was over.  No norm, no max on the
                //    other fifteen passes.
                //  * otherwise the running maximum of |z|^2 over the chunk (an overflowed pass shows as +inf before
                //    any NaN can form).
                constexpr int kAtChunk = FS_AT_CHUNK;
                const bool cycle_watch = FS_AT_CYCLE && A.at_cycle;
                auto chunks = [&](auto lean_tag) {
                    constexpr bool kLean = decltype(lean_tag)::value;
                    if constexpr (sizeof(M) == 4 && FS_AT_PACKED) {
                        // (re, im) travel as one packed pair: squares in one FMUL2, the scale-and-add of c in one FFMA2
                        // imaginary part as fma(RN(re*im), 2s, c.im): fs_at_fast.cuh `advance` has the argument
                        const f32x2 s2 = f2_make(s, s + s), c2 = f2_make(c.re, c.im);
                        CycleWatch<float, IterT> watch(re, im, i);
                        while (at_max - i >= (IterT)kAtChunk) { // i <= at_max always; `i + chunk` could wrap for u32 counts near 2^32
                            const float re0 = re, im0 = im;
                            float worst = 0.0f;
                            f32x2 z2 = f2_make(re, im);
#if FS_AT_WATCH_EVERY_PASS
                            unsigned int seen = 0u; // bit u: the state after pass u of this chunk equals the saved one
#endif
#pragma unroll
                            for (int u = 0; u < kAtChunk; u++) {
                                float rr, ii;
                                f2_split(f2_mul(z2, z2), rr, ii);
                                if (!kLean) worst = fmaxf(worst, rr + ii);
                                else if (u == kAtChunk - 1) worst = rr + ii;
                                z2 = f2_fma(f2_make(rr - ii, re * im), s2, c2);
                                f2_split(z2, re, im);
#if FS_AT_WATCH_EVERY_PASS
                                if (__float_as_uint(re) == __float_as_uint(watch.sre) && __float_as_uint(im) == __float_as_uint(watch.sim))
                                    seen |= 1u << u;
#endif
                            }
                            if (!(worst <= thr)) {
                                re = re0;
                                im = im0;
                                break;
                            }
                            i += kAtChunk;
#if FS_AT_WATCH_EVERY_PASS
                            if (cycle_watch) watch.after_chunk_seen(re, im, i, at_max, at_skipped, seen);
#else
                            if (cycle_watch) watch.after_chunk(re, im, i, at_max, at_skipped);
#endif
                        }
                    } else {
                        const M s_im = s + s;
                        CycleWatch<M, IterT> watch(re, im, i);
                        while (at_max - i >= (IterT)kAtChunk) {
                            const M re0 = re, im0 = im;
                            M worst = M(0);
#pragma unroll
                            for (int u = 0; u < kAtChunk; u++) {
                                const M rr = re * re, ii = im * im;
                                if (!kLean) worst = fmax(worst, rr + ii);
                                else if (u == kAtChunk - 1) worst = rr + ii;
                                const M p = re * im;
                                re = fma_(rr - ii, s, c.re);
                                im = fma_(p, s_im, c.im);
                            }
                            if (!(worst <= thr)) {
                                re = re0;
                                im = im0;
                                break;
                            }
                            i += kAtChunk;
                            if (cycle_watch) watch.after_chunk(re, im, i, at_max, at_skipped);
                        }
                    }
                };
                if (FS_AT_LEAN && plan.mono) chunks(std::true_type{});
                else chunks(std::false_type{});
                for (; i < at_max; i++) {
                    if (atfast::escaped(atfast::norm(re, im), thr)) break;
                    atfast::advance(re, im, s, c.re, c.im);
                }
                z.re = re;
                z.im = im;
                z.e = E; // at_max > 0 and the first pass never escapes (|0|^2 <= R): at least one pass completed
                at_done = true;
            }
        }
        StateWatch<Cplx, IterT> gwatch(z, i);
        const bool gwatch_on = FS_AT_CYCLE && A.at_cycle && !at_done;
        for (; !at_done && i < at_max; i++) {
            // every FS_AT_CHUNK passes: has the state been here before?  (see CycleWatch)
            if (gwatch_on && i != 0 && (i % (IterT)FS_AT_CHUNK) == 0 && gwatch.armed) {
                gwatch.after_chunk(z, i, at_max, at_skipped);
                if (!(i < at_max)) break;
            }
            if constexpr (Num::kDf) {
                // 2x32: every operation is an explicit rounded sequence, evaluated as written (ATInfo.h:166-183)
                Real nsq = norm2(z);
                reduce(nsq);
                if (gt_pr(nsq, A.at.SqrEscapeRadius)) break;
                z = add(mul(z, z), c);
            } else {
            // nvcc shares re*re / im*im between norm_squared and z*z in the reference build:
            //   nsq = rr + ii ; z2.re = rr - ii ; z2.im = fma(re, im, re*im)
            const auto rr = z.re * z.re;
            const auto ii = z.im * z.im;
            Real nsq;
            if constexpr (Num::kHdr) { nsq.m = rr + ii; nsq.e = z.e << 1; reduce(nsq); }
            else { nsq = rr + ii; }
            if (gt_pr(nsq, A.at.SqrEscapeRadius)) break;
            Cplx z2;
            z2.re = rr - ii;
            z2.im = fma_(z.re, z.im, z.re * z.im);
            if constexpr (Num::kHdr) z2.e = imax(z.e + z.e, MIN_BIG);
            z = add(z2, c);
            }
        }
        if (Count) steps_at += i - at_skipped;
#ifdef FS_TILE_TIMING
        if (fs_at_passes) {
            const unsigned int k = atomicAdd(&fs_at_passes_n, 1u);
            fs_at_passes[2 * (size_t)k] = (unsigned int)(i - at_skipped);
            fs_at_passes[2 * (size_t)k + 1] = (unsigned int)i;
        }
#endif
        dz = mul(z, A.at.InvZCoeff);
        reduce(dz);
        iter = i * A.at.StepLength;
    }

}

// ---- LA stages of one pixel (LAKernel.cuh:91-127) ---------------------------------------------------------------
template <class Num, class IterT, bool Count>
FS_D void lav2_stages(const Lav2Args<Num, IterT> &A, const typename Num::Cplx dc, typename Num::Cplx &dz,
                      IterT &RefIteration, IterT &iter, unsigned long long &steps) {
    using Real = typename Num::Real;
    using Cplx = typename Num::Cplx;
    using LA = LaRec<Num, IterT>;
    IterT stage = A.la_valid ? A.la_stage_count : 0;
    while (stage > 0) {
        stage--;
        const IterT LAIndex = A.stages[stage].LAIndex;
        // isLAStageInvalid  GPU_LAReference.h:241-255
        if (ge_pr(cheb(dc), A.las[LAIndex].LAThresholdC)) continue;
        const IterT MacroItCount = A.stages[stage].MacroItCount;
        IterT j = RefIteration;

        while (iter < A.n_iterations) {
            // getLA  GPU_LAReference.h:271-303.  The record is fetched whole with 128-bit loads (the reference, and a
            // field-by-field read here, issue one 32-bit load per member: 15 per step).
            const LA *recp = A.las + (LAIndex + j);
            const LA rec = ldg_rec(recp);
            const IterT l = rec.StepLength;
            bool unusable = true;
            Cplx newdz;
            if (iter + l <= A.n_iterations) {
                // Prepare  GPU_LAInfoDeep.h:90-105: newdz = dz * (2*Ref + dz), reduced
                newdz = mul(dz, add(Num::c_mul2(rec.Ref), dz));
                reduce(newdz);
                unusable = ge_pr(cheb(newdz), rec.LAThreshold);
            }
            if (unusable) {
                RefIteration = rec.NextStageLAIndex;
                break;
            }
            iter += l;
            if (Count) steps++;
            // Evaluate  GPU_LAInfoDeep.h:120-123 ; getZ  LAstep.h:181-185
            dz = add(mul(newdz, rec.ZCoeff), mul(dc, rec.CCoeff));
            const Cplx z = add(recp[1].Ref, dz);
            j++;
            Real zn = cheb(z), dn = cheb(dz);
            reduce(zn);
            reduce(dn);
            if (lt_pr(zn, dn) || j >= MacroItCount) {
                dz = z;
                j = 0;
            }
        }
        if (iter >= A.n_iterations) break;
    }
}

// ---- LA stages of one pixel, float+exponent binary32 (HDRx32): the same walk as lav2_stages above, flattened into one
// loop whose body is a single select-free step (fs_la_fast.cuh).  Why: profiled on View 14, the nested form executes
// ~185 warp-instructions per LA step at 22.6 of 32 lanes -- the operand selects of the three aligned additions, the
// zero/clamp special cases of every operation and the stage-transition code all diverge inside a warp.  Here a lane is
// either between stages (a short divergent loop picks the next stage whose threshold admits dc) or takes exactly one step
// per trip; a step the fast form refuses (exact zeros, exponent gaps in [120,127), non-finite values: rare) is redone
// by the reference-shaped operations, which stay the definition of the result.
// The reference-shaped LA step (Prepare GPU_LAInfoDeep.h:90-105, Evaluate :120-123, getZ LAstep.h:181-185) for the steps the
// select-free form refuses.  Out of line: it runs for ~1 % of the steps and its live values must not cost the fast
// loop registers (inlined, the Full kernel needs 76 registers = 3 CTAs per SM instead of 4).
__device__ __noinline__ void la_step_as_written(HdrC<float> Ref, HdrC<float> ZCoeff, HdrC<float> CCoeff, Hdr<float> LAThreshold,
                                                HdrC<float> nref, HdrC<float> dz, HdrC<float> dc, HdrC<float> &ndz,
                                                HdrC<float> &z, bool &unusable, bool &rebase) {
    using Num = NumHdr<float>;
    HdrC<float> newdz = mul(dz, add(Num::c_mul2(Ref), dz));
    reduce(newdz);
    unusable = ge_pr(cheb(newdz), LAThreshold);
    rebase = false;
    if (!unusable) {
        ndz = add(mul(newdz, ZCoeff), mul(dc, CCoeff));
        z = add(nref, ndz);
        Hdr<float> zn = cheb(z), dn = cheb(ndz);
        reduce(zn);
        reduce(dn);
        rebase = lt_pr(zn, dn);
    }
}

template <class IterT, bool Count>
FS_D void lav2_stages_hdr32(const Lav2Args<NumHdr<float>, IterT> &A, const HdrC<float> dc, HdrC<float> &dz,
                            IterT &RefIteration, IterT &iter, unsigned long long &steps) {
    using Num = NumHdr<float>;
    using Real = Hdr<float>;
    using Cplx = HdrC<float>;
    using LA = LaRec<Num, IterT>;
    IterT stage = A.la_valid ? A.la_stage_count : 0;
    IterT LAIndex = 0, MacroItCount = 0, j = 0;
    bool need_stage = true;
    for (;;) {
        while (need_stage) {
            if (stage == 0) return;
            stage--;
            const StageRec<IterT> sr = A.stages[stage];
            LAIndex = sr.LAIndex;
            // isLAStageInvalid  GPU_LAReference.h:241-255
            if (ge_pr(cheb(dc), A.las[LAIndex].LAThresholdC)) continue;
            MacroItCount = sr.MacroItCount;
            j = RefIteration;
            need_stage = false;
            if (!(iter < A.n_iterations)) return;
        }
        // getLA  GPU_LAReference.h:271-303: the record is fetched whole with 128-bit loads
        const LA *recp = A.las + (LAIndex + j);
        const LA rec = ldg_rec(recp);
        const IterT l = rec.StepLength;
        bool unusable = true, rebase = false;
        Cplx ndz = dz, z = dz;
        if (iter + l <= A.n_iterations) {
            const Cplx nref = recp[1].Ref;
            lafast::StepOut o;
            if (lafast::step(rec.Ref.re, rec.Ref.im, rec.Ref.e, rec.ZCoeff.re, rec.ZCoeff.im, rec.ZCoeff.e, rec.CCoeff.re,
                             rec.CCoeff.im, rec.CCoeff.e, rec.LAThreshold.m, rec.LAThreshold.e, nref.re, nref.im, nref.e,
                             dz.re, dz.im, dz.e, dc.re, dc.im, dc.e, o)) {
                unusable = o.unusable;
                rebase = o.rebase;
                ndz.re = o.dz.re; ndz.im = o.dz.im; ndz.e = o.dz.e;
                z.re = o.z.re; z.im = o.z.im; z.e = o.z.e;
            } else {
                // results come back through locals of this branch only: the loop's own variables stay in registers
                Cplx s_ndz, s_z;
                bool s_unusable, s_rebase;
                la_step_as_written(rec.Ref, rec.ZCoeff, rec.CCoeff, rec.LAThreshold, nref, dz, dc, s_ndz, s_z, s_unusable, s_rebase);
                unusable = s_unusable;
                rebase = s_rebase;
                if (!s_unusable) { ndz = s_ndz; z = s_z; }
            }
        }
        if (unusable) {
            RefIteration = rec.NextStageLAIndex;
            need_stage = true;
            continue;
        }
        iter += l;
        if (Count) steps++;
        j++;
        const bool rb = rebase || j >= MacroItCount;
        dz = rb ? z : ndz;
        j = rb ? (IterT)0 : j;
        if (!(iter < A.n_iterations)) return;
    }
}

// ---- LA stages of one pixel, HDRx32 / 32-bit counts, on la2 records (fs_la_step2.cuh): the walk of lav2_stages above ----
// The reference-shaped step for what la2::step refuses; reads the reference-layout record.  Out of line (rare).
__device__ __noinline__ void la_step_refused(const LaRec<NumHdr<float>, uint32_t> *recp, HdrC<float> dz, HdrC<float> dc,
                                             la2::Out &o) {
    const LaRec<NumHdr<float>, uint32_t> rec = ldg_rec(recp);
    HdrC<float> ndz = dz, z = dz;
    bool unusable, rebase;
    la_step_as_written(rec.Ref, rec.ZCoeff, rec.CCoeff, rec.LAThreshold, recp[1].Ref, dz, dc, ndz, z, unusable, rebase);
    o.unusable = unusable;
    o.rebase = rebase;
    o.dre = ndz.re; o.dim = ndz.im; o.de = ndz.e;
    o.zre = z.re; o.zim = z.im; o.ze = z.e;
}

template <bool Count>
FS_D void lav2_stages_v2(const Lav2Args<NumHdr<float>, uint32_t> &A, const HdrC<float> dc, HdrC<float> &dz,
                         uint32_t &RefIteration, uint32_t &iter, unsigned long long &steps) {
    const uint4 *__restrict__ recs = reinterpret_cast<const uint4 *>(A.las2);
    const uint4 *__restrict__ stages = reinterpret_cast<const uint4 *>(A.stages2);
    const Hdr<float> dcn = cheb(dc);
    uint32_t stage = A.la_valid ? A.la_stage_count : 0;
    while (stage > 0) {
        stage--;
        const uint4 sr = __ldg(stages + stage); // {LAIndex, MacroItCount, LAThresholdC.m, LAThresholdC.e}
        // isLAStageInvalid  GPU_LAReference.h:241-255
        if (ge_pr(dcn, hdr_make<float>((int)sr.w, __uint_as_float(sr.z)))) continue;
        const uint32_t LAIndex = sr.x, MacroItCount = sr.y;
        uint32_t j = RefIteration;
        while (iter < A.n_iterations) {
            // getLA  GPU_LAReference.h:271-303
            const uint4 *rp = recs + 4 * (size_t)(LAIndex + j);
#if FS_LA2_LDG256
            // two 256-bit loads (sm_100 LDG.256): half the L1 wavefronts of four 128-bit ones when the lanes of the warp are
            // on different records
            uint4 q0, q1, q2, q3;
            asm("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                : "=r"(q0.x), "=r"(q0.y), "=r"(q0.z), "=r"(q0.w), "=r"(q1.x), "=r"(q1.y), "=r"(q1.z), "=r"(q1.w) : "l"(rp));
            asm("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8+32];"
                : "=r"(q2.x), "=r"(q2.y), "=r"(q2.z), "=r"(q2.w), "=r"(q3.x), "=r"(q3.y), "=r"(q3.z), "=r"(q3.w) : "l"(rp));
#else
            const uint4 q0 = __ldg(rp), q1 = __ldg(rp + 1), q2 = __ldg(rp + 2), q3 = __ldg(rp + 3);
#endif
#if FS_LA2_PREFETCH
            // the next trip reads the following record unless this one rebases or leaves the stage
            asm volatile("prefetch.global.L1 [%0];" ::"l"(rp + 4));
            asm volatile("prefetch.global.L1 [%0];" ::"l"(rp + 6));
#endif
            // The StepLength test follows the step instead of guarding it: ahead of the step it is the first branch, it reads
            // only the second load, and the compiler sinks the first load below it -- a trip then waits for two load
            // latencies in a row.  A step past the iteration limit (a pixel's last LA step, at most once per stage) is
            // computed and dropped.
            const uint32_t l = q2.w;
            la2::Out o;
            if (!la2::step(q0, q1, q2, q3, dz.re, dz.im, dz.e, dc.re, dc.im, dc.e, o)) {
                // results come back through a local of this branch only: `o` stays in registers
                la2::Out slow;
                la_step_refused(A.las + (LAIndex + j), dz, dc, slow);
                o = slow;
            }
            if (o.unusable || iter + l > A.n_iterations) {
                RefIteration = q3.w;
                break;
            }
            iter += l;
            if (Count) steps++;
            j++;
            const bool rb = o.rebase || j >= MacroItCount;
            dz.re = rb ? o.zre : o.dre;
            dz.im = rb ? o.zim : o.dim;
            dz.e = rb ? o.ze : o.de;
            j = rb ? 0u : j;
        }
        if (iter >= A.n_iterations) break;
    }
}

// Layout Frames renders a zoom batch: A.n_frames frames that share the orbit and the tables, each with its own pixel
// spacing, centre offset and iteration buffer (A.frames).  The queue hands out n_frames x n_tiles tickets, frame-major,
// so the SMs that finish frame k's cheap tiles pick up frame k + 1's while frame k's expensive tiles still run: only the
// last frame's tail is left at the end of the launch.  Tiles of every frame keep the centre-out order and the shard rule.
// No result sink, no probe order.
// Layout ExpMap renders an exponential map: pixel (X, Y) takes dc = expmap_dc(radius[Y], dir_x[X], dir_y[X]) in place of
// the linear map's delta_x / delta_y; everything else -- queue, shard rule, store, result sink, step counters -- is the
// single-frame code.  No probe order (lav2_probe_kernel assumes the linear map).
template <class Num, class IterT, Lav2Mode Mode, bool Count, AtPhase Phase = AtPhase::Fused,
          Lav2Layout Layout = Lav2Layout::Rect>
__global__ void FS_LAV2_BOUNDS(Num) lav2_kernel(const Lav2Args<Num, IterT> A) {
    using Real = typename Num::Real;
    using Cplx = typename Num::Cplx;
    constexpr bool Frames = Layout == Lav2Layout::Frames;
    static_assert(Layout == Lav2Layout::Rect || Phase == AtPhase::Fused, "zoom batches and exp maps run the fused kernel");

    const int lane = threadIdx.x & 31;
    const int tiles_x = (A.width + 7) >> 3;
    const int tiles_y = (((A.height + 3) >> 2) - A.shard_index + A.shard_count - 1) / A.shard_count;
    const unsigned int n_tiles = (unsigned int)tiles_x * (unsigned int)tiles_y;
    const unsigned int n_tickets = Frames ? n_tiles * A.n_frames : n_tiles;
    unsigned long long steps = 0, steps_at = 0, steps_la = 0;

    TileCursor cursor;
    tile_queue_begin(cursor);
    for (;;) {
        unsigned int tile;
        if (!next_tile(A.queue, cursor, n_tickets, tile)) break;
        Real fdx = A.dx, fdy = A.dy, fcx = A.centerX, fcy = A.centerY;
        if constexpr (Frames) {
            const unsigned int frame = tile / n_tiles; // warp-uniform
            tile -= frame * n_tiles;
            const Lav2Frame<Num, IterT> *fr = A.frames + frame;
            fdx = fr->dx;
            fdy = fr->dy;
            fcx = fr->centerX;
            fcy = fr->centerY;
        }

#ifdef FS_TILE_TIMING
        const long long fs_t0 = clock64();
        unsigned long long fs_g0;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(fs_g0));
#endif
        if (Layout == Lav2Layout::Rect && A.order) {
            // two lists filled by lav2_probe_kernel, each in ticket (centre-out) order: expensive tiles, then the rest
            const unsigned int n_first = *(const volatile unsigned int *)(A.order + 2 * (size_t)n_tiles);
            tile = tile < n_first ? __ldg(A.order + tile) : __ldg(A.order + n_tiles + (tile - n_first));
        }
        int X, Y;
        tile_origin(tile, tiles_x, tiles_y, A.shard_count, A.shard_index, X, Y);
        X += lane & 7;
        Y += lane >> 3;
        // lanes outside the image stay with the warp (the perturbation loop is warp-synchronous) and do nothing
        const bool live = X < A.width && Y < A.height;

        IterT iter = 0;
        IterT RefIteration = 0;
        Real dcX, dcY;
        if constexpr (Layout == Lav2Layout::ExpMap) {
            // lanes outside the image read the last row / column: their cells are never stored
            const int tx = X < A.width ? X : A.width - 1, ty = Y < A.height ? Y : A.height - 1;
            expmap_dc<Num>(A.exp_radius[ty], A.exp_dir_x[tx], A.exp_dir_y[tx], dcX, dcY);
        } else {
            // LAKernel.cuh:41-42 (no reduction of the deltas here)
            dcX = Num::delta_x(fdx, X, fcx);
            dcY = Num::delta_y(fdy, Y, fcy);
        }
        const Cplx dc = Num::c_make(dcX, dcY);
        Cplx dz = Num::c_zero();

        if constexpr (Phase == AtPhase::AtOnly) {
            if constexpr (Num::kHdr && !Num::kDf && sizeof(typename Num::Mant) == 4) {
                if (live) {
                    lav2_at<Num, IterT, Count>(A, dc, dz, iter, steps_at);
                    const size_t cell = (size_t)Y * A.pitch + X;
                    A.at_state[cell] = make_float4(dz.re, dz.im, __int_as_float(dz.e), 0.0f);
                    A.out[cell] = iter;
                }
            }
            __syncwarp();
            continue;
        }
        if constexpr (Mode == Lav2Mode::Full || Mode == Lav2Mode::LAO) {
            if (live) {
                if constexpr (Phase == AtPhase::AfterAt && Num::kHdr && !Num::kDf && sizeof(typename Num::Mant) == 4) {
                    const size_t cell = (size_t)Y * A.pitch + X;
                    const float4 st = A.at_state[cell];
                    dz.re = st.x; dz.im = st.y; dz.e = __float_as_int(st.z);
                    iter = A.out[cell];
                } else {
                    lav2_at<Num, IterT, Count>(A, dc, dz, iter, steps_at);
                }
                if constexpr (Num::kHdr && !Num::kDf && sizeof(typename Num::Mant) == 4 && sizeof(IterT) == 4 && FS_LA_STEP2) {
                    if (A.las2 != nullptr) lav2_stages_v2<Count>(A, dc, dz, RefIteration, iter, steps_la);
                    else lav2_stages<Num, IterT, Count>(A, dc, dz, RefIteration, iter, steps_la);
                } else if constexpr (Num::kHdr && !Num::kDf && sizeof(typename Num::Mant) == 4 && FS_LA_FAST)
                    lav2_stages_hdr32<IterT, Count>(A, dc, dz, RefIteration, iter, steps_la);
                else
                    lav2_stages<Num, IterT, Count>(A, dc, dz, RefIteration, iter, steps_la);
            }
        }

        if constexpr (Mode == Lav2Mode::Full || Mode == Lav2Mode::PO) {
            // ---- plain perturbation with rebasing (LAKernel.cuh:130-236) ----
            Real dX = Num::c_re(dz), dY = Num::c_im(dz);
            PerturbLoop<Num, IterT, Count>::run(live, A.orbit, A.orbit_fast, A.orbit_count, A.n_iterations, dcX, dcY, dX, dY,
                                                RefIteration, iter, steps);
        }

        if (live) {
            const size_t cell = (size_t)Y * A.pitch + X;
            if constexpr (Frames) {
                // this tile's ticket is cursor.cur - 1 (next_tile hands out `cur` and advances it): the frame is derived
                // again here rather than held across the tile, which would cost HDRx32 a register beyond its bound of 64
                A.frames[(cursor.cur - 1) / n_tiles].out[cell] = iter;
            } else {
                A.out[cell] = iter;
                if (A.sink) A.sink[cell] = iter; // 8 lanes per row: one 32-byte posted write
            }
        }
#ifdef FS_TILE_TIMING
        if (lane == 0 && fs_tile_times) {
            fs_tile_times[2 * (size_t)tile] = fs_g0;                                  // start, ns (global timer)
            fs_tile_times[2 * (size_t)tile + 1] = (unsigned long long)(clock64() - fs_t0); // duration, SM cycles
        }
#endif
    }

    if (Count && A.step_counter) {
        // one atomic per warp and counter: [0] all executed steps, [1] AT passes, [2] LA steps
        steps += steps_at + steps_la;
        for (int o = 16; o > 0; o >>= 1) {
            steps += __shfl_down_sync(0xffffffffu, steps, o);
            steps_at += __shfl_down_sync(0xffffffffu, steps_at, o);
            steps_la += __shfl_down_sync(0xffffffffu, steps_la, o);
        }
        if (lane == 0 && steps) atomicAdd(A.step_counter, steps);
        if (lane == 0 && steps_at) atomicAdd(A.step_counter + 1, steps_at);
        if (lane == 0 && steps_la) atomicAdd(A.step_counter + 2, steps_la);
    }
}

// ---- cost probe for small shards --------------------------------------------------------------------------------------
// Once a GPU's share of the frame is a handful of tiles per resident warp (8 GPUs on View 14: 6.9), the launch lasts as long
// as its latest-finishing warp, and that is a warp that drew an expensive tile late: the interior pixels next to the set's
// boundary, whose AT passes settle into a cycle only after thousands of passes or never (View 14: 0.5 % of the pixels
// run more than 4,096 of the 18,402 passes; such a tile lasts 0.5 ms of a 0.7 ms launch wherever it starts).  This kernel
// runs the first `A.n_iterations / StepLength` AT passes (the host passes a copy of the arguments with a small limit) of
// the four corner pixels of every tile of the shard and writes the queue order: tiles with a corner that neither escaped
// nor cycled within the limit first, the rest behind them.  Results do not depend on the order; the launch time does.
template <class IterT>
__global__ void __launch_bounds__(256) lav2_probe_kernel(const Lav2Args<NumHdr<float>, IterT> A, unsigned int *order,
                                                         unsigned int *heads) {
    using Num = NumHdr<float>;
    const int tiles_x = (A.width + 7) >> 3;
    const int tiles_y = (((A.height + 3) >> 2) - A.shard_index + A.shard_count - 1) / A.shard_count;
    const unsigned int n_tiles = (unsigned int)tiles_x * (unsigned int)tiles_y;
    const unsigned int t = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned int ticket = t >> 2;
    const int corner = (int)(t & 3u);
    bool slow = false;
    if (ticket < n_tiles) {
        int X, Y;
        tile_origin(ticket, tiles_x, tiles_y, A.shard_count, A.shard_index, X, Y);
        X += (corner & 1) ? 7 : 0;
        Y += (corner & 2) ? 3 : 0;
        if (X < A.width && Y < A.height) {
            const typename Num::Real dcX = Num::delta_x(A.dx, X, A.centerX);
            const typename Num::Real dcY = Num::delta_y(A.dy, Y, A.centerY);
            const typename Num::Cplx dc = Num::c_make(dcX, dcY);
            typename Num::Cplx dz = Num::c_zero();
            IterT iter = 0;
            unsigned long long passes = 0;
            lav2_at<Num, IterT, true>(A, dc, dz, iter, passes);
            slow = passes >= (unsigned long long)(A.n_iterations / A.at.StepLength);
        }
    }
    // the four corners of a tile sit in adjacent lanes
    const unsigned int votes = __ballot_sync(0xffffffffu, slow);
    const bool tile_slow = ((votes >> ((threadIdx.x & 31) & ~3)) & 0xfu) != 0u;
    // flags live in the second list's space until lav2_order_kernel turns them into the two lists
    if (corner == 0 && ticket < n_tiles) order[n_tiles + ticket] = tile_slow ? 1u : 0u;
}

// Stable partition of the tickets by the probe's flag (one CTA; a shard that is probed has a few ten thousand tiles):
// order[0 .. n_first) = flagged tickets, order[n_tiles .. ) = the others, both ascending, i.e. still centre-out -- warps
// that run side by side keep working on neighbouring tiles and find each other's LA records and orbit elements in L1.
__global__ void __launch_bounds__(1024) lav2_order_kernel(unsigned int *order, unsigned int *heads, unsigned int n_tiles) {
    __shared__ unsigned int sums[1024];
    const unsigned int per = (n_tiles + 1023u) / 1024u;
    const unsigned int lo = min(threadIdx.x * per, n_tiles), hi = min(lo + per, n_tiles);
    unsigned int mine = 0;
    for (unsigned int k = lo; k < hi; k++) mine += order[n_tiles + k];
    sums[threadIdx.x] = mine;
    __syncthreads();
    for (unsigned int o = 1; o < 1024u; o <<= 1) { // inclusive scan
        const unsigned int v = threadIdx.x >= o ? sums[threadIdx.x - o] : 0u;
        __syncthreads();
        sums[threadIdx.x] += v;
        __syncthreads();
    }
    unsigned int before = sums[threadIdx.x] - mine; // flagged tickets below `lo`
    // the flags share the second list's space: every thread copies its flags out before anyone writes a slot
    unsigned int local[64];
    const bool fits = per <= 64u;
    if (fits) for (unsigned int k = lo; k < hi; k++) local[k - lo] = order[n_tiles + k];
    __syncthreads();
    if (fits) {
        for (unsigned int k = lo; k < hi; k++) {
            if (local[k - lo]) order[before++] = k;
            else order[n_tiles + (k - before)] = k;
        }
    }
    if (threadIdx.x == 1023) heads[0] = fits ? sums[1023] : 0u;
    if (!fits && threadIdx.x == 0) heads[1] = 1u; // caller never asks for more than 64 * 1024 tiles
}

} // namespace fs
