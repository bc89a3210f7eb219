"""Exact escape-time reference for the direct kernels (Gpu1x32, Gpu1x64, Gpu2x32, Gpu2x64, Gpu4x32, Gpu4x64, GpuHDRx32).

Pure Python, no native code.  For a pixel with c = (cx + X dx, cy + Y dy) -- the coordinate PODs decoded exactly as the
sum of their limbs, Y the kernel's own (flipped) row -- z <- z^2 + c is iterated on integers in fixed point with
ArithModel.ref_bits fraction bits, together with a radius per component ("ball"): every value the kernel's arithmetic
can hold at that step lies in [X - rx, X + rx] x [Y - ry, Y + ry].  Each step the radius grows by the propagated error
(|x^2 - X^2| <= 2|X| rx + rx^2, |xy - XY| <= |X| ry + |Y| rx + rx ry), by the error of the kernel's own step (the
per-type model below, whose per-operation bounds tests/test_exact_escape.py checks against exact arithmetic) and by the
truncation of the fixed-point centre.  While every operand and result of the step is a single limb of the kernel's
type (p-bit significand, normal range), the kernel computes exactly and the radius stays exactly 0.

A pixel is *certified* when at every step where the kernel tests for bailout the whole ball -- including the rounding
of the test itself -- lies on one side of the test.  Its count is then the kernel's count whatever the rounding inside
the ball.  Once the whole ball satisfies |z| >= max(2, |c|) + 1/4 the orbit escapes mathematically and the kernel's
(rounded) orbit grows with it into inf / NaN, which every bailout test reads as escaped: the pixel escapes at the next
decision step and the iteration stops there.
"""
from __future__ import annotations

import math
import multiprocessing as mp
import struct
from dataclasses import dataclass
from fractions import Fraction


@dataclass(frozen=True)
class ArithModel:
    """Error model of one direct kernel's number type.

    limb_bits   significand bits of one limb (binary32: 24, binary64: 53); u = 2^-limb_bits
    limbs       limbs per number (1, 2, 4)
    sub_min     spacing of the limb format's subnormals (the build does not flush to zero)
    eps_add, eps_mul, eps_sqr, eps_scal
                |computed - exact| <= eps * (sum of the operands' magnitudes) for add/sub, eps * |a||b| for products,
                eps * |a|^2 for squares, eps * |a||s| for a number times a limb, each plus floor_op
    floor_op    absolute error floor of one operation (underflow into the subnormal range of the lowest limbs)
    hdr         HDRFloat<CudaDblflt> (GpuHDRx32): fed an HDRFloat<double> POD {f64 m, int32 exp, pad}, which the C-ABI
                splits into head = (float)m, tail = (float)(m - head), renormalised exactly (fs_capi.cu hdr2x32_from_hdr64)
    """
    name: str
    limb_bits: int
    limbs: int
    sub_min: float
    eps_add: float
    eps_mul: float
    eps_sqr: float
    eps_scal: float
    floor_op: float
    hdr: bool = False

    @property
    def u(self) -> float:
        return 2.0 ** -self.limb_bits

    @property
    def ref_bits(self) -> int:
        """Fraction bits of the reference: four times the type's precision plus 64."""
        return 4 * self.limb_bits * self.limbs + 64


_F32_SUB, _F64_SUB = 2.0 ** -149, 2.0 ** -1074
# 1x: the kernels round each FMA downwards: below 1 ulp of the result, i.e. < 2u |result| + the subnormal spacing.
F32 = ArithModel("f32", 24, 1, _F32_SUB, 0.0, 0.0, 0.0, 0.0, _F32_SUB)
F64 = ArithModel("f64", 53, 1, _F64_SUB, 0.0, 0.0, 0.0, 0.0, _F64_SUB)
# double-word (df32 = dblflt, dd64 = dbldbl).  add/sub is AccurateDWPlusDW (Thall's form): relative error
# <= 3u^2 / (1 - 4u) of |a + b| (Joldes, Muller, Popescu, "Tight and rigorous error bounds for basic building blocks of
# double-word arithmetic", ACM TOMS 44(2), 2017, Thm 3.1); stated here against |a| + |b| >= |a + b| as 4u^2.  mul:
# th + err(th) is exact (FMA), the three FMAs that add a.t b.t, a.h b.t and a.t b.h into tt round values of at most
# u|ab|, 2u|ab|, 3u|ab| (each <= u times that), the final Fast2Sum is exact: < 6u^2 |a||b| (1 + O(u)), stated as 8u^2.
# sqr: the same with one product e = a.h a.t rounded and doubled: < 8u^2 |a|^2.  The floor: every rounding of the tail
# chain may fall into the subnormal range.
DF32 = ArithModel("df32", 24, 2, _F32_SUB, 4 * 2.0 ** -48, 8 * 2.0 ** -48, 8 * 2.0 ** -48, 8 * 2.0 ** -48, 8 * _F32_SUB)
DD64 = ArithModel("dd64", 53, 2, _F64_SUB, 4 * 2.0 ** -106, 8 * 2.0 ** -106, 8 * 2.0 ** -106, 8 * 2.0 ** -106, 8 * _F64_SUB)
# four-limb (QD's sloppy operations, fs_qd.cuh).  TwoSum / TwoProd are error-free, so every partial term down to
# order u^3 of the operands is carried exactly; what is rounded or dropped is of order u^4 relative to the operands'
# magnitudes: add -- the rounded b = t2 + t3 of three_sum2, the two roundings of t0 + t1 + t3 and the last `s3 += c4`
# of renorm (<= ~4 u^4 (|a| + |b|)); sloppy mul -- the dropped products a.y b.w, a.z b.z, a.w b.y and smaller, the
# rounded order-u^3 products and their sum, the errors q0, q3..q5 summed in plain arithmetic (<= ~12 u^4 |a||b|);
# sqr the same terms (<= ~12 u^4 |a|^2); times a limb -- a.w b rounded and q2 + p2 (<= ~4 u^4 |a||b|).  Stated with a
# factor 4 of margin.  Against the SUM of the operands' magnitudes, not the result: under cancellation a ~ -b the
# sloppy add keeps this absolute error while the result shrinks (the reference's algorithm, not a port fault).
# The floor: the fourth limb of a Quad<float> is subnormal once |value| < 2^-54 (the third once < 2^-78); every one of
# the ~16 roundings of an operation can then lose up to the subnormal spacing.
QF32 = ArithModel("qf32", 24, 4, _F32_SUB, 16 * 2.0 ** -96, 48 * 2.0 ** -96, 48 * 2.0 ** -96, 16 * 2.0 ** -96, 16 * _F32_SUB)
QD64 = ArithModel("qd64", 53, 4, _F64_SUB, 16 * 2.0 ** -212, 48 * 2.0 ** -212, 48 * 2.0 ** -212, 16 * 2.0 ** -212,
                  16 * _F64_SUB)
# HDR over 2x32 (GpuHDRx32): the mantissa operations are dblflt's (the DF32 bounds, checked through
# fs_selftest_numeric_op 85 as well); the exponent removes underflow.  What is left as an absolute floor: operands
# dropped at exponent gaps >= 120 (below 2^-115 for the values |v| < 32 of an iteration that has not escaped) and
# Reduce's rebasing of a zero tail, which leaves it as 2^(-k - 127) for a head of exponent -k < 0 (fs_df32.cuh
# reduce, the reference's): a relative error below 2^-125 per Reduce.
HDF32 = ArithModel("hdf32", 24, 2, 0.0, 4 * 2.0 ** -48, 8 * 2.0 ** -48, 8 * 2.0 ** -48, 8 * 2.0 ** -48, 2.0 ** -100,
                   hdr=True)
MODELS = {m.name: m for m in (F32, F64, DF32, DD64, QF32, QD64, HDF32)}


@dataclass(frozen=True)
class Kernel:
    """Count convention of one direct kernel, read from fs_direct.cuh / fs_direct_ext.cuh.

    strict      bailout `value < 4` (True) or `value <= 4` (False)
    cap_minus   the limit is n_iterations - (P - 1) (the 1x kernels) instead of n_iterations
    step        which step the kernel executes ('1x', '2x32', '2x64', '4x32', '4x64', 'hdr2x32')
    """
    name: str
    model: ArithModel
    strict: bool
    cap_minus: bool
    step: str
    precisions: tuple


KERNELS = {
    "Gpu1x32": Kernel("Gpu1x32", F32, True, True, "1x", (1, 4, 8, 16)),      # fma(x, x, y*y) < 4
    "Gpu1x64": Kernel("Gpu1x64", F64, True, True, "1x", (1, 4, 8, 16)),
    "Gpu2x32": Kernel("Gpu2x32", DF32, True, False, "2x32", (1, 4, 8, 16)),  # zr.head + zi.head < 4
    "Gpu2x64": Kernel("Gpu2x64", DD64, True, False, "2x64", (1,)),           # __dadd_rn(zr.head, zi.head) < 4
    "Gpu4x32": Kernel("Gpu4x32", QF32, False, False, "4x32", (1,)),          # le(add(zr, zi), 4)
    "Gpu4x64": Kernel("Gpu4x64", QD64, False, False, "4x64", (1,)),
    "GpuHDRx32": Kernel("GpuHDRx32", HDF32, True, False, "hdr2x32", (1, 4, 8, 16)),  # cmp_pr(reduced |z|^2, 4) < 0
}


# ---- coordinate PODs ----------------------------------------------------------------------------------------------
def _f32(v: float) -> float:
    return struct.unpack("<f", struct.pack("<f", v))[0]


def pod_limbs(raw: bytes, model: ArithModel) -> list:
    """The limbs of one coordinate POD (little-endian binary32 / binary64 limbs, most significant first); HDR: the
    head and tail the kernel holds, without the exponent."""
    if model.hdr:
        m = struct.unpack("<d", raw[:8])[0]
        a = _f32(m)
        return [a, _f32(m - a)]
    fmt = "<%d%s" % (model.limbs, "f" if model.limb_bits == 24 else "d")
    return list(struct.unpack(fmt, raw))


def pod_value(raw: bytes, model: ArithModel) -> Fraction:
    """The exact value of a coordinate POD as the kernel holds it: the sum of its limbs as dyadic rationals (HDR: times
    2^exp)."""
    v = sum((Fraction(v) for v in pod_limbs(raw, model)), Fraction(0))
    if model.hdr:
        v *= Fraction(2) ** struct.unpack("<i", raw[8:12])[0]
    return v


def pack_pod(value, model: ArithModel) -> bytes:
    """A POD whose limbs are the greedy round-to-nearest expansion of `value` (exact for dyadic values that fit); HDR:
    of the mantissa in [1, 2), or the zero at MIN_BIG."""
    rest, limbs = Fraction(value), []
    fmt = "f" if model.limb_bits == 24 else "d"
    if model.hdr:
        if rest == 0:
            return struct.pack("<di4x", 0.0, -(2 ** 31) >> 3)
        e = 0
        while abs(rest) >= 2:
            rest, e = rest / 2, e + 1
        while abs(rest) < 1:
            rest, e = rest * 2, e - 1
        return struct.pack("<di4x", float(rest), e)
    for _ in range(model.limbs):
        v = float(rest)
        if fmt == "f":
            v = struct.unpack("<f", struct.pack("<f", v))[0]
        limbs.append(v)
        rest -= Fraction(v)
    return struct.pack("<%d%s" % (model.limbs, fmt), *limbs)


def representable(n: int, P: int, limb_bits: int) -> bool:
    """n / 2^P is 0 or a normal limb value (significand of limb_bits bits, 2^-100 <= |v| < 2^100)."""
    if n == 0:
        return True
    a = abs(n)
    tz = (a & -a).bit_length() - 1
    if (a >> tz).bit_length() > limb_bits:
        return False
    e = a.bit_length() - 1 - P
    return -100 <= e < 100


def _to_fixed(q: Fraction, P: int):
    """floor(q 2^P) and whether it is exact."""
    num, den = q.numerator << P, q.denominator
    n, r = divmod(num, den)
    return n, r == 0


# ---- one pixel --------------------------------------------------------------------------------------------------
_SLOP = 1.0 + 2.0 ** -40   # covers the rounding of the radius arithmetic itself (a handful of binary64 operations)


def _step_errors(k: Kernel, ax: float, ay: float, ax0: float, ay0: float):
    """(error bound of the kernel's new x, of its new y, of its bailout value) for one step from |x| <= ax, |y| <= ay,
    in terms of the per-operation model of k.model (see ArithModel)."""
    m = k.model
    u, fl = m.u, m.floor_op
    x2, y2, xy = ax * ax, ay * ay, ax * ay
    if k.step == "1x":
        # t = fma_rd(-y, y, x0); x' = fma_rd(x, x, t); y' = fma_rd(x + x, y, y0)  (x + x exact)
        ex = 2 * u * (1 + 4 * u) * (x2 + 2 * y2 + 2 * ax0) + 3 * fl
        ey = 2 * u * (1 + 2 * u) * (2 * xy + ay0) + 2 * fl
        # fma(x, x, fl(y*y)): two roundings to nearest
        et = 2 * u * (1 + 2 * u) * (x2 + y2) + 2 * fl
        return ex, ey, et
    if k.step in ("2x32", "2x64", "hdr2x32"):
        eA, eM, eS = m.eps_add, m.eps_mul, m.eps_sqr
        eZ = eS if k.step == "2x32" else eM        # zr = df_sqr(x) / dd_mul(x, x) / mul(x, x)
        mag = (1 + 4 * u)                           # |head| + |tail| vs |value|
        # x' = add(sub(zr, zi), x0): zr, zi carry their own rounding into the next step
        ex = (eZ * (x2 + y2) + eA * 2 * (x2 + y2) * (1 + eZ) + eA * ax0) * mag * mag + 5 * fl
        # y' = add(2 * mul(x, y), y0)  (the doubling is exact)
        ey = (2 * eM * xy + eA * (2 * xy * (1 + eM) + ay0)) * mag * mag + 3 * fl
        if k.step == "hdr2x32":
            # zs = reduced(add(zr, zi)), compared in full (cmp_pr)
            return ex, ey, (eZ * (x2 + y2) + eA * (x2 + y2) * (1 + eZ)) * mag * mag + 3 * fl
        # zr.head + zi.head, rounded: |zr - zr.head| <= u |zr.head|, one more rounding of the sum
        et = (3 * u * (x2 + y2)) * mag * mag + 3 * fl
        return ex, ey, et
    # four limbs
    eA, eM, eS, eQ = m.eps_add, m.eps_mul, m.eps_sqr, m.eps_scal
    eZ = eS if k.step == "4x32" else eM            # zr = sqr(x) / mul(x, x)
    mag = (1 + 4 * u)
    ex = (eZ * (x2 + y2) + eA * 2 * (x2 + y2) * (1 + eZ) + eA * ax0) * mag * mag + 4 * fl
    e2 = 0.0 if k.step == "4x32" else eQ * 2 * xy   # mul_pwr2 is exact, mul(q, 2.0) is modelled
    ey = (2 * eM * xy + 2 * e2 + eA * (2 * xy * (1 + eM) + ay0)) * mag * mag + 4 * fl
    et = (eZ * (x2 + y2) + eA * (x2 + y2) * (1 + eZ)) * mag * mag + 3 * fl
    return ex, ey, et


def _c_radius(k: Kernel, c: Fraction, base: Fraction, delta: Fraction, idx: int) -> float:
    """Bound of |kernel's x0 - c| for x0 computed from base + idx * delta as the kernel does."""
    m = k.model
    ac, ab, ad = abs(float(c)), abs(float(base)), abs(float(delta)) * abs(idx)
    if k.step == "1x":                 # fma(X, dx, cx), rounded to nearest
        return (m.u * ac + m.sub_min) * _SLOP
    # the product delta * idx, then the sum base + product
    prod = (m.eps_scal if k.step == "4x64" else m.eps_mul) * ad
    return ((prod + m.eps_add * (ab + ad * (1 + m.eps_mul))) * (1 + 4 * m.u) + 3 * m.floor_op) * _SLOP


def escape_count(k: Kernel, cx: Fraction, cy: Fraction, dx: Fraction, dy: Fraction, X: int, Y: int, n_iterations: int,
                 precision: int = 1, model: ArithModel | None = None):
    """(count, certified) for the kernel's pixel (X, Y) (Y: the kernel's own, flipped row).  `model` overrides the
    arithmetic model (e.g. to ask what double-double would certify on a window)."""
    if model is not None:
        k = Kernel(k.name, model, k.strict, k.cap_minus, k.step, k.precisions)
    m = k.model
    P = m.ref_bits
    ONE = 1 << P
    INV = 2.0 ** -P
    cap = n_iterations - (precision - 1) if k.cap_minus else n_iterations
    c_re, c_im = cx + X * dx, cy + Y * dy
    Cx, ex_c = _to_fixed(c_re, P)
    Cy, ey_c = _to_fixed(c_im, P)
    lb = m.limb_bits
    exact = ex_c and ey_c and representable(Cx, P, lb) and representable(Cy, P, lb)
    if exact:
        rcx = rcy = 0.0
    else:
        rcx = _c_radius(k, c_re, cx, dx, X) + (0.0 if ex_c else INV)
        rcy = _c_radius(k, c_im, cy, dy, Y) + (0.0 if ey_c else INV)
    acx, acy = abs(float(c_re)) + rcx, abs(float(c_im)) + rcy
    # escape shortcut: |z| >= max(2, |c|) + 1/4 for the whole ball
    esc = max(2.0, math.hypot(acx, acy) * (1 + 2.0 ** -50)) + 0.25
    esc2 = esc * esc
    FOUR = 4 << P
    x = y = 0
    rx = ry = 0.0
    it = 0
    while True:
        # decision step
        if it >= cap:
            return it, True
        if exact and not all(representable(v, 2 * P, lb) for v in (x * x, y * y, x * x + y * y)):
            exact = False                         # the test itself rounds
        if exact:
            v = x * x + y * y                     # exact value of the test at 2P fraction bits
            F4 = FOUR << P
            if v == F4 and m.hdr:
                return it, False                  # a tie: decided by the last-bit residue Reduce leaves (HDF32)
            go_on = v < F4 if k.strict else v <= F4
            if not go_on:
                return it, True
        else:
            fx, fy = abs(x) * INV, abs(y) * INV
            ax, ay = fx + rx, fy + ry
            centre = fx * fx + fy * fy
            d = (2 * fx * rx + rx * rx + 2 * fy * ry + ry * ry + _step_errors(k, ax, ay, acx, acy)[2]) * _SLOP
            d += 8 * centre * 2.0 ** -52          # the binary64 evaluation of `centre`
            lo, hi = centre - d, centre + d
            if k.strict:
                if hi < 4.0:
                    pass
                elif lo >= 4.0:
                    return it, True
                else:
                    return it, False
            else:
                if hi <= 4.0:
                    pass
                elif lo > 4.0:
                    return it, True
                else:
                    return it, False
        # P steps
        for _ in range(precision):
            if exact:
                xx, yy, xy2 = x * x, y * y, 2 * x * y   # 2P fraction bits, exact
                x0s, y0s = Cx << P, Cy << P
                nx2, ny2 = xx - yy + x0s, xy2 + y0s
                vals = (xx, yy, xx - yy, x0s - yy, xy2, nx2, ny2, xx + yy)
                if all(representable(v, 2 * P, lb) for v in vals):
                    x, y = nx2 >> P, ny2 >> P
                    continue
                exact = False                     # this step is the first one that can round
            fx, fy = abs(x) * INV, abs(y) * INV
            ax, ay = fx + rx, fy + ry
            ex, ey, _ = _step_errors(k, ax, ay, acx, acy)
            nrx = (2 * fx * rx + rx * rx + 2 * fy * ry + ry * ry + rcx + ex) * _SLOP + 2 * INV
            nry = (2 * (fx * ry + fy * rx + rx * ry) + rcy + ey) * _SLOP + 2 * INV
            x, y = ((x * x - y * y) >> P) + Cx, ((x * y) >> (P - 1)) + Cy
            rx, ry = nrx, nry
            if rx + ry > 1.0:
                return it, False                  # the ball no longer tells anything
            fx, fy = abs(x) * INV - rx, abs(y) * INV - ry
            lo2 = max(fx, 0.0) ** 2 + max(fy, 0.0) ** 2
            if lo2 >= esc2 * (1 + 2.0 ** -40):
                # escapes mathematically; the kernel reads escaped at the next decision step (or stops at the cap)
                nxt = it + precision
                return nxt, True
        it += precision


# ---- frames -------------------------------------------------------------------------------------------------------
def _work(args):
    kname, coords, pix, n_iterations, precision, mname = args
    k = KERNELS[kname]
    model = MODELS[mname] if mname else None
    cx, cy, dx, dy = coords
    return [escape_count(k, cx, cy, dx, dy, X, Y, n_iterations, precision, model) for X, Y in pix]


def escape_counts(kernel: str, coords, pixels, n_iterations: int, precision: int = 1, model: str | None = None,
                  processes: int | None = None):
    """escape_count over a list of kernel pixels (X, Y), spread over processes of a `spawn` context (safe after CUDA
    initialisation).  coords = (cx, cy, dx, dy) as Fractions.  Returns [(count, certified)]."""
    return map_pixels(_work, lambda part: (kernel, tuple(coords), part, n_iterations, precision, model), pixels,
                      processes)


def map_pixels(work, job, pixels, processes: int | None = None):
    """[work(job(part)) for the parts of `pixels`], flattened, on processes of a `spawn` context (safe after CUDA
    initialisation).  `work` must be a module-level function; job(part) builds its picklable argument."""
    pixels = list(pixels)
    processes = processes or mp.cpu_count()
    chunk = max(1, len(pixels) // (processes * 8))
    jobs = [job(pixels[i:i + chunk]) for i in range(0, len(pixels), chunk)]
    if processes == 1 or len(jobs) == 1:
        res = [work(j) for j in jobs]
    else:
        with mp.get_context("spawn").Pool(processes) as pool:
            res = pool.map(work, jobs)
    return [r for part in res for r in part]
