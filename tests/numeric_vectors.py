"""Operand vectors for the per-operation checks of the device numeric types (SURVEY section 8 row a8): HDRFloat<float>,
HDRFloatComplex<float>, dblflt, dbldbl.  Used by the GPU suite (fs_selftest_numeric_op vs the oracle) and by the CPU suite
(the host build of the same product headers vs the oracle)."""
import math
import struct
from fractions import Fraction

import numpy as np

_HF = np.dtype([("m", "<f4"), ("e", "<i4")])
_HC = np.dtype([("re", "<f4"), ("im", "<f4"), ("e", "<i4")])
_DF = np.dtype([("head", "<f4"), ("tail", "<f4")])
_DD = np.dtype([("head", "<f8"), ("tail", "<f8")])
_MIN_BIG = -(1 << 28)  # MIN_BIG_EXPONENT = INT32_MIN >> 3 (HDRFloat.h:50-58)


def _hdr_mantissas(rng, n, reduced):
    """Signed mantissas: reduced ones in [1, 2); otherwise also what the kernels hold between Reduce calls (products, sums
    after cancellation: anything from 2^-40 to 2^40), zeros and binary32 subnormals."""
    m = rng.uniform(1.0, 2.0, n).astype(np.float32)
    if not reduced:
        m = (m * np.exp2(rng.integers(-40, 41, n)).astype(np.float32)).astype(np.float32)
        k = rng.integers(0, 16, n)
        m[k == 0] = 0.0
        m[k == 1] = np.float32(1e-41)                      # subnormal
        m[k == 2] = np.float32(1.0)
        m[k == 3] = np.nextafter(np.float32(2.0), np.float32(0.0))
    return (m * rng.choice(np.array([-1.0, 1.0], np.float32), n)).astype(np.float32)


def _hdr_exponents(rng, n, base):
    """Exponents around `base` with every gap the alignment code distinguishes (0, +-1, +-119..+-121, +-126..+-129, far)."""
    gaps = np.array([0, 1, -1, 2, -2, 23, -24, 30, -30, 119, -119, 120, -120, 121, -121, 126, -126, 127, -127, 128, -128, 129, -129,
                     1000, -1000], np.int64)
    e = base + rng.choice(gaps, n) + rng.integers(-3, 4, n)
    k = rng.integers(0, 24, n)
    e[k == 0] = _MIN_BIG
    e[k == 1] = _MIN_BIG + rng.integers(0, 200, n)[k == 1]
    return np.clip(e, _MIN_BIG, 20_000_000).astype(np.int32)


def _hf_operands(rng, n, reduced):
    a = np.zeros(n, _HF)
    a["m"] = _hdr_mantissas(rng, n, reduced)
    a["e"] = _hdr_exponents(rng, n, int(rng.integers(-5000, 5000)))
    z = a["m"] == 0
    a["e"][z & (rng.integers(0, 2, n) == 0)] = _MIN_BIG   # the canonical zero, and zeros that kept an exponent
    return a


def _hc_operands(rng, n, reduced):
    a = np.zeros(n, _HC)
    a["re"] = _hdr_mantissas(rng, n, reduced)
    a["im"] = _hdr_mantissas(rng, n, False) * np.exp2(-rng.integers(0, 30, n)).astype(np.float32)
    a["e"] = _hdr_exponents(rng, n, int(rng.integers(-5000, 5000)))
    return a


def _dd_operands(rng, n, dtype, eps_bits):
    a = np.zeros(n, dtype)
    ft = dtype["head"].type
    head = (rng.uniform(1.0, 2.0, n) * np.exp2(rng.integers(-30, 31, n)) * rng.choice([-1.0, 1.0], n)).astype(ft)
    tail = (head.astype(np.float64) * np.exp2(-eps_bits - rng.integers(0, 8, n)) * rng.uniform(-1.0, 1.0, n)).astype(ft)
    k = rng.integers(0, 12, n)
    head[k == 0] = 0
    tail[k <= 1] = 0
    a["head"], a["tail"] = head, tail
    return a



OPS = [
    (0, "HDRFloat add"), (1, "HDRFloat subtract"), (2, "HDRFloat multiply"), (3, "HDRFloat square"), (4, "HDRFloat Reduce"),
    (5, "HDRFloat divide"), (6, "HDRFloat compareToBothPositiveReduced"),
    (10, "HDRFloatComplex plus"), (11, "HDRFloatComplex times"), (12, "HDRFloatComplex Reduce"),
    (13, "HDRFloatComplex chebychevNorm"), (14, "HDRFloatComplex times HDRFloat"),
    (20, "dblflt add"), (21, "dblflt sub"), (22, "dblflt mul"), (23, "dblflt sqr"),
    (30, "dbldbl add"), (31, "dbldbl sub"), (32, "dbldbl mul"),
    (40, "HDRx32 perturbation step (custom_perturb2)"),
    (50, "HDRFloat<double> add"), (51, "HDRFloat<double> subtract"), (52, "HDRFloat<double> multiply"),
    (53, "HDRFloat<double> square"), (54, "HDRFloat<double> Reduce"), (55, "HDRFloat<double> divide"),
    (56, "HDRFloat<double> compareToBothPositiveReduced"),
]
_HD = np.dtype([("m", "<f8"), ("e", "<i4"), ("pad", "<i4")])


def _hd_operands(rng, n, reduced):
    """HDRFloat<double> operands: as _hf_operands, with 53-bit mantissas (unreduced ones from 2^-300 to 2^300, subnormals)."""
    a = np.zeros(n, _HD)
    m = rng.uniform(1.0, 2.0, n)
    if not reduced:
        m = m * np.exp2(rng.integers(-300, 301, n).astype(np.float64))
        k = rng.integers(0, 16, n)
        m[k == 0] = 0.0
        m[k == 1] = 5e-320                                   # subnormal
        m[k == 2] = 1.0
        m[k == 3] = np.nextafter(2.0, 0.0)
    a["m"] = m * rng.choice(np.array([-1.0, 1.0]), n)
    a["e"] = _hdr_exponents(rng, n, int(rng.integers(-5000, 5000)))
    z = a["m"] == 0
    a["e"][z & (rng.integers(0, 2, n) == 0)] = _MIN_BIG
    return a
_STEP = np.dtype([("m0", "<f4"), ("e0", "<i4"), ("m1", "<f4"), ("e1", "<i4"), ("m2", "<f4"), ("e2", "<i4")])


def operands(op, n):
    """Operand pairs for `op`, aimed at the code's case distinctions: exponent gaps 0, +-1, +-119..121, +-126..129, far apart,
    the MIN_BIG exponent, zeros with and without it, unreduced and subnormal mantissas."""
    rng = np.random.default_rng(1000 + op)
    if 50 <= op <= 56:
        reduced = op == 56
        a, b = _hd_operands(rng, n, reduced), _hd_operands(rng, n, reduced)
        if op == 55:
            b["m"][b["m"] == 0] = 1.5
        if op == 56:
            a["m"], b["m"] = np.abs(a["m"]), np.abs(b["m"])
            same = rng.integers(0, 3, n) == 0
            b["e"][same] = a["e"][same]
        return a, b
    if op == 40:
        # reduced dX, dY, Zx, Zy, cX, cY (what the kernels hold at a step): exponents so that the two product sums and the
        # added c meet at every gap the alignment distinguishes, including the 127 rule of custom_perturb2
        a, b = np.zeros(n, _STEP), np.zeros(n, _STEP)
        for arr in (a, b):
            for k in range(3):
                h = _hf_operands(rng, n, True)
                arr["m%d" % k] = h["m"]
                arr["e%d" % k] = h["e"]
        # orbit elements Zx, Zy live near exponent 0..-60; deltas and c far below or near them
        a["e2"] = rng.integers(-60, 2, n).astype(np.int32)
        b["e0"] = rng.integers(-60, 2, n).astype(np.int32)
        near = rng.integers(0, 2, n) == 0
        for arr, f in ((a, "e0"), (a, "e1"), (b, "e1"), (b, "e2")):
            arr[f] = np.where(near, rng.integers(-140, 2, n), arr[f]).astype(np.int32)
        return a, b
    if op <= 6:
        reduced = op == 6  # the comparison is specified for reduced operands only
        a, b = _hf_operands(rng, n, reduced), _hf_operands(rng, n, reduced)
        if op == 5:
            b["m"][b["m"] == 0] = np.float32(1.5)          # x / 0 is not an operation the kernels perform
        if op == 6:
            a["m"], b["m"] = np.abs(a["m"]), np.abs(b["m"])
            same = rng.integers(0, 3, n) == 0              # equal exponents: the mantissas decide
            b["e"][same] = a["e"][same]
    elif op <= 14:
        a, b = _hc_operands(rng, n, False), _hc_operands(rng, n, False)
        if op == 14:
            b["re"] = _hdr_mantissas(rng, n, True)
    elif op <= 23:
        a, b = _dd_operands(rng, n, _DF, 24), _dd_operands(rng, n, _DF, 24)
    else:
        a, b = _dd_operands(rng, n, _DD, 53), _dd_operands(rng, n, _DD, 53)
    return a, b


def mismatches(got, want):
    """Indices where the results differ.  Not compared: the sign of an exactly-zero mantissa (where the reference returns an
    operand untouched -- exponent gap >= 120 -- it keeps that operand's -0, the library's forms give +0; no consumer can tell:
    zeros are tested with == 0, compared, multiplied or passed through |x|, and Reduce / the exponent extraction return
    before looking at a zero's bits) and NaN payloads (a NaN result is a NaN result)."""
    got, want = got.copy(), want.copy()
    n = got.shape[0]
    for f in got.dtype.names:
        if got.dtype[f].kind == "f":
            got[f][got[f] == 0] = 0
            want[f][want[f] == 0] = 0
            both = np.isnan(got[f]) & np.isnan(want[f])
            got[f][both] = 0
            want[f][both] = 0
    return np.flatnonzero((got.view(np.uint8).reshape(n, -1) != want.view(np.uint8).reshape(n, -1)).any(axis=1))


# ---- Quad<F> (fs_qd.cuh) --------------------------------------------------------------------------------------------
# Listed apart from OPS: these operations have no bit-exact restatement in the oracle by design (the port splits products
# with an FMA where the reference leaves a Dekker split to the compiler).  They are checked against exact arithmetic
# within the bounds of tests/exact_escape.py, and the device against the host build of fs_qd.cuh bit for bit.
QUAD_OPS = [
    (60, "Quad<double> add"), (61, "Quad<double> sub"), (62, "Quad<double> mul(q, q)"), (63, "Quad<double> mul(q, scalar)"),
    (64, "Quad<double> sqr"), (65, "Quad<double> mul_pwr2"), (66, "Quad<double> le(q, q)"), (67, "Quad<double> le(q, scalar)"),
    (70, "Quad<float> add"), (71, "Quad<float> sub"), (72, "Quad<float> mul(q, q)"), (73, "Quad<float> mul(q, scalar)"),
    (74, "Quad<float> sqr"), (75, "Quad<float> mul_pwr2"), (76, "Quad<float> le(q, q)"), (77, "Quad<float> le(q, scalar)"),
]
_Q64 = np.dtype([("x", "<f8"), ("y", "<f8"), ("z", "<f8"), ("w", "<f8")])
_Q32 = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("w", "<f4")])


def quad_dtype(op):
    return _Q64 if op < 70 else _Q32


def _expansion(value, ft):
    """Greedy round-to-nearest four-limb expansion of the Fraction `value` (normalised: each limb rounds what is left)."""
    limbs, rest = [], value
    for _ in range(4):
        v = ft(float(rest)) if rest != 0 else ft(0.0)
        limbs.append(v)
        rest -= Fraction(float(v))
    return limbs


def quad_operands(op, n):
    """Operand pairs for the Quad<F> operation `op`, aimed at the case distinctions of fs_qd.cuh: zero limbs (the zero
    shortcuts of two_sum / quick_two_sum / renorm in the double flavour), cancellation a ~ -b to every limb depth,
    overlapping and widely spaced limbs, sums and squares around the bailout |z|^2 ~ 4, tiny magnitudes where the low
    limbs of Quad<float> are subnormal, signed zeros, and for le equal heads (and equal second / third limbs).
    The scalar operand of ops 3, 5, 7 is b.x."""
    rng = np.random.default_rng(2000 + op)
    k = op % 10
    dt = quad_dtype(op)
    ft = dt["x"].type
    p = 53 if op < 70 else 24
    a, b = np.zeros(n, dt), np.zeros(n, dt)

    def rand_value(lo, hi):
        # a value with far more bits than four limbs hold, magnitude 2^[lo, hi)
        m = Fraction(int(rng.integers(1 << 62, 1 << 63)), 1 << 62) + Fraction(int(rng.integers(0, 1 << 62)), 1 << 124)
        m += Fraction(int(rng.integers(0, 1 << 62)), 1 << 186) + Fraction(int(rng.integers(0, 1 << 62)), 1 << 248)
        m *= Fraction(2) ** int(rng.integers(lo, hi))
        return m if rng.integers(0, 2) else -m

    tiny_lo = -140 if op >= 70 else -300
    for i in range(n):
        kind = int(rng.integers(0, 10))
        if kind == 6 and op >= 70:
            lo, hi = tiny_lo, -40                         # Quad<float>: third / fourth limbs subnormal
        elif kind == 5:
            lo, hi = 0, 2                                 # around the bailout: |a|, |b| in [1, 4)
        else:
            lo, hi = -12, 4
        va, vb = rand_value(lo, hi), rand_value(lo, hi)
        la, lb = _expansion(va, ft), _expansion(vb, ft)
        if kind == 0:                                     # zero limbs
            for L in (la, lb):
                for j in range(1, 4):
                    if rng.integers(0, 2):
                        L[j] = ft(0.0)
            if rng.integers(0, 4) == 0:
                la = [ft(0.0)] * 4
        elif kind == 1 and k in (0, 1):                   # cancellation a ~ -b (add) / a ~ b (sub) down to limb `d`
            d = int(rng.integers(1, 5))
            s = -1 if k == 0 else 1
            lb = [ft(s * v) for v in la[:d]] + lb[d:] if d < 4 else [ft(s * v) for v in la]
            if d < 4:
                rest = _expansion(rand_value(lo - p * d, hi - p * d), ft)
                lb = lb[:d] + rest[:4 - d]
        elif kind == 2:                                   # overlapping limbs: y within 2^-8 of x's magnitude
            la[1] = ft(float(la[0]) * float(rng.uniform(-1, 1)) * 2.0 ** -int(rng.integers(1, 9)))
        elif kind == 3:                                   # widely spaced limbs
            for j in range(1, 4):
                la[j] = ft(float(la[j]) * 2.0 ** -int(rng.integers(0, 2 * p)))
        elif kind == 4:                                   # signed zeros: trailing limbs (or all four) +-0
            for L in (la, lb):
                d = int(rng.integers(0, 4))
                for j in range(d, 4):
                    L[j] = ft(-0.0) if rng.integers(0, 2) else ft(0.0)
        if k in (6, 7):                                   # the comparison is specified on normalised expansions
            la = _expansion(sum((Fraction(float(v)) for v in la), Fraction(0)), ft)
            lb = _expansion(sum((Fraction(float(v)) for v in lb), Fraction(0)), ft)
            if rng.integers(0, 2):                        # equal heads, and equal second / third / fourth limbs
                d = int(rng.integers(1, 5))
                vb = sum((Fraction(float(v)) for v in la[:d]), Fraction(0))
                if d < 4 and la[d - 1] != 0 and rng.integers(0, 4):
                    vb += rand_value(-2 * p, -p - 1) * Fraction(abs(float(la[d - 1])))
                lb = _expansion(vb, ft)
            if kind == 4:
                la = [ft(-0.0) if v == 0 else v for v in la]
        a[i] = tuple(la)
        b[i] = tuple(lb)
    if k == 5:                                            # mul_pwr2: the kernel doubles; halving may round subnormals
        b["x"] = rng.choice(np.array([2.0, 2.0, 2.0, -2.0, 4.0, 0.5]), n).astype(ft)
    if k == 7:
        b["x"] = np.where(rng.integers(0, 2, n) == 0, a["x"], b["x"])   # le(q, scalar) with a.x == b
    return a, b


# ---- perturbation-step records (fs_num.cuh perturb_selftest, ops 80-85) ---------------------------------------------
PERTURB_OPS = {"f32": 80, "f64": 81, "hdr32": 82, "hdr64": 83, "2x32": 84, "hdr2x32": 85}
_CELL = {"f32": "<f", "f64": "<d", "2x32": "<ff", "hdr32": "<fi", "hdr64": "<di4x", "hdr2x32": "<ffi"}
_GAPS = [0, 1, -1, 119, 120, 121, 126, 127, 128]


def _f32(v):
    return struct.unpack("<f", struct.pack("<f", v))[0]


def _number(rng, tname, scale, zero_e=None):
    """(cell bytes, exact value) of one number of about 2^scale; with zero_e an exact zero instead (HDR: at exponent
    zero_e, or at the canonical MIN_BIG for zero_e == "canon")."""
    hdr = tname.startswith("hdr")
    sign = -1.0 if rng.integers(0, 2) else 1.0
    if zero_e is not None:
        if hdr:
            e = _MIN_BIG if zero_e == "canon" else int(zero_e)
            vals = {"hdr32": (0.0, e), "hdr64": (0.0, e), "hdr2x32": (0.0, 0.0, e)}[tname]
        else:
            vals = {"f32": (sign * 0.0,), "f64": (sign * 0.0,), "2x32": (0.0, 0.0)}[tname]
        return struct.pack(_CELL[tname], *vals).ljust(16, b"\0"), Fraction(0)
    if hdr:
        # reduced mantissa in [1, 2), or an unreduced one in [2^-24, 8) as the kernels hold between Reduce calls
        m = float(rng.uniform(1.0, 2.0)) if rng.integers(0, 3) else float(rng.uniform(1.0, 2.0)) * 2.0 ** int(rng.integers(-24, 3))
        m *= sign
        if tname == "hdr32":
            m = _f32(m)
            vals, v = (m, scale), Fraction(m) * Fraction(2) ** scale
        elif tname == "hdr64":
            vals, v = (m, scale), Fraction(m) * Fraction(2) ** scale
        else:
            h = _f32(m)
            t = _f32(h * float(rng.uniform(-1, 1)) * 2.0 ** -25)
            vals, v = (h, t, scale), (Fraction(h) + Fraction(t)) * Fraction(2) ** scale
        return struct.pack(_CELL[tname], *vals).ljust(16, b"\0"), v
    x = sign * float(rng.uniform(1.0, 2.0)) * 2.0 ** scale
    if tname == "f32":
        x = _f32(x)
        return struct.pack("<f", x).ljust(16, b"\0"), Fraction(x)
    if tname == "f64":
        return struct.pack("<d", x).ljust(16, b"\0"), Fraction(x)
    h = _f32(x)
    t = _f32(h * float(rng.uniform(-1, 1)) * 2.0 ** -25)
    return struct.pack("<ff", h, t).ljust(16, b"\0"), Fraction(h) + Fraction(t)


def perturb_records(tname, n, seed=80):
    """n records of perturb_selftest for the type and their exact operand values [(dx, dy, zx, zy, cx, cy, X, Y)],
    aimed at the case distinctions of the step: exponent gaps 0, +-1, 119-121, 126-128 between the orbit, the delta and
    dc; exact zeros (HDR: canonical, and at exponents up to the largest operand's, where a cancellation leaves them);
    unreduced HDR mantissas;
    subnormal results for the plain types; cancellation 2Z ~ -d and dc ~ -d (2Z + d)."""
    rng = np.random.default_rng(seed)
    hdr = tname.startswith("hdr")
    lo = {"f32": -140, "2x32": -100, "f64": -1000}.get(tname, -100000)
    rec = np.zeros((n, 128), np.uint8)
    vals = []
    for i in range(n):
        sz = int(rng.integers(-40, 2)) if rng.integers(0, 4) == 0 else int(rng.integers(-2, 2))
        g = _GAPS[int(rng.integers(0, len(_GAPS)))] if rng.integers(0, 2) else int(rng.integers(2, 60))
        sd = max(sz - g, lo)
        g2 = _GAPS[int(rng.integers(0, len(_GAPS)))] if rng.integers(0, 3) == 0 else int(rng.integers(-3, 4))
        sc = max(min(sd + g2, 1), lo)
        cells, v = [], []
        for k, s in enumerate((sd, sd + int(rng.integers(-3, 4)), sz, sz + int(rng.integers(-3, 1)), sc, sc)):
            s = max(s, lo)
            z = None
            if rng.integers(0, 12) == 0:
                z = "canon" if (not hdr or rng.integers(0, 2)) else max(sz, sd, sc) + int(rng.integers(-200, 1))
            c, x = _number(rng, tname, s, z)
            cells.append(c)
            v.append(x)
        kind = int(rng.integers(0, 7))
        if kind == 0 and v[2] != 0:     # 2 Zx ~ -dx: the delta cancels the orbit
            tgt = -2 * v[2] * (1 + Fraction(int(rng.integers(-4, 5)), 1 << 30))
            cells[0], v[0] = _pack_value(tname, tgt)
        elif kind == 1:                 # dc ~ -d (2Z + d): the step cancels to nearly nothing
            dx, dy, zx, zy = v[0], v[1], v[2], v[3]
            ex = dx * (2 * zx + dx) - dy * (2 * zy + dy)
            ey = dx * (2 * zy + dy) + dy * (2 * zx + dx)
            if ex != 0:
                cells[4], v[4] = _pack_value(tname, -ex)
            if ey != 0:
                cells[5], v[5] = _pack_value(tname, -ey)
        X, Y = int(rng.integers(0, 5000)), int(rng.integers(0, 5000))
        buf = b"".join(cells) + struct.pack("<ii", X, Y)
        rec[i, :len(buf)] = np.frombuffer(buf, np.uint8)
        vals.append((*v, X, Y))
    return rec, vals


def _pack_value(tname, q):
    """(cell, exact value) of the type's nearest representation of the rational q (HDR: reduced mantissa)."""
    if q == 0:
        return _number(np.random.default_rng(0), tname, 0, "canon")
    if tname in ("f32", "f64"):
        x = _f32(float(q)) if tname == "f32" else float(q)
        return struct.pack(_CELL[tname], x).ljust(16, b"\0"), Fraction(x)
    if tname == "2x32":
        h = _f32(float(q))
        t = _f32(float(q - Fraction(h)))
        return struct.pack("<ff", h, t).ljust(16, b"\0"), Fraction(h) + Fraction(t)
    e = math.floor(math.log2(abs(q))) if abs(q) > 0 else 0
    while abs(q) >= Fraction(2) ** (e + 1):
        e += 1
    while abs(q) < Fraction(2) ** e:
        e -= 1
    m = q / Fraction(2) ** e
    if tname == "hdr32":
        mm = _f32(float(m))
        return struct.pack("<fi", mm, e).ljust(16, b"\0"), Fraction(mm) * Fraction(2) ** e
    if tname == "hdr64":
        mm = float(m)
        return struct.pack("<di4x", mm, e).ljust(16, b"\0"), Fraction(mm) * Fraction(2) ** e
    h = _f32(float(m))
    t = _f32(float(m - Fraction(h)))
    return struct.pack("<ffi", h, t, e).ljust(16, b"\0"), (Fraction(h) + Fraction(t)) * Fraction(2) ** e
