"""Exact reference for the perturbation-only kernels (Gpu{1x32,2x32,1x64,HDRx32,HDRx64,HDRx2x32}PerturbedLAv2PO).

Pure Python, no native code, on the principles of tests/exact_escape.py (its fixed-point helpers and process pool).

Truth.  Pixel (X, Y) of a w x h frame is c = (minX + X dx, maxY - Y dy), exact rationals of the view after
SquareAspectRatio; the reference point is the exact centre C.  The reference orbit Z_n of C is iterated in fixed point
with P fraction bits (the window's depth plus at least 160) and a radius R_n of its own truncation.

The kernel's inputs are read as exact values, not trusted: the orbit bytes it is given (every element layout decoded),
whose distance from Z_n enters the model element by element (it absorbs the mpf centre, the GMP loop and the rounding
into the type), and the coordinate PODs dx, dy, center_x, center_y, from which the kernel forms
dc = (X dx - center_x, -Y dy - center_y) with one rounding bound per operation.

State per pixel: the kernel's orbit index m, which the model follows; the centre of a ball around the true
delta = z_n - Z_m; a radius e that bounds both |kernel's delta - centre| and |true delta - centre| (complex modulus).
Each step adds to e the propagated error e |2Z + 2 delta| + e^2 + 2 (|delta| + e) |Z~_m - Z_m|, the dc error, the
rounding of the step (the per-type bounds below, which tests/test_exact_perturb.py checks against exact rationals)
and the truncation of the fixed-point centre.  After a rebase the new delta is z~ = fl(Z~_{m+1} + delta~'), with the
radius of z~, and m = 0 (Z_0 = 0 exactly).

Decisions, in the order of PerturbLoop::run / hdr32fast::step (step, test, ++iter; iter = m = 0 and delta = 0 at the
start):
- `iter < n_iterations` is deterministic; once it fails the count is n_iterations whatever |z|.
- bailout: |z|^2 < 256 (strict) for f32 / f64 / 2x32 (fs_num.cuh lt_bailout, fs_df32.cuh); for the HDR types the
  reduced test `e < 1 || (e == 1 && m < 256)` is |z|^2 < 4 (strict), fs_types.cuh lt_bailout.  The test reads the
  kernel's rounded norm: the ball's [lo, hi] of |z|^2 widened by the norm's rounding must lie on one side.
- rebase: |z~|^2 < |delta~'|^2 (strict), decided by the balls of both norms, or forced when m >= count - 1 (the end of
  the orbit).  If the balls overlap and m < count - 1 the pixel is not certified.
A pixel is certified when every decision was decided by the ball; its count is then the kernel's count, whatever the
rounding inside the ball, and the count of the true orbit of c.
"""
from __future__ import annotations

import math
import struct
from dataclasses import dataclass
from fractions import Fraction

from exact_escape import DF32, F32, F64, ArithModel, _to_fixed, map_pixels

MIN_BIG = -(2 ** 31) >> 3


@dataclass(frozen=True)
class PerturbType:
    """Numeric policy of one PO kernel and the error bounds of its operations.

    numeric      the fs_numeric tag of the PODs and the orbit (include/fs_gpu.h)
    hdr          float+exponent (NumHdr, NumHdr2x32): no underflow, reduced bailout test |z|^2 < 4
    limbs        the mantissa format (exact_escape.ArithModel: limb precision, subnormal spacing)
    bailout      the strict bound of |z|^2
    pod, elem    struct formats of a coordinate POD and of one orbit element
    eps_step     perturb: per component |error| <= eps_step * P + eps_c * |dc| + floor, P = |dx| Sx + |dy| Sy for x and
    eps_c        |dx| Sy + |dy| Sx for y, Sx = 2|Zx| + |dx|, Sy = 2|Zy| + |dy| (all of the kernel's operands)
    eps_norm     norm2(x, y): eps_norm * (x^2 + y^2) + floor
    eps_add      add(a, b): eps_add * (|a| + |b|) + floor
    eps_delta    delta_x / delta_y: eps_delta * (|X| |d| + |center|) + floor
    floor        absolute floor per operation (the plain types' subnormal range; 0 for HDR)
    """
    name: str
    numeric: int
    hdr: bool
    limbs: ArithModel
    bailout: int
    pod: str
    elem: str
    eps_step: float
    eps_c: float
    eps_norm: float
    eps_add: float
    eps_delta: float
    floor: float


_U32, _U64 = 2.0 ** -24, 2.0 ** -53
_F32_SUB, _F64_SUB = F32.sub_min, F64.sub_min
# Plain binary32 / binary64 (NumPlain): sx, sy one FMA each (u Sx, u Sy), t = sy * d rounded, one FMA, the add of dc:
# every term of P is rounded at most four times (< 4u P (1 + O(u))), dc once (u |dc|), stated as 5u and 2u.  norm2 =
# fma(x, x, y*y): two roundings.  delta = fma(X, d, -center): one.  The floor: each of the eight roundings may fall into
# the subnormal range (<= half its spacing) and the floors of sx, sy are multiplied by |d| <= 1.
# NumHdr<float>: the same sequence with every alignment by an exact power of two (fused3), so the same bounds;
# operands are dropped only at exponent gaps >= 120 / 127 (below 2^-90 of the result for the mantissas in [2^-24, 8)
# the kernel holds), covered by the margin of 5u over 4u.
# NumHdr<double>: fused3 calls the binary32 FMA (fmaf_as_ref): the products, the orbit and dc are rounded to binary32
# and every FMA rounds to binary32, so the step has binary32's precision (eps with u = 2^-24).  Its adds (2Z + d,
# Z + d), norm2 and the deltas run in binary64.
# 2x32 (Num2x32 plain arm, NumHdr2x32 custom_perturb3) with u^2 = 2^-48: 2Z exact, s = 2Z + d one add (4u^2 S), each of
# the four products 8u^2, sub/add of the products 4u^2 P, the add of dc 4u^2 (P + |dc|): < 20u^2 P + 4u^2 |dc| (1 +
# O(u)), stated as 24u^2 and 8u^2.  norm2 = add(mul, mul): 8u^2 + 4u^2.  delta = sub(mul(d, X), center): 8u^2 + 4u^2.
# The floor of the plain arm: every rounding of the tail chains may fall into the subnormal range.
_DW = 2.0 ** -48
TYPES = {
    "f32": PerturbType("f32", 0, False, F32, 256, "<f", "<ff", 5 * _U32, 2 * _U32, 3 * _U32, 2 * _U32, 2 * _U32,
                       8 * _F32_SUB),
    "f64": PerturbType("f64", 1, False, F64, 256, "<d", "<dd", 5 * _U64, 2 * _U64, 3 * _U64, 2 * _U64, 2 * _U64,
                       8 * _F64_SUB),
    "2x32": PerturbType("2x32", 2, False, DF32, 256, "<ff", "<ffff", 24 * _DW, 8 * _DW, 16 * _DW, 8 * _DW, 16 * _DW,
                        64 * _F32_SUB),
    "hdr32": PerturbType("hdr32", 3, True, F32, 4, "<fi", "<fiif", 5 * _U32, 2 * _U32, 3 * _U32, 2 * _U32, 3 * _U32,
                         0.0),
    "hdr64": PerturbType("hdr64", 4, True, F64, 4, "<di4x", "<di4xi4xd", 5 * _U32, 2 * _U32, 3 * _U64, 2 * _U64,
                         3 * _U64, 0.0),
    "hdr2x32": PerturbType("hdr2x32", 5, True, DF32, 4, "<ffi", "<ffiiff", 24 * _DW, 8 * _DW, 16 * _DW, 8 * _DW,
                           16 * _DW, 0.0),
}


def _hdr(m, e) -> Fraction:
    if m == 0:
        return Fraction(0)
    return Fraction(m) * (Fraction(2) ** e)


def pod_value(tname: str, raw: bytes) -> Fraction:
    """The exact value of a coordinate POD of the type."""
    v = struct.unpack(TYPES[tname].pod, raw)
    if tname in ("f32", "f64"):
        return Fraction(v[0])
    if tname == "2x32":
        return Fraction(v[0]) + Fraction(v[1])
    if tname in ("hdr32", "hdr64"):
        return _hdr(v[0], v[1])
    return _hdr(Fraction(v[0]) + Fraction(v[1]), v[2])


def orbit_values(tname: str, elements) -> list:
    """[(x, y)] exact values of the orbit elements (rows of Orbit.as_numpy()) in the type's layout."""
    fmt = TYPES[tname].elem
    out = []
    for row in elements:
        v = struct.unpack(fmt, bytes(row))
        if tname in ("f32", "f64"):
            out.append((Fraction(v[0]), Fraction(v[1])))
        elif tname == "2x32":
            out.append((Fraction(v[0]) + Fraction(v[1]), Fraction(v[2]) + Fraction(v[3])))
        elif tname in ("hdr32", "hdr64"):
            out.append((_hdr(v[0], v[1]), _hdr(v[3], v[2])))   # {x.m, x.e, y.e, y.m}
        else:
            out.append((_hdr(Fraction(v[0]) + Fraction(v[1]), v[2]), _hdr(Fraction(v[4]) + Fraction(v[5]), v[3])))
    return out


# ---- per-operation bounds (checked by tests/test_exact_perturb.py) --------------------------------------------------
# The bounds take operand magnitudes.  An HDR zero at a non-canonical exponent e (fused3 and the adds leave exact
# cancellations there) still aligns its partners to 2^e, and its square or product to 2^2e, and drops what lies 120 /
# 127 binades below, so it counts as magnitude 2^(e - 30) (bound_mag).  The model carries the rule (po_count): a
# component of delta' whose ball holds 0 may be such a zero.  Its exponent is that of the largest term of the step
# (a product dx.m s.m or dc), and a term of magnitude T has an exponent of at most log2 T + 2 p + 4 for mantissas of at
# least 2^-p (a reduced one, or an unreduced one the kernel holds: the exact difference of two aligned p-bit mantissas
# after a rebase or in dc; p = 24, 53, 48 for HDRx32, HDRx64, HDRx2x32).  So the component enters the next bounds with
# magnitude at least T 2^(2p - 26) (ZERO_LIFT).
ZERO_LIFT = {"hdr32": 2.0 ** (2 * 24 - 26), "hdr64": 2.0 ** (2 * 53 - 26), "hdr2x32": 2.0 ** (2 * 48 - 26)}


def bound_mag(tname: str, raw: bytes) -> float:
    """The magnitude a number enters the bounds with: |value|, or 2^(e - 30) for an HDR zero at exponent e."""
    t = TYPES[tname]
    v = abs(float(pod_value(tname, raw)))
    if t.hdr and v == 0.0:
        e = struct.unpack(t.pod, raw[:struct.calcsize(t.pod)])[-1]
        return 0.0 if e == MIN_BIG else math.ldexp(1.0, max(e - 30, -1100))
    return v


def perturb_bound(t: PerturbType, dx, dy, zx, zy, cx, cy):
    """(bound x, bound y) of |perturb - exact| from the operands' magnitudes."""
    A, B = abs(dx), abs(dy)
    Sx, Sy = 2 * abs(zx) + A, 2 * abs(zy) + B
    return (t.eps_step * (A * Sx + B * Sy) + t.eps_c * abs(cx) + t.floor,
            t.eps_step * (A * Sy + B * Sx) + t.eps_c * abs(cy) + t.floor)


def norm_bound(t: PerturbType, x, y):
    return t.eps_norm * (x * x + y * y) + t.floor


def add_bound(t: PerturbType, a, b):
    return t.eps_add * (abs(a) + abs(b)) + t.floor


def delta_bound(t: PerturbType, d, X, center):
    return t.eps_delta * (abs(X) * abs(d) + abs(center)) + t.floor


# ---- one window ---------------------------------------------------------------------------------------------------
_SLOP = 1.0 + 2.0 ** -40   # the binary64 evaluation of the radii and of the ball's norms


def _f(x: int, P: int) -> float:
    """x 2^-P as a float (relative error 2^-53)."""
    b = x.bit_length()
    if b > 1000:
        s = b - 64
        return math.ldexp(float(x >> s) if x >= 0 else -float((-x) >> s), s - P)
    return math.ldexp(float(x), -P)


@dataclass(frozen=True)
class Window:
    """Everything the model needs about one (type, view, w, h, n_iterations): picklable."""
    tname: str
    P: int
    zx: tuple           # fixed-point centre of the true orbit Z_n of C, n < count
    zy: tuple
    zerr: tuple         # |Z~_n - Z_n| bound: kernel element vs fixed point + R_n
    zabs: tuple         # |Z~_n| upper bound (float)
    count: int
    n_iterations: int
    w: int
    h: int
    dx: Fraction        # exact pixel spacing of the view
    dy: Fraction
    pdx: Fraction       # the PODs' exact values
    pdy: Fraction
    pcx: Fraction
    pcy: Fraction


def true_orbit(cx: Fraction, cy: Fraction, count: int, P: int):
    """Fixed-point orbit of C = cx + i cy, n < count, with the radius R_n of its truncation (floats)."""
    Cx, ex = _to_fixed(cx, P)
    Cy, ey = _to_fixed(cy, P)
    x = y = 0
    R = 0.0
    xs, ys, rs = [], [], []
    tr = math.ldexp(3.0, -P)
    for _ in range(count):
        xs.append(x)
        ys.append(y)
        rs.append(R)
        fx, fy = _f(x, P), _f(y, P)
        R = (2 * math.hypot(fx, fy) * R + R * R + tr) * _SLOP
        x, y = ((x * x - y * y) >> P) + Cx, ((x * y) >> (P - 1)) + Cy
    return xs, ys, rs


def make_window(tname: str, view_coords, pods: dict, elements, n_iterations: int, w: int, h: int,
                depth_bits: int) -> Window:
    """view_coords = (minX, minY, dx, dy) exact (test_exact_escape.exact_view_coords); pods = View.coords(numeric);
    elements = Orbit.as_numpy(); depth_bits >= -log2 of the pixel spacing."""
    mnx, mny, dx, dy = view_coords
    cx, cy = mnx + w * dx / 2, mny + h * dy / 2
    zt = orbit_values(tname, elements)
    count = len(zt)
    P = depth_bits + 160
    while True:
        xs, ys, rs = true_orbit(cx, cy, count, P)
        if max(rs) < 2.0 ** -(depth_bits + 64):
            break
        P += 128   # the orbit's derivative ate the margin: more bits
    zerr, zabs = [], []
    INV = 2.0 ** -P
    for (ux, uy), x, y, r in zip(zt, xs, ys, rs):
        ex = abs(ux - Fraction(x, 1 << P))
        ey = abs(uy - Fraction(y, 1 << P))
        zerr.append((math.hypot(float(ex), float(ey)) + r + INV) * _SLOP)
        zabs.append(math.hypot(float(ux), float(uy)) * _SLOP)
    v = {k: pod_value(tname, pods[k]) for k in ("dx", "dy", "center_x", "center_y")}
    return Window(tname, P, tuple(xs), tuple(ys), tuple(zerr), tuple(zabs), count, n_iterations, w, h, dx, dy,
                  v["dx"], v["dy"], v["center_x"], v["center_y"])


def po_count(win: Window, X: int, Y: int, bailout: int | None = None, mirror: bool = False):
    """(count, certified) of kernel pixel (X, Y).  `bailout` overrides the type's bound of |z|^2 and `mirror` maps row
    Y to the row h - 1 - Y of the view (wrong conventions, to show that the comparison would see them)."""
    t = TYPES[win.tname]
    P = win.P
    INV = math.ldexp(1.0, -P)
    B = float(bailout if bailout is not None else t.bailout)
    Yv = win.h - 1 - Y if mirror else Y
    # dc: the truth, and the kernel's from the PODs with its rounding
    tdx = X * win.dx - win.w * win.dx / 2
    tdy = win.h * win.dy / 2 - Yv * win.dy
    kdx = X * win.pdx - win.pcx
    kdy = -Yv * win.pdy - win.pcy
    rcx = float(abs(kdx - tdx)) + delta_bound(t, float(win.pdx), X, float(win.pcx))
    rcy = float(abs(kdy - tdy)) + delta_bound(t, float(win.pdy), Yv, float(win.pcy))
    Dx, _ = _to_fixed(tdx, P)
    Dy, _ = _to_fixed(tdy, P)
    rc = (math.hypot(rcx, rcy) + 2 * INV) * _SLOP
    acx, acy = abs(float(kdx)), abs(float(kdy))
    zx, zy, zerr, zabs = win.zx, win.zy, win.zerr, win.zabs
    last = win.count - 1
    n = win.n_iterations
    ex_, ey_ = 0, 0   # delta's centre (fixed point)
    e = 0.0           # radius
    zmx = zmy = 0.0   # HDR: least magnitude a component enters the bounds with (a possible non-canonical zero)
    lift = ZERO_LIFT.get(win.tname, 0.0)
    m = 0
    it = 0
    while True:
        # ---- step: delta' = delta (2 Z_m + delta) + dc
        Zx, Zy, oe = zx[m], zy[m], zerr[m]
        sx, sy = 2 * Zx + ex_, 2 * Zy + ey_
        fdx, fdy = _f(ex_, P), _f(ey_, P)
        ad = math.hypot(fdx, fdy)
        g = math.hypot(_f(sx + ex_, P), _f(sy + ey_, P))           # |2Z + 2 delta|
        A, Bm = max(abs(fdx) + e, zmx), max(abs(fdy) + e, zmy)
        azx, azy = abs(_f(Zx, P)) + oe, abs(_f(Zy, P)) + oe
        rx, ry = perturb_bound(t, A, Bm, azx, azy, acx + rcx, acy + rcy)
        e = (e * g + e * e + 2 * (ad + e) * oe + rc + math.hypot(rx, ry)) * _SLOP + 3 * INV
        ex_, ey_ = ((ex_ * sx - ey_ * sy) >> P) + Dx, ((ex_ * sy + ey_ * sx) >> P) + Dy
        if lift:
            # the largest term of each component: the products and dc (see ZERO_LIFT)
            Sx, Sy = 2 * azx + A, 2 * azy + Bm
            tx = max(A * Sx, Bm * Sy, acx + rcx)
            ty = max(A * Sy, Bm * Sx, acy + rcy)
            zmx = lift * tx if abs(_f(ex_, P)) <= e else 0.0
            zmy = lift * ty if abs(_f(ey_, P)) <= e else 0.0
        m += 1
        # ---- z = Z_{m} + delta'
        Zx, Zy, oe = zx[m], zy[m], zerr[m]
        wx, wy = Zx + ex_, Zy + ey_
        fdx, fdy = _f(ex_, P), _f(ey_, P)
        ad = math.hypot(fdx, fdy)
        bx = add_bound(t, abs(_f(Zx, P)) + oe, max(abs(fdx) + e, zmx))
        by = add_bound(t, abs(_f(Zy, P)) + oe, max(abs(fdy) + e, zmy))
        rz = (e + oe + math.hypot(bx, by)) * _SLOP
        if it >= n:
            return it, True
        az = math.hypot(_f(wx, P), _f(wy, P))
        zlo, zhi = max(az - rz, 0.0), az + rz
        n2lo = zlo * zlo * (1 - t.eps_norm) / _SLOP - t.floor
        n2hi = zhi * zhi * (1 + t.eps_norm) * _SLOP + t.floor
        if n2lo >= B:
            return it, True                          # escaped: `lt_bailout(n2)` is false for the whole ball
        if n2hi >= B:
            return it, False
        if rz > 1.0:
            return it, False                         # the ball no longer tells anything
        # ---- rebase?
        if m >= last:
            rebase = True
        else:
            dlo, dhi = max(ad - e, 0.0), ad + e
            zn = t.eps_norm * (zmx * zmx + zmy * zmy)
            d2lo = dlo * dlo * (1 - t.eps_norm) / _SLOP - t.floor - zn
            d2hi = dhi * dhi * (1 + t.eps_norm) * _SLOP + t.floor + zn
            if n2hi < d2lo:
                rebase = True
            elif n2lo >= d2hi:
                rebase = False
            else:
                return it, False
        it += 1
        if rebase:
            # z = add(Z, delta') keeps a zero delta component only when Z's lies 120 binades below it
            ex_, ey_, e, m = wx, wy, rz, 0


def _work(args):
    win, part, bailout, mirror = args
    return [po_count(win, X, Y, bailout, mirror) for X, Y in part]


def po_counts(win: Window, pixels, bailout: int | None = None, mirror: bool = False, processes: int | None = None):
    """po_count over a list of kernel pixels (X, Y) on a process pool.  Returns [(count, certified)]."""
    return map_pixels(_work, lambda part: (win, part, bailout, mirror), pixels, processes)
