"""The direct escape-time kernels and their arithmetic against exact arithmetic (tests/exact_escape.py).

Parity with the reference's kernels cannot check what a frame is meant to contain, and for the four-limb kernels -- the
one place this library is deliberately not bit-identical -- there is no reference kernel that resolves their windows.
Here the kernels' counts are compared with escape counts computed on integers, wherever the ball model certifies that the
kernel's arithmetic cannot change the count; the per-operation bounds the model rests on are checked against exact
rationals.  CPU tests run the oracle's restatements of the 1x / 2x kernels and the host build of the four-limb loop
(fs_qd.cuh quad_escape_count); GPU tests run the kernels."""
import os
import sys
from fractions import Fraction

import numpy as np
import pytest

import exact_escape as E
import numeric_vectors as nv
import oracle_cpu
from fractalshark_b200 import Numeric
from fractalshark_b200 import RenderAlgorithm as A
from fractalshark_b200.views import PRESETS, VIEW1, ViewPreset

ALGS = {"Gpu1x32": A.Gpu1x32, "Gpu1x64": A.Gpu1x64, "Gpu2x32": A.Gpu2x32, "Gpu2x64": A.Gpu2x64, "Gpu4x32": A.Gpu4x32,
        "Gpu4x64": A.Gpu4x64, "GpuHDRx32": A.GpuHDRx32}
TAGS = {"Gpu1x32": Numeric.F32, "Gpu1x64": Numeric.F64, "Gpu2x32": Numeric.X2_32, "Gpu2x64": Numeric.X2_64,
        "Gpu4x32": Numeric.X4_32, "Gpu4x64": Numeric.X4_64, "GpuHDRx32": Numeric.HDR64}
# GpuHDRx32 (HDR over 2x32) has no CPU restatement: its arithmetic is device-only, so it is checked on the GPU
CPU_KERNELS = [k for k in TAGS if k != "GpuHDRx32"]
WORKERS = max(1, min(8, os.cpu_count() or 1))


def _report(line):
    sys.stderr.write(line + "\n")


# ---- coordinates ------------------------------------------------------------------------------------------------
def exact_view_coords(p: ViewPreset, w: int, h: int):
    """(cx, cy, dx, dy) of a preset at w x h as Fractions: the decimal strings, SquareAspectRatio
    (PointZoomBBConverter.cpp:271-312) restated, cx = minX, cy = minY, dx = (maxX - minX) / w, dy = (maxY - minY) / h."""
    mnx, mny, mxx, mxy = (Fraction(s) for s in (p.min_x, p.min_y, p.max_x, p.max_y))
    ratio = Fraction(w, h)
    mwidth = (mxx - mnx) / ratio
    height = mxy - mny
    if height > mwidth:
        t = (height - mwidth) * ratio / 2
        mnx, mxx = mnx - t, mxx + t
    elif height < mwidth:
        t = (mwidth - height) / 2
        mny, mxy = mny - t, mxy + t
    return mnx, mny, (mxx - mnx) / w, (mxy - mny) / h


# The perturbation kernels' PODs (fs_host.cpp fsh_view_coords): numeric tag, exact_perturb type, relative precision
# (F32 / HDR32 round the mpf through binary64 to binary32: < 2^-23; F64 / HDR64: < 2^-52; X2_32 splits the binary64
# value into head + rounded tail: < 2^-47; HDR2X32 splits the truncated 53-bit mpf mantissa into head and
# (float)(m - head) without renormalising or reducing: the tail's rounding, 2^-24 of |m - head| <= 2^-24 |m|, and the
# truncation, < 2^-47 of the value in all), subnormal floor.
PO_TAGS = {"PO-F32": (Numeric.F32, "f32", 23, 2.0 ** -149), "PO-F64": (Numeric.F64, "f64", 52, 2.0 ** -1074),
           "PO-X2_32": (Numeric.X2_32, "2x32", 47, 2 * 2.0 ** -149), "PO-HDR32": (Numeric.HDR32, "hdr32", 23, 0.0),
           "PO-HDR64": (Numeric.HDR64, "hdr64", 52, 0.0), "PO-HDR2X32": (Numeric.HDR2X32, "hdr2x32", 47, 0.0)}


@pytest.mark.parametrize("kernel", list(TAGS) + list(PO_TAGS))
@pytest.mark.parametrize("view_id", [0, 1, 102, 103, 104])
def test_view_coordinate_pods_hold_the_view_within_the_type_precision(built, kernel, view_id):
    """View.coords: each POD (the numeric tag the direct kernel is fed: F32, F64, MattDblflt 0x102, X2_64, X4_32, X4_64,
    HDR64 split into 2x32 as GpuHDRx32 holds it) equals the exact coordinate within the type's precision: L limbs of p bits, each limb the
    conversion of what the
    limbs before it left (truncated then rounded: < 2^-(p-1) relative per limb), plus one subnormal spacing per limb,
    plus the error of the generator's own mpf arithmetic at View.precision_bits.  The perturbation kernels' PODs
    (PO-*: F32, F64, X2_32 as CudaDblflt, HDR32, HDR64, HDR2X32) are checked the same way, with center_x = C_x - minX
    and center_y = C_y - maxY (C the view's centre): they are the exact model's starting radius (exact_perturb.py)."""
    from fractalshark_b200.host_inputs import View
    w, h = 320, 180
    p = PRESETS[view_id]
    view = View(p.min_x, p.min_y, p.max_x, p.max_y, w, h)
    scale = max(abs(Fraction(s)) for s in (p.min_x, p.min_y, p.max_x, p.max_y))
    mpf_err = 16 * scale * Fraction(1, 2 ** view.precision_bits)
    cx, cy, dx, dy = exact_view_coords(p, w, h)
    if kernel in PO_TAGS:
        import exact_perturb as EP
        tag, tname, bits, sub = PO_TAGS[kernel]
        pods = view.coords(tag)
        want = {"cx": cx, "cy": cy, "dx": dx, "dy": dy, "center_x": w * dx / 2, "center_y": -h * dy / 2}
        for name, v in want.items():
            got = EP.pod_value(tname, pods[name])
            tol = abs(v) * Fraction(1, 2 ** bits) + Fraction(sub) + mpf_err
            assert abs(got - v) <= tol, (name, float(got), float(v), float(abs(got - v) / tol))
        return
    pods = view.coords(TAGS[kernel], direct=True)
    m = E.KERNELS[kernel].model
    for name, want in zip(("cx", "cy", "dx", "dy"), (cx, cy, dx, dy)):
        got = E.pod_value(pods[name], m)
        tol = abs(want) * Fraction(1, 2 ** (m.limbs * (m.limb_bits - 1))) + m.limbs * Fraction(m.sub_min) + mpf_err
        assert abs(got - want) <= tol, (name, float(got), float(want), float(abs(got - want) / tol))


# ---- per-operation bounds -----------------------------------------------------------------------------------------
def _fr(v):
    return Fraction(float(v))


def _quad_value(q):
    return _fr(q["x"]) + _fr(q["y"]) + _fr(q["z"]) + _fr(q["w"])


def _quad_mag(q):
    return abs(_fr(q["x"])) + abs(_fr(q["y"])) + abs(_fr(q["z"])) + abs(_fr(q["w"]))


def nonoverlapping(q, p):
    """Every limb at most 2^-(p-1) of the last non-zero limb before it: the expansions renorm produces, the coordinate
    PODs and make(X, 0, 0, 0) -- every Quad the kernels hold.  The bounds are stated for these."""
    prev = None
    for f in ("x", "y", "z", "w"):
        v = abs(float(q[f]))
        if prev is not None and v > prev * 2.0 ** -(p - 1):
            return False                                 # overlapping, or a zero head above a non-zero limb
        prev = v if prev is None or v else prev
    return True


def quad_op_errors(op, a, b, got):
    """[(|got - exact|, bound)] of the Quad op on every operand pair of non-overlapping expansions (others: skipped); for
    the comparisons |got - exact| is 0 or 1 and the bound 0."""
    m = E.QD64 if op < 70 else E.QF32
    k = op % 10
    out = []
    for i in range(a.shape[0]):
        if not (nonoverlapping(a[i], m.limb_bits) and nonoverlapping(b[i], m.limb_bits)):
            out.append((Fraction(0), Fraction(0)))
            continue
        va, vb, r = _quad_value(a[i]), _quad_value(b[i]), _quad_value(got[i])
        ma, mb, s = _quad_mag(a[i]), _quad_mag(b[i]), _fr(b[i]["x"])
        if k in (6, 7):
            want = int(va <= (vb if k == 6 else s))
            out.append((abs(int(r) - want), 0))
            continue
        fl = Fraction(m.floor_op)
        if k == 0:
            ex, bound = va + vb, Fraction(m.eps_add) * (ma + mb) + fl
        elif k == 1:
            ex, bound = va - vb, Fraction(m.eps_add) * (ma + mb) + fl
        elif k == 2:
            ex, bound = va * vb, Fraction(m.eps_mul) * ma * mb + fl
        elif k == 3:
            ex, bound = va * s, Fraction(m.eps_scal) * ma * abs(s) + fl
        elif k == 4:
            ex, bound = va * va, Fraction(m.eps_sqr) * ma * ma + fl
        else:
            ex, bound = va * s, fl                       # times a power of two: exact up to underflow
        out.append((abs(r - ex), bound))
    return out


def _worst(errs):
    ratio = max((float(e / bd) if bd else (float("inf") if e else 0.0) for e, bd in errs), default=0.0)
    err = max((float(e) for e, _ in errs), default=0.0)
    return err, ratio


N_QUAD = 3000


@pytest.fixture(scope="module")
def quad_vectors():
    return {op: nv.quad_operands(op, N_QUAD) for op, _ in nv.QUAD_OPS}


@pytest.mark.parametrize("op,name", nv.QUAD_OPS, ids=[n for _, n in nv.QUAD_OPS])
def test_host_quad_operations_within_their_bounds_of_exact_arithmetic(built, quad_vectors, op, name):
    """The host build of fs_qd.cuh (QuadOps is FS_HD; g++ without contraction, FMA via fma(), no FTZ: the device's
    bits) on operand vectors aimed at its branches: every result within the bound tests/exact_escape.py assumes."""
    a, b = quad_vectors[op]
    got = oracle_cpu.lockstep_quad_op(op, a, b)
    errs = quad_op_errors(op, a, b, got)
    err, ratio = _worst(errs)
    _report(f"{name}: worst |error| {err:.3e}, worst error / bound {ratio:.3e}")
    bad = [i for i, (e, bd) in enumerate(errs) if e > bd]
    assert not bad, (len(bad), bad[:5], a[bad[0]], b[bad[0]], got[bad[0]])


DW_OPS = [(20, "dblflt add"), (21, "dblflt sub"), (22, "dblflt mul"), (23, "dblflt sqr"), (30, "dbldbl add"),
          (31, "dbldbl sub"), (32, "dbldbl mul")]


@pytest.mark.parametrize("op,name", DW_OPS, ids=[n for _, n in DW_OPS])
def test_double_word_operations_within_their_bounds_of_exact_arithmetic(built, op, name):
    """dblflt / dbldbl through the oracle's restatement (pinned bit for bit to the device by the parity suite): every
    result within the double-word bounds of tests/exact_escape.py."""
    m = E.DF32 if op < 30 else E.DD64
    a, b = nv.operands(op, 20000)
    got = oracle_cpu.numeric_op(op, a, b)
    errs = []
    for i in range(a.shape[0]):
        va, vb = _fr(a[i]["head"]) + _fr(a[i]["tail"]), _fr(b[i]["head"]) + _fr(b[i]["tail"])
        ma, mb = abs(_fr(a[i]["head"])) + abs(_fr(a[i]["tail"])), abs(_fr(b[i]["head"])) + abs(_fr(b[i]["tail"]))
        r = _fr(got[i]["head"]) + _fr(got[i]["tail"])
        k = op % 10
        if k == 0:
            ex, bd = va + vb, Fraction(m.eps_add) * (ma + mb)
        elif k == 1:
            ex, bd = va - vb, Fraction(m.eps_add) * (ma + mb)
        elif k == 2:
            ex, bd = va * vb, Fraction(m.eps_mul) * ma * mb
        else:
            ex, bd = va * va, Fraction(m.eps_sqr) * ma * ma
        errs.append((abs(r - ex), bd + Fraction(m.floor_op)))
    err, ratio = _worst(errs)
    _report(f"{name}: worst |error| {err:.3e}, worst error / bound {ratio:.3e}")
    bad = [i for i, (e, bd) in enumerate(errs) if e > bd]
    assert not bad, (len(bad), a[bad[0]], b[bad[0]], got[bad[0]])


@pytest.mark.gpu
@pytest.mark.parametrize("op,name", nv.QUAD_OPS, ids=[n for _, n in nv.QUAD_OPS])
def test_device_quad_operations_equal_the_host_build(built, quad_vectors, op, name):
    """fs_selftest_numeric_op 60-67 / 70-77 on the GPU: bit for bit what the host build gives (whose results the CPU
    test above holds to exact arithmetic)."""
    from fractalshark_b200 import _native
    a, b = quad_vectors[op]
    got = np.zeros_like(a)
    rc = _native.gpu_lib().fs_selftest_numeric_op(0, op, a.ctypes.data, b.ctypes.data, got.ctypes.data, a.shape[0])
    assert rc == 0, rc
    want = oracle_cpu.lockstep_quad_op(op, a, b)
    diff = np.flatnonzero((got.view(np.uint8).reshape(a.shape[0], -1) != want.view(np.uint8).reshape(a.shape[0], -1)).any(axis=1))
    assert diff.size == 0, (diff.size, a[diff[0]], b[diff[0]], got[diff[0]], want[diff[0]])
    assert all(e <= bd for e, bd in quad_op_errors(op, a, b, got))


# ---- edge points --------------------------------------------------------------------------------------------------
EDGE_W = EDGE_H = 17                 # ragged against the 8 x 4 tiles
EDGE_LIMITS = (1, 2, 3, 37)          # with P and P + 1 below


def edge_coords(kernel):
    """cx = cy = -2, dx = dy = 1/4, packed exactly: every c of the 17 x 17 grid is exact in every type."""
    m = E.KERNELS[kernel].model
    return {"cx": E.pack_pod(-2, m), "cy": E.pack_pod(-2, m), "dx": E.pack_pod(Fraction(1, 4), m),
            "dy": E.pack_pod(Fraction(1, 4), m)}


def edge_cases():
    out = []
    for kernel, k in E.KERNELS.items():
        for P in k.precisions:
            for n in sorted(set(EDGE_LIMITS + (P, P + 1))):
                if k.cap_minus and n < P:   # n_iterations - (P - 1) is unsigned (see DESIGN.md section 2)
                    continue
                out.append((kernel, P, n))
    return out


EDGE_CASES = edge_cases()
CPU_EDGE_CASES = [c for c in EDGE_CASES if c[0] in CPU_KERNELS]
_EDGE_MODEL = {}


def edge_model(kernel, P, n):
    """Model counts of the edge frame, indexed [Yout, X]; certified mask."""
    key = (kernel, P, n)
    if key not in _EDGE_MODEL:
        q = Fraction(1, 4)
        pix = [(X, EDGE_H - 1 - yo) for yo in range(EDGE_H) for X in range(EDGE_W)]
        res = E.escape_counts(kernel, (Fraction(-2), Fraction(-2), q, q), pix, n, P, processes=1)
        cnt = np.array([r[0] for r in res], np.int64).reshape(EDGE_H, EDGE_W)
        cert = np.array([r[1] for r in res], bool).reshape(EDGE_H, EDGE_W)
        _EDGE_MODEL[key] = (cnt, cert)
    return _EDGE_MODEL[key]


def _cap(kernel, P, n):
    k = E.KERNELS[kernel]
    first = n - (P - 1) if k.cap_minus else n
    return -(-first // P) * P


# c -> expected count for P = 1: (1x and 2x kernels, 4x kernels); None = the cap
EDGE_TABLE = {(-2, 0): (1, None), (0, 2): (1, 2), (2, 0): (1, 2), (1, 0): (2, 3), (-1, 1): (3, 3), (0, 1): (None, None),
              (-1, 0): (None, None), (0, 0): (None, None)}
# the entries decided by a tie |z|^2 = 4: GpuHDRx32's Reduce leaves a last-bit residue in zero tails (exact_escape HDF32),
# so the model does not certify ties for it
EDGE_TIES = {(-2, 0), (0, 2), (2, 0), (1, 0)}


def test_edge_table_is_what_the_exact_model_gives():
    """The table of the issue's edge points, from exact arithmetic alone (no kernel): strict bailout makes c = -2, 2i, 2
    escape at the first test where |z|^2 = 4; the non-strict quad test keeps iterating; i, -1, 0 never escape."""
    for kernel in E.KERNELS:
        four = kernel.startswith("Gpu4")
        for n in (1, 2, 3, 37):
            cnt, cert = edge_model(kernel, 1, n)
            for (re, im), want in EDGE_TABLE.items():
                if E.KERNELS[kernel].model.hdr and (re, im) in EDGE_TIES:
                    continue
                X, Y = (re + 2) * 4, (im + 2) * 4
                w = want[1 if four else 0]
                w = n if w is None else min(w, n)
                assert cert[EDGE_H - 1 - Y, X] and cnt[EDGE_H - 1 - Y, X] == w, (kernel, n, re, im, cnt[EDGE_H - 1 - Y, X])
    # every non-exact pixel went through the ball model: some of them are certified, some are not
    cnt, cert = edge_model("Gpu1x32", 1, 37)
    assert cert.sum() > 100 and not cert.all()


def _check_certified(got, cnt, cert, what):
    bad = np.argwhere(cert & (got != cnt))
    assert bad.size == 0, (what, len(bad), [(tuple(i), int(got[tuple(i)]), int(cnt[tuple(i)])) for i in bad[:6]])


def _cpu_edge(kernel, P, n, ib):
    coords = edge_coords(kernel)
    if kernel.startswith("Gpu4"):
        X = np.tile(np.arange(EDGE_W), EDGE_H)
        Y = EDGE_H - 1 - np.repeat(np.arange(EDGE_H), EDGE_W)
        return oracle_cpu.quad_escape_counts(4 if kernel == "Gpu4x32" else 8, coords, n, X, Y, ib).reshape(EDGE_H, EDGE_W)
    out, _ = oracle_cpu.render_direct(ALGS[kernel], EDGE_W, EDGE_H, coords, n, P, iter_bytes=ib)
    return out[:EDGE_H, :EDGE_W]


@pytest.mark.parametrize("kernel,P,n", CPU_EDGE_CASES, ids=["%s-p%d-n%d" % c for c in CPU_EDGE_CASES])
def test_edge_points_cpu(built, kernel, P, n):
    """The oracle's restatement (1x, 2x) / the host build of the four-limb loop on the exact 17 x 17 grid: every
    certified pixel equals the exact count, for 32- and 64-bit iteration types."""
    cnt, cert = edge_model(kernel, P, n)
    assert (cnt[cert] <= _cap(kernel, P, n)).all()
    for ib in (4, 8):
        _check_certified(_cpu_edge(kernel, P, n, ib).astype(np.int64), cnt, cert, (kernel, P, n, ib))


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,P,n", EDGE_CASES, ids=["%s-p%d-n%d" % c for c in EDGE_CASES])
def test_edge_points_gpu(built, kernel, P, n):
    """The kernel on the exact 17 x 17 grid: every certified pixel equals the exact count (u32 and u64)."""
    import cases
    from fractalshark_b200.gpu_renderer import GPURenderer
    cnt, cert = edge_model(kernel, P, n)
    for ib in (4, 8):
        got, _, _ = cases.render(GPURenderer, EDGE_W, EDGE_H, ALGS[kernel], edge_coords(kernel), None, None, n, ib,
                                 precision=P)
        _check_certified(got[:EDGE_H, :EDGE_W].astype(np.int64), cnt, cert, (kernel, P, n, ib))


# ---- windows at each type's resolution limit ------------------------------------------------------------------------
def _around_view1(width):
    """A square window of the given width around View #1's centre."""
    cx = (Fraction(VIEW1.min_x) + Fraction(VIEW1.max_x)) / 2
    cy = (Fraction(VIEW1.min_y) + Fraction(VIEW1.max_y)) / 2
    half = Fraction(width) / 2
    return ViewPreset(_dec(cx - half), _dec(cy - half), _dec(cx + half), _dec(cy + half), 20000)


def _dec(v: Fraction, digits=80):
    sign = "-" if v < 0 else ""
    v = abs(v)
    i = int(v)
    f = int((v - i) * 10 ** digits)
    return "%s%d.%0*d" % (sign, i, digits, f)


WIN_W, WIN_H, WIN_N, WIN_SAMPLE = 320, 180, 20000, 1200
# (id, kernel, preset, floor of the certified fraction, least number of distinct certified counts).  Pixel spacing
# 10-30 bits above each type's precision at |c| ~ 1.76: f32 2^-12, f64 2^-36, df32 2^-30 (View 104 is below 2x32's
# resolution: its 48 bits see that window as a handful of points), dd64 View 102 (2^-88), qd64 Views 102 and 103
# (2^-88, 2^-181), qf32 View 104 (2^-75).
WINDOWS = [
    ("1x32-v1w8e-2", "Gpu1x32", _around_view1(Fraction(8, 100)), 0.9, 12),
    ("1x64-v1w5e-9", "Gpu1x64", _around_view1(Fraction(5, 10 ** 9)), 0.9, 12),
    ("2x32-v1w3e-7", "Gpu2x32", _around_view1(Fraction(3, 10 ** 7)), 0.9, 12),
    ("2x64-v102", "Gpu2x64", PRESETS[102], 0.9, 12),
    ("4x64-v102", "Gpu4x64", PRESETS[102], 0.9, 12),
    ("4x64-v103", "Gpu4x64", PRESETS[103], 0.9, 12),
    ("4x32-v104", "Gpu4x32", PRESETS[104], 0.9, 12),
    ("hdrx32-v1w3e-7", "GpuHDRx32", _around_view1(Fraction(3, 10 ** 7)), 0.9, 12),   # 2x32's 48 bits, as Gpu2x32
]
WIN_IDS = [w[0] for w in WINDOWS]


def window_precisions(kernel):
    return E.KERNELS[kernel].precisions


WIN_CASES = [(w[0], P) for w in WINDOWS for P in window_precisions(w[1])]
CPU_WIN_CASES = [c for c in WIN_CASES if WINDOWS[WIN_IDS.index(c[0])][1] in CPU_KERNELS]


def window_pixels():
    """The seeded sample of (X, Yout) the windows are checked on."""
    rng = np.random.default_rng(104)
    idx = rng.choice(WIN_W * WIN_H, WIN_SAMPLE, replace=False)
    return idx % WIN_W, idx // WIN_W


_WIN = {}


def window(win_id, P, model=None):
    """(coords PODs, sample X, sample Yout, model counts, certified) of a window, computed once per session."""
    key = (win_id, P, model)
    if key not in _WIN:
        from fractalshark_b200.host_inputs import View
        _, kernel, p, _, _ = WINDOWS[WIN_IDS.index(win_id)]
        view = View(p.min_x, p.min_y, p.max_x, p.max_y, WIN_W, WIN_H)
        pods = view.coords(TAGS[kernel], direct=True)
        m = E.KERNELS[kernel].model
        c = tuple(E.pod_value(pods[k], m) for k in ("cx", "cy", "dx", "dy"))
        X, Yo = window_pixels()
        res = E.escape_counts(kernel, c, list(zip(X.tolist(), (WIN_H - 1 - Yo).tolist())), WIN_N, P, model=model,
                              processes=WORKERS)
        cnt = np.array([r[0] for r in res], np.int64)
        cert = np.array([r[1] for r in res], bool)
        _WIN[key] = (pods, X, Yo, cnt, cert)
    return _WIN[key]


@pytest.mark.parametrize("win_id,P", WIN_CASES, ids=["%s-p%d" % c for c in WIN_CASES])
def test_window_model_is_not_vacuous(built, win_id, P):
    """From the ball model alone: a window certifies at least a floor of its sampled pixels, with at least K distinct
    counts (K / P with P iterations per bailout test), so that the comparisons below test something."""
    _, kernel, _, floor, K = WINDOWS[WIN_IDS.index(win_id)]
    K = max(2, K // P)
    _, _, _, cnt, cert = window(win_id, P)
    frac, distinct = float(cert.mean()), len(set(cnt[cert].tolist()))
    _report(f"{win_id} P={P}: certified {frac:.3f} of {cert.size}, {distinct} distinct counts")
    assert frac >= floor and distinct >= K, (frac, distinct)


def test_view_103_needs_four_limbs(built):
    """View 103 tells four limbs from two: under the double-double model almost nothing of it is certified."""
    _, _, _, _, cert4 = window("4x64-v103", 1)
    _, _, _, _, cert2 = window("4x64-v103", 1, model="dd64")
    _report(f"4x64-v103 under the dd64 model: certified {float(cert2.mean()):.3f} (qd64: {float(cert4.mean()):.3f})")
    assert cert2.mean() <= 0.02 and cert4.mean() >= 0.5


def _cpu_window(kernel, pods, X, Yo, P, ib):
    if kernel.startswith("Gpu4"):
        return oracle_cpu.quad_escape_counts(4 if kernel == "Gpu4x32" else 8, pods, WIN_N, X, WIN_H - 1 - Yo, ib,
                                             threads=WORKERS).astype(np.int64)
    out, _ = oracle_cpu.render_direct(ALGS[kernel], WIN_W, WIN_H, pods, WIN_N, P, iter_bytes=ib,
                                      threads=WORKERS)
    return out[Yo, X].astype(np.int64)


@pytest.mark.parametrize("win_id,P", CPU_WIN_CASES, ids=["%s-p%d" % c for c in CPU_WIN_CASES])
def test_window_cpu(built, win_id, P):
    """The oracle's restatement (1x, 2x) / the host-built four-limb loop: every certified sampled pixel equals the
    exact count."""
    _, kernel, _, _, _ = WINDOWS[WIN_IDS.index(win_id)]
    pods, X, Yo, cnt, cert = window(win_id, P)
    got = _cpu_window(kernel, pods, X, Yo, P, 4)
    bad = np.flatnonzero(cert & (got != cnt))
    assert bad.size == 0, (bad.size, [(int(X[i]), int(Yo[i]), int(got[i]), int(cnt[i])) for i in bad[:6]])


@pytest.mark.gpu
@pytest.mark.parametrize("win_id,P", WIN_CASES, ids=["%s-p%d" % c for c in WIN_CASES])
def test_window_gpu(built, win_id, P):
    """The kernel on the whole window (u32 and u64): every certified sampled pixel equals the exact count; the
    four-limb kernels' frame equals the host build of their loop on the sample."""
    import cases
    from fractalshark_b200.gpu_renderer import GPURenderer
    _, kernel, _, _, _ = WINDOWS[WIN_IDS.index(win_id)]
    pods, X, Yo, cnt, cert = window(win_id, P)
    for ib in (4, 8):
        frame, _, _ = cases.render(GPURenderer, WIN_W, WIN_H, ALGS[kernel], pods, None, None, WIN_N, ib, precision=P)
        got = frame[Yo, X].astype(np.int64)
        bad = np.flatnonzero(cert & (got != cnt))
        assert bad.size == 0, (ib, bad.size, [(int(X[i]), int(Yo[i]), int(got[i]), int(cnt[i])) for i in bad[:6]])
        if kernel.startswith("Gpu4"):
            np.testing.assert_array_equal(got, _cpu_window(kernel, pods, X, Yo, P, ib))
