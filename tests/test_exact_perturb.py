"""The perturbation-only kernels (…PerturbedLAv2PO) against exact arithmetic (tests/exact_perturb.py).

Every other check on these kernels is a parity check (reference kernels, fixtures, recordings, the library's own slower
paths); an A/B pair shares the pixel -> c mapping, the orbit, the rebase rule, the orbit wrap, the bailout and the count
convention, so a fault in any of them passes both arms.  Here the counts are compared with the escape counts of the
true orbits of the pixels' c, wherever the ball model certifies that the kernel's arithmetic cannot change the count.
CPU tests run the oracle's HDRx32 PO restatement; GPU tests run all six PO kernels with the library's defaults."""
import math
import os
import struct
import sys
import time
from fractions import Fraction

import numpy as np
import pytest

import exact_perturb as EP
from fractalshark_b200 import RenderAlgorithm as A
from fractalshark_b200.views import PRESETS

WORKERS = max(1, min(8, os.cpu_count() or 1))
W, H, SAMPLE = 48, 27, 300
ALGS = {"f32": A.Gpu1x32PerturbedLAv2PO, "f64": A.Gpu1x64PerturbedLAv2PO, "2x32": A.Gpu2x32PerturbedLAv2PO,
        "hdr32": A.GpuHDRx32PerturbedLAv2PO, "hdr64": A.GpuHDRx64PerturbedLAv2PO,
        "hdr2x32": A.GpuHDRx2x32PerturbedLAv2PO}
# (type, view) -> (floor of the certified fraction, least number of distinct certified counts), from what the model
# certifies on the sample of the 48 x 27 frame (300 seeded pixels and the 144 of the partial tiles of rows 24-26, 409
# in all; floors a few points below the measured fraction).  The deltas must be representable in the type: f32 / 2x32
# get views 101 and 100, f64 100 / 102 / 1.  On view 100 (orbits of ~2,000 steps) HDRx32 / HDRx64 certify little:
# binary32 precision, and each time a component's ball holds 0 the model allows for a zero at a non-canonical exponent
# (exact_perturb.ZERO_LIFT).
WINDOWS = {
    ("f32", 101): (0.58, 30), ("f32", 100): (0.15, 15),
    ("f64", 100): (0.94, 80), ("f64", 102): (0.97, 8), ("f64", 1): (0.97, 8),
    ("2x32", 101): (0.94, 60), ("2x32", 100): (0.92, 80),
    ("hdr32", 1): (0.97, 8), ("hdr32", 100): (0.08, 25), ("hdr32", 102): (0.97, 8), ("hdr32", 103): (0.97, 8),
    ("hdr64", 1): (0.97, 8), ("hdr64", 100): (0.10, 25), ("hdr64", 102): (0.97, 8), ("hdr64", 103): (0.97, 8),
    ("hdr2x32", 1): (0.97, 8), ("hdr2x32", 100): (0.94, 80), ("hdr2x32", 102): (0.97, 8), ("hdr2x32", 103): (0.97, 8),
}
# one ragged frame per type: partial 8 x 4 tiles and lanes that are not live in the warp-synchronous loop
RAGGED_W, RAGGED_H = 50, 37


def _report(line):
    sys.stderr.write(line + "\n")


def sample_pixels(w, h, k=SAMPLE, seed=2):
    """A seeded sample of (X, Y), plus every pixel of the partial 8 x 4 tiles of a ragged frame (the last columns when w
    is not a multiple of 8, the last rows when h is not a multiple of 4)."""
    rng = np.random.default_rng(seed)
    idx = set(rng.choice(w * h, min(k, w * h), replace=False).tolist())
    idx |= {Y * w + X for Y in range(h) for X in range(w) if X >= w - w % 8 or Y >= h - h % 4}
    idx = np.array(sorted(idx))
    return idx % w, idx // w


_WIN = {}


def window(tname, view_id, w=W, h=H, iter_bytes=4):
    """(coords, orbit, la, n, Window, X, Y) of a (type, view, size), computed once per session."""
    import cases
    from test_exact_escape import exact_view_coords
    key = (tname, view_id, w, h, iter_bytes)
    if key not in _WIN:
        view, coords, orbit, la, n = cases.make_inputs(view_id, w, h, ALGS[tname], None, iter_bytes)
        vc = exact_view_coords(PRESETS[view_id], w, h)
        depth = -math.floor(math.log2(float(min(vc[2], vc[3]))))
        win = EP.make_window(tname, vc, coords, orbit.as_numpy(), n, w, h, depth)
        X, Y = sample_pixels(w, h)
        _WIN[key] = (coords, orbit, la, n, win, X, Y)
    return _WIN[key]


_MODEL = {}


def model(tname, view_id, w=W, h=H, **kw):
    """(counts, certified) of the sampled pixels, and the seconds it took."""
    key = (tname, view_id, w, h, tuple(sorted(kw.items())))
    if key not in _MODEL:
        _, _, _, _, win, X, Y = window(tname, view_id, w, h)
        t0 = time.time()
        res = EP.po_counts(win, list(zip(X.tolist(), Y.tolist())), processes=WORKERS, **kw)
        _MODEL[key] = (np.array([r[0] for r in res], np.int64), np.array([r[1] for r in res], bool), time.time() - t0)
    return _MODEL[key]


def _check(got, cnt, cert, X, Y, what):
    bad = np.flatnonzero(cert & (got != cnt))
    assert bad.size == 0, (what, bad.size, [(int(X[i]), int(Y[i]), int(got[i]), int(cnt[i])) for i in bad[:6]])


# ---- non-vacuity -----------------------------------------------------------------------------------------------------
WIN_IDS = ["%s-v%d" % k for k in WINDOWS]


@pytest.mark.parametrize("tname,view_id", list(WINDOWS), ids=WIN_IDS)
def test_model_is_not_vacuous(built, tname, view_id):
    """From the model alone: the window certifies at least a floor of its sampled pixels, with at least K distinct
    counts, so that the comparisons below test something."""
    floor, K = WINDOWS[(tname, view_id)]
    cnt, cert, secs = model(tname, view_id)
    frac, distinct = float(cert.mean()), len(set(cnt[cert].tolist()))
    _report(f"{tname} view {view_id} {W}x{H}: certified {frac:.3f} of {cert.size}, {distinct} distinct counts, "
            f"{secs:.1f} s")
    assert frac >= floor and distinct >= K, (frac, distinct)


# ---- CPU: the oracle's HDRx32 PO restatement --------------------------------------------------------------------------
CPU_VIEWS = [1, 100, 102, 103]


def _oracle(view_id, ib, w=W, h=H):
    import oracle_cpu
    coords, orbit, la, n, _, _, _ = window("hdr32", view_id, w, h)
    out, _ = oracle_cpu.render_lav2(ALGS["hdr32"], w, h, coords, orbit, la, n, iter_bytes=ib, threads=WORKERS)
    return out


@pytest.mark.parametrize("ib", [4, 8], ids=["u32", "u64"])
@pytest.mark.parametrize("view_id", CPU_VIEWS)
def test_oracle_hdr32_po_equals_the_exact_count(built, view_id, ib):
    """oracle_cpu.render_lav2 (HDRx32 PO, bit-identical to the fixtures): every certified pixel has the exact count.
    This also pins the model's count convention (step, test, ++iter) against code the fixtures hold."""
    _, _, _, _, _, X, Y = window("hdr32", view_id)
    cnt, cert, _ = model("hdr32", view_id)
    got = _oracle(view_id, ib)[Y, X].astype(np.int64)
    _check(got, cnt, cert, X, Y, ("hdr32", view_id, ib))


@pytest.mark.parametrize("view_id", CPU_VIEWS)
def test_wrong_conventions_would_be_seen(built, view_id):
    """The model under a wrong convention -- rows mirrored (c_y running up from minY, as the direct kernels' flipped
    rows would give), or the plain types' bailout |z|^2 < 256 for this HDR kernel -- disagrees with the oracle's frame
    on certified pixels: the comparison above would catch either fault."""
    _, _, _, _, _, X, Y = window("hdr32", view_id)
    got = _oracle(view_id, 4)[Y, X].astype(np.int64)
    for kw in ({"mirror": True}, {"bailout": 256}):
        cnt, cert, _ = model("hdr32", view_id, **kw)
        wrong = int((cert & (got != cnt)).sum())
        _report(f"hdr32 view {view_id} under {kw}: {wrong} certified pixels disagree")
        assert wrong >= 10, (kw, wrong)


# ---- GPU: the six PO kernels ------------------------------------------------------------------------------------------
def _gpu(tname, view_id, ib, w=W, h=H):
    import cases
    from fractalshark_b200.gpu_renderer import GPURenderer
    coords, orbit, la, n, _, _, _ = window(tname, view_id, w, h, ib)
    frame, _, _ = cases.render(GPURenderer, w, h, ALGS[tname], coords, orbit, la, n, ib)
    return frame


@pytest.mark.gpu
@pytest.mark.parametrize("ib", [4, 8], ids=["u32", "u64"])
@pytest.mark.parametrize("tname,view_id", list(WINDOWS), ids=WIN_IDS)
def test_po_kernel_equals_the_exact_count(built, tname, view_id, ib):
    """The PO kernel with the library's defaults (HDRx32: scaled chunks and the float+exponent fallback): every
    certified sampled pixel has the exact count."""
    _, _, _, _, _, X, Y = window(tname, view_id)
    cnt, cert, _ = model(tname, view_id)
    got = _gpu(tname, view_id, ib)[Y, X].astype(np.int64)
    _check(got, cnt, cert, X, Y, (tname, view_id, ib))


RAGGED = [("f32", 101), ("f64", 102), ("2x32", 101), ("hdr32", 102), ("hdr64", 102), ("hdr2x32", 102)]


@pytest.mark.gpu
@pytest.mark.parametrize("tname,view_id", RAGGED, ids=["%s-v%d" % k for k in RAGGED])
def test_po_kernel_ragged_frame(built, tname, view_id):
    """A 50 x 37 frame (u64): partial tiles and idle lanes; every certified sampled pixel -- the sample holds every pixel
    of the partial tiles (columns 48-49, row 36) -- has the exact count, and the model certifies most of them."""
    _, _, _, _, _, X, Y = window(tname, view_id, RAGGED_W, RAGGED_H)
    cnt, cert, _ = model(tname, view_id, RAGGED_W, RAGGED_H)
    edge = (X >= RAGGED_W - RAGGED_W % 8) | (Y >= RAGGED_H - RAGGED_H % 4)
    _report(f"{tname} view {view_id} {RAGGED_W}x{RAGGED_H}: certified {float(cert.mean()):.3f} of {cert.size}, "
            f"partial-tile pixels {int((cert & edge).sum())} of {int(edge.sum())} certified")
    assert cert.mean() >= 0.5 and (cert & edge).sum() >= 0.5 * edge.sum(), (cert.mean(), (cert & edge).sum())
    got = _gpu(tname, view_id, 8, RAGGED_W, RAGGED_H)[Y, X].astype(np.int64)
    _check(got, cnt, cert, X, Y, (tname, view_id, "ragged"))


# ---- per-step bounds against exact rationals ------------------------------------------------------------------------
N_REC = 4000
STEP_OPS = ("perturb", "norm2", "delta_x", "delta_y", "add")


def step_errors(tname, rec, vals, out, t=None):
    """{op: [(|result - exact|, bound)]} of perturb_selftest records (the bounds of exact_perturb.py, or of `t`)."""
    t = t or EP.TYPES[tname]
    nb = struct.calcsize(t.pod)
    errs = {k: [] for k in STEP_OPS}
    for i, (dx, dy, zx, zy, cx, cy, X, Y) in enumerate(vals):
        r = [EP.pod_value(tname, bytes(out[i, 16 * k:16 * k + nb])) for k in range(6)]
        f = [EP.bound_mag(tname, bytes(rec[i, 16 * k:16 * k + nb])) for k in range(6)]
        bx, by = EP.perturb_bound(t, *f)
        ex = dx * (2 * zx + dx) - dy * (2 * zy + dy) + cx
        ey = dx * (2 * zy + dy) + dy * (2 * zx + dx) + cy
        errs["perturb"] += [(abs(r[0] - ex), Fraction(bx)), (abs(r[1] - ey), Fraction(by))]
        errs["norm2"].append((abs(r[2] - (dx * dx + dy * dy)), Fraction(EP.norm_bound(t, f[0], f[1]))))
        errs["delta_x"].append((abs(r[3] - (X * zx - cx)), Fraction(EP.delta_bound(t, f[2], X, f[4]))))
        errs["delta_y"].append((abs(r[4] - (-Y * zy - cy)), Fraction(EP.delta_bound(t, f[3], Y, f[5]))))
        errs["add"].append((abs(r[5] - (zx + dx)), Fraction(EP.add_bound(t, f[2], f[0]))))
    return errs


def _assert_within(tname, errs):
    for op, lst in errs.items():
        ratio = max((float(e / b) if b else (float("inf") if e else 0.0) for e, b in lst), default=0.0)
        _report(f"{tname} {op}: worst error / bound {ratio:.3e}")
        bad = [i for i, (e, b) in enumerate(lst) if e > b]
        assert not bad, (tname, op, len(bad), bad[:5])


HOST_TYPES = ["f32", "f64", "hdr32", "hdr64"]


@pytest.mark.parametrize("tname", HOST_TYPES)
def test_step_bounds_host(built, tname):
    """NumPlain<float/double>, NumHdr<float/double> (FS_HD; host build, the device's bits): perturb, norm2, delta_x,
    delta_y and add within the bounds exact_perturb.py assumes, on records aimed at the step's case distinctions."""
    import numeric_vectors as nv
    import oracle_cpu
    rec, vals = nv.perturb_records(tname, N_REC)
    out = oracle_cpu.lockstep_numeric_op(nv.PERTURB_OPS[tname], rec, rec)
    _assert_within(tname, step_errors(tname, rec, vals, out))


def test_hdr64_step_has_binary32_precision(built):
    """NumHdr<double>::perturb rounds through the binary32 FMA (fs_num.cuh fmaf_as_ref): its bound is stated with
    binary32's epsilon, and the same bound with binary64's epsilon is exceeded."""
    import dataclasses
    import numeric_vectors as nv
    import oracle_cpu
    t = EP.TYPES["hdr64"]
    assert t.eps_step == 5 * 2.0 ** -24 and t.eps_c == 2 * 2.0 ** -24
    rec, vals = nv.perturb_records("hdr64", N_REC)
    out = oracle_cpu.lockstep_numeric_op(nv.PERTURB_OPS["hdr64"], rec, rec)
    as64 = dataclasses.replace(t, eps_step=5 * 2.0 ** -53, eps_c=2 * 2.0 ** -53)
    errs = step_errors("hdr64", rec, vals, out, as64)["perturb"]
    over = sum(e > b for e, b in errs)
    _report(f"hdr64 perturb under a binary64 epsilon: {over} of {len(errs)} results outside the bound")
    assert over > N_REC // 10, over


@pytest.mark.gpu
@pytest.mark.parametrize("tname", ["2x32", "hdr2x32"] + HOST_TYPES)
def test_step_bounds_device(built, tname):
    """fs_selftest_numeric_op 80-85 on the GPU: the df32 policies (Num2x32 plain arm, NumHdr2x32 custom_perturb3,
    device-only) within their bounds; the FS_HD policies bit for bit what the host build gives."""
    import numeric_vectors as nv
    from fractalshark_b200 import _native
    rec, vals = nv.perturb_records(tname, N_REC)
    got = np.zeros_like(rec)
    rc = _native.gpu_lib().fs_selftest_numeric_op(0, nv.PERTURB_OPS[tname], rec.ctypes.data, rec.ctypes.data,
                                                  got.ctypes.data, rec.shape[0])
    assert rc == 0, rc
    _assert_within(tname, step_errors(tname, rec, vals, got))
    if tname in HOST_TYPES:
        import oracle_cpu
        want = oracle_cpu.lockstep_numeric_op(nv.PERTURB_OPS[tname], rec, rec)
        nb = struct.calcsize(EP.TYPES[tname].pod.replace("4x", ""))   # HDRx64: not the padding
        for k in range(6):
            np.testing.assert_array_equal(got[:, 16 * k:16 * k + nb], want[:, 16 * k:16 * k + nb])
