"""Exponential maps (fs_render_perturb_lav2_expmap + fsh_view_expmap): one frame whose pixel (X, Y) lies at
dc = radius[Y] * (dir_x[X], dir_y[X]) from the reference point.  Every cell must be the cell a single render of that dc
gives: a sampled pixel is rendered again as pixel (0, 0) of a frame centred at -dc (delta_x / delta_y at X = Y = 0 give
back dc's bits exactly, which the self-test ops check first), 64 such frames per zoom batch."""
import hashlib
import math
import os
import struct
import subprocess
import sys
from fractions import Fraction

import numpy as np
import pytest

import cases
import oracle_cpu
from fractalshark_b200 import LAv2Mode, Numeric, traits
from fractalshark_b200 import RenderAlgorithm as A
from fractalshark_b200 import _native
from fractalshark_b200.gpu_renderer import GPURenderer
from fractalshark_b200.host_inputs import POD_BYTES, View
from fractalshark_b200.views import PRESETS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNSUPPORTED = 10100
PERTURB_OPS = {Numeric.F32: 80, Numeric.F64: 81, Numeric.HDR32: 82, Numeric.HDR64: 83, Numeric.X2_32: 84,
               Numeric.HDR2X32: 85}
EXPMAP_OPS = {Numeric.F32: 86, Numeric.F64: 87, Numeric.HDR32: 88, Numeric.HDR64: 89, Numeric.X2_32: 90,
              Numeric.HDR2X32: 91}
HOST_NUMERICS = [Numeric.F32, Numeric.F64, Numeric.HDR32, Numeric.HDR64]
# bytes holding the sign bit of every float of a POD (the 2x32 types negate head and tail)
SIGN_BYTES = {Numeric.F32: (3,), Numeric.F64: (7,), Numeric.X2_32: (3, 7), Numeric.HDR32: (3,), Numeric.HDR64: (7,),
              Numeric.HDR2X32: (3, 7)}
# bytes of a POD that hold its value (HDRx64: 4 bytes of padding behind the exponent)
VALUE_BYTES = {Numeric.F32: 4, Numeric.F64: 8, Numeric.X2_32: 8, Numeric.HDR32: 8, Numeric.HDR64: 12, Numeric.HDR2X32: 12}
# views whose range each type covers, as the parity cases use them
VIEW_OF = {Numeric.F32: 101, Numeric.F64: 101, Numeric.X2_32: 101, Numeric.HDR32: 14, Numeric.HDR64: 14,
           Numeric.HDR2X32: 14}


def _neg(numeric, pod: bytes) -> bytes:
    b = bytearray(pod)
    for k in SIGN_BYTES[numeric]:
        b[k] ^= 0x80
    return bytes(b)


def _pod(table: bytes, numeric, k: int) -> bytes:
    nb = POD_BYTES[numeric]
    return table[k * nb:(k + 1) * nb]


def _expmap_operands(em, numeric, xs, ys):
    """Elements of ops 86-91 for pixels (xs[i], ys[i]): a = {radius[Y], -}, b = {dir_x[X], dir_y[X]}."""
    nb = POD_BYTES[numeric]
    a = np.zeros((len(xs), 32), np.uint8)
    b = np.zeros((len(xs), 32), np.uint8)
    for i, (x, y) in enumerate(zip(xs, ys)):
        a[i, :nb] = np.frombuffer(_pod(em["radius"], numeric, y), np.uint8)
        b[i, :nb] = np.frombuffer(_pod(em["dir_x"], numeric, x), np.uint8)
        b[i, 16:16 + nb] = np.frombuffer(_pod(em["dir_y"], numeric, x), np.uint8)
    return a, b


def _split_dc(out, numeric, nb=None):
    nb = nb or POD_BYTES[numeric]
    return [bytes(row[:nb]) for row in out], [bytes(row[16:16 + nb]) for row in out]


def _assert_deltas_give_dc(out, numeric, dcx, dcy):
    """Slots 3 / 4 of perturb_selftest records hold dcX / dcY, compared on the bytes that hold the value."""
    vb = VALUE_BYTES[numeric]
    assert [bytes(r[48:48 + vb]) for r in out] == [x[:vb] for x in dcx]
    assert [bytes(r[64:64 + vb]) for r in out] == [y[:vb] for y in dcy]


def _delta_records(numeric, coords, dcx, dcy):
    """perturb_selftest records whose slots 3 / 4 are delta_x(dx, 0, -dcX) / delta_y(dy, 0, -dcY): pixel (0, 0) of a
    frame with the view's spacing, centred at -dc."""
    nb = POD_BYTES[numeric]
    rec = np.zeros((len(dcx), 128), np.uint8)
    for i, (x, y) in enumerate(zip(dcx, dcy)):
        rec[i, 32:32 + nb] = np.frombuffer(coords["dx"], np.uint8)
        rec[i, 48:48 + nb] = np.frombuffer(coords["dy"], np.uint8)
        rec[i, 64:64 + nb] = np.frombuffer(_neg(numeric, x), np.uint8)
        rec[i, 80:80 + nb] = np.frombuffer(_neg(numeric, y), np.uint8)
    return rec


def _host_expmap_op(op, a, b):
    out = np.zeros_like(a)
    rc = _native.host_lib().fsh_selftest_numeric_op(op, a.ctypes.data, b.ctypes.data, out.ctypes.data, a.shape[0])
    assert rc == 0
    return out


# ---- CPU -----------------------------------------------------------------------------------------------------------------
def test_expmap_entries_are_bound(built):
    assert callable(_native.gpu_lib().fs_render_perturb_lav2_expmap)
    assert callable(_native.host_lib().fsh_view_expmap)
    assert callable(_native.host_lib().fsh_selftest_numeric_op)
    assert callable(GPURenderer.RenderPerturbLAv2ExpMap) and callable(View.exp_map)


def test_bad_expmap_renders_are_refused_without_touching_cuda(built):
    """A NULL renderer or table, a mode other than Full / PO / LAO and a renderer without initialized memory are refused
    before any CUDA call: in a fresh process the CUDA driver library is not even loaded afterwards."""
    code = ("import ctypes, sys; sys.path.insert(0, %r)\n"
            "from fractalshark_b200 import _native\n"
            "lib = _native.gpu_lib()\n"
            "t = ctypes.create_string_buffer(8 * 64)\n"
            "r = lib.fs_create(0)\n"
            "go = lambda h, mode, a, b, c: lib.fs_render_perturb_lav2_expmap(h, 3, 3, mode, 0, a, b, c, 1000)\n"
            "rcs = [go(None, 1, t, t, t), go(r, 1, None, t, t), go(r, 1, t, None, t), go(r, 1, t, t, None),\n"
            "       go(r, 0, t, t, t), go(r, 4, t, t, t), go(r, 1, t, t, t), go(r, 2, t, t, t), go(r, 3, t, t, t)]\n"
            "lib.fs_destroy(r)\n"
            "maps = open('/proc/self/maps').read()\n"
            "print(*rcs, int('libcuda.so' in maps))\n" % ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    *rcs, cuda_loaded = map(int, out.stdout.split())
    assert rcs == [UNSUPPORTED] * 9
    assert cuda_loaded == 0


def test_exp_map_refuses_types_it_has_no_table_for(built):
    p = PRESETS[5]
    v = View(p.min_x, p.min_y, p.max_x, p.max_y, 64, 36)
    with pytest.raises(ValueError):
        v.exp_map(Numeric.X4_64, 8)
    assert _native.host_lib().fsh_selftest_numeric_op(90, None, None, None, 0) == -1


def _log2(q: Fraction):
    """log2 q as (integer, float) parts, exact up to the float's rounding."""
    k = q.numerator.bit_length() - q.denominator.bit_length()
    return k, math.log2(float(q / Fraction(2) ** k))


def _value(numeric, pod: bytes) -> Fraction:
    if numeric == Numeric.F64:
        return Fraction(struct.unpack("<d", pod)[0])
    m, e = struct.unpack("<di4x", pod)
    return Fraction(m) * Fraction(2) ** e


@pytest.mark.parametrize("numeric,view_id", [(Numeric.F64, 5), (Numeric.F64, 1), (Numeric.HDR64, 5),
                                             (Numeric.HDR64, 14)],
                         ids=["f64_v5", "f64_v1", "hdr64_v5", "hdr64_v14"])
def test_exp_map_tables_follow_the_map(built, numeric, view_id):
    """Radii and directions, checked with exact arithmetic from the view's own dx / dy PODs: radius0 = half-diagonal *
    e^(-pi/W), log2 radius[Y] = log2 radius0 - Y 2 pi / (W ln 2), |dir| = 1."""
    w, h, rows = 256, 144, 64
    p = PRESETS[view_id]
    v = View(p.min_x, p.min_y, p.max_x, p.max_y, w, h)
    em = v.exp_map(numeric, rows)
    coords = v.coords(numeric)
    dx, dy = _value(numeric, coords["dx"]), _value(numeric, coords["dy"])
    d2 = (dx * w / 2) ** 2 + (dy * h / 2) ** 2
    k2, f2 = _log2(d2)
    step = 2 * math.pi / (w * math.log(2))
    want_k, want_f = k2 // 2, (k2 % 2 + f2) / 2 - step / 2
    assert em["log2_row_step"] == pytest.approx(-step, rel=1e-15)
    assert em["log2_radius0"] == pytest.approx(want_k + want_f, rel=1e-12)
    radii = [_value(numeric, _pod(em["radius"], numeric, y)) for y in range(rows)]
    assert all(a > b for a, b in zip(radii, radii[1:]))
    for y, rho in enumerate(radii):
        k, f = _log2(rho)
        assert abs((k - want_k) + (f - (want_f - y * step))) < 2.0 ** -40, y
    for x in range(w):
        ux, uy = (_value(numeric, _pod(em[t], numeric, x)) for t in ("dir_x", "dir_y"))
        assert abs(ux * ux + uy * uy - 1) <= 8 * Fraction(2) ** -52, x
    # column X at angle 2 pi (X + 1/2) / W, counter-clockwise from the positive real axis
    ux, uy = (float(_value(numeric, _pod(em[t], numeric, w // 8))) for t in ("dir_x", "dir_y"))
    assert math.atan2(uy, ux) == pytest.approx(2 * math.pi * (w // 8 + 0.5) / w, rel=1e-14)


# sha256 of radius + dir_x + dir_y of View 1 at 16x9, 8 rows: a change of conventions (rounding, reduction, angle
# origin, row 0) shows here even where the checks above would still hold
PINNED = {
    Numeric.F32: "f7a81a847198d0248439c6a14db3a9e326ceac0052c3ae741b4e5735f4870f7b",
    Numeric.F64: "ee5cf8bf8be53255bdca14784ec67523dbc6da3022af424b75e7d43023c1df53",
    Numeric.X2_32: "d6c07e91307c04613127f1457694c94d4a4cc098bf4aaa1e465f78bc5f76211f",
    Numeric.HDR32: "c3489c813ec8e749a4fcb7b3016f4977f47dbbd67fd1b4c5f60b8a539afcfc66",
    Numeric.HDR64: "15f287af89216c5de5d62fa7fdc744c0beae82d783a4e31e060a0d45b7bb9dbc",
    Numeric.HDR2X32: "c7b359b45cde653dc33b2144a846d9df272ee19c78882b602e6efc2b72d01f77",
}


@pytest.mark.parametrize("numeric", list(PINNED), ids=[t.name for t in PINNED])
def test_small_exp_map_tables_are_pinned(built, numeric):
    p = PRESETS[1]
    em = View(p.min_x, p.min_y, p.max_x, p.max_y, 16, 9).exp_map(numeric, 8)
    assert len(em["radius"]) == 8 * POD_BYTES[numeric] and len(em["dir_x"]) == 16 * POD_BYTES[numeric]
    assert hashlib.sha256(em["radius"] + em["dir_x"] + em["dir_y"]).hexdigest() == PINNED[numeric]


@pytest.mark.parametrize("numeric,view_id", [(Numeric.F32, 101), (Numeric.F64, 100), (Numeric.HDR32, 14),
                                             (Numeric.HDR32, 5), (Numeric.HDR64, 14), (Numeric.HDR64, 5)],
                         ids=["f32_v101", "f64_v100", "hdr32_v14", "hdr32_v5", "hdr64_v14", "hdr64_v5"])
def test_pixel_zero_of_a_frame_centred_at_minus_dc_has_that_dc(built, numeric, view_id):
    """Host build of the policies: delta_x(dx, 0, -dcX) and delta_y(dy, 0, -dcY) (ops 80-83, slots 3 / 4) return the bits
    of expmap_dc (ops 86-89) for every pixel of a 64 x 64 map -- what the GPU check below renders with."""
    p = PRESETS[view_id]
    v = View(p.min_x, p.min_y, p.max_x, p.max_y, 64, 36)
    em, coords = v.exp_map(numeric, 64), v.coords(numeric)
    ys, xs = np.divmod(np.arange(64 * 64), 64)
    out = _host_expmap_op(EXPMAP_OPS[numeric], *_expmap_operands(em, numeric, xs, ys))
    dcx, dcy = _split_dc(out, numeric)
    nb = POD_BYTES[numeric]
    # the construction needs dc != 0 (a zero's sign or HDR exponent is not carried through): no row underflows here
    mant = "<f" if numeric in (Numeric.F32, Numeric.HDR32) else "<d"
    assert all(struct.unpack_from(mant, c)[0] != 0 for c in dcx + dcy)
    got = oracle_cpu.lockstep_numeric_op(PERTURB_OPS[numeric], *[_delta_records(numeric, coords, dcx, dcy)] * 2)
    _assert_deltas_give_dc(got, numeric, dcx, dcy)


# ---- GPU -----------------------------------------------------------------------------------------------------------------
W, ROWS, VIEW_H = 64, 64, 36
ALGS = {
    Numeric.F32: (A.Gpu1x32PerturbedLAv2, A.Gpu1x32PerturbedLAv2PO, A.Gpu1x32PerturbedLAv2LAO),
    Numeric.F64: (A.Gpu1x64PerturbedLAv2, A.Gpu1x64PerturbedLAv2PO, A.Gpu1x64PerturbedLAv2LAO),
    Numeric.X2_32: (A.Gpu2x32PerturbedLAv2, A.Gpu2x32PerturbedLAv2PO, A.Gpu2x32PerturbedLAv2LAO),
    Numeric.HDR32: (A.GpuHDRx32PerturbedLAv2, A.GpuHDRx32PerturbedLAv2PO, A.GpuHDRx32PerturbedLAv2LAO),
    Numeric.HDR64: (A.GpuHDRx64PerturbedLAv2, A.GpuHDRx64PerturbedLAv2PO, A.GpuHDRx64PerturbedLAv2LAO),
    Numeric.HDR2X32: (A.GpuHDRx2x32PerturbedLAv2, A.GpuHDRx2x32PerturbedLAv2PO, A.GpuHDRx2x32PerturbedLAv2LAO),
}
RC_ALGS = (A.GpuHDRx32PerturbedRCLAv2, A.GpuHDRx32PerturbedRCLAv2PO, A.GpuHDRx32PerturbedRCLAv2LAO)


def _n_iter(alg):
    """PO on View 14 stops at 3,000 (no LA: every interior pixel would run the preset's 2^31); the rest use the preset."""
    t = traits(alg)
    return 3000 if VIEW_OF[t.numeric] == 14 and t.mode == LAv2Mode.PO else None


# (algorithm, iteration bytes): six numeric types x Full / PO / LAO x u32 / u64, and the RC orbits of HDRx32
GPU_CASES = [(alg, ib) for algs in ALGS.values() for alg in algs for ib in (4, 8)] + [(alg, ib) for alg in RC_ALGS
                                                                                    for ib in (4, 8)]
GPU_IDS = [f"{alg.name}_u{8 * ib}" for alg, ib in GPU_CASES]


def _setup(alg, ib, view_id=None, n_iter=None):
    numeric = traits(alg).numeric
    view_id = VIEW_OF[numeric] if view_id is None else view_id
    view, coords, orbit, la, n = cases.make_inputs(view_id, W, VIEW_H, alg, n_iter or _n_iter(alg), ib)
    return view, coords, orbit, la, n, view.exp_map(numeric, ROWS)


def _renderer(w, h, ib, orbit, la, aa=1, make=GPURenderer, shard=None):
    r = make()
    assert r.InitializeMemory(w, h, aa, iter_bytes=ib) == 0
    if shard is not None:
        assert r.SetShard(*shard) == 0
    assert r.InitializePerturb(1, orbit, 0, None, la) == 0
    r.ClearMemory()
    return r


def _render_expmap(r, alg, em, n, colours=False):
    rc = r.RenderPerturbLAv2ExpMap(alg, em, n)
    assert rc == 0, GPURenderer.ConvertErrorToString(rc)
    rc, iters, col, red = r.RenderCurrent(n, want_colors=colours)
    assert rc == 0
    return iters, col, red


def _samples(cells, n, rng):
    """>= 256 pixels: the first and last row and column, escaped pixels and pixels at the limit where there are any,
    and random ones."""
    h, w = cells.shape
    picks = []
    for k in np.linspace(0, w - 1, 16).astype(int):
        picks += [(int(k), 0), (int(k), h - 1)]
    for k in np.linspace(0, h - 1, 16).astype(int):
        picks += [(0, int(k)), (w - 1, int(k))]
    for where in (np.argwhere(cells < n), np.argwhere(cells >= n)):
        for y, x in where[rng.permutation(len(where))[:64]]:
            picks.append((int(x), int(y)))
    while len(set(picks)) < 256:
        picks.append((int(rng.integers(0, w)), int(rng.integers(0, h))))
    picks = sorted(set(picks))
    return [x for x, _ in picks], [y for _, y in picks]


def _device_op(op, a, b):
    out = np.zeros_like(a)
    rc = _native.gpu_lib().fs_selftest_numeric_op(0, op, a.ctypes.data, b.ctypes.data, out.ctypes.data, a.shape[0])
    assert rc == 0
    return out


def _single_cells(alg, ib, orbit, la, coords, dcx, dcy, n):
    """Pixel (0, 0) of one frame per dc, centred at -dc with the view's spacing: 64 frames per zoom batch on an 8x4
    renderer with the same uploads."""
    numeric = traits(alg).numeric
    r = _renderer(8, 4, ib, orbit, la)
    out = []
    for k in range(0, len(dcx), 64):
        frames = [{"cx": coords["cx"], "cy": coords["cy"], "dx": coords["dx"], "dy": coords["dy"],
                   "center_x": _neg(numeric, x), "center_y": _neg(numeric, y)}
                  for x, y in zip(dcx[k:k + 64], dcy[k:k + 64])]
        rc = r.RenderPerturbLAv2Frames(alg, frames, n)
        assert rc == 0, GPURenderer.ConvertErrorToString(rc)
        for f in range(len(frames)):
            assert r.SelectFrame(f) == 0
            rc, iters, _, _ = r.RenderCurrent(n)
            assert rc == 0
            out.append(int(iters[0, 0]))
    r.close()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("alg,ib", GPU_CASES, ids=GPU_IDS)
def test_every_exp_map_cell_is_the_single_render_of_its_dc(alg, ib):
    numeric = traits(alg).numeric
    _, coords, orbit, la, n, em = _setup(alg, ib)
    r = _renderer(W, ROWS, ib, orbit, la)
    iters, _, _ = _render_expmap(r, alg, em, n)
    r.close()
    cells = iters[:ROWS, :W]
    xs, ys = _samples(cells, n, np.random.default_rng(int(alg) * 8 + ib))
    assert len(xs) >= 256
    if traits(alg).mode == LAv2Mode.Full:
        assert (cells < n).any() and (cells >= n).any()  # both kinds of pixel are among the samples
    dcx, dcy = _split_dc(_device_op(EXPMAP_OPS[numeric], *_expmap_operands(em, numeric, xs, ys)), numeric)
    rec = _delta_records(numeric, coords, dcx, dcy)
    _assert_deltas_give_dc(_device_op(PERTURB_OPS[numeric], rec, rec), numeric, dcx, dcy)
    want = _single_cells(alg, ib, orbit, la, coords, dcx, dcy, n)
    got = [int(cells[y, x]) for x, y in zip(xs, ys)]
    bad = [(x, y, g, w) for x, y, g, w in zip(xs, ys, got, want) if g != w]
    assert not bad, f"{len(bad)} of {len(xs)} cells differ, first (X, Y, exp map, single): {bad[:5]}"


@pytest.mark.gpu
@pytest.mark.parametrize("aa", [1, 2])
@pytest.mark.parametrize("alg,ib", [(A.GpuHDRx32PerturbedLAv2, 4), (A.Gpu1x64PerturbedLAv2, 8)],
                         ids=["GpuHDRx32PerturbedLAv2_u32", "Gpu1x64PerturbedLAv2_u64"])
def test_groups_and_shards_return_the_single_renderers_bytes(alg, ib, aa):
    """A group {0, 0} and two renderers with fs_set_shard(2, i) give one renderer's cells, colours and Min/Max/Sum."""
    _, _, orbit, la, n, em = _setup(alg, ib)
    r = _renderer(W, ROWS, ib, orbit, la, aa=aa)
    want_it, want_col, want_red = _render_expmap(r, alg, em, n, colours=True)
    r.close()
    g = _renderer(W, ROWS, ib, orbit, la, aa=aa, make=lambda: GPURenderer(devices=[0, 0]))
    got_it, got_col, got_red = _render_expmap(g, alg, em, n, colours=True)
    g.close()
    np.testing.assert_array_equal(got_it, want_it)
    np.testing.assert_array_equal(got_col, want_col)
    assert got_red == want_red
    it = np.zeros_like(want_it)
    col = np.zeros_like(want_col)
    mins, maxs, sums = [], [], 0
    for s in range(2):
        sh = _renderer(W, ROWS, ib, orbit, la, aa=aa, shard=(2, s))
        assert sh.RenderPerturbLAv2ExpMap(alg, em, n) == 0
        rc, red = sh.RenderCurrentShard(n, it, colors_out=col)
        assert rc == 0
        mins.append(red["Min"]); maxs.append(red["Max"]); sums += red["Sum"]
        sh.close()
    np.testing.assert_array_equal(it, want_it)
    n_cells = (ROWS // aa) * (W // aa)
    np.testing.assert_array_equal(col.reshape(-1, 4)[:n_cells], want_col.reshape(-1, 4)[:n_cells])
    assert (min(mins), max(maxs), sums) == (want_red["Min"], want_red["Max"], want_red["Sum"])


@pytest.mark.gpu
def test_the_result_sink_holds_the_exp_map():
    alg, ib = A.GpuHDRx32PerturbedLAv2, 4
    _, _, orbit, la, n, em = _setup(alg, ib)
    r = _renderer(W, ROWS, ib, orbit, la)
    sink = np.full(r.buffer_shape(), 7, np.uint32)
    assert r.SetResultSink(sink) == 0
    assert r.EnableStepCounter(True) == 0
    before = r.KernelLaunchCount()
    assert r.RenderPerturbLAv2ExpMap(alg, em, n) == 0
    assert r.SyncComputeStream() == 0
    assert r.KernelLaunchCount() - before == 1
    assert r.ReadStepCounters()["total"] > 0 and r.LastRenderMs() > 0
    streamed = sink.copy()
    assert r.SetResultSink(None) == 0
    rc, iters, _, _ = r.RenderCurrent(n)
    assert rc == 0
    np.testing.assert_array_equal(streamed, iters)
    assert (streamed[:ROWS, :W] != 7).all()
    r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("alg,ib", [(A.GpuHDRx32PerturbedLAv2, 4), (A.GpuHDRx2x32PerturbedLAv2LAO, 8)],
                         ids=["GpuHDRx32PerturbedLAv2_u32", "GpuHDRx2x32PerturbedLAv2LAO_u64"])
def test_an_exp_map_is_one_frame_and_leaves_the_renderer_as_a_single_render_does(alg, ib):
    view_id = VIEW_OF[traits(alg).numeric]
    p = PRESETS[view_id]
    _, _, orbit, la, n, em = _setup(alg, ib)
    coords = View(p.min_x, p.min_y, p.max_x, p.max_y, W, ROWS).coords(traits(alg).numeric)
    fresh = _renderer(W, ROWS, ib, orbit, la)
    assert fresh.RenderPerturbLAv2(alg, coords, n) == 0
    want = fresh.RenderCurrent(n, want_colors=True)
    fresh.close()
    r = _renderer(W, ROWS, ib, orbit, la)
    _render_expmap(r, alg, em, n)
    assert r.SelectFrame(1) == UNSUPPORTED
    assert r.SelectFrame(0) == 0
    assert r.RenderPerturbLAv2(alg, coords, n) == 0
    got = r.RenderCurrent(n, want_colors=True)
    r.close()
    assert got[0] == want[0] == 0
    np.testing.assert_array_equal(got[1], want[1])
    np.testing.assert_array_equal(got[2], want[2])
    assert got[3] == want[3]
