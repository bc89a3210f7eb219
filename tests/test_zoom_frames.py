"""Zoom batches (fs_render_perturb_lav2_frames + fs_select_frame): frames of one orbit and LA table rendered in one launch
return, frame by frame, exactly the bytes a single-frame render of the same coordinates returns -- iteration cells (whole
padded buffers), colours and Min/Max/Sum.  The frames come from View.zoomed, which keeps the centre and therefore the
reference orbit."""
import os
import struct
import subprocess
import sys

import numpy as np
import pytest

import cases
from fractalshark_b200 import LAv2Mode, Numeric, traits
from fractalshark_b200 import RenderAlgorithm as A
from fractalshark_b200 import _native
from fractalshark_b200.gpu_renderer import GPURenderer
from fractalshark_b200.host_inputs import View
from fractalshark_b200.views import PRESETS
from test_device_group import GROUP_IDS, GROUPS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNSUPPORTED = 10100
PERTURB_NUMERICS = [Numeric.F32, Numeric.F64, Numeric.X2_32, Numeric.HDR32, Numeric.HDR64, Numeric.HDR2X32]

# scale 1, zoom-outs, one zoom-in and a repeated frame
SCALES = ["1", "2", "1.5", "0.5", "1", "4"]


# ---- CPU -----------------------------------------------------------------------------------------------------------------
def test_frame_entries_are_bound(built):
    lib = _native.gpu_lib()
    assert callable(lib.fs_render_perturb_lav2_frames)
    assert callable(lib.fs_select_frame)
    assert callable(_native.host_lib().fsh_view_zoom)


def test_bad_batches_and_selections_are_refused_without_touching_cuda(built):
    """n_frames 0 and 65 and a NULL renderer are refused before any CUDA call, as is fs_select_frame on a handle that has
    rendered nothing: in a fresh process the CUDA driver library is not even loaded afterwards."""
    code = ("import ctypes, sys; sys.path.insert(0, %r)\n"
            "from fractalshark_b200 import _native\n"
            "lib = _native.gpu_lib()\n"
            "pod = ctypes.create_string_buffer(8 * 65)\n"
            "r = lib.fs_create(0)\n"
            "args = lambda n: (3, 3, 1, 0, n, pod, pod, pod, pod, pod, pod, 1000)\n"
            "rcs = [lib.fs_render_perturb_lav2_frames(r, *args(0)), lib.fs_render_perturb_lav2_frames(r, *args(65)),\n"
            "       lib.fs_render_perturb_lav2_frames(None, *args(1)), lib.fs_select_frame(r, 0),\n"
            "       lib.fs_select_frame(r, 1), lib.fs_select_frame(None, 0)]\n"
            "lib.fs_destroy(r)\n"
            "maps = open('/proc/self/maps').read()\n"
            "print(*rcs, int('libcuda.so' in maps))\n" % ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    *rcs, cuda_loaded = map(int, out.stdout.split())
    assert rcs == [UNSUPPORTED] * 6
    assert cuda_loaded == 0


@pytest.mark.parametrize("view_id", [0, 1, 5, 14, 100, 101])
@pytest.mark.parametrize("size", [(96, 54, 1), (100, 270, 1), (150, 270, 3)], ids=["96x54", "100x270", "150x270_aa3"])
def test_zoomed_by_one_is_the_parent_view(built, view_id, size):
    p = PRESETS[view_id]
    v = View(p.min_x, p.min_y, p.max_x, p.max_y, *size)
    z = v.zoomed("1")
    assert (z.width, z.height, z.antialiasing, z.precision_bits) == (v.width, v.height, v.antialiasing, v.precision_bits)
    for t in PERTURB_NUMERICS:
        assert z.coords(t) == v.coords(t), t.name


_HDR_LAYOUT = {Numeric.HDR32: "<fi", Numeric.HDR64: "<di4x", Numeric.HDR2X32: "<ffi"}


@pytest.mark.parametrize("view_id", [1, 5, 14, 100])
def test_zoomed_by_two_doubles_the_pixel_spacing_exactly(built, view_id):
    """HDR types: the same mantissa, exponent + 1."""
    p = PRESETS[view_id]
    v = View(p.min_x, p.min_y, p.max_x, p.max_y, 100, 270)
    z = v.zoomed("2")
    for t, fmt in _HDR_LAYOUT.items():
        a, b = v.coords(t), z.coords(t)
        for k in ("dx", "dy"):
            *ma, ea = struct.unpack(fmt, a[k])
            *mb, eb = struct.unpack(fmt, b[k])
            assert ma == mb and eb == ea + 1, (t.name, k)


def test_zoomed_refuses_a_scale_that_is_not_a_positive_number(built):
    p = PRESETS[0]
    v = View(p.min_x, p.min_y, p.max_x, p.max_y, 64, 36)
    for bad in ("", "x", "0", "-1"):
        with pytest.raises(ValueError):
            v.zoomed(bad)


# ---- GPU -----------------------------------------------------------------------------------------------------------------
# (view id, w, h, algorithm, n_iter (None = preset), iter_bytes, antialiasing): every LAv2 numeric type with Full / PO / LAO
# and RC, u32 and u64, on the views the parity cases use for that type; ragged sizes, AA 1 and AA 3
CASES = [
    (5, 96, 54, A.GpuHDRx32PerturbedLAv2, None, 4, 1),
    (5, 100, 270, A.GpuHDRx32PerturbedLAv2PO, 3000, 8, 1),
    (14, 150, 270, A.GpuHDRx32PerturbedLAv2, None, 4, 3),
    (1, 96, 54, A.GpuHDRx32PerturbedLAv2LAO, None, 4, 1),
    (5, 100, 270, A.GpuHDRx32PerturbedRCLAv2, None, 8, 1),
    (5, 64, 36, A.GpuHDRx64PerturbedLAv2, None, 4, 1),
    (5, 150, 270, A.GpuHDRx64PerturbedRCLAv2PO, 3000, 8, 3),
    (100, 96, 54, A.Gpu1x64PerturbedLAv2, None, 4, 1),
    (1, 96, 54, A.Gpu1x64PerturbedRCLAv2LAO, None, 8, 3),
    (101, 96, 54, A.Gpu1x32PerturbedLAv2, None, 4, 1),
    (101, 100, 270, A.Gpu1x32PerturbedRCLAv2PO, None, 8, 1),
    (100, 96, 54, A.Gpu2x32PerturbedLAv2LAO, None, 4, 1),
    (101, 150, 270, A.Gpu2x32PerturbedRCLAv2, None, 8, 3),
    (5, 96, 54, A.GpuHDRx2x32PerturbedLAv2PO, 3000, 4, 1),
    (1, 100, 270, A.GpuHDRx2x32PerturbedRCLAv2, None, 8, 1),
    (5, 96, 54, A.GpuHDRx2x32PerturbedLAv2LAO, None, 4, 3),
]
CASE_IDS = [f"v{c[0]}_{c[3].name}_{c[1]}x{c[2]}_u{8 * c[5]}_aa{c[6]}" for c in CASES]


def _inputs(case, scales=SCALES):
    view_id, w, h, alg, n_iter, ib, aa = case
    view, _, orbit, la, n = cases.make_inputs(view_id, w, h, alg, n_iter, ib)  # w, h: super-sampled, as in cases.render
    numeric = traits(alg).numeric
    return [view.zoomed(s).coords(numeric) for s in scales], orbit, la, n


def _renderer(case, orbit, la, make=GPURenderer, shard=None):
    _, w, h, _, _, ib, aa = case
    r = make()
    assert r.InitializeMemory(w, h, aa, iter_bytes=ib) == 0
    if shard is not None:
        assert r.SetShard(*shard) == 0
    assert r.InitializePerturb(1, orbit, 0, None, la) == 0
    r.ClearMemory()
    return r


def _result(r, n):
    rc, iters, colors, red = r.RenderCurrent(n, want_colors=True)
    assert rc == 0
    return iters, colors, red


def _singles(case, frames, orbit, la, n):
    """The reference: a fresh single-frame render of every frame's coordinates with the same orbit and LA table."""
    alg = case[3]
    out = []
    for coords in frames:
        r = _renderer(case, orbit, la)
        rc = r.RenderPerturbLAv2(alg, coords, n)
        assert rc == 0, GPURenderer.ConvertErrorToString(rc)
        out.append(_result(r, n))
        r.close()
    return out


def _batch_results(r, n_frames, n):
    out = []
    for k in range(n_frames):
        assert r.SelectFrame(k) == 0
        out.append(_result(r, n))
    return out


def _batch(r, case, frames, n):
    rc = r.RenderPerturbLAv2Frames(case[3], frames, n)
    assert rc == 0, GPURenderer.ConvertErrorToString(rc)
    return _batch_results(r, len(frames), n)


def _assert_same(got, want):
    assert len(got) == len(want)
    for k, ((gi, gc, gr), (wi, wc, wr)) in enumerate(zip(got, want)):
        np.testing.assert_array_equal(gi, wi, err_msg=f"frame {k}: iterations")
        np.testing.assert_array_equal(gc, wc, err_msg=f"frame {k}: colours")
        assert gr == wr, f"frame {k}: reduction"


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_every_frame_of_a_batch_equals_its_single_render(case):
    frames, orbit, la, n = _inputs(case)
    want = _singles(case, frames, orbit, la, n)
    r = _renderer(case, orbit, la)
    got = _batch(r, case, frames, n)
    assert r.SelectFrame(len(frames)) == UNSUPPORTED
    r.close()
    _assert_same(got, want)
    # the frames really differ, so a batch that rendered frame 0 six times would not pass.  Checked where the full algorithm
    # runs on a frame with any structure: a frame that is interior at the iteration cap everywhere (View 5 at 3,000 PO
    # iterations) looks the same at every scale, and an LA-only count can be the same at scales 1 and 2 (View 1, f64 LAO).
    _, w, h, alg = case[:4]
    if traits(alg).mode == LAv2Mode.Full and np.unique(want[0][0][:h, :w]).size > 1:
        assert not np.array_equal(want[0][0], want[1][0])


@pytest.mark.gpu
@pytest.mark.parametrize("case", [CASES[0], CASES[8], CASES[13]], ids=[CASE_IDS[0], CASE_IDS[8], CASE_IDS[13]])
def test_a_batch_of_one_frame_is_the_single_render(case):
    frames, orbit, la, n = _inputs(case, ["1.25"])
    r = _renderer(case, orbit, la)
    assert r.RenderPerturbLAv2(case[3], frames[0], n) == 0
    want = [_result(r, n)]
    r.ClearMemory()
    got = _batch(r, case, frames, n)
    assert r.SelectFrame(1) == UNSUPPORTED
    r.close()
    _assert_same(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("case", [CASES[0], CASES[4], CASES[11]], ids=[CASE_IDS[0], CASE_IDS[4], CASE_IDS[11]])
def test_sharded_batches_assemble_the_unsharded_frames(case):
    """fs_set_shard applies per frame: three shards' RenderCurrentShard of frame k fill frame k."""
    frames, orbit, la, n = _inputs(case)
    r = _renderer(case, orbit, la)
    want = _batch(r, case, frames, n)
    r.close()
    shards = [_renderer(case, orbit, la, shard=(3, i)) for i in range(3)]
    for s in shards:
        assert s.RenderPerturbLAv2Frames(case[3], frames, n) == 0
    dt = np.uint32 if case[5] == 4 else np.uint64
    for k in range(len(frames)):
        whole = np.zeros(shards[0].buffer_shape(), dt)
        for s in shards:
            assert s.SelectFrame(k) == 0
            rc, _ = s.RenderCurrentShard(n, whole)
            assert rc == 0
        np.testing.assert_array_equal(whole, want[k][0], err_msg=f"frame {k}")
    for s in shards:
        s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("devices", GROUPS, ids=GROUP_IDS)
@pytest.mark.parametrize("case", [CASES[0], CASES[2], CASES[12]], ids=[CASE_IDS[0], CASE_IDS[2], CASE_IDS[12]])
def test_groups_return_the_single_renderers_bytes_for_every_frame(case, devices):
    """AA 1 colours and reductions meet on the lead; AA 3 frames are gathered there from the selected frame's bands."""
    frames, orbit, la, n = _inputs(case)
    r = _renderer(case, orbit, la)
    want = _batch(r, case, frames, n)
    r.close()
    g = _renderer(case, orbit, la, make=lambda: GPURenderer(devices=devices))
    got = _batch(g, case, frames, n)
    assert g.SelectFrame(len(frames)) == UNSUPPORTED
    g.close()
    _assert_same(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("case", [CASES[0], CASES[7]], ids=[CASE_IDS[0], CASE_IDS[7]])
def test_batch_step_counters_are_the_sum_of_the_single_renders(case):
    frames, orbit, la, n = _inputs(case)
    counts = []
    for batch in (False, True):
        r = _renderer(case, orbit, la)
        assert r.EnableStepCounter(True) == 0
        before = r.KernelLaunchCount()
        if batch:
            assert r.RenderPerturbLAv2Frames(case[3], frames, n) == 0
        else:
            for coords in frames:
                assert r.RenderPerturbLAv2(case[3], coords, n) == 0
        counts.append(r.ReadStepCounters())
        launches = r.KernelLaunchCount() - before
        r.close()
    assert counts[1] == counts[0]
    assert counts[1]["total"] > 0
    assert launches == 1  # the whole batch is one kernel


@pytest.mark.gpu
def test_a_batch_leaves_the_result_sink_unfilled_and_render_current_copies():
    case = CASES[0]
    frames, orbit, la, n = _inputs(case)
    want = _singles(case, frames, orbit, la, n)
    r = _renderer(case, orbit, la)
    sink = np.full(r.buffer_shape(), 7, np.uint32)
    assert r.SetResultSink(sink) == 0
    assert r.RenderPerturbLAv2Frames(case[3], frames, n) == 0
    assert r.SyncComputeStream() == 0
    assert (sink == 7).all()
    for k in (0, 2):
        assert r.SelectFrame(k) == 0
        rc, got, _, red = r.RenderCurrent(n, iters_out=sink)
        assert rc == 0 and got is sink
        np.testing.assert_array_equal(sink, want[k][0])
        assert red == want[k][2]
    assert r.SetResultSink(None) == 0
    r.close()


@pytest.mark.gpu
def test_a_single_render_after_a_batch_resets_the_selection():
    case = CASES[0]
    frames, orbit, la, n = _inputs(case)
    want = _singles(case, frames[:2], orbit, la, n)
    r = _renderer(case, orbit, la)
    assert r.RenderPerturbLAv2Frames(case[3], frames, n) == 0
    base = r.DeviceIterBuffer()
    assert r.SelectFrame(3) == 0
    assert r.RenderPerturbLAv2(case[3], frames[1], n) == 0
    assert r.DeviceIterBuffer() == base  # frame 0 again: the iteration buffer
    assert r.SelectFrame(1) == UNSUPPORTED
    _assert_same([_result(r, n)], want[1:2])
    r.close()


@pytest.mark.gpu
def test_selection_moves_the_device_iteration_buffer_and_refusal_keeps_it():
    case = CASES[0]
    frames, orbit, la, n = _inputs(case, SCALES[:3])
    r = _renderer(case, orbit, la)
    assert r.RenderPerturbLAv2Frames(case[3], frames, n) == 0
    base = r.DeviceIterBuffer()
    assert r.SelectFrame(2) == 0
    second = r.DeviceIterBuffer()
    assert second not in (0, base)
    assert r.SelectFrame(3) == UNSUPPORTED
    assert r.DeviceIterBuffer() == second
    r.close()


@pytest.mark.gpu
def test_progressive_render_current_during_a_batch():
    """A progressive RenderCurrent while the batch runs returns at once with frame 0's cells as far as they are done; the
    final RenderCurrent has every frame."""
    case = (14, 480, 270, A.GpuHDRx32PerturbedLAv2, None, 4, 1)
    frames, orbit, la, n = _inputs(case, SCALES[:4])
    want = _singles(case, frames, orbit, la, n)
    r = _renderer(case, orbit, la)
    assert r.RenderPerturbLAv2Frames(case[3], frames, n) == 0
    rc, partial, _, _ = r.RenderCurrent(n, progressive=True)
    assert rc == 0
    done = partial != 0
    np.testing.assert_array_equal(partial[done], want[0][0][done])
    got = _batch_results(r, len(frames), n)
    r.close()
    _assert_same(got, want)

