"""Device groups (fs_create_group / fs_create_default): one handle that renders every frame on several devices returns
exactly the bytes one renderer returns.  Groups of one GPU repeated k times exercise the whole path on a one-GPU host; on a
host with more GPUs the groups also span them."""
import ctypes
import os
import subprocess
import sys
import time

import numpy as np
import pytest

import cases
from fractalshark_b200 import RenderAlgorithm as A
from fractalshark_b200 import _native
from fractalshark_b200.gpu_renderer import GPURenderer
from test_gpu_parity import SHARDED_CASES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _groups():
    groups = [[0] * 2, [0] * 3, [0] * 8]
    try:
        import torch
        n = torch.cuda.device_count()
    except Exception:
        n = 0
    if n > 1:
        groups += [list(range(n)), [0, 1, 0]]
    return groups


GROUPS = _groups()
GROUP_IDS = ["-".join(map(str, g)) for g in GROUPS]


def _grouped(devices):
    return lambda: GPURenderer(devices=devices)


# ---- CPU: the device list of fs_create_default --------------------------------------------------------------------------
MALFORMED = ["", "0,,1", "a", "-1", "0,", ",0", "0 ,1", ",".join(["0"] * 65)]


@pytest.mark.parametrize("value", MALFORMED, ids=["empty", "empty_item", "letter", "negative", "trailing_comma",
                                                  "leading_comma", "space", "65_ids"])
def test_malformed_device_lists_are_refused_without_touching_cuda(built, value):
    """A malformed FS_GPU_DEVICES gives NULL before any CUDA call: in a fresh process the CUDA driver library is not even
    loaded afterwards (the runtime loads it on its first call)."""
    code = ("import ctypes, sys; sys.path.insert(0, %r)\n"
            "from fractalshark_b200 import _native\n"
            "h = _native.gpu_lib().fs_create_default()\n"
            "maps = open('/proc/self/maps').read()\n"
            "print(int(h or 0), int('libcuda.so' in maps))\n" % ROOT)
    env = dict(os.environ, FS_GPU_DEVICES=value)
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    handle, cuda_loaded = map(int, out.stdout.split())
    assert handle == 0
    assert cuda_loaded == 0


def test_group_entries_are_bound(built):
    lib = _native.gpu_lib()
    assert lib.fs_device_count(None) == 0
    assert lib.fs_create_group(None, 0) is None


# ---- GPU ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("devices", GROUPS, ids=GROUP_IDS)
@pytest.mark.parametrize("case", SHARDED_CASES, ids=[f"v{c[0]}_{c[3].name}_{c[1]}x{c[2]}_u{8 * c[5]}" for c in SHARDED_CASES])
def test_group_renders_every_kernel_family_like_one_renderer(case, devices):
    """Iteration cells, colours and Min/Max/Sum of a group equal one renderer's, whole padded buffers."""
    view_id, w, h, alg, n_iter, ib, prec, _ = case
    _, coords, orbit, la, n = cases.make_inputs(view_id, w, h, alg, n_iter, ib)
    want, want_col, want_red = cases.render(GPURenderer, w, h, alg, coords, orbit, la, n, ib, want_colors=True, precision=prec)
    got, got_col, got_red = cases.render(_grouped(devices), w, h, alg, coords, orbit, la, n, ib, want_colors=True,
                                         precision=prec)
    np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(got_col, want_col)
    assert got_red == want_red


# (antialiasing, super-sampled width, height): ragged last bands (268, 270 rows) and widths off the 16-column padding
AA_FRAMES = [(1, 100, 270), (2, 192, 268), (2, 74, 270), (3, 150, 270), (3, 96, 54), (4, 100, 272), (4, 384, 268)]


@pytest.mark.gpu
@pytest.mark.parametrize("devices", GROUPS, ids=GROUP_IDS)
@pytest.mark.parametrize("aa,w,h", AA_FRAMES, ids=[f"aa{a}_{w}x{h}" for a, w, h in AA_FRAMES])
def test_group_colours_at_every_antialiasing_like_one_renderer(aa, w, h, devices):
    """AA 1/2/4 colour and reduce on every member; AA 3 cells straddle the members' bands and are coloured on the lead."""
    alg, n = A.Gpu1x64, 300
    _, coords, _, _, _ = cases.make_inputs(0, w, h, alg, n, 4)
    out = []
    for make in (GPURenderer, _grouped(devices)):
        r = make()
        assert r.InitializeMemory(w, h, aa, iter_bytes=4) == 0
        r.ClearMemory()
        assert r.Render(alg, coords, n, 1) == 0
        rc, it, col, red = r.RenderCurrent(n, want_colors=True)
        assert rc == 0
        out.append((it, col, red))
        r.close()
    (want, want_col, want_red), (got, got_col, got_red) = out
    np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(got_col, want_col)
    assert got_red == want_red


@pytest.mark.gpu
@pytest.mark.parametrize("devices", GROUPS[1:2] + GROUPS[3:], ids=GROUP_IDS[1:2] + GROUP_IDS[3:])
def test_group_with_antialiasing_3_renders_a_perturbation_frame_like_one_renderer(devices):
    w, h, alg = 288, 162, A.GpuHDRx32PerturbedLAv2
    _, coords, orbit, la, n = cases.make_inputs(14, w, h, alg, None, 4)
    want = cases.render(GPURenderer, w, h, alg, coords, orbit, la, n, 4, want_colors=True, aa=3)
    got = cases.render(_grouped(devices), w, h, alg, coords, orbit, la, n, 4, want_colors=True, aa=3)
    for a, b in zip(got[:2], want[:2]):
        np.testing.assert_array_equal(a, b)
    assert got[2] == want[2]


@pytest.mark.gpu
@pytest.mark.parametrize("devices", GROUPS, ids=GROUP_IDS)
@pytest.mark.parametrize("aa", [1, 3])
def test_group_result_sink_holds_the_frame(devices, aa):
    """Every member streams its own bands into the one host frame; RenderCurrent(iters_out=sink) returns it, with the
    colours and Min/Max/Sum of one renderer."""
    _, view_id, w, h, alg, n_iter, ib = next(c for c in cases.ALL_SMALL_CASES if c[0] == "v5_hdr32_lav2")
    _, coords, orbit, la, n = cases.make_inputs(view_id, w, h, alg, n_iter, ib)
    want, want_col, want_red = cases.render(GPURenderer, w, h, alg, coords, orbit, la, n, ib, want_colors=True, aa=aa)
    r = GPURenderer(devices=devices)
    assert r.InitializeMemory(w, h, aa, iter_bytes=ib) == 0
    assert r.InitializePerturb(1, orbit, 0, None, la) == 0
    sink = np.zeros(r.buffer_shape(), np.uint32)
    assert r.SetResultSink(sink) == 0
    for _ in range(2):   # twice: the second render streams into the frame the first one filled
        sink[:] = 0
        r.ClearMemory()
        assert r.RenderPerturbLAv2(alg, coords, n) == 0
        assert r.SyncComputeStream() == 0
        np.testing.assert_array_equal(sink, want)
        rc, got, col, red = r.RenderCurrent(n, iters_out=sink, want_colors=True)
        assert rc == 0 and got is sink
        np.testing.assert_array_equal(got, want)
        np.testing.assert_array_equal(col, want_col)
        assert red == want_red
    assert r.SetResultSink(None) == 0
    r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("devices", GROUPS, ids=GROUP_IDS)
def test_group_done_callback_fires_once_after_every_member(devices):
    """The callback runs once, and when it runs every member's bands have arrived in the result sink."""
    w, h, alg = 960, 540, A.GpuHDRx32PerturbedLAv2
    _, coords, orbit, la, n = cases.make_inputs(14, w, h, alg, None, 4)
    want, _, _ = cases.render(GPURenderer, w, h, alg, coords, orbit, la, n, 4)
    r = GPURenderer(devices=devices)
    assert r.InitializeMemory(w, h, 1, iter_bytes=4) == 0
    assert r.InitializePerturb(1, orbit, 0, None, la) == 0
    sink = np.zeros(r.buffer_shape(), np.uint32)
    assert r.SetResultSink(sink) == 0
    seen = []
    r.ClearMemory()
    assert r.RenderPerturbLAv2(alg, coords, n) == 0
    assert r.EnqueueComputeDoneCallback(lambda: seen.append(int(sink.astype(np.uint64).sum()))) == 0
    t0 = time.time()
    while r.QueryComputeStream() == 600:   # cudaErrorNotReady while any member is busy
        assert time.time() - t0 < 60
        time.sleep(0.001)
    assert r.QueryComputeStream() == 0
    assert seen == [int(want.astype(np.uint64).sum())]
    assert r.SyncComputeStream() == 0 and r.QueryComputeStream() == 0
    assert seen == [int(want.astype(np.uint64).sum())]
    assert r.SetResultSink(None) == 0
    r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("devices", GROUPS[1:2] + GROUPS[3:], ids=GROUP_IDS[1:2] + GROUP_IDS[3:])
@pytest.mark.parametrize("aa", [1, 3])
def test_group_progressive_render_current_during_a_render(devices, aa):
    """A progressive RenderCurrent while the members render succeeds; each of its cells is 0 or final; the final frame
    is the undisturbed one.  At AA 3 the progressive colours come from the lead's gather on the display streams."""
    w, h, alg = 1920, 1080, A.GpuHDRx32PerturbedLAv2PO
    r = GPURenderer(devices=devices)
    assert r.InitializeMemory(w, h, aa, iter_bytes=4) == 0
    for n_iter in (60000, 250000, 1000000):
        _, coords, orbit, la, n = cases.make_inputs(5, w, h, alg, n_iter, 4)
        assert r.InitializePerturb(n_iter, orbit, 0, None, la) == 0
        r.ClearMemory()
        assert r.RenderPerturbLAv2(alg, coords, n) == 0
        rc, want, want_col, want_red = r.RenderCurrent(n, want_colors=True)
        assert rc == 0
        full_ms = r.LastRenderMs()
        if full_ms >= 40.0:
            break
    r.ClearMemory()
    assert r.SyncComputeStream() == 0
    assert r.RenderPerturbLAv2(alg, coords, n) == 0
    time.sleep(0.25 * full_ms * 1e-3)
    rc, part, _, red = r.RenderCurrent(n, want_colors=True, progressive=True)
    assert rc == 0
    filled = part != 0
    np.testing.assert_array_equal(part[filled], want[filled])
    assert red["Sum"] <= want_red["Sum"]
    assert r.SyncComputeStream() == 0
    rc, got, got_col, got_red = r.RenderCurrent(n, want_colors=True)
    assert rc == 0
    np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(got_col, want_col)
    assert got_red == want_red
    r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("devices", GROUPS, ids=GROUP_IDS)
@pytest.mark.parametrize("aa", [1, 3])
def test_group_result_calls_back_to_back_without_a_synchronise(devices, aa):
    """Render, RenderCurrent, ClearMemory, Render, RenderCurrent, ... enqueued from one thread into page-locked buffers,
    with one synchronise at the end: every frame's cells, colours and Min/Max/Sum are those of one renderer.  (Members
    write into lead-owned memory only after the lead has read what the previous call left there.)"""
    import torch
    w, h, alg = 288, 162, A.Gpu1x64
    limits = (300, 2000, 700)
    _, coords, _, _, _ = cases.make_inputs(0, w, h, alg, 300, 4)

    def pinned(shape, dtype):
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        return torch.empty(nbytes, dtype=torch.uint8, pin_memory=True).numpy().view(dtype).reshape(shape)

    out = []
    for make in (GPURenderer, _grouped(devices)):
        r = make()
        assert r.InitializeMemory(w, h, aa, iter_bytes=4) == 0
        hp, wp = r.buffer_shape()
        frames = []
        for n in limits:
            it = pinned((hp, wp), np.uint32)
            col = pinned((-(-(h // aa) // 8) * 8, -(-(w // aa) // 16) * 16, 4), np.uint16)
            red = pinned((3,), np.uint64)
            r.ClearMemory()
            assert r.Render(alg, coords, n, 1) == 0
            assert r._lib.fs_render_current(r._h, n, it.ctypes.data, col.ctypes.data,
                                            ctypes.cast(red.ctypes.data, ctypes.POINTER(_native.FsReduction)), 0) == 0
            frames.append((it, col, red))
        assert r.SyncComputeStream() == 0
        out.append([tuple(a.copy() for a in f) for f in frames])
        r.close()
    for (want_it, want_col, want_red), (got_it, got_col, got_red) in zip(*out):
        np.testing.assert_array_equal(got_it, want_it)
        np.testing.assert_array_equal(got_col, want_col)
        np.testing.assert_array_equal(got_red, want_red)
    assert not np.array_equal(out[0][0][2], out[0][1][2])   # the frames differ, so a mix-up would show


@pytest.mark.gpu
def test_group_counters_are_the_sums_of_its_members_and_sharding_entries_are_refused():
    """Step counters and launch counts of a group of three equal the sums over three renderers sharded (3, i)."""
    _, view_id, w, h, alg, n_iter, ib = next(c for c in cases.ALL_SMALL_CASES if c[0] == "v5_hdr32_lav2")
    _, coords, orbit, la, n = cases.make_inputs(view_id, w, h, alg, n_iter, ib)

    def run(r, shard=None):
        assert r.InitializeMemory(w, h, 1, iter_bytes=ib) == 0
        if shard is not None:
            assert r.SetShard(3, shard) == 0
        assert r.InitializePerturb(1, orbit, 0, None, la) == 0
        assert r.EnableStepCounter(True) == 0
        r.ClearMemory()
        assert r.RenderPerturbLAv2(alg, coords, n) == 0
        assert r.SyncComputeStream() == 0
        return r.ReadStepCounters(), r.ReadStepCounter(), r.KernelLaunchCount()

    singles = []
    for s in range(3):
        r = GPURenderer()
        singles.append(run(r, s))
        r.close()
    g = GPURenderer(devices=[0, 0, 0])
    kinds, steps, launches = run(g)
    assert kinds == {k: sum(s[0][k] for s in singles) for k in kinds}
    assert steps == sum(s[1] for s in singles) and steps > 0
    assert launches == sum(s[2] for s in singles)
    assert g.LastRenderMs() > 0
    assert g.SetShard(3, 1) == 10100
    assert g.RenderCurrentShard(n, np.zeros(g.buffer_shape(), np.uint32))[0] == 10100
    g.close()


@pytest.mark.gpu
def test_group_handles_and_the_default_renderer(monkeypatch):
    """FS_GPU_DEVICES=0,0 makes fs_create_default a group of two that renders fs_create(0)'s frame; one id is a plain
    renderer; an id outside the machine's devices is refused."""
    assert GPURenderer().DeviceCount() == 1
    assert GPURenderer(devices=[0]).DeviceCount() == 1
    assert GPURenderer(devices=[0, 0, 0]).DeviceCount() == 3
    with pytest.raises(MemoryError):
        GPURenderer(devices=[0, 4096])
    assert _native.gpu_lib().fs_create_group((ctypes.c_int32 * 1)(0), 0) is None
    w, h, alg, n = 200, 133, A.Gpu1x64, 500
    _, coords, _, _, _ = cases.make_inputs(0, w, h, alg, n, 4)
    want, _, want_red = cases.render(GPURenderer, w, h, alg, coords, None, None, n, 4)
    monkeypatch.setenv("FS_GPU_DEVICES", "0,0")

    def default_renderer():
        r = GPURenderer()   # then swap its handle for fs_create_default's
        r.close()
        r._h = _native.gpu_lib().fs_create_default()
        assert r._h
        return r

    assert default_renderer().DeviceCount() == 2
    got, _, got_red = cases.render(default_renderer, w, h, alg, coords, None, None, n, 4)
    np.testing.assert_array_equal(got, want)
    assert got_red == want_red
