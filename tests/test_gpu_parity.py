"""GPU parity tests (run on the B200 box): every call goes through the C-ABI of libfsgpu.so."""
import os
import sys

import numpy as np
import pytest

import cases
import oracle_cpu
import ref_renderer
from fractalshark_b200 import RenderAlgorithm as A
from fractalshark_b200 import Numeric, traits
from fractalshark_b200.gpu_renderer import GPURenderer, default_palette
from fractalshark_b200.sharding import merge_shards, rows_of_shard

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "ref_gpu_small.npz")


@pytest.fixture(scope="module")
def golden():
    return cases.load_goldens()


@pytest.mark.parametrize("case", cases.ALL_SMALL_CASES, ids=[c[0] for c in cases.ALL_SMALL_CASES])
def test_small_cases_bit_exact_vs_oracle_and_golden(golden, case):
    """Bit-exact against the committed reference-kernel fixtures and (where restated) the CPU oracle."""
    name, view_id, w, h, alg, n_iter, ib = case
    _, coords, orbit, la, n = cases.make_inputs(view_id, w, h, alg, n_iter, ib)
    prec = cases.CASE_PRECISION.get(name, 1)
    got, _, red = cases.render(GPURenderer, w, h, alg, coords, orbit, la, n, ib, precision=prec)
    if name in cases.NOT_BIT_EXACT:
        assert float((got[:h, :w] == golden[name]).mean()) >= cases.NOT_BIT_EXACT[name]
    else:
        np.testing.assert_array_equal(got[:h, :w], golden[name])
    want = cases.oracle_render(alg, w, h, coords, orbit, la, n, ib, precision=prec)
    if want is not None:
        np.testing.assert_array_equal(got[:h, :w], want[:h, :w])
    assert red["Sum"] == int(got[:h, :w].astype(np.uint64).sum())
    assert red["Min"] == int(got[:h, :w].min()) and red["Max"] == int(got[:h, :w].max())
    # cells outside width x height stay cleared
    assert not got[h:, :].any() and not got[:, w:].any()


FULL_CASES = [
    ("v0_gpu1x64_full", 0, 3840, 2160, A.Gpu1x64, 65536, 4, 1.0),          # FP64 direct: bit-exact required
    ("v0_gpu1x32_full", 0, 3840, 2160, A.Gpu1x32, 65536, 4, 1.0),
    ("v5_hdr32_lav2_full", 5, 3840, 2160, A.GpuHDRx32PerturbedLAv2, None, 4, 1.0),   # north_star tolerance
    ("v5_hdr32_lav2_po_full", 5, 1920, 1080, A.GpuHDRx32PerturbedLAv2PO, 20000, 4, 1.0),
    ("v5_hdr32_lav2_u64_full", 5, 1920, 1080, A.GpuHDRx32PerturbedLAv2, None, 8, 1.0),
    ("v1_hdr32_lav2_full", 1, 3840, 2160, A.GpuHDRx32PerturbedLAv2, None, 4, 1.0),
    ("v5_hdr32_bla_full", 5, 3840, 2160, A.GpuHDRx32PerturbedBLA, None, 4, 1.0),       # BASELINE configs[2]
    ("v5_hdr64_bla_full", 5, 1920, 1080, A.GpuHDRx64PerturbedBLA, None, 4, 1.0),
    ("v100_f64_bla_full", 100, 3840, 2160, A.Gpu1x64PerturbedBLA, None, 4, 1.0),          # FP64 perturbation: bit-exact
    ("v100_f64_lav2_full", 100, 3840, 2160, A.Gpu1x64PerturbedLAv2, None, 4, 1.0),
    ("v100_f64_lav2_po_full", 100, 1920, 1080, A.Gpu1x64PerturbedLAv2PO, None, 8, 1.0),
    ("v5_hdr64_lav2_full", 5, 1920, 1080, A.GpuHDRx64PerturbedLAv2, None, 4, 1.0),
    ("v101_f32_lav2_full", 101, 3840, 2160, A.Gpu1x32PerturbedLAv2, None, 4, 1.0),
    ("v100_2x32_lav2_full", 100, 1920, 1080, A.Gpu2x32PerturbedLAv2, None, 4, 1.0),
    ("v100_2x32_lav2_po_full", 100, 1920, 1080, A.Gpu2x32PerturbedLAv2PO, None, 4, 1.0),
    ("v5_hdr2x32_lav2_full", 5, 1920, 1080, A.GpuHDRx2x32PerturbedLAv2, None, 4, 1.0),
    ("v1_hdr2x32_lav2_u64_full", 1, 1920, 1080, A.GpuHDRx2x32PerturbedLAv2, None, 8, 1.0),
    ("v100_scaled_f64_full", 100, 3840, 2160, A.Gpu1x32PerturbedScaled, None, 4, 1.0),
    ("v5_scaled_hdr32_full", 5, 1920, 1080, A.GpuHDRx32PerturbedScaled, 50000, 4, 1.0),
    ("v19_scaled_hdr32_bad_full", 19, 960, 540, A.GpuHDRx32PerturbedScaled, 1000000, 4, 1.0),
    ("v19_scaled_f64_bad_full", 19, 960, 540, A.Gpu1x32PerturbedScaled, 1000000, 8, 1.0),
    ("v0_gpu2x32_full", 0, 3840, 2160, A.Gpu2x32, 4096, 4, 1.0),
    ("v0_gpu2x64_full", 0, 1920, 1080, A.Gpu2x64, 2048, 4, 1.0),
    ("v102_gpu2x64_full", 102, 1920, 1080, A.Gpu2x64, 20000, 4, 1.0),
    ("v100_gpuhdrx32_full", 100, 960, 540, A.GpuHDRx32, 5000, 4, 1.0),
    ("v14_hdr32_lav2_full", 14, 3840, 2160, A.GpuHDRx32PerturbedLAv2, None, 4, 1.0),   # north_star target view
    ("v14_hdr2x32_lav2_full", 14, 1920, 1080, A.GpuHDRx2x32PerturbedLAv2, None, 4, 1.0),
    ("v14_hdr32_rclav2_u64_full", 14, 1920, 1080, A.GpuHDRx32PerturbedRCLAv2, None, 8, 1.0),
    ("v14_hdr64_lav2_full", 14, 960, 540, A.GpuHDRx64PerturbedLAv2, None, 4, 1.0),
    ("v19_hdr32_lav2_full", 19, 3840, 2160, A.GpuHDRx32PerturbedLAv2, None, 4, 1.0),
    ("v5_hdr32_rclav2_full", 5, 3840, 2160, A.GpuHDRx32PerturbedRCLAv2, None, 4, 1.0),
    ("v19_hdr32_rclav2_full", 19, 960, 540, A.GpuHDRx32PerturbedRCLAv2, 3000000, 4, 1.0),
    ("v100_f64_rclav2_full", 100, 1920, 1080, A.Gpu1x64PerturbedRCLAv2, None, 4, 1.0),
    ("v5_hdr2x32_rclav2_po_full", 5, 960, 540, A.GpuHDRx2x32PerturbedRCLAv2PO, 20000, 8, 1.0),
    # iteration_precision 4 / 8 / 16 (GPU_Render.cu:633-668): name suffix _pN, limits not multiples of N
    ("v0_gpu1x32_p4_full", 0, 3840, 2160, A.Gpu1x32, 65533, 4, 1.0),
    ("v0_gpu1x32_p16_full", 0, 1920, 1080, A.Gpu1x32, 65535, 8, 1.0),
    ("v0_gpu1x64_p8_full", 0, 3840, 2160, A.Gpu1x64, 65531, 4, 1.0),
    ("v0_gpu1x64_p16_full", 0, 1920, 1080, A.Gpu1x64, 65536, 4, 1.0),
    ("v0_gpu2x32_p4_full", 0, 1920, 1080, A.Gpu2x32, 4095, 4, 1.0),
    ("v0_gpu2x32_p16_full", 0, 1920, 1080, A.Gpu2x32, 4099, 8, 1.0),
    ("v100_gpuhdrx32_p8_full", 100, 960, 540, A.GpuHDRx32, 5003, 4, 1.0),
    ("v0_gpuhdrx32_p4_full", 0, 960, 540, A.GpuHDRx32, 1023, 4, 1.0),
    ("v0_gpu4x32_full", 0, 960, 540, A.Gpu4x32, 1024, 4, -0.999),   # negative: exactness floor only, see NOT_BIT_EXACT
    ("v0_gpu4x64_full", 0, 960, 540, A.Gpu4x64, 1024, 4, -0.999),
]


@pytest.mark.skipif(not ref_renderer.available(), reason="oracle/_ref (reference CUDA kernels) not built")
@pytest.mark.parametrize("case", FULL_CASES, ids=[c[0] for c in FULL_CASES])
def test_full_size_vs_reference_cuda_kernels(case):
    """BASELINE.json sizes against the reference's own kernels on the same GPU and inputs.
    north_star asks for FP64/FP32 direct bit-exact and HDRx32/2x32/LA >= 99.9 % exact with |d iter| <= 1 elsewhere;
    every case here is held to bit-exactness (1.0) except the four-limb direct kernels (DESIGN.md section 2)."""
    name, view_id, w, h, alg, n_iter, ib, min_exact = case
    prec = cases.full_case_precision(name)
    _, coords, orbit, la, n = cases.make_inputs(view_id, w, h, alg, n_iter, ib)
    got, _, red = cases.render(GPURenderer, w, h, alg, coords, orbit, la, n, ib, precision=prec)
    ref, _, ref_red = cases.render(ref_renderer.RefGPURenderer, w, h, alg, coords, orbit, la, n, ib, precision=prec)
    a, b = got[:h, :w].astype(np.int64), ref[:h, :w].astype(np.int64)
    exact = float((a == b).mean())
    assert exact >= abs(min_exact), exact
    if 0 < min_exact < 1.0:
        assert int(np.abs(a - b).max()) <= 1
    assert (red["Min"], red["Max"], red["Sum"]) == (ref_red["Min"], ref_red["Max"], ref_red["Sum"]) or min_exact < 1.0


def test_four_limb_kernels_resolve_what_double_double_resolves():
    """Property for Gpu4x64 where the reference's own 4x64 kernel cannot serve as the checker (on windows of
    width 1e-24 its frame is one constant -- it resolves less than its 2x64 kernel): the four-double kernel
    must agree with the double-double kernel (itself bit-exact against the reference) on a window both resolve."""
    w, h, n = 480, 270, 20000
    _, c2, _, _, _ = cases.make_inputs(102, w, h, A.Gpu2x64, n, 4)
    _, c4, _, _, _ = cases.make_inputs(102, w, h, A.Gpu4x64, n, 4)
    i2, _, _ = cases.render(GPURenderer, w, h, A.Gpu2x64, c2, None, None, n, 4)
    i4, _, _ = cases.render(GPURenderer, w, h, A.Gpu4x64, c4, None, None, n, 4)
    assert float((i2[:h, :w] == i4[:h, :w]).mean()) >= 0.999
    assert int(i4[:h, :w].max()) > int(i4[:h, :w].min())


def test_full_size_properties_without_reference():
    """Size-independent properties at 3840x2160: idempotence, sharded == unsharded, checksum of checksums,
    u32 == u64, sampled rows == oracle."""
    w, h, alg = 3840, 2160, A.GpuHDRx32PerturbedLAv2
    _, coords, orbit, la, n = cases.make_inputs(5, w, h, alg, None, 4)
    r = GPURenderer()
    assert r.InitializeMemory(w, h, 1, iter_bytes=4) == 0
    assert r.InitializePerturb(7, orbit, 0, None, la) == 0
    outs = []
    for _ in range(2):
        r.ClearMemory()
        assert r.RenderPerturbLAv2(alg, coords, n) == 0
        rc, it, _, red = r.RenderCurrent(n)
        assert rc == 0
        outs.append(it.copy())
        assert red["Sum"] == int(it[:h, :w].astype(np.uint64).sum())
    np.testing.assert_array_equal(outs[0], outs[1])                       # idempotent / deterministic
    # three shards merge to the unsharded frame; the shard Sums add up (checksum of checksums)
    bufs, sums = [], 0
    for s in range(3):
        assert r.SetShard(3, s) == 0
        r.ClearMemory()
        assert r.RenderPerturbLAv2(alg, coords, n) == 0
        rc, it, _, red = r.RenderCurrent(n)
        rows = rows_of_shard(h, 3, s)
        other = np.setdiff1d(np.arange(h), rows)
        assert not it[other].any()                                        # other shards' cells untouched
        bufs.append(it.copy())
        sums += red["Sum"]
    assert r.SetShard(1, 0) == 0
    np.testing.assert_array_equal(merge_shards(bufs, h)[:h, :w], outs[0][:h, :w])
    assert sums == int(outs[0][:h, :w].astype(np.uint64).sum())
    # the sharded result call fills ONE host frame band by band (no merge step); rows it does not own stay untouched
    frame = np.full_like(outs[0], 0xDEADBEEF)
    for s in range(3):
        assert r.SetShard(3, s) == 0
        r.ClearMemory()
        assert r.RenderPerturbLAv2(alg, coords, n) == 0
        before = frame.copy()
        rc, red = r.RenderCurrentShard(n, frame)
        assert rc == 0
        rows = rows_of_shard(h, 3, s)
        other = np.setdiff1d(np.arange(frame.shape[0]), np.concatenate([rows, np.arange(h, frame.shape[0])]))
        np.testing.assert_array_equal(frame[other], before[other])
        assert red["Sum"] == int(frame[rows, :w].astype(np.uint64).sum())
    np.testing.assert_array_equal(frame[:h, :w], outs[0][:h, :w])
    # result sink: the kernel streams finished pixels into a host frame while it renders; RenderCurrent on the same
    # frame then skips its copy.  A render entry that does not stream (here: after ClearMemory alone) copies as usual.
    assert r.SetShard(1, 0) == 0
    sink = np.full_like(outs[0], 0xDEADBEEF)
    assert r.SetResultSink(sink) == 0
    r.ClearMemory()
    assert r.RenderPerturbLAv2(alg, coords, n) == 0
    assert r.SyncComputeStream() == 0
    np.testing.assert_array_equal(sink[:h, :w], outs[0][:h, :w])          # arrived before any RenderCurrent
    rc, it, _, red = r.RenderCurrent(n, iters_out=sink)
    assert rc == 0 and it is sink and red["Sum"] == int(outs[0][:h, :w].astype(np.uint64).sum())
    r.ClearMemory()
    rc, it, _, red = r.RenderCurrent(n, iters_out=sink)                   # nothing streamed since the clear: plain copy
    assert rc == 0 and not sink[:h, :w].any()
    for s_ in range(2):                                                   # two shards stream into the one frame
        assert r.SetShard(2, s_) == 0
        r.ClearMemory()
        assert r.RenderPerturbLAv2(alg, coords, n) == 0
        rc, red = r.RenderCurrentShard(n, sink)
        assert rc == 0
    np.testing.assert_array_equal(sink[:h, :w], outs[0][:h, :w])
    assert r.SetResultSink(None) == 0
    # sampled rows against the CPU oracle
    want, _ = oracle_cpu.render_lav2(alg, w, h, coords, orbit, la, n, rows=(0, h), row_step=270, col_step=7,
                                     threads=oracle_cpu.hardware_threads())
    np.testing.assert_array_equal(outs[0][0:h:270, 0:w:7], want[0:h:270, 0:w:7])
    r.close()
    # 64-bit iteration type gives the same counts
    _, coords8, orbit8, la8, _ = cases.make_inputs(5, 960, 540, alg, None, 8)
    it8, _, _ = cases.render(GPURenderer, 960, 540, alg, coords8, orbit8, la8, n, 8)
    _, coords4, orbit4, la4, _ = cases.make_inputs(5, 960, 540, alg, None, 4)
    it4, _, _ = cases.render(GPURenderer, 960, 540, alg, coords4, orbit4, la4, n, 4)
    np.testing.assert_array_equal(it8.astype(np.uint64), it4.astype(np.uint64))


@pytest.mark.parametrize("aa", [1, 2, 3, 4])
def test_antialiasing_palette_reduction(aa):
    """RenderCurrent: AA box filter + palette + Min/Max/Sum vs the oracle (and the reference when present)."""
    w, h, alg, n = 96 * aa, 48 * aa, A.Gpu1x64, 300
    _, coords, _, _, _ = cases.make_inputs(0, w, h, alg, n, 4)
    iters, colors, red = cases.render(GPURenderer, w, h, alg, coords, None, None, n, 4, want_colors=True, aa=aa)
    want_c, want_r = oracle_cpu.post(iters, w, h, aa, default_palette(), 0, n)
    assert red == want_r
    np.testing.assert_array_equal(colors.reshape(-1, 4)[: (h // aa) * (w // aa)].reshape(h // aa, w // aa, 4), want_c)
    if ref_renderer.available():
        _, rcol, rred = cases.render(ref_renderer.RefGPURenderer, w, h, alg, coords, None, None, n, 4, want_colors=True, aa=aa)
        assert rred == red
        np.testing.assert_array_equal(rcol.reshape(-1, 4)[: (h // aa) * (w // aa)], colors.reshape(-1, 4)[: (h // aa) * (w // aa)])


@pytest.mark.parametrize("view_id,w,h,alg,n_iter", [
    (5, 1920, 1080, A.GpuHDRx32PerturbedLAv2, None),
    (5, 960, 540, A.GpuHDRx32PerturbedLAv2PO, 20000),
    (1, 1920, 1080, A.GpuHDRx32PerturbedLAv2PO, None),
    (19, 960, 540, A.GpuHDRx32PerturbedLAv2, 3000000),
])
def test_scaled_chunks_equal_float_exponent_loop(view_id, w, h, alg, n_iter):
    """A/B inside the library: the scaled plain-float chunks (default) and the pure float+exponent loop give
    the same iteration buffer, and the scaled form executes the same number of algorithmic steps."""
    _, coords, orbit, la, n = cases.make_inputs(view_id, w, h, alg, n_iter, 4)
    outs, steps = [], []
    for scaled in (True, False):
        r = GPURenderer()
        assert r.InitializeMemory(w, h, 1, iter_bytes=4) == 0
        assert r.SetScaledSteps(scaled) == 0
        assert r.InitializePerturb(1, orbit, 0, None, la) == 0
        assert r.EnableStepCounter(True) == 0
        r.ClearMemory()
        assert r.RenderPerturbLAv2(alg, coords, n) == 0
        rc, it, _, _ = r.RenderCurrent(n)
        assert rc == 0
        outs.append(it.copy())
        steps.append(r.ReadStepCounter())
        r.close()
    np.testing.assert_array_equal(outs[0], outs[1])
    assert steps[0] == steps[1]


def test_split_and_fused_at_launches_agree():
    """The two-launch form of the HDRx32 LAv2 path (AT shortcut first) gives the same frame as the fused launch."""
    w, h, alg = 960, 540, A.GpuHDRx32PerturbedLAv2
    for view_id in (14, 5):
        _, coords, orbit, la, n = cases.make_inputs(view_id, w, h, alg, None, 4)
        outs = []
        for split in (True, False):
            r = GPURenderer()
            assert r.SetSplitAt(split) == 0
            assert r.InitializeMemory(w, h, 1, iter_bytes=4) == 0
            assert r.InitializePerturb(1, orbit, 0, None, la) == 0
            r.ClearMemory()
            assert r.RenderPerturbLAv2(alg, coords, n) == 0
            rc, it, _, _ = r.RenderCurrent(n)
            assert rc == 0
            outs.append(it.copy())
            r.close()
        np.testing.assert_array_equal(outs[0], outs[1])


def _render_lav2(view_id, w, h, alg, n_iter, iter_bytes, switches, count=False):
    _, coords, orbit, la, n = cases.make_inputs(view_id, w, h, alg, n_iter, iter_bytes)
    r = GPURenderer()
    for name, value in switches.items():
        assert getattr(r, name)(value) == 0
    assert r.InitializeMemory(w, h, 1, iter_bytes=iter_bytes) == 0
    assert r.InitializePerturb(1, orbit, 0, None, la) == 0
    if count:
        assert r.EnableStepCounter(True) == 0
    r.ClearMemory()
    assert r.RenderPerturbLAv2(alg, coords, n) == 0
    rc, it, _, red = r.RenderCurrent(n)
    assert rc == 0
    steps = r.ReadStepCounters() if count else None
    r.close()
    return it.copy(), red, steps


@pytest.mark.parametrize("view_id,w,h,alg,n_iter,iter_bytes", [
    (14, 3840, 2160, A.GpuHDRx32PerturbedLAv2, None, 4),   # interior pixels: 18,402 AT passes each in the reference
    (14, 960, 540, A.GpuHDRx32PerturbedLAv2LAO, None, 8),
    (14, 960, 540, A.GpuHDRx64PerturbedLAv2, None, 4),     # binary64 mantissa: the unpacked form of the loop
    (14, 640, 360, A.GpuHDRx2x32PerturbedLAv2, None, 4),   # 2x32 mantissa: the watch on the general loop's whole state
    (100, 640, 360, A.Gpu1x64PerturbedLAv2, None, 4),
    (101, 640, 360, A.Gpu2x32PerturbedLAv2, None, 8),
    (5, 960, 540, A.GpuHDRx32PerturbedLAv2, None, 4),
    (19, 960, 540, A.GpuHDRx32PerturbedLAv2, None, 4),
    (100, 640, 360, A.GpuHDRx32PerturbedLAv2, None, 4),
])
def test_at_cycle_detection_skips_passes_not_results(view_id, w, h, alg, n_iter, iter_bytes):
    """The AT shortcut with cycle detection (default) gives the frame of the loop that executes every pass of
    ATInfo::PerformAT, and never executes more passes than it."""
    on, red_on, st_on = _render_lav2(view_id, w, h, alg, n_iter, iter_bytes, {"SetAtCycleDetection": True}, count=True)
    off, red_off, st_off = _render_lav2(view_id, w, h, alg, n_iter, iter_bytes, {"SetAtCycleDetection": False}, count=True)
    np.testing.assert_array_equal(on, off)
    assert red_on == red_off
    assert st_on["at"] <= st_off["at"]                        # AT passes executed
    assert st_on["la"] == st_off["la"]                        # identical walk afterwards
    assert st_on["perturbation"] == st_off["perturbation"]
    if view_id == 14 and alg in (A.GpuHDRx32PerturbedLAv2, A.GpuHDRx2x32PerturbedLAv2):
        assert st_on["at"] * 4 < st_off["at"], "View 14: the interior pixels should settle long before 18,402 passes"


@pytest.mark.parametrize("view_id,w,h,alg,iter_bytes", [
    (14, 640, 360, A.GpuHDRx32PerturbedBLA, 4),    # interior pixels: 18,402 periods of the reference orbit each
    (14, 320, 180, A.GpuHDRx64PerturbedBLA, 8),
    (5, 960, 540, A.GpuHDRx32PerturbedBLA, 4),
    (1, 960, 540, A.GpuHDRx32PerturbedBLA, 4),
    (100, 640, 360, A.Gpu1x64PerturbedBLA, 4),
])
def test_bla_cycle_detection_skips_periods_not_results(view_id, w, h, alg, iter_bytes):
    """The BLA kernels with cycle detection at rebase events (default) give the frame of the loop that executes every
    period, and never execute more steps than it."""
    _, coords, orbit, table, n = cases.make_inputs(view_id, w, h, alg, None, iter_bytes)
    outs, steps = [], []
    for on in (True, False):
        r = GPURenderer()
        assert r.SetAtCycleDetection(on) == 0
        assert r.InitializeMemory(w, h, 1, iter_bytes=iter_bytes) == 0
        assert r.EnableStepCounter(True) == 0
        r.ClearMemory()
        assert r.RenderPerturbBLA(alg, orbit, table, coords, n) == 0
        rc, it, _, red = r.RenderCurrent(n)
        assert rc == 0
        outs.append((it.copy(), red))
        steps.append(r.ReadStepCounter())
        r.close()
    np.testing.assert_array_equal(outs[0][0], outs[1][0])
    assert outs[0][1] == outs[1][1]
    assert steps[0] <= steps[1]
    if view_id == 14:
        assert steps[0] * 2 < steps[1], "View 14: interior pixels should settle long before 18,402 periods"


@pytest.mark.parametrize("view_id,w,h,n_iter,iter_bytes", [
    (5, 1920, 1080, None, 4), (14, 640, 360, None, 4), (1, 960, 540, None, 8), (19, 640, 360, 3000000, 4), (100, 640, 360, None, 4),
])
def test_select_free_bla_loop_equals_reference_shaped(view_id, w, h, n_iter, iter_bytes):
    """A/B inside the library: the select-free HDRx32 BLA loop (bla_pixel_hdr32, default) and the loop on the
    reference-shaped float+exponent operators give the same iteration buffer and execute the same steps."""
    alg = A.GpuHDRx32PerturbedBLA
    _, coords, orbit, table, n = cases.make_inputs(view_id, w, h, alg, n_iter, iter_bytes)
    outs, steps = [], []
    for fast in (True, False):
        r = GPURenderer()
        assert r.SetLaStep2(fast) == 0   # the switch of the select-free forms
        assert r.InitializeMemory(w, h, 1, iter_bytes=iter_bytes) == 0
        assert r.EnableStepCounter(True) == 0
        r.ClearMemory()
        assert r.RenderPerturbBLA(alg, orbit, table, coords, n) == 0
        rc, it, _, red = r.RenderCurrent(n)
        assert rc == 0
        outs.append((it.copy(), red))
        steps.append(r.ReadStepCounter())
        r.close()
    np.testing.assert_array_equal(outs[0][0], outs[1][0])
    assert outs[0][1] == outs[1][1] and steps[0] == steps[1]


@pytest.mark.parametrize("view_id,w,h,alg,n_iter", [
    (14, 3840, 2160, A.GpuHDRx32PerturbedLAv2, None),
    (5, 1920, 1080, A.GpuHDRx32PerturbedLAv2, None),
    (5, 1920, 1080, A.GpuHDRx32PerturbedLAv2LAO, None),
    (19, 1920, 1080, A.GpuHDRx32PerturbedLAv2, None),
    (1, 1920, 1080, A.GpuHDRx32PerturbedLAv2, None),
    (100, 640, 360, A.GpuHDRx32PerturbedLAv2, None),
    (101, 640, 360, A.GpuHDRx32PerturbedLAv2, None),
])
def test_step_shaped_la_records_equal_reference_shaped(view_id, w, h, alg, n_iter):
    """A/B inside the library: the LA walk on la2 records (fs_la_step2.cuh, default) and on reference-shaped records
    give the same iteration buffer and execute the same steps."""
    a, _, st_a = _render_lav2(view_id, w, h, alg, n_iter, 4, {"SetLaStep2": True}, count=True)
    b, _, st_b = _render_lav2(view_id, w, h, alg, n_iter, 4, {"SetLaStep2": False}, count=True)
    np.testing.assert_array_equal(a, b)
    assert st_a == st_b


@pytest.mark.parametrize("view_id,w,h,alg,n_iter,iter_bytes", [
    (14, 1920, 1080, A.GpuHDRx32PerturbedLAv2, None, 4),
    (5, 960, 540, A.GpuHDRx32PerturbedLAv2, None, 4),
    (5, 960, 540, A.GpuHDRx32PerturbedLAv2PO, 20000, 4),
    (5, 960, 540, A.GpuHDRx32PerturbedLAv2LAO, None, 8),
    (19, 960, 540, A.GpuHDRx32PerturbedLAv2, None, 8),
    (1, 100, 37, A.GpuHDRx32PerturbedLAv2, None, 4),       # ragged: partial tiles on both edges
])
def test_lane_refill_kernel_equals_tile_kernel(view_id, w, h, alg, n_iter, iter_bytes):
    """A/B inside the library: the lane-refill kernel (fs_lav2_pool.cuh, off by default) gives the tile kernel's frame."""
    a, red_a, _ = _render_lav2(view_id, w, h, alg, n_iter, iter_bytes, {"SetPoolKernel": True})
    b, red_b, _ = _render_lav2(view_id, w, h, alg, n_iter, iter_bytes, {"SetPoolKernel": False})
    np.testing.assert_array_equal(a, b)
    assert red_a == red_b


def test_error_behaviour_matches_reference():
    """Error codes and no-op-before-init behaviour (GPU_Render.cu:322-332, 626-628, 1007-1022)."""
    r = GPURenderer()
    _, coords, orbit, la, n = cases.make_inputs(1, 64, 32, A.GpuHDRx32PerturbedLAv2, None, 4)
    assert r.RenderPerturbLAv2(A.GpuHDRx32PerturbedLAv2, coords, n) == 0      # not initialised: returns success, does nothing
    assert r.InitializeMemory(64, 32, 5) == 10002                             # bad antialiasing
    assert r.InitializeMemory(65, 32, 2) == 10003
    assert r.InitializeMemory(64, 33, 2) == 10004
    assert r.InitializeMemory(64, 32, 1) == 0
    assert r.RenderPerturbLAv2(A.GpuHDRx32PerturbedLAv2, coords, n) == 10005  # no orbit uploaded
    assert r.InitializePerturb(3, orbit, 0, None, la) == 0
    assert r.RenderPerturbLAv2(A.GpuHDRx32PerturbedLAv2, coords, n) == 0
    assert r.InitializeMemory(128, 32, 1) == 0                                # geometry change drops the cached orbit
    assert r.RenderPerturbLAv2(A.GpuHDRx32PerturbedLAv2, coords, n) == 10005
    assert "antialiasing" in GPURenderer.ConvertErrorToString(10002)
    done = []
    assert r.EnqueueComputeDoneCallback(lambda: done.append(1)) == 0
    assert r.SyncComputeStream() == 0 and done == [1]
    assert r.QueryComputeStream() == 0
    r.close()


EDGE_CASES = [
    # (view, w, h, algorithm, n_iter, iter_bytes): degenerate and ragged frames, iteration limits 0/1/2, tiny orbits
    (5, 1, 1, A.GpuHDRx32PerturbedLAv2, None, 4),
    (5, 17, 9, A.GpuHDRx32PerturbedLAv2, None, 8),
    (5, 33, 5, A.GpuHDRx32PerturbedRCLAv2, None, 4),
    (5, 16, 8, A.GpuHDRx32PerturbedLAv2, 1, 4),
    (5, 16, 8, A.GpuHDRx32PerturbedLAv2PO, 2, 4),
    (5, 16, 8, A.GpuHDRx32PerturbedBLA, 3, 4),
    (100, 19, 7, A.Gpu1x32PerturbedScaled, 5, 4),
    (19, 9, 3, A.GpuHDRx32PerturbedScaled, 50000, 8),
    (100, 15, 9, A.Gpu2x32PerturbedRCLAv2LAO, None, 4),
    (0, 7, 3, A.Gpu2x32, 64, 4),
    (0, 3, 5, A.Gpu4x64, 32, 8),
    (0, 1, 1, A.Gpu1x64, 10, 4),
]


EDGE_IDS = [f"v{c[0]}_{c[1]}x{c[2]}_{c[3].name}_{c[4]}" for c in EDGE_CASES]


@pytest.mark.skipif(not ref_renderer.available(), reason="oracle/_ref (reference CUDA kernels) not built")
@pytest.mark.parametrize("case", EDGE_CASES, ids=EDGE_IDS)
def test_edge_shapes_and_limits_vs_reference_kernels(case):
    """1x1 and ragged frames (not multiples of the 16x8 padding or of the 8x4 work tile), iteration limits of a
    few steps, both iteration widths: same buffers as the reference kernels, padding cells left cleared."""
    view_id, w, h, alg, n_iter, ib = case
    _, coords, orbit, la, n = cases.make_inputs(view_id, w, h, alg, n_iter, ib)
    got, _, red = cases.render(GPURenderer, w, h, alg, coords, orbit, la, n, ib)
    ref, _, ref_red = cases.render(ref_renderer.RefGPURenderer, w, h, alg, coords, orbit, la, n, ib)
    np.testing.assert_array_equal(got[:h, :w], ref[:h, :w])
    assert not got[h:, :].any() and not got[:, w:].any()
    assert (red["Min"], red["Max"], red["Sum"]) == (ref_red["Min"], ref_red["Max"], ref_red["Sum"])


def test_scaled_and_compressed_entry_points_reject_what_the_reference_does_not_instantiate():
    _, coords, orbit, la, n = cases.make_inputs(100, 32, 16, A.Gpu1x32PerturbedScaled, None, 4)
    r = GPURenderer()
    assert r.RenderPerturbBLAScaled(A.Gpu1x32PerturbedScaled, orbit, la, coords, n) == 0   # not initialised: no-op
    assert r.InitializeMemory(32, 16, 1) == 0
    assert r.RenderPerturbBLAScaled(A.Gpu1x32PerturbedScaled, orbit, la, coords, n) == 0
    # orbits of different length (GPU_Render.cu / Fractal.cpp:2909-2912 "Mismatch on size")
    _, _, orbit2, la2, _ = cases.make_inputs(101, 32, 16, A.Gpu1x32PerturbedScaled, None, 4)
    assert r.RenderPerturbBLAScaled(A.Gpu1x32PerturbedScaled, orbit, la2, coords, n) == 10100
    # a compressed orbit without OrbitXLow/YLow cannot be replayed
    _, c5, o5, l5, n5 = cases.make_inputs(5, 32, 16, A.GpuHDRx32PerturbedRCLAv2, None, 4)
    d = o5.descriptor()
    d.orbit_x_low = None
    import ctypes as C
    rc = r._lib.fs_initialize_perturb(r._h, 4, int(o5.numeric), 2, 9, C.byref(d), 0, 0, None, None)
    assert rc == 10005
    r.close()


SHARDED_CASES = [
    # (view, w, h, algorithm, n_iter, iter_bytes, precision, shard_count): every kernel family that takes fs_set_shard
    (0, 480, 270, A.Gpu1x32, 2000, 4, 1, 2),
    (0, 480, 270, A.Gpu1x64, 2000, 4, 4, 3),
    (0, 200, 133, A.Gpu1x64, 500, 8, 1, 8),     # ragged height, more shards than some frames have full bands
    (0, 240, 136, A.Gpu2x32, 500, 4, 8, 2),
    (0, 240, 136, A.Gpu2x64, 500, 4, 1, 3),
    (0, 96, 54, A.Gpu4x64, 128, 4, 1, 2),
    (100, 240, 135, A.GpuHDRx32, 2000, 4, 1, 3),
    (5, 240, 135, A.GpuHDRx32PerturbedBLA, None, 4, 1, 3),
    (100, 240, 135, A.Gpu1x64PerturbedBLA, None, 8, 1, 2),
    (5, 160, 90, A.GpuHDRx64PerturbedBLA, None, 4, 1, 8),
    (100, 240, 135, A.Gpu1x32PerturbedScaled, None, 4, 1, 3),
    (19, 160, 90, A.GpuHDRx32PerturbedScaled, 200000, 4, 1, 2),
    (100, 240, 135, A.Gpu2x32PerturbedLAv2, None, 4, 1, 3),
    (14, 240, 135, A.GpuHDRx2x32PerturbedLAv2, None, 4, 1, 8),
    (5, 160, 90, A.GpuHDRx32PerturbedRCLAv2, None, 8, 1, 2),
]


@pytest.mark.parametrize("case", SHARDED_CASES, ids=[f"v{c[0]}_{c[3].name}_n{c[7]}" for c in SHARDED_CASES])
def test_sharded_renders_of_every_kernel_family_merge_to_the_unsharded_frame(case):
    """fs_set_shard applies to every render entry: each shard writes exactly its own 4-row bands of the OUTPUT frame
    (the direct kernels flip rows, LowPrecisionKernels.cuh:309), the other rows stay cleared, the merged frame and the
    sum of the shard reductions equal the unsharded render, and RenderCurrentShard assembles the same frame."""
    view_id, w, h, alg, n_iter, ib, prec, count = case
    _, coords, orbit, la, n = cases.make_inputs(view_id, w, h, alg, n_iter, ib)
    whole, _, whole_red = cases.render(GPURenderer, w, h, alg, coords, orbit, la, n, ib, precision=prec)
    bufs, total = [], 0
    for s in range(count):
        it, _, red = cases.render(GPURenderer, w, h, alg, coords, orbit, la, n, ib, precision=prec, shard=(count, s))
        rows = rows_of_shard(h, count, s)
        other = np.setdiff1d(np.arange(it.shape[0]), rows)
        assert not it[other].any()
        np.testing.assert_array_equal(it[rows, :w], whole[rows, :w])
        bufs.append(it)
        total += red["Sum"]
    np.testing.assert_array_equal(merge_shards(bufs, h)[:h, :w], whole[:h, :w])
    assert total == whole_red["Sum"]


@pytest.mark.parametrize("aa,h_ss", [(1, 270), (2, 272), (4, 272), (2, 268)])
def test_sharded_colour_frame_assembles_to_the_unsharded_one(aa, h_ss):
    """RenderCurrentShard with a colour buffer: every shard colours the cells of its own 4-row bands and copies exactly
    those (iterations and Color16) into whole-frame host buffers; three shards fill the frames the unsharded
    RenderCurrent produces, and Min/Max/Sum combine to the frame's.  268 rows: the last band is cut by the frame edge."""
    w, h, alg, n = 96 * aa, h_ss, A.Gpu1x64, 300
    _, coords, _, _, _ = cases.make_inputs(0, w, h, alg, n, 4)
    r = GPURenderer()
    assert r.InitializeMemory(w, h, aa, iter_bytes=4) == 0
    r.ClearMemory()
    assert r.Render(alg, coords, n, 1) == 0
    rc, want_it, want_col, want_red = r.RenderCurrent(n, want_colors=True)
    assert rc == 0
    it = np.full_like(want_it, 0xDEADBEEF)
    col = np.zeros_like(want_col)
    mins, maxs, sums = [], [], 0
    for s in range(3):
        assert r.SetShard(3, s) == 0
        r.ClearMemory()
        assert r.Render(alg, coords, n, 1) == 0
        rc, red = r.RenderCurrentShard(n, it, colors_out=col)
        assert rc == 0
        mins.append(red["Min"]); maxs.append(red["Max"]); sums += red["Sum"]
    np.testing.assert_array_equal(it[:h, :w], want_it[:h, :w])
    n_cells = (h // aa) * (w // aa)
    np.testing.assert_array_equal(col.reshape(-1, 4)[:n_cells], want_col.reshape(-1, 4)[:n_cells])
    assert (min(mins), max(maxs), sums) == (want_red["Min"], want_red["Max"], want_red["Sum"])
    r.close()


def test_sharded_colours_with_antialiasing_3_are_refused():
    """3x3 antialiasing cells straddle the 4-row bands the shards own: a colour buffer is refused, iterations still flow."""
    w, h, alg, n = 96, 54, A.Gpu1x64, 100
    _, coords, _, _, _ = cases.make_inputs(0, w, h, alg, n, 4)
    r = GPURenderer()
    assert r.InitializeMemory(w, h, 3, iter_bytes=4) == 0
    assert r.SetShard(2, 1) == 0
    r.ClearMemory()
    assert r.Render(alg, coords, n, 1) == 0
    hp, wp = r.buffer_shape()
    it = np.zeros((hp, wp), np.uint32)
    col = np.zeros((24, 32, 4), np.uint16)
    rc, _ = r.RenderCurrentShard(n, it, colors_out=col)
    assert rc == 10100
    rc, _ = r.RenderCurrentShard(n, it)
    assert rc == 0 and it.any()
    r.close()


def test_progressive_render_current_returns_during_a_running_render():
    """RenderCurrent(progressive=true) is called by the reference's pool once a second WHILE the render kernel runs
    (RenderThreadPool.cpp:915-959, 1923-1948): it must come back with the partial frame (finished pixels, zeros
    elsewhere) long before the render ends, and the finished frame must be unaffected by the slots it borrowed."""
    import time
    w, h, alg = 3840, 2160, A.GpuHDRx32PerturbedLAv2PO
    r = GPURenderer()
    assert r.InitializeMemory(w, h, 1, iter_bytes=4) == 0
    # the undisturbed frame and its duration; the iteration limit is raised until the render lasts >= 150 ms
    for n_iter in (60000, 250000, 1000000, 4000000):
        _, coords, orbit, la, n = cases.make_inputs(5, w, h, alg, n_iter, 4)
        assert r.InitializePerturb(n_iter, orbit, 0, None, la) == 0
        r.ClearMemory()
        assert r.RenderPerturbLAv2(alg, coords, n) == 0
        rc, want, _, want_red = r.RenderCurrent(n)
        assert rc == 0
        full_ms = r.LastRenderMs()
        if full_ms >= 150.0:
            break
    assert full_ms >= 150.0, f"workload too short to observe a progressive frame ({full_ms:.1f} ms)"
    # now with progressive frames pulled while it runs
    r.ClearMemory()
    assert r.SyncComputeStream() == 0
    t0 = time.perf_counter()
    assert r.RenderPerturbLAv2(alg, coords, n) == 0
    time.sleep(0.25 * full_ms * 1e-3)
    partials = []
    for _ in range(2):
        rc, part, colors, red = r.RenderCurrent(n, want_colors=True, progressive=True)   # syncs the display stream only
        t_back = (time.perf_counter() - t0) * 1e3
        still_running = r.QueryComputeStream() == 600                                      # cudaErrorNotReady
        assert rc == 0
        partials.append((t_back, still_running, part.copy(), red))
        time.sleep(0.1 * full_ms * 1e-3)
    assert r.SyncComputeStream() == 0
    t_done = (time.perf_counter() - t0) * 1e3
    rc, got, _, got_red = r.RenderCurrent(n)
    assert rc == 0
    np.testing.assert_array_equal(got, want)                       # borrowing SM slots changes nothing in the result
    assert got_red == want_red
    for t_back, still_running, part, red in partials:
        assert still_running, f"progressive frame came back at {t_back:.1f} ms, render finished by then ({t_done:.1f} ms)"
        filled = part[:h, :w] != 0
        assert filled.any() and not filled.all()                   # a partial frame
        np.testing.assert_array_equal(part[:h, :w][filled], want[:h, :w][filled])   # finished pixels are final
        assert 0 < red["Sum"] < want_red["Sum"]
    # asked for a quarter of the way in, back well before the end -- even though every warp-tile of this workload
    # (interior pixels first, each running to the iteration limit) outlasts the wait
    assert partials[0][0] < 0.6 * t_done, (partials[0][0], t_done)
    # the render that lent its slots is not much slower (8 of ~600 CTAs)
    assert r.LastRenderMs() < 1.25 * full_ms
    r.close()


def test_tables_in_page_locked_host_memory_render_the_same_frame(monkeypatch):
    """The reference keeps orbit and LA tables in page-locked host memory when device memory runs out (Perturb.cuh:50-61,
    GPU_LAReference.h:90-113); the same fallback here (forced through FS_FORCE_HOST_TABLES) gives the same frames."""
    for name in ("v5_hdr32_lav2", "v5_hdr32_rclav2", "v5_hdr32_bla", "v100_f64_lav2"):
        _, view_id, w, h, alg, n_iter, ib = next(c for c in cases.ALL_SMALL_CASES if c[0] == name)
        _, coords, orbit, la, n = cases.make_inputs(view_id, w, h, alg, n_iter, ib)
        want, _, want_red = cases.render(GPURenderer, w, h, alg, coords, orbit, la, n, ib)
        monkeypatch.setenv("FS_FORCE_HOST_TABLES", "1")
        got, _, got_red = cases.render(GPURenderer, w, h, alg, coords, orbit, la, n, ib)
        monkeypatch.delenv("FS_FORCE_HOST_TABLES")
        np.testing.assert_array_equal(got, want)
        assert got_red == want_red


def test_native_library_is_the_one_loaded():
    """The CUDA path is the one that ran: libfsgpu.so is mapped into this process."""
    maps = open("/proc/self/maps").read()
    assert "libfsgpu.so" in maps


# ---- per-operation vectors of the device numeric types (SURVEY section 8 row a8) ---------------------------------------
import numeric_vectors


@pytest.mark.gpu
@pytest.mark.parametrize("op,name", numeric_vectors.OPS)
def test_device_numeric_operations_match_the_reference_restatement(built, op, name):
    """Row a8 on its own: every operation of HDRFloat<float>, HDRFloatComplex<float>, dblflt and dbldbl the kernels are built
    from, evaluated on the GPU by the very functions the kernels call (fs_selftest_numeric_op) on 400,000 operand pairs
    aimed at the code's case distinctions (numeric_vectors.operands) against oracle_cpu.cpp's restatement of
    HDRFloat.h:432-448, 624-636, 829-884, 974-1065, 1150-1167, HDRFloatComplex.h:219-283, 334-348, 473-527, 691-695,
    dblflt.cuh:91-219 and dbldbl.cuh:86-203.  Bit for bit (numeric_vectors.mismatches says what is not compared)."""
    import oracle_cpu
    from fractalshark_b200 import _native
    n = 400_000
    a, b = numeric_vectors.operands(op, n)
    out = np.zeros_like(a)
    rc = _native.gpu_lib().fs_selftest_numeric_op(0, op, a.ctypes.data, b.ctypes.data, out.ctypes.data, n)
    assert rc == 0, rc
    want = oracle_cpu.numeric_op(op, a, b)
    bad = numeric_vectors.mismatches(out, want)
    assert bad.size == 0, (name, int(bad.size), a[bad[:3]], b[bad[:3]], out[bad[:3]], want[bad[:3]])
