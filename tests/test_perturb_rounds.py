"""HDRx32 perturbation chunks (fs_scaled_loop.cuh fast_round) on the headline view, View 14, whose pixels rebase about
every 8 steps.  A rebase whose Z' + d' is exact but outside the range a chunk may start from is committed and re-centred;
these cases check that the committed states stay identical to the float+exponent steps and that such chunks are no
longer thrown away."""
import numpy as np
import pytest

import cases
import oracle_cpu
from fractalshark_b200 import RenderAlgorithm as A
from fractalshark_b200.gpu_renderer import GPURenderer


def test_view14_chunks_match_float_exponent_steps_in_lockstep(built):
    """Identical by value to the float+exponent restatement after every committed chunk, identical counts, and few
    chunks discarded: a rebase out of the chunk's start range is re-centred instead of rejected."""
    alg, stride, w, h = A.GpuHDRx32PerturbedLAv2, 24, 3840, 2160
    _, coords, orbit, la, n = cases.make_inputs(14, w, h, alg, None, 4)
    want, _ = oracle_cpu.render_lav2(alg, w, h, coords, orbit, la, n, row_step=stride, col_step=stride,
                                     threads=oracle_cpu.hardware_threads())
    got, st = oracle_cpu.lockstep_lav2(alg, w, h, coords, orbit, la, n, col_step=stride, row_step=stride,
                                       threads=oracle_cpu.hardware_threads())
    assert st["mismatches"] == 0, st
    np.testing.assert_array_equal(got, want)
    assert st["fast_steps"] > 100 * st["slow_steps"], st
    assert st["chunks_rejected"] * 40 < st["chunks_committed"], st


@pytest.mark.gpu
@pytest.mark.parametrize("view_id,w,h,alg,n_iter", [
    (14, 960, 540, A.GpuHDRx32PerturbedLAv2, None),
    (5, 960, 540, A.GpuHDRx32PerturbedLAv2PO, 20007),
])
def test_chunks_equal_float_exponent_loop_on_gpu(view_id, w, h, alg, n_iter):
    """The scaled chunks and the library's pure float+exponent loop give the same iteration buffer and execute the
    same number of algorithmic steps, on the headline view and with a limit that most pixels reach mid-chunk."""
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
    assert int((outs[0][:h, :w] == n).sum()) > 0
