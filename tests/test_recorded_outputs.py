"""This library's own outputs, pinned: the LA / BLA tables of the in-tree builders and the frames of the full-size and
edge-shape cases, against what tests/golden/record_library_outputs.py recorded from this library.  These are regression
pins, not reference comparisons: the checks against the reference's own builders and kernels (test_table_construction.py,
test_full_size_vs_reference_cuda_kernels, test_edge_shapes_and_limits_vs_reference_kernels) need oracle/_ref, built from
the FractalShark sources, and this module keeps the same cases checked where that is not available.  A deliberate change
of an output is re-recorded with the script."""
import numpy as np
import pytest

import cases
import test_gpu_parity as P
from fractalshark_b200 import RenderAlgorithm as A

LA_CASES = [(1, 4), (1, 8), (5, 4), (5, 8), (19, 4), (14, 4), (14, 8), (100, 4)]
BLA_VIEWS = [1, 5, 14, 100]


def la_key(view_id, iter_bytes):
    return "v%d_u%d" % (view_id, 8 * iter_bytes)


@pytest.mark.parametrize("view_id,iter_bytes", LA_CASES)
def test_la_table_equals_the_recorded_one(built, view_id, iter_bytes):
    _, _, _, la, _ = cases.make_inputs(view_id, 192, 108, A.GpuHDRx32PerturbedLAv2, None, iter_bytes)
    assert cases.la_digest(la) == cases.load_recorded("tables.json")["la"][la_key(view_id, iter_bytes)]


@pytest.mark.parametrize("view_id", BLA_VIEWS)
def test_bla_table_equals_the_recorded_one(built, view_id):
    _, _, _, bl, _ = cases.make_inputs(view_id, 192, 108, A.GpuHDRx32PerturbedBLA, None, 4)
    assert cases.bla_digest(bl) == cases.load_recorded("tables.json")["bla"]["v%d" % view_id]


@pytest.mark.gpu
@pytest.mark.parametrize("case", P.FULL_CASES, ids=[c[0] for c in P.FULL_CASES])
def test_full_size_frame_equals_the_recorded_one(case):
    """Same inputs (CRC32), same sampled rows, same SHA-256 of the whole iteration buffer, same Min/Max/Sum."""
    from fractalshark_b200.gpu_renderer import GPURenderer
    name, view_id, w, h, alg, n_iter, ib, _ = case
    _, coords, orbit, la, n = cases.make_inputs(view_id, w, h, alg, n_iter, ib)
    got, _, red = cases.render(GPURenderer, w, h, alg, coords, orbit, la, n, ib, precision=cases.full_case_precision(name))
    rec = cases.load_recorded("frames_full.json")[name]
    rows = cases.load_recorded("frames_full_rows.npz")
    assert cases.inputs_crc(coords, orbit, la) == rec["inputs_crc32"], "input generator drifted from the recording"
    np.testing.assert_array_equal(got[rows[name + "__rows"], :w], rows[name])
    assert cases.sha256_of(got[:h, :w]) == rec["sha256"]
    assert (red["Min"], red["Max"], red["Sum"]) == (rec["min"], rec["max"], rec["sum"])
    assert not got[h:, :].any() and not got[:, w:].any()


@pytest.mark.gpu
@pytest.mark.parametrize("case", P.EDGE_CASES, ids=P.EDGE_IDS)
def test_edge_shape_frame_equals_the_recorded_one(case):
    from fractalshark_b200.gpu_renderer import GPURenderer
    view_id, w, h, alg, n_iter, ib = case
    _, coords, orbit, la, n = cases.make_inputs(view_id, w, h, alg, n_iter, ib)
    got, _, red = cases.render(GPURenderer, w, h, alg, coords, orbit, la, n, ib)
    rec = cases.load_recorded("frames_edge.npz")
    case_id = P.EDGE_IDS[P.EDGE_CASES.index(case)]
    np.testing.assert_array_equal(got[:h, :w], rec[case_id])
    assert [red["Min"], red["Max"], red["Sum"]] == rec[case_id + "__red"].tolist()
    assert not got[h:, :].any() and not got[:, w:].any()
