"""Records this library's own outputs for tests/test_recorded_outputs.py, which pins them.  These recordings are
snapshots of this library, not of the reference: the checks against the reference's builders and kernels need oracle/_ref,
built from the FractalShark sources, which are not part of this repository.  Where oracle/_ref is built, every table and
frame is first held to the reference's (as the tests that compare with it do) and nothing is written unless all agree.

    tables.json           LA and BLA tables of the in-tree builders: sizes and SHA-256 digests (cases.la_digest /
                          cases.bla_digest; View 14's LA table alone is 2 MB)
    frames_full.json      frames of FULL_CASES (tests/test_gpu_parity.py): SHA-256 of the iteration buffer, Min / Max / Sum
                          and the CRC32 of the inputs (cases.inputs_crc)
    frames_full_rows.npz  two whole rows of every such frame, chosen with a fixed seed, so that a failure shows where
    frames_edge.npz       frames of EDGE_CASES (tests/test_gpu_parity.py), whole, with Min / Max / Sum

    python tests/golden/record_library_outputs.py tables [OUT_DIR]   # CPU
    python tests/golden/record_library_outputs.py frames [OUT_DIR]   # needs a CUDA device

OUT_DIR defaults to tests/golden/.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import cases  # noqa: E402
import ref_host  # noqa: E402
import ref_renderer  # noqa: E402

ROW_SEED = 7


def _write_json(path, obj):
    with open(path, "w") as f:
        json.dump(obj, f, indent=1, sort_keys=True)
        f.write("\n")


def record_tables(out_dir):
    import test_recorded_outputs as T
    from fractalshark_b200 import RenderAlgorithm as A
    out = {"la": {}, "bla": {}}
    for view_id, ib in T.LA_CASES:
        _, _, orbit, la, n = cases.make_inputs(view_id, 192, 108, A.GpuHDRx32PerturbedLAv2, None, ib)
        out["la"][T.la_key(view_id, ib)] = cases.la_digest(la)
        if ref_host.available():
            ref = ref_host.RefLaTable(orbit, ib, n, 0)
            theirs = ref.las.copy()
            if ib == 8:
                theirs[:, 60:64] = 0
            assert cases.sha256_of(theirs) == out["la"][T.la_key(view_id, ib)]["las_sha256"], (view_id, ib)
            assert cases.sha256_of(ref.stages[: ref.stage_count]) == out["la"][T.la_key(view_id, ib)]["stages_sha256"]
            assert cases.sha256_of(ref.at) == out["la"][T.la_key(view_id, ib)]["at_sha256"]
    for view_id in T.BLA_VIEWS:
        _, _, orbit, bl, n = cases.make_inputs(view_id, 192, 108, A.GpuHDRx32PerturbedBLA, None, 4)
        out["bla"]["v%d" % view_id] = cases.bla_digest(bl)
        if ref_host.available():
            ref = ref_host.RefLaTable(orbit, 4, n, 1, with_blas=True)
            assert ref.blas_lm2 == bl.lm2 and [cases.sha256_of(a) for a in ref.blas_levels] == \
                out["bla"]["v%d" % view_id]["levels_sha256"], view_id
    _write_json(os.path.join(out_dir, "tables.json"), out)


def record_frames(out_dir):
    import test_gpu_parity as P
    from fractalshark_b200.gpu_renderer import GPURenderer
    full, rows = {}, {}
    rng = np.random.default_rng(ROW_SEED)
    for name, view_id, w, h, alg, n_iter, ib, min_exact in P.FULL_CASES:
        _, coords, orbit, la, n = cases.make_inputs(view_id, w, h, alg, n_iter, ib)
        got, _, red = cases.render(GPURenderer, w, h, alg, coords, orbit, la, n, ib,
                                   precision=cases.full_case_precision(name))
        if ref_renderer.available():
            ref, _, _ = cases.render(ref_renderer.RefGPURenderer, w, h, alg, coords, orbit, la, n, ib,
                                     precision=cases.full_case_precision(name))
            assert float((got[:h, :w] == ref[:h, :w]).mean()) >= abs(min_exact), name
        full[name] = {"sha256": cases.sha256_of(got[:h, :w]), "min": red["Min"], "max": red["Max"], "sum": red["Sum"],
                      "inputs_crc32": int(cases.inputs_crc(coords, orbit, la))}
        pick = np.sort(rng.choice(h, size=2, replace=False))
        rows[name], rows[name + "__rows"] = got[pick, :w].copy(), pick
        print(name, full[name], flush=True)
    _write_json(os.path.join(out_dir, "frames_full.json"), full)
    np.savez_compressed(os.path.join(out_dir, "frames_full_rows.npz"), **rows)
    edge = {}
    for case_id, (view_id, w, h, alg, n_iter, ib) in zip(P.EDGE_IDS, P.EDGE_CASES):
        _, coords, orbit, la, n = cases.make_inputs(view_id, w, h, alg, n_iter, ib)
        got, _, red = cases.render(GPURenderer, w, h, alg, coords, orbit, la, n, ib)
        if ref_renderer.available():
            ref, _, _ = cases.render(ref_renderer.RefGPURenderer, w, h, alg, coords, orbit, la, n, ib)
            np.testing.assert_array_equal(got[:h, :w], ref[:h, :w])
        edge[case_id] = got[:h, :w].copy()
        edge[case_id + "__red"] = np.array([red["Min"], red["Max"], red["Sum"]], dtype=np.uint64)
    np.savez_compressed(os.path.join(out_dir, "frames_edge.npz"), **edge)


if __name__ == "__main__":
    what = sys.argv[1]
    out = sys.argv[2] if len(sys.argv) > 2 else HERE
    os.makedirs(out, exist_ok=True)
    {"tables": record_tables, "frames": record_frames}[what](out)
