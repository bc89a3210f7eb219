"""Shared parity cases: (name, view id, w, h, algorithm, n_iter (None = preset), iter_bytes)."""
from fractalshark_b200 import RenderAlgorithm as A

SMALL_CASES = [
    ("v0_gpu1x64", 0, 96, 54, A.Gpu1x64, 1024, 4),
    ("v0_gpu1x32", 0, 96, 54, A.Gpu1x32, 1024, 4),
    ("v0_gpu1x64_u64", 0, 50, 37, A.Gpu1x64, 300, 8),          # ragged size (not a multiple of 16x8)
    ("v5_hdr32_lav2", 5, 96, 54, A.GpuHDRx32PerturbedLAv2, None, 4),
    ("v5_hdr32_lav2_u64", 5, 50, 37, A.GpuHDRx32PerturbedLAv2, None, 8),
    ("v5_hdr32_lav2_po", 5, 64, 36, A.GpuHDRx32PerturbedLAv2PO, 3000, 4),
    ("v5_hdr32_lav2_lao", 5, 96, 54, A.GpuHDRx32PerturbedLAv2LAO, None, 4),
    ("v1_hdr32_lav2", 1, 96, 54, A.GpuHDRx32PerturbedLAv2, None, 4),
    ("v1_hdr32_lav2_po", 1, 96, 54, A.GpuHDRx32PerturbedLAv2PO, None, 4),
    ("v19_hdr32_lav2_capped", 19, 64, 36, A.GpuHDRx32PerturbedLAv2, 200000, 4),
]

# second fixture file (tests/golden/ref_gpu_small2.npz): BLA kernels and the other numeric variants of LAv2
SMALL_CASES_2 = [
    ("v5_hdr32_bla", 5, 96, 54, A.GpuHDRx32PerturbedBLA, None, 4),
    ("v5_hdr32_bla_u64", 5, 50, 37, A.GpuHDRx32PerturbedBLA, None, 8),
    ("v1_hdr32_bla", 1, 96, 54, A.GpuHDRx32PerturbedBLA, None, 4),
    ("v100_hdr32_bla", 100, 96, 54, A.GpuHDRx32PerturbedBLA, None, 4),
    ("v100_f64_bla", 100, 96, 54, A.Gpu1x64PerturbedBLA, None, 4),
    ("v1_f64_bla_u64", 1, 50, 37, A.Gpu1x64PerturbedBLA, None, 8),
    ("v5_hdr64_bla", 5, 64, 36, A.GpuHDRx64PerturbedBLA, None, 4),
    ("v5_hdr64_lav2", 5, 64, 36, A.GpuHDRx64PerturbedLAv2, None, 4),
    ("v5_hdr64_lav2_po", 5, 64, 36, A.GpuHDRx64PerturbedLAv2PO, 3000, 4),
    ("v100_f64_lav2", 100, 96, 54, A.Gpu1x64PerturbedLAv2, None, 4),
    ("v100_f64_lav2_po", 100, 96, 54, A.Gpu1x64PerturbedLAv2PO, None, 4),
    ("v1_f64_lav2", 1, 96, 54, A.Gpu1x64PerturbedLAv2, None, 4),
    ("v101_f32_lav2", 101, 96, 54, A.Gpu1x32PerturbedLAv2, None, 4),
    ("v100_hdr32_lav2", 100, 96, 54, A.GpuHDRx32PerturbedLAv2, None, 4),
]
# third fixture file (tests/golden/ref_gpu_small3.npz): 2x32 (CudaDblflt) and HDRx2x32 LAv2 variants
SMALL_CASES_3 = [
    ("v100_2x32_lav2", 100, 96, 54, A.Gpu2x32PerturbedLAv2, None, 4),
    ("v100_2x32_lav2_po", 100, 64, 36, A.Gpu2x32PerturbedLAv2PO, None, 4),
    ("v100_2x32_lav2_lao", 100, 96, 54, A.Gpu2x32PerturbedLAv2LAO, None, 4),
    ("v101_2x32_lav2_u64", 101, 50, 37, A.Gpu2x32PerturbedLAv2, None, 8),
    ("v5_hdr2x32_lav2", 5, 96, 54, A.GpuHDRx2x32PerturbedLAv2, None, 4),
    ("v5_hdr2x32_lav2_po", 5, 64, 36, A.GpuHDRx2x32PerturbedLAv2PO, 3000, 4),
    ("v5_hdr2x32_lav2_lao", 5, 96, 54, A.GpuHDRx2x32PerturbedLAv2LAO, None, 4),
    ("v1_hdr2x32_lav2_u64", 1, 50, 37, A.GpuHDRx2x32PerturbedLAv2, None, 8),
    ("v19_hdr2x32_lav2_capped", 19, 64, 36, A.GpuHDRx2x32PerturbedLAv2, 200000, 4),
]
# fourth fixture file (tests/golden/ref_gpu_small4.npz): scaled kernels (views 19: orbit elements flagged `bad`)
# and the extended-precision direct kernels
SMALL_CASES_4 = [
    ("v100_scaled_f64", 100, 96, 54, A.Gpu1x32PerturbedScaled, None, 4),
    ("v101_scaled_f64_u64", 101, 50, 37, A.Gpu1x32PerturbedScaled, None, 8),
    ("v19_scaled_f64_bad", 19, 64, 36, A.Gpu1x32PerturbedScaled, 200000, 4),
    ("v1_scaled_hdr32", 1, 96, 54, A.GpuHDRx32PerturbedScaled, None, 4),
    ("v5_scaled_hdr32", 5, 64, 36, A.GpuHDRx32PerturbedScaled, 20000, 4),
    ("v19_scaled_hdr32_bad_u64", 19, 50, 37, A.GpuHDRx32PerturbedScaled, 200000, 8),
    ("v0_gpu2x32", 0, 96, 54, A.Gpu2x32, 1024, 4),
    ("v100_gpu2x32_u64", 100, 50, 37, A.Gpu2x32, 20000, 8),
    ("v0_gpu2x64", 0, 96, 54, A.Gpu2x64, 1024, 4),
    ("v102_gpu2x64_u64", 102, 50, 37, A.Gpu2x64, 20000, 8),
    ("v0_gpuhdrx32", 0, 96, 54, A.GpuHDRx32, 512, 4),
    ("v100_gpuhdrx32_u64", 100, 50, 37, A.GpuHDRx32, 5000, 8),
    ("v0_gpu4x32", 0, 96, 54, A.Gpu4x32, 256, 4),
    ("v0_gpu4x64", 0, 96, 54, A.Gpu4x64, 256, 4),
]
# fifth fixture file (tests/golden/ref_gpu_small5.npz): RC algorithms (compressed orbits, PerturbExtras::SimpleCompression)
SMALL_CASES_5 = [
    ("v5_hdr32_rclav2", 5, 96, 54, A.GpuHDRx32PerturbedRCLAv2, None, 4),
    ("v5_hdr32_rclav2_po_u64", 5, 50, 37, A.GpuHDRx32PerturbedRCLAv2PO, 3000, 8),
    ("v5_hdr32_rclav2_lao", 5, 96, 54, A.GpuHDRx32PerturbedRCLAv2LAO, None, 4),
    ("v19_hdr32_rclav2_capped", 19, 64, 36, A.GpuHDRx32PerturbedRCLAv2, 200000, 4),
    ("v100_f64_rclav2", 100, 96, 54, A.Gpu1x64PerturbedRCLAv2, None, 4),
    ("v100_f64_rclav2_po_u64", 100, 50, 37, A.Gpu1x64PerturbedRCLAv2PO, None, 8),
    ("v101_f32_rclav2", 101, 96, 54, A.Gpu1x32PerturbedRCLAv2, None, 4),
    ("v5_hdr64_rclav2", 5, 64, 36, A.GpuHDRx64PerturbedRCLAv2, None, 4),
    ("v100_2x32_rclav2", 100, 96, 54, A.Gpu2x32PerturbedRCLAv2, None, 4),
    ("v5_hdr2x32_rclav2", 5, 64, 36, A.GpuHDRx2x32PerturbedRCLAv2, None, 4),
    ("v1_hdr2x32_rclav2_lao_u64", 1, 50, 37, A.GpuHDRx2x32PerturbedRCLAv2LAO, None, 8),
]
# sixth fixture file (tests/golden/ref_gpu_small6.npz): View 14, the north_star target view (21.7-kbit orbit)
SMALL_CASES_6 = [
    ("v14_hdr32_lav2", 14, 96, 54, A.GpuHDRx32PerturbedLAv2, None, 4),
    ("v14_hdr32_lav2_lao_u64", 14, 50, 37, A.GpuHDRx32PerturbedLAv2LAO, None, 8),
    ("v14_hdr32_rclav2", 14, 64, 36, A.GpuHDRx32PerturbedRCLAv2, None, 4),
    ("v14_hdr32_bla", 14, 64, 36, A.GpuHDRx32PerturbedBLA, None, 4),
]
# seventh fixture file (tests/golden/ref_gpu_small7.npz): direct kernels at iteration_precision 4 / 8 / 16 -- P steps
# per bailout test and `n_iterations -= P-1` (GPU_Render.cu:633-668, LowPrecisionKernels.cuh:317,707).  Iteration
# limits are chosen NOT to be multiples of P so the shortened limit and the chunked overshoot both show.
SMALL_CASES_7 = [
    ("v0_gpu1x32_p4", 0, 96, 54, A.Gpu1x32, 1023, 4),
    ("v0_gpu1x32_p8", 0, 96, 54, A.Gpu1x32, 1021, 4),
    ("v0_gpu1x32_p16_u64", 0, 50, 37, A.Gpu1x32, 1000, 8),
    ("v0_gpu1x64_p4_u64", 0, 50, 37, A.Gpu1x64, 301, 8),
    ("v0_gpu1x64_p8", 0, 96, 54, A.Gpu1x64, 1023, 4),
    ("v0_gpu1x64_p16", 0, 96, 54, A.Gpu1x64, 1030, 4),
    ("v0_gpu2x32_p4", 0, 96, 54, A.Gpu2x32, 1023, 4),
    ("v100_gpu2x32_p8_u64", 100, 50, 37, A.Gpu2x32, 20001, 8),
    ("v0_gpu2x32_p16", 0, 96, 54, A.Gpu2x32, 1030, 4),
    ("v0_gpuhdrx32_p4", 0, 96, 54, A.GpuHDRx32, 511, 4),
    ("v100_gpuhdrx32_p8_u64", 100, 50, 37, A.GpuHDRx32, 5003, 8),
    ("v0_gpuhdrx32_p16", 0, 96, 54, A.GpuHDRx32, 520, 4),
    ("v0_gpu1x32_p16_tiny", 0, 16, 8, A.Gpu1x32, 17, 4),       # limit barely above P: one chunk at most
]
# iteration_precision of a case (default 1)
CASE_PRECISION = {c[0]: int(c[0].split("_p")[1].split("_")[0]) for c in SMALL_CASES_7}
# Gpu4x32 / Gpu4x64: the four-limb products are split exactly here (one FMA) while the reference build leaves a
# Dekker split to the compiler's contraction (fs_qd.cuh); frames agree to >= 99.9 % of pixels, not bit for bit.
NOT_BIT_EXACT = {"v0_gpu4x32": 0.999, "v0_gpu4x64": 0.999}
ALL_SMALL_CASES = (SMALL_CASES + SMALL_CASES_2 + SMALL_CASES_3 + SMALL_CASES_4 + SMALL_CASES_5 + SMALL_CASES_6 +
                   SMALL_CASES_7)
CASE_SETS = {"1": SMALL_CASES, "2": SMALL_CASES_2, "3": SMALL_CASES_3, "4": SMALL_CASES_4, "5": SMALL_CASES_5,
             "6": SMALL_CASES_6, "7": SMALL_CASES_7}
GOLDEN_FILES = {"1": "ref_gpu_small.npz", "2": "ref_gpu_small2.npz", "3": "ref_gpu_small3.npz",
                "4": "ref_gpu_small4.npz", "5": "ref_gpu_small5.npz", "6": "ref_gpu_small6.npz",
                "7": "ref_gpu_small7.npz"}


def golden_file_of(name):
    import os
    here = os.path.dirname(os.path.abspath(__file__))
    which = next(k for k, cs in CASE_SETS.items() if any(c[0] == name for c in cs))
    return os.path.join(here, "golden", GOLDEN_FILES[which])


def load_goldens():
    """All committed reference-kernel fixtures merged into one dict."""
    import os
    import numpy as np
    here = os.path.dirname(os.path.abspath(__file__))
    out = {}
    for f in GOLDEN_FILES.values():
        out.update(np.load(os.path.join(here, "golden", f)))
    return out


def inputs_crc(coords, orbit, table):
    """CRC32 of everything fed to the kernels, stored beside each golden buffer."""
    import zlib
    crc = 0
    for k in sorted(coords):
        crc = zlib.crc32(coords[k], crc)
    if orbit is not None:
        crc = zlib.crc32(orbit.as_numpy().tobytes(), crc)
    if table is not None and hasattr(table, "num_las") and table.num_las:
        las = table.las_numpy()
        if las.shape[1] in (128, 136):
            # LAInfoDeep<HDRFloat<double>>: 4 padding bytes after every int32 exponent (3 complex {re,im,exp}
            # of 24 B, 3 reals {m,exp} of 16 B) are indeterminate in the generator's C++ structs
            las = las.copy()
            for off in (20, 44, 68, 84, 100, 116):
                las[:, off:off + 4] = 0
        crc = zlib.crc32(las.tobytes(), crc)
        crc = zlib.crc32(table.stages_numpy().tobytes(), crc)
    if table is not None and hasattr(table, "as_numpy"):   # scaled kernel: the binary32 orbit
        crc = zlib.crc32(table.as_numpy().tobytes(), crc)
    if table is not None and hasattr(table, "level_counts"):
        for lv in range(table.num_levels):
            crc = zlib.crc32(table.level_numpy(lv).tobytes(), crc)
    return crc


def sha256_of(a):
    import hashlib
    import numpy as np
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def la_digest(la):
    """Sizes and SHA-256 digests of an LA table (LAInfoDeep[] with its indeterminate padding cleared, the LAStageCount
    stage records, the ATInfo bytes), as stored in tests/golden/tables.json."""
    import ctypes as C
    import numpy as np
    las = la.las_numpy().copy()
    if la.iter_bytes == 8:
        las[:, 60:64] = 0   # LAInfoDeep<uint64_t, ...>: 4 padding bytes between MinMag (ends at 60) and LAi (at 64)
    at = np.frombuffer((C.c_ubyte * la.at_bytes).from_address(la.descriptor().at), dtype=np.uint8)
    return {"num_las": la.num_las, "stage_count": la.stage_count, "use_at": bool(la.use_at), "is_valid": bool(la.is_valid),
            "las_elem_bytes": la.las_elem_bytes, "at_bytes": la.at_bytes, "las_sha256": sha256_of(las),
            "stages_sha256": sha256_of(la.stages_numpy()[: la.stage_count]), "at_sha256": sha256_of(at)}


def bla_digest(bl):
    """Level count, LM2 and the SHA-256 of every level of a BLA table, as stored in tests/golden/tables.json."""
    return {"num_levels": bl.num_levels, "lm2": bl.lm2,
            "levels_sha256": [sha256_of(bl.level_numpy(lv)) for lv in range(bl.num_levels)]}


def full_case_precision(name):
    """iteration_precision of a full-size case: the N of a `_pN` name suffix, else 1."""
    return int(name.split("_p")[1].split("_")[0]) if "_p" in name and name.split("_p")[1][0].isdigit() else 1


def load_recorded(name):
    """A recording of tests/golden/record_library_outputs.py: .json as a dict, .npz as a dict of arrays."""
    import json
    import os
    import numpy as np
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name)
    if name.endswith(".json"):
        with open(path) as f:
            return json.load(f)
    return dict(np.load(path))


def oracle_render(alg, w, h, coords, orbit, table, n, ib, precision=1, **kw):
    """CPU oracle for a case, or None when the oracle has no restatement of that variant."""
    import oracle_cpu
    from fractalshark_b200 import traits
    fam = traits(alg).family
    kw.setdefault("threads", oracle_cpu.hardware_threads())
    try:
        if fam == "lav2":
            return oracle_cpu.render_lav2(alg, w, h, coords, orbit, table, n, iter_bytes=ib, **kw)[0]
        if fam == "bla":
            return oracle_cpu.render_bla(alg, w, h, coords, orbit, table, n, iter_bytes=ib, **kw)[0]
        if fam == "scaled":
            return oracle_cpu.render_scaled(alg, w, h, coords, orbit, table, n, iter_bytes=ib, **kw)[0]
        return oracle_cpu.render_direct(alg, w, h, coords, n, precision, iter_bytes=ib, threads=kw["threads"])[0]
    except NotImplementedError:
        return None


_ORBIT_CACHE = {}


def _cached_orbit(view, view_id, numeric, n_iter):
    """The reference orbit depends on the view's centre, radius (after the aspect-ratio squaring of the bounds) and
    precision, not on the pixel count: computed once per (view, aspect ratio, numeric type, iteration cap) --
    View 14's 21.7-kbit orbit takes several seconds."""
    from fractions import Fraction
    from fractalshark_b200.host_inputs import Orbit
    key = (view_id, Fraction(view.width, view.height), int(numeric), int(n_iter))
    if key not in _ORBIT_CACHE:
        if len(_ORBIT_CACHE) > 12:
            _ORBIT_CACHE.clear()
        _ORBIT_CACHE[key] = Orbit(view, numeric, n_iter, True)
    return _ORBIT_CACHE[key]


def make_inputs(view_id, w, h, alg, n_iter, iter_bytes):
    from fractalshark_b200 import traits
    from fractalshark_b200.host_inputs import LaTable, View
    from fractalshark_b200.views import PRESETS

    def Orbit(view, numeric, n, _periodicity):
        return _cached_orbit(view, view_id, numeric, n)

    p = PRESETS[view_id]
    n_iter = n_iter or p.num_iterations
    t = traits(alg)
    view = View(p.min_x, p.min_y, p.max_x, p.max_y, w, h)
    coords = view.coords(t.numeric, direct=(t.family == "direct"))
    orbit = la = None
    if t.family == "lav2":
        orbit = Orbit(view, t.numeric, n_iter, True)
        if int(t.pextras) == 2:   # RC algorithms: waypoints only, LA table from the host replay
            orbit = orbit.compress()
        la = LaTable(orbit, iter_bytes)
    elif t.family == "bla":
        from fractalshark_b200.host_inputs import BlaTable
        orbit = Orbit(view, t.numeric, n_iter, True)
        la = BlaTable(orbit)   # rides in the `la` slot of the case tuple
    elif t.family == "scaled":
        base = Orbit(view, t.numeric, n_iter, True)
        orbit = base.with_bad()             # GPUReferenceIter<T, Bad>
        la = base.with_bad(to_float=True)   # its binary32 copy rides in the `la` slot
    return view, coords, orbit, la, n_iter


def render(renderer_cls, w, h, alg, coords, orbit, la, n_iter, iter_bytes, want_colors=False, aa=1, precision=1,
           shard=None):
    from fractalshark_b200 import traits
    r = renderer_cls()
    rc = r.InitializeMemory(w, h, aa, iter_bytes=iter_bytes)
    assert rc == 0, rc
    if shard is not None:
        assert r.SetShard(*shard) == 0
    fam = traits(alg).family
    if orbit is not None and fam == "lav2":
        rc = r.InitializePerturb(1, orbit, 0, None, la)
        assert rc == 0, rc
    r.ClearMemory()
    if fam == "lav2":
        rc = r.RenderPerturbLAv2(alg, coords, n_iter)
    elif fam == "bla":
        rc = r.RenderPerturbBLA(alg, orbit, la, coords, n_iter)
    elif fam == "scaled":
        rc = r.RenderPerturbBLAScaled(alg, orbit, la, coords, n_iter)
    else:
        rc = r.Render(alg, coords, n_iter, precision)
    assert rc == 0, rc
    rc, iters, colors, red = r.RenderCurrent(n_iter, want_colors=want_colors)
    assert rc == 0, rc
    r.close()
    return iters, colors, red
