"""TEST INFRASTRUCTURE: ctypes wrapper of oracle/liboracle.so (CPU restatement of the reference kernels)."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from fractalshark_b200.algorithms import traits
from fractalshark_b200.gpu_renderer import NB_THREADS_H, NB_THREADS_W, _round_up

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_LIB = os.path.join(ROOT, "oracle", "liboracle.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(ORACLE_LIB)
        V, I, U64 = C.c_void_p, C.c_int, C.c_uint64
        L.orc_render_lav2.restype = U64
        L.orc_render_lav2.argtypes = [I, I, I, V, U64, V, V, V, U64, I, I, I, I, V, V, V, V, U64, V, I, I, I, I, I]
        L.orc_render_direct.restype = U64
        L.orc_render_direct.argtypes = [I, I, I, I, V, V, V, V, U64, I, V, I, I, I]
        L.orc_render_bla.restype = U64
        L.orc_render_bla.argtypes = [I, I, V, U64, V, I, I, I, V, V, V, V, U64, V, I, I, I, I, I]
        L.orc_post.restype = None
        L.orc_post.argtypes = [I, V, I, I, I, V, C.c_uint32, C.c_uint32, U64, V, V]
        L.orc_hardware_threads.restype = I
        _lib = L
    return _lib


def _buf(b: bytes):
    return C.cast(C.create_string_buffer(b, len(b)), C.c_void_p)


def hardware_threads() -> int:
    return int(lib().orc_hardware_threads())


def numeric_op(op: int, a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """One operation of the reference's device numeric types on operand arrays (oracle_cpu.cpp orc_numeric_op); operands and
    results as raw bytes in structured arrays of the element layout of `op`."""
    L = lib()
    L.orc_numeric_op.restype = C.c_int
    L.orc_numeric_op.argtypes = [C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
    a = np.ascontiguousarray(a)
    b = np.ascontiguousarray(b)
    out = np.zeros_like(a)
    rc = L.orc_numeric_op(op, a.ctypes.data, b.ctypes.data, out.ctypes.data, a.shape[0])
    assert rc == 0, rc
    return out


def render_lav2(alg, w, h, coords, orbit, la, n_iter, iter_bytes=4, rows=None, col_step=1, row_step=1, threads=1, out=None):
    """Returns (iters[hp, wp], executed_steps). Only rows in `rows` / every col_step-th column are computed."""
    t = traits(alg)
    hp, wp = _round_up(h, NB_THREADS_H), _round_up(w, NB_THREADS_W)
    dt = np.uint32 if iter_bytes == 4 else np.uint64
    if out is None:
        out = np.zeros((hp, wp), dtype=dt)
    rb, re = rows if rows is not None else (0, h)
    d = orbit.descriptor()
    elements = d.elements
    if getattr(orbit, "pextras", 0) == 2:
        # compressed orbit: replay the waypoints with the device arithmetic first (Perturb.cuh:246-326)
        full = np.zeros((d.uncompressed_count, 16), dtype=np.uint8)
        fn = lib().orc_expand_orbit
        fn.restype = C.c_uint64
        fn.argtypes = [C.c_int, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]
        if fn(int(t.numeric), d.elements, d.compressed_count, d.uncompressed_count, d.orbit_x_low, d.orbit_y_low,
              full.ctypes.data) != 0:
            raise NotImplementedError(f"oracle has no compressed-orbit replay for {alg!r}")
        elements = full.ctypes.data
    if la is not None:
        l = la.descriptor()
        largs = (l.las, l.stages, l.at, l.la_stage_count, l.use_at, l.is_valid)
    else:
        largs = (None, None, None, 0, 0, 0)
    steps = lib().orc_render_lav2(int(t.numeric), iter_bytes, int(t.mode), elements, d.uncompressed_count, *largs,
                                  w, h, _buf(coords["dx"]), _buf(coords["dy"]), _buf(coords["center_x"]),
                                  _buf(coords["center_y"]), n_iter, out.ctypes.data, rb, re, col_step, row_step, threads)
    if steps == 2 ** 64 - 1:
        raise NotImplementedError(f"oracle has no restatement for {alg!r}")
    return out, int(steps)


def render_bla(alg, w, h, coords, orbit, blas, n_iter, iter_bytes=4, rows=None, col_step=1, row_step=1, threads=1):
    """mandel_1xHDR_float_perturb_bla / mandel_1x_double_perturb_bla restated on the CPU."""
    t = traits(alg)
    hp, wp = _round_up(h, NB_THREADS_H), _round_up(w, NB_THREADS_W)
    out = np.zeros((hp, wp), dtype=np.uint32 if iter_bytes == 4 else np.uint64)
    rb, re = rows if rows is not None else (0, h)
    d, b = orbit.descriptor(), blas.descriptor()
    steps = lib().orc_render_bla(int(t.numeric), iter_bytes, d.elements, d.uncompressed_count,
                                 C.cast(b.levels, C.c_void_p), b.lm2, w, h, _buf(coords["dx"]), _buf(coords["dy"]),
                                 _buf(coords["center_x"]), _buf(coords["center_y"]), n_iter, out.ctypes.data, rb, re,
                                 col_step, row_step, threads)
    if steps == 2 ** 64 - 1:
        raise NotImplementedError(f"oracle has no restatement for {alg!r}")
    return out, int(steps)


def render_scaled(alg, w, h, coords, orbit_t, orbit_f, n_iter, iter_bytes=4, rows=None, col_step=1, row_step=1,
                  threads=1):
    """CPU restatement of mandel_1x_float_perturb_scaled (both orbits in the Bad layout)."""
    t = traits(alg)
    hp, wp = _round_up(h, NB_THREADS_H), _round_up(w, NB_THREADS_W)
    out = np.zeros((hp, wp), dtype=np.uint32 if iter_bytes == 4 else np.uint64)
    rb, re = rows if rows is not None else (0, h)
    fn = lib().orc_render_scaled
    fn.restype = C.c_uint64
    fn.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                   C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    steps = fn(int(t.numeric), iter_bytes, orbit_t.data_ptr, orbit_f.data_ptr, orbit_t.count, w, h, _buf(coords["dx"]),
               _buf(coords["dy"]), _buf(coords["center_x"]), _buf(coords["center_y"]), n_iter, out.ctypes.data, rb, re,
               col_step, row_step, threads)
    if steps == 2 ** 64 - 1:
        raise NotImplementedError(f"oracle has no restatement for {alg!r}")
    return out, int(steps)


def render_direct(alg, w, h, coords, n_iter, prec=1, iter_bytes=4, rows=None, threads=1):
    t = traits(alg)
    hp, wp = _round_up(h, NB_THREADS_H), _round_up(w, NB_THREADS_W)
    out = np.zeros((hp, wp), dtype=np.uint32 if iter_bytes == 4 else np.uint64)
    rb, re = rows if rows is not None else (0, h)
    steps = lib().orc_render_direct(int(t.numeric), iter_bytes, w, h, _buf(coords["cx"]), _buf(coords["cy"]),
                                    _buf(coords["dx"]), _buf(coords["dy"]), n_iter, prec, out.ctypes.data, rb, re,
                                    threads)
    if steps == 2 ** 64 - 1:
        raise NotImplementedError(f"oracle has no restatement for {alg!r}")
    return out, int(steps)


def post(iters, w, h, aa, palette, aux_depth, n_iter):
    iter_bytes = iters.dtype.itemsize
    palette = np.ascontiguousarray(palette, dtype=np.uint16)
    colors = np.zeros((h // aa, w // aa, 4), dtype=np.uint16)
    red = np.zeros(3, dtype=np.uint64)
    lib().orc_post(iter_bytes, iters.ctypes.data, w, h, aa, palette.ctypes.data, palette.shape[0], aux_depth, n_iter,
                   colors.ctypes.data, red.ctypes.data)
    return colors, {"Min": int(red[0]), "Max": int(red[1]), "Sum": int(red[2])}


LOCKSTEP_LIB = os.path.join(ROOT, "oracle", "liblockstep.so")
_lock = None


def lockstep_lav2(alg, w, h, coords, orbit, la, n_iter, col_step=1, row_step=1, threads=1):
    """Runs the product's scaled plain-float chunks (fs_scaled_loop.cuh, host build) in lockstep with the
    float+exponent oracle.  Returns (iters, stats dict); stats["mismatches"] must be 0."""
    global _lock
    if _lock is None:
        _lock = C.CDLL(LOCKSTEP_LIB)
    V, I, U64 = C.c_void_p, C.c_int, C.c_uint64
    _lock.lockstep_render_lav2.restype = U64
    _lock.lockstep_render_lav2.argtypes = [I, V, U64, V, V, V, U64, I, I, I, I, V, V, V, V, U64, V, I, I, I, V]
    t = traits(alg)
    hp, wp = _round_up(h, NB_THREADS_H), _round_up(w, NB_THREADS_W)
    out = np.zeros((hp, wp), dtype=np.uint32)
    d, l = orbit.descriptor(), la.descriptor()
    stats = (C.c_uint64 * 8)()
    _lock.lockstep_render_lav2(int(t.mode), d.elements, d.uncompressed_count, l.las, l.stages, l.at, l.la_stage_count,
                               l.use_at, l.is_valid, w, h, _buf(coords["dx"]), _buf(coords["dy"]),
                               _buf(coords["center_x"]), _buf(coords["center_y"]), n_iter, out.ctypes.data, col_step,
                               row_step, threads, stats)
    keys = ("fast_steps", "slow_steps", "chunks_committed", "chunks_rejected", "entries_refused", "mismatches",
            "finished_in_chunk")
    return out, dict(zip(keys, [int(x) for x in stats]))


def lockstep_at(w, h, coords, la, n_iter, max_passes=20000, col_step=1, row_step=1):
    """Runs the product's AT mantissa recurrence (fs_at_fast.cuh, host build) pass by pass against the oracle's
    float+exponent AT loop for every sampled pixel of the frame.  Returns the stats dict (mismatches must be 0)."""
    global _lock
    if _lock is None:
        _lock = C.CDLL(LOCKSTEP_LIB)
    fn = _lock.lockstep_at
    fn.restype = C.c_uint64
    fn.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                   C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_void_p]
    l = la.descriptor()
    stats = (C.c_uint64 * 6)()
    fn(l.at, l.use_at, l.is_valid, w, h, _buf(coords["dx"]), _buf(coords["dy"]), _buf(coords["center_x"]),
       _buf(coords["center_y"]), n_iter, max_passes, col_step, row_step, stats)
    return dict(zip(("pixels", "refused", "passes", "mismatches", "escaped", "mono"), (int(v) for v in stats)))


def lockstep_at_cycle(w, h, coords, la, n_iter, col_step=1, row_step=1):
    """The cycle watch of the chunked AT loop (fs_at_fast.cuh CycleWatch, host build) against the loop that executes every
    pass, for every sampled pixel: same pass count and same z, bit for bit (mismatches must be 0)."""
    global _lock
    if _lock is None:
        _lock = C.CDLL(LOCKSTEP_LIB)
    fn = _lock.lockstep_at_cycle
    fn.restype = C.c_uint64
    fn.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                   C.c_uint64, C.c_int, C.c_int, C.c_void_p]
    l = la.descriptor()
    stats = (C.c_uint64 * 5)()
    fn(l.at, l.use_at, l.is_valid, w, h, _buf(coords["dx"]), _buf(coords["dy"]), _buf(coords["center_x"]),
       _buf(coords["center_y"]), n_iter, col_step, row_step, stats)
    return dict(zip(("pixels", "cycles_found", "passes_with_watch", "passes_without", "mismatches"), (int(v) for v in stats)))


def at_plan(cre, cim, ce, rm, re_):
    """(ok, mono, E, thr) of the plan the kernel's AT shortcut makes for c = (cre, cim) x 2^ce, R = rm x 2^re_."""
    global _lock
    if _lock is None:
        _lock = C.CDLL(LOCKSTEP_LIB)
    out = (C.c_int * 3)()
    thr = C.c_float()
    _lock.lockstep_at_plan.restype = None
    _lock.lockstep_at_plan.argtypes = [C.c_float, C.c_float, C.c_int, C.c_float, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_float)]
    _lock.lockstep_at_plan(cre, cim, ce, rm, re_, out, C.byref(thr))
    return bool(out[0]), bool(out[1]), int(out[2]), float(thr.value)


def at_growth(cre, cim, ce, rm, re_, zre, zim, passes):
    """(first escaped pass or -1, every later pass still reads escaped) for the mantissa recurrence started at z."""
    global _lock
    if _lock is None:
        _lock = C.CDLL(LOCKSTEP_LIB)
    stays = C.c_int()
    _lock.lockstep_at_growth.restype = C.c_int
    _lock.lockstep_at_growth.argtypes = [C.c_float, C.c_float, C.c_int, C.c_float, C.c_int, C.c_float, C.c_float, C.c_int,
                                         C.POINTER(C.c_int)]
    first = _lock.lockstep_at_growth(cre, cim, ce, rm, re_, zre, zim, passes, C.byref(stays))
    return int(first), bool(stays.value)


def twice_product_identity_mismatches(count, seed=1):
    """fma(a, b, RN(a*b)) == 2*RN(a*b) on `count` random binary32 and binary64 pairs (lockstep_check.cpp)."""
    L = C.CDLL(LOCKSTEP_LIB)
    L.lockstep_twice_product_identity.restype = C.c_uint64
    L.lockstep_twice_product_identity.argtypes = [C.c_uint64, C.c_uint64]
    return int(L.lockstep_twice_product_identity(count, seed))


def lockstep_la(w, h, coords, la, n_iter, iter_bytes=4, col_step=1, row_step=1):
    """Runs the product's select-free LA step (fs_la_fast.cuh, host build) on the inputs of every LA step the oracle
    attempts for the sampled pixels.  Returns {"steps", "refused", "mismatches", "unusable"}; mismatches must be 0."""
    global _lock
    if _lock is None:
        _lock = C.CDLL(LOCKSTEP_LIB)
    fn = _lock.lockstep_la
    fn.restype = None
    V, I, U64 = C.c_void_p, C.c_int, C.c_uint64
    fn.argtypes = [V, V, V, U64, I, I, I, I, V, V, V, V, U64, I, I, I, V]
    l = la.descriptor()
    out = (C.c_uint64 * 6)()
    fn(l.las, l.stages, l.at, l.la_stage_count, l.use_at, l.is_valid, w, h, _buf(coords["dx"]), _buf(coords["dy"]),
       _buf(coords["center_x"]), _buf(coords["center_y"]), n_iter, iter_bytes, col_step, row_step, out)
    # refused2 / mismatches2: the same inputs through the step on step-shaped records (fs_la_step2.cuh)
    return dict(zip(("steps", "refused", "mismatches", "unusable", "refused2", "mismatches2"), (int(v) for v in out)))


def lockstep_la2_fuzz(count, seed=1):
    """la2::step (fs_la_step2.cuh, host build) against the oracle's reference-shaped LA step on synthetic inputs aimed at
    its guards (exponent gaps around 120..127, exact zeros, un-reduced mantissas, thresholds one ulp off).
    Returns {"cases", "accepted", "refused", "mismatches"}; mismatches must be 0."""
    global _lock
    if _lock is None:
        _lock = C.CDLL(LOCKSTEP_LIB)
    fn = _lock.lockstep_la2_fuzz
    fn.restype = None
    fn.argtypes = [C.c_uint64, C.c_uint64, C.c_void_p]
    out = (C.c_uint64 * 4)()
    fn(count, seed, out)
    return dict(zip(("cases", "accepted", "refused", "mismatches"), (int(v) for v in out)))


def lockstep_numeric_op(op: int, a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """The host build of the product's HDRFloat<float> / HDRFloatComplex<float> operations (fs_types.cuh) on operand arrays."""
    global _lock
    if _lock is None:
        _lock = C.CDLL(LOCKSTEP_LIB)
    fn = _lock.lockstep_numeric_op
    fn.restype = C.c_int
    fn.argtypes = [C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
    a = np.ascontiguousarray(a)
    b = np.ascontiguousarray(b)
    out = np.zeros_like(a)
    rc = fn(op, a.ctypes.data, b.ctypes.data, out.ctypes.data, a.shape[0])
    assert rc == 0, rc
    return out


def lockstep_quad_op(op: int, a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """The host build of the Quad<F> operations (fs_qd.cuh quad_selftest_op, ops 60-67 / 70-77) on operand arrays."""
    global _lock
    if _lock is None:
        _lock = C.CDLL(LOCKSTEP_LIB)
    fn = _lock.lockstep_quad_op
    fn.restype = C.c_int
    fn.argtypes = [C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
    a = np.ascontiguousarray(a)
    b = np.ascontiguousarray(b)
    out = np.zeros_like(a)
    rc = fn(op, a.ctypes.data, b.ctypes.data, out.ctypes.data, a.shape[0])
    assert rc == 0, rc
    return out


def quad_escape_counts(limb_bytes, coords, n_iter, X, Y, iter_bytes=4, threads=1):
    """The escape-time loop of Gpu4x32 (limb_bytes 4) / Gpu4x64 (8) -- fs_qd.cuh quad_escape_count, host build -- for the
    kernel pixels (X[i], Y[i]) (Y: the kernel's own, flipped row).  Returns the counts as uint64."""
    global _lock
    if _lock is None:
        _lock = C.CDLL(LOCKSTEP_LIB)
    fn = _lock.lockstep_quad_pixels
    fn.restype = C.c_int
    V = C.c_void_p
    fn.argtypes = [C.c_int, C.c_int, V, V, V, V, C.c_uint64, V, V, C.c_uint64, V, C.c_int]
    X = np.ascontiguousarray(X, dtype=np.int32)
    Y = np.ascontiguousarray(Y, dtype=np.int32)
    out = np.zeros(X.shape[0], np.uint64)
    rc = fn(limb_bytes, iter_bytes, _buf(coords["cx"]), _buf(coords["cy"]), _buf(coords["dx"]), _buf(coords["dy"]), n_iter,
            X.ctypes.data, Y.ctypes.data, X.shape[0], out.ctypes.data, threads)
    assert rc == 0, rc
    return out
