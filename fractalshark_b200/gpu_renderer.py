"""``GPURenderer`` -- host-side mirror of the reference class over the C-ABI.

Method names, argument meaning and error behaviour follow FractalSharkLib/GPU_Render.h:20-227: every
method returns the ``uint32_t`` status (0 = success, else ``cudaError_t`` or ``FractalSharkError``
10000+); render calls only enqueue; results are pulled with ``RenderCurrent``.  Template arguments of
the reference (``IterType``, ``T``, ``Mode``, ``PExtras``) are explicit keyword arguments here.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as N
from .algorithms import LAv2Mode, Numeric, PerturbExtras, RenderAlgorithm, traits

NB_THREADS_W = 16  # GPU_Render.h:116-120
NB_THREADS_H = 8


def _round_up(v: int, m: int) -> int:
    return (v + m - 1) // m * m


def _buf(b: bytes):
    return C.cast(C.create_string_buffer(b, len(b)), C.c_void_p)


class GPURenderer:
    def __init__(self, device: int = 0, devices=None):
        """``devices``: a list of device ids makes a device group (``fs_create_group``): one handle whose every call
        renders the frame on all of them, member i rendering the 4-row bands b % n == i; ids may repeat."""
        self._lib = N.gpu_lib()
        if devices is None:
            self._h = self._lib.fs_create(device)
        else:
            ids = (C.c_int32 * len(devices))(*devices)
            self._h = self._lib.fs_create_group(ids, len(devices))
        if not self._h:
            raise MemoryError("fs_create failed" if devices is None else f"fs_create_group({list(devices)}) failed")
        self._iter_bytes = 4
        self._keep = []  # host buffers borrowed by in-flight async copies
        self._cb = None

    def close(self):
        if getattr(self, "_h", None):
            self._lib.fs_destroy(self._h)
            self._h = None

    __del__ = close

    # ---- statics -------------------------------------------------------------------------------
    @staticmethod
    def TestCudaIsWorking() -> int:
        return int(N.gpu_lib().fs_test_cuda_is_working())

    @staticmethod
    def ConvertErrorToString(err: int) -> str:
        return N.gpu_lib().fs_convert_error_to_string(err).decode()

    # ---- lifecycle -----------------------------------------------------------------------------
    def InitializeMemory(self, w: int, h: int, antialiasing: int = 1, palette: np.ndarray | None = None,
                         palette_aux_depth: int = 0, palette_generation: int = 1, expected_reuse: bool = False,
                         iter_bytes: int = 4) -> int:
        """``w``/``h`` are the super-sampled sizes (screen size x antialiasing), GPU_Render.h:91-100."""
        if palette is None:
            palette = default_palette()
        palette = np.ascontiguousarray(palette, dtype=np.uint16).reshape(-1, 4)
        self._palette = palette
        self._iter_bytes = iter_bytes
        self._antialiasing = antialiasing
        return int(self._lib.fs_initialize_memory(self._h, iter_bytes, w, h, antialiasing,
                                                  palette.ctypes.data, palette.shape[0], palette_aux_depth,
                                                  palette_generation, int(expected_reuse)))

    def InitializePerturb(self, generation1: int, perturb1, generation2: int = 0, perturb2=None, la=None,
                          pextras: PerturbExtras | None = None) -> int:
        """``perturb1``/``perturb2`` are :class:`host_inputs.Orbit`, ``la`` a :class:`host_inputs.LaTable`.
        ``pextras`` defaults to the layout of ``perturb1`` (Disable, or SimpleCompression for ``Orbit.compress()``)."""
        if pextras is None:
            pextras = PerturbExtras(getattr(perturb1, "pextras", 0))
        d1 = perturb1.descriptor()
        d2 = perturb2.descriptor() if perturb2 is not None else None
        dl = la.descriptor() if la is not None else None
        # page-locked sources are read asynchronously (include/fs_gpu.h): keep them alive until the next upload
        self._keep = [perturb1, perturb2, la, d1, d2, dl]
        return int(self._lib.fs_initialize_perturb(
            self._h, self._iter_bytes, int(perturb1.numeric), int(pextras), generation1, C.byref(d1),
            int(perturb2.numeric) if perturb2 is not None else 0, generation2,
            C.byref(d2) if d2 is not None else None, C.byref(dl) if dl is not None else None))

    def ClearMemory(self) -> None:
        self._lib.fs_clear_memory(self._h)

    # ---- render calls --------------------------------------------------------------------------
    def Render(self, algorithm: RenderAlgorithm, coords: dict, n_iterations: int, iteration_precision: int = 1) -> int:
        t = traits(algorithm)
        return int(self._lib.fs_render(self._h, int(algorithm), int(t.numeric), _buf(coords["cx"]), _buf(coords["cy"]),
                                       _buf(coords["dx"]), _buf(coords["dy"]), n_iterations, iteration_precision))

    def RenderPerturbLAv2(self, algorithm: RenderAlgorithm, coords: dict, n_iterations: int) -> int:
        t = traits(algorithm)
        return int(self._lib.fs_render_perturb_lav2(
            self._h, int(algorithm), int(t.numeric), int(t.mode), int(t.pextras), _buf(coords["cx"]), _buf(coords["cy"]),
            _buf(coords["dx"]), _buf(coords["dy"]), _buf(coords["center_x"]), _buf(coords["center_y"]), n_iterations))

    def RenderPerturbLAv2Frames(self, algorithm: RenderAlgorithm, coords_list, n_iterations: int) -> int:
        """A zoom batch (``fs_render_perturb_lav2_frames``): one frame per entry of ``coords_list`` (dicts as
        ``View.coords`` returns, 1 to 64 of them), all with the uploaded orbit and LA table, in one launch.  Frame 0
        lands in the iteration buffer; ``SelectFrame(k)`` picks the frame ``RenderCurrent`` returns."""
        t = traits(algorithm)
        coords_list = list(coords_list)

        def cat(key):
            return _buf(b"".join(c[key] for c in coords_list)) if coords_list else None
        return int(self._lib.fs_render_perturb_lav2_frames(
            self._h, int(algorithm), int(t.numeric), int(t.mode), int(t.pextras), len(coords_list), cat("cx"), cat("cy"),
            cat("dx"), cat("dy"), cat("center_x"), cat("center_y"), n_iterations))

    def RenderPerturbLAv2ExpMap(self, algorithm: RenderAlgorithm, expmap: dict, n_iterations: int) -> int:
        """An exponential map (``fs_render_perturb_lav2_expmap``) around the uploaded orbit's reference point: ``expmap``
        is what ``View.exp_map`` returns, with as many radii as the initialized height and as many directions as the
        width.  One frame; every cell is the cell a single render of its own dc gives."""
        t = traits(algorithm)
        return int(self._lib.fs_render_perturb_lav2_expmap(
            self._h, int(algorithm), int(t.numeric), int(t.mode), int(t.pextras), _buf(expmap["radius"]),
            _buf(expmap["dir_x"]), _buf(expmap["dir_y"]), n_iterations))

    def SelectFrame(self, k: int) -> int:
        """Frame of the last render that ``RenderCurrent`` / ``RenderCurrentShard`` / ``DeviceIterBuffer`` read."""
        return int(self._lib.fs_select_frame(self._h, k))

    def RenderPerturbBLA(self, algorithm: RenderAlgorithm, perturb, blas, coords: dict, n_iterations: int,
                         iteration_precision: int = 1) -> int:
        """``perturb`` is a :class:`host_inputs.Orbit`, ``blas`` a :class:`host_inputs.BlaTable`; both are uploaded
        by this call, as in the reference (GPU_Render.cu:1440-1570)."""
        t = traits(algorithm)
        d, b = perturb.descriptor(), blas.descriptor()
        return int(self._lib.fs_render_perturb_bla(
            self._h, int(algorithm), int(t.numeric), C.byref(d), C.byref(b), _buf(coords["cx"]), _buf(coords["cy"]),
            _buf(coords["dx"]), _buf(coords["dy"]), _buf(coords["center_x"]), _buf(coords["center_y"]), n_iterations,
            iteration_precision))

    def RenderPerturbBLAScaled(self, algorithm: RenderAlgorithm, double_perturb, float_perturb, coords: dict,
                               n_iterations: int, iteration_precision: int = 1) -> int:
        """``double_perturb`` / ``float_perturb``: :class:`host_inputs.Orbit` objects in the ``Bad`` layout
        (``Orbit.with_bad()`` / ``Orbit.with_bad(to_float=True)``), both uploaded by this call as in the
        reference (GPU_Render.cu:1302-1377)."""
        t = traits(algorithm)
        d, f = double_perturb.descriptor(), float_perturb.descriptor()
        return int(self._lib.fs_render_perturb_bla_scaled(
            self._h, int(algorithm), int(t.numeric), C.byref(d), C.byref(f), _buf(coords["cx"]), _buf(coords["cy"]),
            _buf(coords["dx"]), _buf(coords["dy"]), _buf(coords["center_x"]), _buf(coords["center_y"]), n_iterations,
            iteration_precision))

    # ---- results -------------------------------------------------------------------------------
    def buffer_shape(self) -> tuple[int, int]:
        w, h = self.GetWidth(), self.GetHeight()
        return _round_up(h, NB_THREADS_H), _round_up(w, NB_THREADS_W)

    def RenderCurrent(self, n_iterations: int, want_iters: bool = True, want_colors: bool = False,
                      progressive: bool = False, iters_out=None):
        """Returns ``(status, iters, colors, reduction)``; arrays are padded like the reference's buffers.
        ``iters_out``: caller-owned host array of the padded shape to receive the iteration buffer (e.g. pinned
        memory); the C-ABI borrows whatever pointer it is given, as the reference does (GPU_Render.cu:1768-1788)."""
        hp, wp = self.buffer_shape()
        dt = np.uint32 if self._iter_bytes == 4 else np.uint64
        if iters_out is not None:
            assert iters_out.shape == (hp, wp) and iters_out.dtype == dt and iters_out.flags["C_CONTIGUOUS"]
            iters, want_iters = iters_out, True
        else:
            iters = np.empty((hp, wp), dtype=dt) if want_iters else None
        colors = None
        if want_colors:
            aa = self._aa()
            colors = np.empty((_round_up(self.GetHeight() // aa, NB_THREADS_H),
                               _round_up(self.GetWidth() // aa, NB_THREADS_W), 4), dtype=np.uint16)
        red = N.FsReduction()
        rc = int(self._lib.fs_render_current(self._h, n_iterations, iters.ctypes.data if want_iters else None,
                                             colors.ctypes.data if want_colors else None, C.byref(red),
                                             int(progressive)))
        if rc == 0:
            rc = self.SyncDisplayStream() if progressive else self.SyncComputeStream()
        return rc, iters, colors, {"Min": int(red.Min), "Max": int(red.Max), "Sum": int(red.Sum)}

    def RenderCurrentShard(self, n_iterations: int, iters_out, progressive: bool = False, colors_out=None):
        """Multi-GPU form: copies only the 4-row bands this shard rendered (``SetShard``) into the same positions of
        ``iters_out`` -- a caller-owned whole-frame host array, typically one shared-memory frame every rank writes
        into -- and leaves the other rows untouched; ``colors_out`` (whole-frame colour array, shape of
        ``RenderCurrent``'s) receives the Color16 cells of those bands the same way.
        Returns ``(status, reduction over this shard's cells)``."""
        hp, wp = self.buffer_shape()
        dt = np.uint32 if self._iter_bytes == 4 else np.uint64
        assert iters_out.shape == (hp, wp) and iters_out.dtype == dt and iters_out.flags["C_CONTIGUOUS"]
        if colors_out is not None:
            assert colors_out.dtype == np.uint16 and colors_out.flags["C_CONTIGUOUS"]
        red = N.FsReduction()
        rc = int(self._lib.fs_render_current_shard(self._h, n_iterations, iters_out.ctypes.data,
                                                   colors_out.ctypes.data if colors_out is not None else None,
                                                   C.byref(red), int(progressive)))
        if rc == 0:
            rc = self.SyncDisplayStream() if progressive else self.SyncComputeStream()
        return rc, {"Min": int(red.Min), "Max": int(red.Max), "Sum": int(red.Sum)}

    def SetResultSink(self, frame) -> int:
        """``frame``: whole-frame host array of the padded shape (page-locked, or registered by the call) the LAv2
        kernels stream finished pixels into while they render; ``RenderCurrent(iters_out=frame)`` /
        ``RenderCurrentShard(n, frame)`` then skip their copy.  ``None`` removes the sink."""
        if frame is None:
            self._sink = None
            return int(self._lib.fs_set_result_sink(self._h, None, 0))
        hp, wp = self.buffer_shape()
        dt = np.uint32 if self._iter_bytes == 4 else np.uint64
        assert frame.shape == (hp, wp) and frame.dtype == dt and frame.flags["C_CONTIGUOUS"]
        self._sink = frame  # keep the mapping alive as long as the device may write into it
        return int(self._lib.fs_set_result_sink(self._h, frame.ctypes.data, frame.nbytes))

    def _aa(self) -> int:
        return getattr(self, "_antialiasing", 1)

    def SyncComputeStream(self) -> int:
        return int(self._lib.fs_sync_compute_stream(self._h))

    def SyncDisplayStream(self) -> int:
        return int(self._lib.fs_sync_display_stream(self._h))

    def QueryComputeStream(self) -> int:
        return int(self._lib.fs_query_compute_stream(self._h))

    def EnqueueComputeDoneCallback(self, fn) -> int:
        self._cb = N.DONE_CALLBACK(lambda _user: fn())
        return int(self._lib.fs_enqueue_compute_done_callback(self._h, self._cb, None))

    def GetWidth(self) -> int:
        return int(self._lib.fs_get_width(self._h))

    def GetHeight(self) -> int:
        return int(self._lib.fs_get_height(self._h))

    # ---- additions (measurement / sharding) ----------------------------------------------------
    def SetShard(self, shard_count: int, shard_index: int) -> int:
        """Render only the 4-row tile bands b with b % shard_count == shard_index (multi-GPU sharding)."""
        return int(self._lib.fs_set_shard(self._h, shard_count, shard_index))

    @staticmethod
    def MeasureFp32IssuePeak(device: int = 0) -> float:
        v = C.c_double(0)
        rc = N.gpu_lib().fs_measure_fp32_issue_peak(device, C.byref(v))
        if rc:
            raise RuntimeError(GPURenderer.ConvertErrorToString(rc))
        return float(v.value)

    @staticmethod
    def MeasureFp64IssuePeak(device: int = 0) -> float:
        v = C.c_double(0)
        rc = N.gpu_lib().fs_measure_fp64_issue_peak(device, C.byref(v))
        if rc:
            raise RuntimeError(GPURenderer.ConvertErrorToString(rc))
        return float(v.value)

    def LastRenderMs(self) -> float:
        ms = C.c_float(0)
        rc = self._lib.fs_last_render_ms(self._h, C.byref(ms))
        if rc:
            raise RuntimeError(self.ConvertErrorToString(rc))
        return float(ms.value)

    def EnableStepCounter(self, enable: bool = True) -> int:
        return int(self._lib.fs_enable_step_counter(self._h, int(enable)))

    def ReadStepCounters(self) -> dict:
        """Executed steps of the renders since EnableStepCounter(True), split by kind."""
        v = (C.c_uint64 * 3)()
        rc = self._lib.fs_read_step_counters(self._h, v)
        if rc:
            raise RuntimeError(self.ConvertErrorToString(rc))
        total, at, la = int(v[0]), int(v[1]), int(v[2])
        return {"total": total, "at": at, "la": la, "perturbation": total - at - la}

    def ReadStepCounter(self) -> int:
        v = C.c_uint64(0)
        rc = self._lib.fs_read_step_counter(self._h, C.byref(v))
        if rc:
            raise RuntimeError(self.ConvertErrorToString(rc))
        return int(v.value)

    def SetScaledSteps(self, enable: bool = True) -> int:
        """A/B switch of the HDRx32 perturbation loop (same results either way); applies to the next upload."""
        return int(self._lib.fs_set_scaled_steps(self._h, int(enable)))

    def SetSplitAt(self, enable: bool = True) -> int:
        """A/B switch: AT shortcut of the HDRx32 LAv2 path in its own launch (default) or fused (same results)."""
        return int(self._lib.fs_set_split_at(self._h, int(enable)))

    def SetAtCycleDetection(self, enable: bool = True) -> int:
        """A/B switch of the AT shortcut: skip whole periods once the passes repeat exactly (default) or execute every
        pass like the reference (same results)."""
        return int(self._lib.fs_set_at_cycle_detection(self._h, int(enable)))

    def SetLaStep2(self, enable: bool = True) -> int:
        """A/B switch of the HDRx32 / 32-bit LA walk: step-shaped records (default) or reference-shaped (same results)."""
        return int(self._lib.fs_set_la_step2(self._h, int(enable)))

    def SetPoolKernel(self, enable: bool = True) -> int:
        """A/B switch of the HDRx32 LAv2 path: lane-refill kernel (default) or one tile per warp (same results)."""
        return int(self._lib.fs_set_pool_kernel(self._h, int(enable)))

    def DeviceCount(self) -> int:
        """1 for a single renderer, n for a device group."""
        return int(self._lib.fs_device_count(self._h))

    def DeviceIterBuffer(self) -> int:
        return int(self._lib.fs_device_iter_buffer(self._h) or 0)

    def KernelLaunchCount(self) -> int:
        return int(self._lib.fs_kernel_launch_count(self._h))


def default_palette(n: int = 4096) -> np.ndarray:
    """A deterministic RGBA16 palette (the reference's palettes are UI data, FractalPalette.cpp)."""
    i = np.arange(n, dtype=np.float64)
    pal = np.empty((n, 4), dtype=np.uint16)
    pal[:, 0] = (32767.5 * (1 + np.sin(i * 0.0123))).astype(np.uint16)
    pal[:, 1] = (32767.5 * (1 + np.sin(i * 0.0211 + 2.0))).astype(np.uint16)
    pal[:, 2] = (32767.5 * (1 + np.sin(i * 0.0337 + 4.0))).astype(np.uint16)
    pal[:, 3] = 65535
    return pal
