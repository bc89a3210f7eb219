"""Inputs of the render path: view coordinates, reference orbit, LA table (libfshost.so).

These are what the reference's host code hands to ``GPURenderer`` (coordinates: Fractal.cpp:1789-1844,
2831-2840; orbit: RefOrbitCalc.cpp:415-647; LA table: LAReference.cpp:28-1074), in the reference's
own memory layouts.  They are inputs -- not part of the timed GPU path.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as N
from .algorithms import Numeric

# bytes of one coordinate POD per numeric tag (SURVEY.md section 2.2)
POD_BYTES = {Numeric.F32: 4, Numeric.F64: 8, Numeric.X2_32: 8, Numeric.HDR32: 8, Numeric.HDR64: 16,
             Numeric.HDR2X32: 12, Numeric.X2_64: 16, Numeric.X4_32: 16, Numeric.X4_64: 32}


class View:
    """A view rectangle at a given super-sampled size (PointZoomBBConverter + SquareAspectRatio)."""

    def __init__(self, min_x: str, min_y: str, max_x: str, max_y: str, width: int, height: int,
                 antialiasing: int = 1, square_aspect: bool = True):
        self._lib = N.host_lib()
        self.width, self.height, self.antialiasing = width, height, antialiasing
        self._h = self._lib.fsh_view_create(min_x.encode(), min_y.encode(), max_x.encode(), max_y.encode(),
                                            width, height, antialiasing, int(square_aspect))
        if not self._h:
            raise ValueError("could not parse view coordinates")

    def __del__(self):
        if getattr(self, "_h", None):
            self._lib.fsh_view_destroy(self._h)
            self._h = None

    def zoomed(self, scale: str) -> "View":
        """A frame of a zoom sequence around this view's centre: the same centre, precision, size and antialiasing,
        bounds = centre -/+ this view's half-extents x ``scale`` (a decimal string; "2" shows twice the extent).  Such
        frames share this view's reference orbit and LA table (``GPURenderer.RenderPerturbLAv2Frames``)."""
        h = self._lib.fsh_view_zoom(self._h, scale.encode())
        if not h:
            raise ValueError(f"bad zoom scale {scale!r}")
        z = View.__new__(View)
        z._lib, z._h = self._lib, h
        z.width, z.height, z.antialiasing = self.width, self.height, self.antialiasing
        return z

    @property
    def precision_bits(self) -> int:
        return int(self._lib.fsh_view_precision_bits(self._h))

    def coords(self, numeric: Numeric, direct: bool = False) -> dict:
        """cx, cy, dx, dy, centerX, centerY as raw PODs of ``numeric`` (FillGpuCoords / FillCoord).
        ``direct`` selects the MattDblflt flavour of the 2x32 POD that the direct kernel Gpu2x32 is fed
        (Fractal.cpp:1805-1810) instead of the CudaDblflt one of the perturbation kernels (:1820-1824)."""
        nb = POD_BYTES[Numeric(numeric)]
        bufs = {k: C.create_string_buffer(nb) for k in ("cx", "cy", "dx", "dy", "center_x", "center_y")}
        tag = 0x102 if (direct and Numeric(numeric) == Numeric.X2_32) else int(numeric)
        rc = self._lib.fsh_view_coords(self._h, tag, *[C.cast(b, C.c_void_p) for b in bufs.values()])
        if rc != 0:
            raise ValueError(f"numeric {numeric!r} not supported by the input generator")
        return {k: bytes(b.raw) for k, b in bufs.items()}

    def exp_map(self, numeric: Numeric, rows: int) -> dict:
        """Tables of an exponential map around this view's centre (``fsh_view_expmap``) for
        ``GPURenderer.RenderPerturbLAv2ExpMap``, W = the super-sampled width: ``dir_x`` / ``dir_y`` (W PODs of ``numeric``
        each) = cos / sin of the angle 2 pi (X + 1/2) / W, ``radius`` (``rows`` PODs) = radius0 * exp(-2 pi Y / W) with
        radius0 = the half-diagonal * exp(-pi / W), row 0 outermost; ``log2_radius0`` and ``log2_row_step`` as floats.
        A zoom by Z needs W ln Z / (2 pi) rows."""
        nb = POD_BYTES[Numeric(numeric)]
        w = self.width * self.antialiasing
        radius, dir_x, dir_y = C.create_string_buffer(nb * rows), C.create_string_buffer(nb * w), C.create_string_buffer(nb * w)
        l0, step = C.c_double(), C.c_double()
        rc = self._lib.fsh_view_expmap(self._h, int(numeric), int(rows), C.cast(radius, C.c_void_p),
                                       C.cast(dir_x, C.c_void_p), C.cast(dir_y, C.c_void_p), C.byref(l0), C.byref(step))
        if rc != 0:
            raise ValueError(f"numeric {numeric!r} not supported by the exp-map builder")
        return {"radius": bytes(radius.raw), "dir_x": bytes(dir_x.raw), "dir_y": bytes(dir_y.raw),
                "log2_radius0": l0.value, "log2_row_step": step.value}


class Orbit:
    """High-precision reference orbit stored as GPUReferenceIter<T, Disable>[count]."""

    def __init__(self, view: View, numeric: Numeric, max_iterations: int, periodicity: bool = True):
        self._lib = N.host_lib()
        self.numeric = Numeric(numeric)
        self._view = view
        self._h = self._lib.fsh_orbit_compute(view._h, int(numeric), int(max_iterations), int(periodicity))
        if not self._h:
            raise ValueError(f"numeric {numeric!r} not supported by the input generator")
        self.count = int(self._lib.fsh_orbit_count(self._h))
        self.period = int(self._lib.fsh_orbit_period(self._h))
        self.elem_bytes = int(self._lib.fsh_orbit_elem_bytes(self._h))
        self.uncompressed_count = self.count

    pextras = 0  # PerturbExtras of the element layout (0 Disable, 1 Bad, 2 SimpleCompression)

    @classmethod
    def _wrap(cls, view, numeric, handle):
        o = cls.__new__(cls)
        o._lib = N.host_lib()
        o.numeric = Numeric(numeric)
        o._view = view
        o._h = handle
        o.count = int(o._lib.fsh_orbit_count(handle))
        o.period = int(o._lib.fsh_orbit_period(handle))
        o.elem_bytes = int(o._lib.fsh_orbit_elem_bytes(handle))
        o.uncompressed_count = int(o._lib.fsh_orbit_uncompressed_count(handle))
        return o

    def compress(self, error_exp: int = 20) -> "Orbit":
        """``GPUReferenceIter<T, PerturbExtras::SimpleCompression>[]``: the waypoints RefOrbitCompressor keeps for a
        relative replay error of 10^-error_exp (default 20, Fractal.h:138-141).  ``count`` is then the compressed
        size, ``uncompressed_count`` the number of orbit entries; LaTable() of such an orbit is built from its host
        replay with the reference's coarser period divisor."""
        h = self._lib.fsh_orbit_compress(self._h, int(error_exp))
        if not h:
            raise ValueError("orbit cannot be compressed")
        o = Orbit._wrap(self._view, self.numeric, h)
        o.pextras = 2
        return o

    def with_bad(self, to_float: bool = False) -> "Orbit":
        """``GPUReferenceIter<T, PerturbExtras::Bad>[count]`` for the scaled kernel: the same orbit with the
        underflow flag of RefOrbitCalc.cpp:550-562, or (``to_float``) its binary32 copy
        (RefOrbitCalc::CopyUsefulPerturbationResults)."""
        h = self._lib.fsh_orbit_with_bad(self._h, int(to_float))
        if not h:
            raise ValueError("Bad-flagged orbits exist for double and HDRFloat<float> only")
        return Orbit._wrap(self._view, Numeric.F32 if to_float else self.numeric, h)

    def __del__(self):
        if getattr(self, "_h", None):
            self._lib.fsh_orbit_destroy(self._h)
            self._h = None

    @property
    def data_ptr(self) -> int:
        return int(self._lib.fsh_orbit_data(self._h))

    def as_numpy(self) -> np.ndarray:
        buf = (C.c_ubyte * (self.count * self.elem_bytes)).from_address(self.data_ptr)
        return np.frombuffer(buf, dtype=np.uint8).reshape(self.count, self.elem_bytes)

    def descriptor(self) -> N.FsOrbit:
        return N.FsOrbit(self.data_ptr, self.count, self.uncompressed_count, self.period,
                         int(self._lib.fsh_orbit_x_low(self._h)), int(self._lib.fsh_orbit_y_low(self._h)))


class LaTable:
    """LAv2 table (LAInfoDeep[], LAStageInfo[], ATInfo) built from an orbit."""

    def __init__(self, orbit: Orbit, iter_bytes: int):
        self._lib = N.host_lib()
        self._orbit = orbit
        self.iter_bytes = iter_bytes
        self._h = self._lib.fsh_la_build(orbit._h, iter_bytes)
        if not self._h:
            raise ValueError("LA build failed")
        L = self._lib
        self.num_las = int(L.fsh_la_num_las(self._h))
        self.num_stages = int(L.fsh_la_num_stages(self._h))
        self.stage_count = int(L.fsh_la_stage_count(self._h))
        self.use_at = bool(L.fsh_la_use_at(self._h))
        self.is_valid = bool(L.fsh_la_is_valid(self._h))
        self.at_bytes = int(L.fsh_la_at_bytes(self._h))

    def __del__(self):
        if getattr(self, "_h", None):
            self._lib.fsh_la_destroy(self._h)
            self._h = None

    def descriptor(self) -> N.FsLaReference:
        L = self._lib
        return N.FsLaReference(int(L.fsh_la_las(self._h) or 0), self.num_las, int(L.fsh_la_stages(self._h) or 0),
                               self.num_stages, int(L.fsh_la_at(self._h) or 0), self.stage_count,
                               int(self.use_at), int(self.is_valid))

    def las_numpy(self) -> np.ndarray:
        if self.num_las == 0:
            return np.zeros((0, 0), np.uint8)
        ptr = int(self._lib.fsh_la_las(self._h))
        eb = self.las_elem_bytes
        buf = (C.c_ubyte * (self.num_las * eb)).from_address(ptr)
        return np.frombuffer(buf, dtype=np.uint8).reshape(self.num_las, eb)

    @property
    def las_elem_bytes(self) -> int:
        table = {(Numeric.HDR32, 4): 68, (Numeric.HDR32, 8): 80, (Numeric.F32, 4): 44, (Numeric.F32, 8): 56,
                 (Numeric.F64, 4): 80, (Numeric.F64, 8): 88, (Numeric.HDR64, 4): 128, (Numeric.HDR64, 8): 136,
                 (Numeric.X2_32, 4): 80, (Numeric.X2_32, 8): 88, (Numeric.HDR2X32, 4): 104, (Numeric.HDR2X32, 8): 112}
        return table[(self._orbit.numeric, self.iter_bytes)]

    def stages_numpy(self) -> np.ndarray:
        ptr = int(self._lib.fsh_la_stages(self._h))
        dt = np.uint32 if self.iter_bytes == 4 else np.uint64
        buf = (C.c_ubyte * (self.num_stages * 2 * self.iter_bytes)).from_address(ptr)
        return np.frombuffer(buf, dtype=dt).reshape(self.num_stages, 2)


class BlaTable:
    """BLA table (``BLAS<IterType, T>::Init(count, MaxRadius)``, BLAS.cpp:212-254) built from an orbit:
    per-level arrays of ``BLA<T>`` records in the reference layout (BLA.h:7-14)."""

    def __init__(self, orbit: Orbit):
        self._lib = N.host_lib()
        self._orbit = orbit
        self._h = self._lib.fsh_blas_build(orbit._h)
        if not self._h:
            raise ValueError("BLA build failed")
        L = self._lib
        self.num_levels = int(L.fsh_blas_num_levels(self._h))
        self.lm2 = int(L.fsh_blas_lm2(self._h))
        self.elem_bytes = int(L.fsh_blas_elem_bytes(self._h))
        counts = L.fsh_blas_level_counts(self._h)
        self.level_counts = [int(counts[i]) for i in range(self.num_levels)]

    def __del__(self):
        if getattr(self, "_h", None):
            self._lib.fsh_blas_destroy(self._h)
            self._h = None

    def descriptor(self) -> N.FsBlas:
        L = self._lib
        return N.FsBlas(L.fsh_blas_levels(self._h), L.fsh_blas_level_counts(self._h), self.num_levels, 2, self.lm2)

    def level_numpy(self, level: int) -> np.ndarray:
        n = self.level_counts[level]
        if n == 0:
            return np.zeros((0, self.elem_bytes), np.uint8)
        ptr = self._lib.fsh_blas_levels(self._h)[level]
        buf = (C.c_ubyte * (n * self.elem_bytes)).from_address(ptr)
        return np.frombuffer(buf, dtype=np.uint8).reshape(n, self.elem_bytes)


class ReplicatedInputs:
    """Orbit + LA table + coordinates as plain byte blobs, the form in which they travel between ranks
    (``pack`` on the rank that produced them, ``unpack`` on the receivers).  The unpacked object offers the
    ``descriptor()`` / size attributes of :class:`Orbit` and :class:`LaTable`, so the renderer uploads straight from
    the received host buffers; nothing is recomputed on the receiving rank."""

    class _Orbit:
        pextras = 0

        def __init__(self, meta, data: np.ndarray, x_low: np.ndarray, y_low: np.ndarray):
            self.numeric = Numeric(meta["numeric"])
            self.count = meta["count"]
            self.uncompressed_count = meta["uncompressed_count"]
            self.period = meta["period"]
            self.elem_bytes = meta["elem_bytes"]
            self.pextras = meta["pextras"]
            self._data, self._x, self._y = data, x_low, y_low

        def as_numpy(self):
            return self._data.reshape(self.count, self.elem_bytes)

        def descriptor(self):
            return N.FsOrbit(self._data.ctypes.data, self.count, self.uncompressed_count, self.period,
                             self._x.ctypes.data, self._y.ctypes.data)

    class _La:
        def __init__(self, meta, las: np.ndarray, stages: np.ndarray, at: np.ndarray):
            self.num_las, self.num_stages, self.stage_count = meta["num_las"], meta["num_stages"], meta["stage_count"]
            self.use_at, self.is_valid = meta["use_at"], meta["is_valid"]
            self.las_elem_bytes, self.at_bytes, self.iter_bytes = meta["las_elem_bytes"], meta["at_bytes"], meta["iter_bytes"]
            self._las, self._stages, self._at = las, stages, at

        def descriptor(self):
            return N.FsLaReference(self._las.ctypes.data if self.num_las else None, self.num_las,
                                   self._stages.ctypes.data if self.num_stages else None, self.num_stages,
                                   self._at.ctypes.data if self.at_bytes else None, self.stage_count,
                                   int(self.use_at), int(self.is_valid))

    @staticmethod
    def pack(coords: dict, orbit: "Orbit", la: "LaTable", n_iter: int):
        """-> (meta dict, [uint8 arrays]) ; the arrays are copies, safe to hand to a collective."""
        lib = orbit._lib
        def grab(ptr, nbytes):
            if not ptr or not nbytes:
                return np.zeros(0, np.uint8)
            return np.frombuffer((C.c_ubyte * nbytes).from_address(ptr), dtype=np.uint8).copy()
        pod = POD_BYTES[orbit.numeric]
        blobs = [grab(orbit.data_ptr, orbit.count * orbit.elem_bytes),
                 grab(int(lib.fsh_orbit_x_low(orbit._h)), pod), grab(int(lib.fsh_orbit_y_low(orbit._h)), pod),
                 grab(int(lib.fsh_la_las(la._h) or 0), la.num_las * la.las_elem_bytes),
                 grab(int(lib.fsh_la_stages(la._h) or 0), la.num_stages * 2 * la.iter_bytes),
                 grab(int(lib.fsh_la_at(la._h) or 0), la.at_bytes)]
        meta = {"numeric": int(orbit.numeric), "count": orbit.count, "uncompressed_count": orbit.uncompressed_count,
                "period": orbit.period, "elem_bytes": orbit.elem_bytes, "pextras": int(orbit.pextras),
                "num_las": la.num_las, "num_stages": la.num_stages, "stage_count": la.stage_count,
                "use_at": bool(la.use_at), "is_valid": bool(la.is_valid), "las_elem_bytes": la.las_elem_bytes,
                "at_bytes": la.at_bytes, "iter_bytes": la.iter_bytes, "n_iter": int(n_iter),
                "coords": {k: bytes(v) for k, v in coords.items()}, "sizes": [int(b.size) for b in blobs]}
        return meta, blobs

    @staticmethod
    def unpack(meta: dict, blobs):
        """-> (coords, orbit-like, la-like, n_iter) from what ``pack`` produced."""
        o = ReplicatedInputs._Orbit(meta, blobs[0], blobs[1], blobs[2])
        l = ReplicatedInputs._La(meta, blobs[3], blobs[4], blobs[5])
        return dict(meta["coords"]), o, l, meta["n_iter"]
