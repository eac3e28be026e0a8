"""ctypes binding of libcwipc_util_cuda, mirroring the part of the reference's python/cwipc/util.py
that touches the filter hot path: same names, same argument meaning, same error behaviour
(ref: python/cwipc/util.py:260-300 point types, :368-553 signatures, :573-740 wrapper class,
:1135-1330 module functions).

The unchanged reference binding can load this library too (install lib/libcwipc_util.so on
LD_LIBRARY_PATH / CWIPC_LIBRARY_DIR, or call cwipc.util.cwipc_util_dll_load(<abs path>) first);
this module exists so that the repo's tests and bench run on a GPU box where /root/reference is absent.

There is no CPU fallback: if the CUDA library is missing or no device is present, calls fail loudly.
"""
from __future__ import annotations

import ctypes
import os
from collections.abc import Mapping
from typing import Any, Iterable, List, Optional, Sequence, Union

import numpy

__all__ = [
    "CWIPC_API_VERSION", "CWIPC_FLAGS_BINARY", "CwipcError",
    "CWIPC_LOG_LEVEL_NONE", "CWIPC_LOG_LEVEL_ERROR", "CWIPC_LOG_LEVEL_WARNING", "CWIPC_LOG_LEVEL_TRACE", "CWIPC_LOG_LEVEL_DEBUG",
    "cwipc_point", "cwipc_point_array", "cwipc_point_numpy_dtype", "cwipc_pointcloud_wrapper", "cwipc_activesource_wrapper",
    "cwipc_util_dll_load", "cwipc_get_version", "cwipc_log_configure", "cwipc_dangling_allocations",
    "cwipc_read", "cwipc_write", "cwipc_read_debugdump", "cwipc_write_debugdump",
    "cwipc_from_points", "cwipc_from_numpy_array", "cwipc_from_numpy_matrix", "cwipc_from_packet", "cwipc_synthetic",
    "cwipc_downsample", "cwipc_remove_outliers", "cwipc_tilefilter", "cwipc_tilemap", "cwipc_colormap", "cwipc_crop",
    "cwipc_join", "cwipc_join_multi", "cwipc_tilefilter_masked", "cwipc_downsample_pertile", "cwipc_transform",
    "cuda_device_count", "cuda_set_device", "cuda_synchronize", "cuda_kernel_launches",
]

CWIPC_API_VERSION = 0x20260129
CWIPC_FLAGS_BINARY = 1
CWIPC_LOG_LEVEL_NONE, CWIPC_LOG_LEVEL_ERROR, CWIPC_LOG_LEVEL_WARNING, CWIPC_LOG_LEVEL_TRACE, CWIPC_LOG_LEVEL_DEBUG = 0, 1, 2, 3, 4


class CwipcError(RuntimeError):
    pass


class cwipc_point(ctypes.Structure):
    """x,y,z float coordinates, r,g,b colour 0..255, tile (8 bit).  16 bytes, the HBM layout."""
    _fields_ = [("x", ctypes.c_float), ("y", ctypes.c_float), ("z", ctypes.c_float),
                ("r", ctypes.c_ubyte), ("g", ctypes.c_ubyte), ("b", ctypes.c_ubyte), ("tile", ctypes.c_ubyte)]

    def __eq__(self, other: Any) -> bool:
        return isinstance(other, cwipc_point) and all(getattr(self, f[0]) == getattr(other, f[0]) for f in self._fields_)

    def __ne__(self, other: Any) -> bool:
        return not self.__eq__(other)


cwipc_point_numpy_dtype = numpy.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("r", "u1"), ("g", "u1"), ("b", "u1"), ("tile", "u1")])
assert cwipc_point_numpy_dtype.itemsize == ctypes.sizeof(cwipc_point) == 16


def cwipc_point_array(*, count: Optional[int] = None, values: Any = None) -> ctypes.Array:
    """Create an array of cwipc_point from a count, a sequence of 7-tuples, or a bytes-like buffer."""
    if count is None:
        count = len(values) if values is not None else 0
    atype = cwipc_point * count
    if values is None:
        return atype()
    if isinstance(values, (bytes, bytearray, memoryview)):
        if isinstance(values, bytearray):
            return atype.from_buffer(values)
        return atype.from_buffer_copy(values)
    return atype(*[v if isinstance(v, cwipc_point) else cwipc_point(*v) for v in values])


class _p(ctypes.c_void_p):
    pass


class cwipc_pointcloud_p(_p):
    pass


class cwipc_source_p(_p):
    pass


_LOG_CALLBACK = ctypes.CFUNCTYPE(None, ctypes.c_int, ctypes.c_char_p)
_dll: Optional[ctypes.CDLL] = None
_log_callback_ref = None


def _default_library_path() -> str:
    here = os.path.dirname(os.path.abspath(__file__))
    return os.path.join(here, "lib", "libcwipc_util_cuda.so")


def cwipc_util_dll_load(libname: Optional[str] = None) -> ctypes.CDLL:
    """Load libcwipc_util_cuda and declare the signatures (ref: python/cwipc/util.py:368-553)."""
    global _dll
    if _dll is not None:
        return _dll
    path = libname or os.environ.get("CWIPC_CUDA_LIBRARY") or _default_library_path()
    if not os.path.exists(path) and not libname and not os.environ.get("CWIPC_CUDA_LIBRARY"):
        # a fresh checkout (the .so is not in the history): build it in-tree with nvcc; this is still the CUDA library or nothing
        try:
            from . import build as _build
            _build.build_library()
        except Exception as e:  # pragma: no cover
            raise RuntimeError(f"libcwipc_util_cuda not found at {path} and building it failed: {e}") from e
    if not os.path.exists(path):
        raise RuntimeError(f"libcwipc_util_cuda not found at {path}: build it with `python -m cwipc_util_b200.build` (there is no CPU fallback)")
    d = ctypes.CDLL(path)
    c_err = ctypes.POINTER(ctypes.c_char_p)
    sigs = {
        "cwipc_get_version": ([], ctypes.c_char_p),
        "cwipc_log_configure": ([ctypes.c_int, _LOG_CALLBACK], None),
        "_cwipc_log_emit": ([ctypes.c_int, ctypes.c_char_p, ctypes.c_char_p], None),
        "cwipc_dangling_allocations": ([ctypes.c_bool], ctypes.c_int),
        "cwipc_read": ([ctypes.c_char_p, ctypes.c_ulonglong, c_err, ctypes.c_ulonglong], cwipc_pointcloud_p),
        "cwipc_write": ([ctypes.c_char_p, cwipc_pointcloud_p, c_err], ctypes.c_int),
        "cwipc_write_ext": ([ctypes.c_char_p, cwipc_pointcloud_p, ctypes.c_int, c_err], ctypes.c_int),
        "cwipc_from_points": ([ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_ulonglong, c_err, ctypes.c_ulonglong], cwipc_pointcloud_p),
        "cwipc_cuda_from_points_async": ([ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_ulonglong, c_err, ctypes.c_ulonglong], cwipc_pointcloud_p),
        "cwipc_from_packet": ([ctypes.c_void_p, ctypes.c_size_t, c_err, ctypes.c_ulonglong], cwipc_pointcloud_p),
        "cwipc_read_debugdump": ([ctypes.c_char_p, c_err, ctypes.c_ulonglong], cwipc_pointcloud_p),
        "cwipc_write_debugdump": ([ctypes.c_char_p, cwipc_pointcloud_p, c_err], ctypes.c_int),
        "cwipc_pointcloud_free": ([cwipc_pointcloud_p], None),
        "cwipc_pointcloud__shallowcopy": ([cwipc_pointcloud_p], cwipc_pointcloud_p),
        "cwipc_pointcloud_timestamp": ([cwipc_pointcloud_p], ctypes.c_ulonglong),
        "cwipc_pointcloud_cellsize": ([cwipc_pointcloud_p], ctypes.c_float),
        "cwipc_pointcloud__set_cellsize": ([cwipc_pointcloud_p, ctypes.c_float], None),
        "cwipc_pointcloud__set_timestamp": ([cwipc_pointcloud_p, ctypes.c_ulonglong], None),
        "cwipc_pointcloud_count": ([cwipc_pointcloud_p], ctypes.c_int),
        "cwipc_pointcloud_get_uncompressed_size": ([cwipc_pointcloud_p], ctypes.c_size_t),
        "cwipc_pointcloud_copy_uncompressed": ([cwipc_pointcloud_p, ctypes.c_void_p, ctypes.c_size_t], ctypes.c_int),
        "cwipc_pointcloud_copy_packet": ([cwipc_pointcloud_p, ctypes.c_void_p, ctypes.c_size_t], ctypes.c_size_t),
        "cwipc_synthetic": ([ctypes.c_int, ctypes.c_int, c_err, ctypes.c_ulonglong], cwipc_source_p),
        "cwipc_source_get": ([cwipc_source_p], cwipc_pointcloud_p),
        "cwipc_source_free": ([cwipc_source_p], None),
        "cwipc_source_eof": ([cwipc_source_p], ctypes.c_bool),
        "cwipc_source_available": ([cwipc_source_p, ctypes.c_bool], ctypes.c_bool),
        "cwipc_activesource_start": ([cwipc_source_p], ctypes.c_bool),
        "cwipc_activesource_stop": ([cwipc_source_p], None),
        "cwipc_activesource_maxtile": ([cwipc_source_p], ctypes.c_int),
        "cwipc_activesource_auxiliary_operation": ([cwipc_source_p, ctypes.c_char_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t], ctypes.c_bool),
        "cwipc_downsample": ([cwipc_pointcloud_p, ctypes.c_float], cwipc_pointcloud_p),
        "cwipc_remove_outliers": ([cwipc_pointcloud_p, ctypes.c_int, ctypes.c_float, ctypes.c_bool], cwipc_pointcloud_p),
        "cwipc_tilefilter": ([cwipc_pointcloud_p, ctypes.c_int], cwipc_pointcloud_p),
        "cwipc_cuda_tilefilter_masked": ([cwipc_pointcloud_p, ctypes.c_int], cwipc_pointcloud_p),
        "cwipc_cuda_downsample_pertile": ([cwipc_pointcloud_p, ctypes.c_float], cwipc_pointcloud_p),
        "cwipc_cuda_transform": ([cwipc_pointcloud_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int], cwipc_pointcloud_p),
        "cwipc_tilemap": ([cwipc_pointcloud_p, ctypes.c_char_p], cwipc_pointcloud_p),
        "cwipc_colormap": ([cwipc_pointcloud_p, ctypes.c_uint32, ctypes.c_uint32], cwipc_pointcloud_p),
        "cwipc_crop": ([cwipc_pointcloud_p, ctypes.POINTER(ctypes.c_float)], cwipc_pointcloud_p),
        "cwipc_join": ([cwipc_pointcloud_p, cwipc_pointcloud_p], cwipc_pointcloud_p),
        "cwipc_cuda_device_count": ([], ctypes.c_int),
        "cwipc_cuda_set_device": ([ctypes.c_int], ctypes.c_int),
        "cwipc_cuda_get_device": ([], ctypes.c_int),
        "cwipc_cuda_synchronize": ([], ctypes.c_int),
        "cwipc_cuda_host_alloc": ([ctypes.c_size_t], ctypes.c_void_p),
        "cwipc_cuda_host_free": ([ctypes.c_void_p], None),
        "cwipc_cuda_pointcloud_device": ([cwipc_pointcloud_p], ctypes.c_int),
        "cwipc_cuda_pointcloud_device_ptr": ([cwipc_pointcloud_p], ctypes.c_void_p),
        "cwipc_cuda_knn_mean_distances": ([cwipc_pointcloud_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t], ctypes.c_int),
        "cwipc_cuda_downsample_keys": ([cwipc_pointcloud_p, ctypes.c_float, ctypes.c_void_p, ctypes.c_size_t], ctypes.c_int),
        "cwipc_cuda_octree_replay": ([cwipc_pointcloud_p, ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p], ctypes.c_int),
        "cwipc_cuda_downsample_planned": ([cwipc_pointcloud_p, ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p], cwipc_pointcloud_p),
        "cwipc_cuda_from_device_points": ([ctypes.c_void_p, ctypes.c_int, ctypes.c_ulonglong], cwipc_pointcloud_p),
        "cwipc_cuda_knn_query": ([cwipc_pointcloud_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p], ctypes.c_int),
        "cwipc_cuda_knn_lists": ([cwipc_pointcloud_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p], ctypes.c_int),
        "cwipc_cuda_knn_merge_lists": ([ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p], ctypes.c_int),
        "cwipc_cuda_distance_stats": ([ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p], ctypes.c_int),
        "cwipc_cuda_outlier_threshold": ([ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_float], ctypes.c_double),
        "cwipc_cuda_filter_by_distance": ([cwipc_pointcloud_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_double], cwipc_pointcloud_p),
        "cwipc_cuda_knn_query_open": ([cwipc_pointcloud_p, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_float, ctypes.c_void_p], ctypes.c_void_p),
        "cwipc_cuda_distances_open": ([ctypes.c_void_p, cwipc_pointcloud_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p], ctypes.c_int),
        "cwipc_cuda_distances_patch": ([ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int], ctypes.c_int),
        "cwipc_cuda_distances_stats": ([ctypes.c_void_p, ctypes.c_void_p], ctypes.c_int),
        "cwipc_cuda_distances_filter": ([cwipc_pointcloud_p, ctypes.c_void_p, ctypes.c_double], cwipc_pointcloud_p),
        "cwipc_cuda_distances_free": ([ctypes.c_void_p], None),
        "cwipc_cuda_sort_u64": ([ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_int], ctypes.c_int),
        "cwipc_cuda_timer_create": ([], ctypes.c_void_p),
        "cwipc_cuda_timer_destroy": ([ctypes.c_void_p], None),
        "cwipc_cuda_timer_start": ([ctypes.c_void_p], None),
        "cwipc_cuda_timer_stop": ([ctypes.c_void_p], None),
        "cwipc_cuda_timer_elapsed_ms": ([ctypes.c_void_p], ctypes.c_float),
        "cwipc_cuda_timer_span_ms": ([ctypes.c_void_p, ctypes.c_void_p], ctypes.c_float),
        "cwipc_cuda_kernel_launches": ([], ctypes.c_uint64),
        "cwipc_cuda_profile_enable": ([ctypes.c_int], None),
        "cwipc_cuda_profile_reset": ([], None),
        "cwipc_cuda_profile_report": ([ctypes.c_char_p, ctypes.c_size_t], ctypes.c_size_t),
        "cwipc_cuda_flush_l2": ([], None),
        "cwipc_cuda_trim": ([], ctypes.c_int),
        "cwipc_cuda_comm_unique_id": ([ctypes.c_void_p], ctypes.c_int),
        "cwipc_cuda_comm_create": ([ctypes.c_void_p, ctypes.c_int, ctypes.c_int], ctypes.c_void_p),
        "cwipc_cuda_comm_free": ([ctypes.c_void_p], None),
        "cwipc_cuda_comm_rank": ([ctypes.c_void_p], ctypes.c_int),
        "cwipc_cuda_comm_size": ([ctypes.c_void_p], ctypes.c_int),
        "cwipc_cuda_slab_downsample": ([cwipc_pointcloud_p, ctypes.c_float, ctypes.c_void_p], cwipc_pointcloud_p),
        "cwipc_cuda_slab_remove_outliers": ([cwipc_pointcloud_p, ctypes.c_int, ctypes.c_float, ctypes.c_bool, ctypes.c_float, ctypes.c_void_p], cwipc_pointcloud_p),
        "cwipc_cuda_slab_tilefilter": ([cwipc_pointcloud_p, ctypes.c_int, ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64)], cwipc_pointcloud_p),
    }
    for name, (argtypes, restype) in sigs.items():
        fn = getattr(d, name)
        fn.argtypes = argtypes
        fn.restype = restype
    _dll = d
    return d


def _raise_or_none(err: ctypes.c_char_p) -> None:
    if err and err.value:
        raise CwipcError(err.value.decode("utf8"))


class cwipc_pointcloud_wrapper:
    """Pointcloud as an opaque object living on the GPU (ref: python/cwipc/util.py:573-740)."""

    def __init__(self, _cwipc: Optional[cwipc_pointcloud_p] = None):
        if _cwipc is not None and not isinstance(_cwipc, cwipc_pointcloud_p):
            raise CwipcError("Invalid cwipc_pointcloud_p pointer passed to cwipc_pointcloud_wrapper")
        self._cwipc = _cwipc if _cwipc else None
        self._bytes: Optional[bytearray] = None
        self._points = None
        self._must_be_freed = True

    def __del__(self):
        if getattr(self, "_must_be_freed", False):
            self.free()

    def as_cwipc_p(self) -> cwipc_pointcloud_p:
        assert self._cwipc
        return self._cwipc

    def free(self) -> None:
        if self._cwipc and self._must_be_freed:
            cwipc_util_dll_load().cwipc_pointcloud_free(self._cwipc)
        self._cwipc = None
        self._must_be_freed = False

    def clone(self) -> "cwipc_pointcloud_wrapper":
        return cwipc_pointcloud_wrapper(cwipc_util_dll_load().cwipc_pointcloud__shallowcopy(self.as_cwipc_p()))

    def timestamp(self) -> int:
        return cwipc_util_dll_load().cwipc_pointcloud_timestamp(self.as_cwipc_p())

    def cellsize(self) -> float:
        return cwipc_util_dll_load().cwipc_pointcloud_cellsize(self.as_cwipc_p())

    def _set_cellsize(self, cellsize: float) -> None:
        cwipc_util_dll_load().cwipc_pointcloud__set_cellsize(self.as_cwipc_p(), cellsize)

    def _set_timestamp(self, timestamp: int) -> None:
        cwipc_util_dll_load().cwipc_pointcloud__set_timestamp(self.as_cwipc_p(), timestamp)

    def count(self) -> int:
        return cwipc_util_dll_load().cwipc_pointcloud_count(self.as_cwipc_p())

    def get_uncompressed_size(self) -> int:
        return cwipc_util_dll_load().cwipc_pointcloud_get_uncompressed_size(self.as_cwipc_p())

    def _initialize_points_and_bytes(self) -> None:
        d = cwipc_util_dll_load()
        nbytes = d.cwipc_pointcloud_get_uncompressed_size(self.as_cwipc_p())
        buffer = bytearray(nbytes)
        if nbytes:
            arg = (ctypes.c_byte * nbytes).from_buffer(buffer)
            npoints = d.cwipc_pointcloud_copy_uncompressed(self.as_cwipc_p(), ctypes.addressof(arg), nbytes)
            if npoints < 0:
                raise CwipcError("cwipc_pointcloud_copy_uncompressed failed")
        else:
            npoints = 0
        self._bytes = buffer
        self._points = cwipc_point_array(count=npoints, values=buffer)

    def get_points(self) -> ctypes.Array:
        if self._points is None:
            self._initialize_points_and_bytes()
        return self._points

    def get_bytes(self) -> bytearray:
        if self._bytes is None:
            self._initialize_points_and_bytes()
        return self._bytes

    def get_numpy_array(self) -> numpy.ndarray:
        """The points as a numpy record array (dtype cwipc_point_numpy_dtype); one D2H copy."""
        return numpy.frombuffer(self.get_bytes(), dtype=cwipc_point_numpy_dtype)

    def get_numpy_matrix(self, onlyGeometry: bool = False) -> numpy.ndarray:
        a = self.get_numpy_array()
        m = numpy.zeros((a.shape[0], 3 if onlyGeometry else 7), numpy.float32)
        m[:, 0], m[:, 1], m[:, 2] = a["x"], a["y"], a["z"]
        if not onlyGeometry:
            m[:, 3], m[:, 4], m[:, 5], m[:, 6] = a["r"], a["g"], a["b"], a["tile"]
        return m

    def get_packet(self) -> bytearray:
        d = cwipc_util_dll_load()
        nbytes = d.cwipc_pointcloud_copy_packet(self.as_cwipc_p(), None, 0)
        buffer = bytearray(nbytes)
        arg = (ctypes.c_byte * nbytes).from_buffer(buffer)
        rv = d.cwipc_pointcloud_copy_packet(self.as_cwipc_p(), ctypes.addressof(arg), nbytes)
        assert rv == nbytes
        return buffer


class cwipc_activesource_wrapper:
    def __init__(self, _src: cwipc_source_p):
        self._src = _src

    def __del__(self):
        self.free()

    def free(self) -> None:
        if self._src:
            cwipc_util_dll_load().cwipc_source_free(self._src)
        self._src = None

    def start(self) -> bool:
        return cwipc_util_dll_load().cwipc_activesource_start(self._src)

    def stop(self) -> None:
        cwipc_util_dll_load().cwipc_activesource_stop(self._src)

    def eof(self) -> bool:
        return cwipc_util_dll_load().cwipc_source_eof(self._src)

    def available(self, wait: bool) -> bool:
        return cwipc_util_dll_load().cwipc_source_available(self._src, wait)

    def maxtile(self) -> int:
        return cwipc_util_dll_load().cwipc_activesource_maxtile(self._src)

    def get(self) -> Optional[cwipc_pointcloud_wrapper]:
        rv = cwipc_util_dll_load().cwipc_source_get(self._src)
        return cwipc_pointcloud_wrapper(rv) if rv else None

    def set_angle(self, angle: float) -> bool:
        """test hook of the synthetic source (ref: src/cwipc_synthetic.cpp:169-179)"""
        a, b = ctypes.c_float(angle), ctypes.c_float(0)
        return cwipc_util_dll_load().cwipc_activesource_auxiliary_operation(self._src, b"test-setangle", ctypes.byref(a), 4, ctypes.byref(b), 4)

    def host_generate(self, angle: float, npoints: int) -> numpy.ndarray:
        """libcwipc_util_cuda only: the HOST generator's points for `angle` (the checker of the device-side generator);
        the next get() uses the same angle instead of the wall clock."""
        a = ctypes.c_float(angle)
        out = numpy.zeros(npoints, cwipc_point_numpy_dtype)
        ok = cwipc_util_dll_load().cwipc_activesource_auxiliary_operation(self._src, b"cuda-host-generate", ctypes.byref(a), 4, out.ctypes.data, out.nbytes)
        if not ok:
            raise CwipcError("cuda-host-generate refused (wrong point count?)")
        return out


# ---- module functions, same names as the reference binding -------------------------------------
def cwipc_get_version() -> str:
    return cwipc_util_dll_load().cwipc_get_version().decode("utf8")


def cwipc_log_configure(level: int, callback=None) -> None:
    global _log_callback_ref
    _log_callback_ref = _LOG_CALLBACK(callback) if callback else _LOG_CALLBACK(0)
    cwipc_util_dll_load().cwipc_log_configure(level, _log_callback_ref)


def cwipc_dangling_allocations(log: bool) -> int:
    return cwipc_util_dll_load().cwipc_dangling_allocations(log)


def _wrap(rv, err: ctypes.c_char_p, what: str) -> cwipc_pointcloud_wrapper:
    _raise_or_none(err)
    if rv:
        return cwipc_pointcloud_wrapper(rv)
    raise CwipcError(f"{what}: no pointcloud, but no specific error returned from C library")


def cwipc_read(filename: str, timestamp: int) -> cwipc_pointcloud_wrapper:
    err = ctypes.c_char_p()
    rv = cwipc_util_dll_load().cwipc_read(filename.encode("utf8"), timestamp, ctypes.byref(err), CWIPC_API_VERSION)
    return _wrap(rv, err, "cwipc_read")


def cwipc_write(filename: str, pointcloud: cwipc_pointcloud_wrapper, flags: int = 0) -> int:
    err = ctypes.c_char_p()
    rv = cwipc_util_dll_load().cwipc_write_ext(filename.encode("utf8"), pointcloud.as_cwipc_p(), flags, ctypes.byref(err))
    _raise_or_none(err)
    return rv


def cwipc_read_debugdump(filename: str) -> cwipc_pointcloud_wrapper:
    err = ctypes.c_char_p()
    rv = cwipc_util_dll_load().cwipc_read_debugdump(filename.encode("utf8"), ctypes.byref(err), CWIPC_API_VERSION)
    return _wrap(rv, err, "cwipc_read_debugdump")


def cwipc_write_debugdump(filename: str, pointcloud: cwipc_pointcloud_wrapper) -> int:
    err = ctypes.c_char_p()
    rv = cwipc_util_dll_load().cwipc_write_debugdump(filename.encode("utf8"), pointcloud.as_cwipc_p(), ctypes.byref(err))
    _raise_or_none(err)
    return rv


def cwipc_from_points(points: Any, timestamp: int) -> cwipc_pointcloud_wrapper:
    """Create a cwipc from a cwipc_point_array or a list/tuple of (x,y,z,r,g,b,tile)."""
    if not isinstance(points, ctypes.Array):
        points = cwipc_point_array(values=points)
    err = ctypes.c_char_p()
    rv = cwipc_util_dll_load().cwipc_from_points(ctypes.addressof(points), ctypes.sizeof(points), len(points), timestamp, ctypes.byref(err), CWIPC_API_VERSION)
    return _wrap(rv, err, "cwipc_from_points")


def cwipc_from_numpy_array(np_points: numpy.ndarray, timestamp: int) -> cwipc_pointcloud_wrapper:
    np_points = numpy.ascontiguousarray(np_points, dtype=cwipc_point_numpy_dtype)
    n = np_points.shape[0]
    err = ctypes.c_char_p()
    rv = cwipc_util_dll_load().cwipc_from_points(np_points.ctypes.data, n * 16, n, timestamp, ctypes.byref(err), CWIPC_API_VERSION)
    return _wrap(rv, err, "cwipc_from_numpy_array")


def cwipc_from_numpy_matrix(m: numpy.ndarray, timestamp: int) -> cwipc_pointcloud_wrapper:
    count = m.shape[0]
    assert m.shape == (count, 7)
    a = numpy.zeros(count, cwipc_point_numpy_dtype)
    a["x"], a["y"], a["z"] = m[:, 0], m[:, 1], m[:, 2]
    a["r"], a["g"], a["b"], a["tile"] = m[:, 3].astype(numpy.uint8), m[:, 4].astype(numpy.uint8), m[:, 5].astype(numpy.uint8), m[:, 6].astype(numpy.uint8)
    return cwipc_from_numpy_array(a, timestamp)


def cwipc_from_packet(packet: Union[bytes, bytearray]) -> cwipc_pointcloud_wrapper:
    n = len(packet)
    buf = (ctypes.c_char * n).from_buffer_copy(bytes(packet))
    err = ctypes.c_char_p()
    rv = cwipc_util_dll_load().cwipc_from_packet(ctypes.addressof(buf), n, ctypes.byref(err), CWIPC_API_VERSION)
    return _wrap(rv, err, "cwipc_from_packet")


def cwipc_synthetic(fps: int = 0, npoints: int = 0) -> cwipc_activesource_wrapper:
    err = ctypes.c_char_p()
    rv = cwipc_util_dll_load().cwipc_synthetic(fps, npoints, ctypes.byref(err), CWIPC_API_VERSION)
    _raise_or_none(err)
    if rv:
        return cwipc_activesource_wrapper(rv)
    raise CwipcError("cwipc_synthetic: cannot create synthetic source")


def cwipc_downsample(pc: cwipc_pointcloud_wrapper, voxelsize: float) -> cwipc_pointcloud_wrapper:
    """Pointcloud voxelized to cubes of the given size (negative: single global grid)."""
    return cwipc_pointcloud_wrapper(cwipc_util_dll_load().cwipc_downsample(pc.as_cwipc_p(), voxelsize))


def cwipc_remove_outliers(pc: cwipc_pointcloud_wrapper, kNeighbors: int, stdDesvMultThresh: float, perTile: bool) -> cwipc_pointcloud_wrapper:
    return cwipc_pointcloud_wrapper(cwipc_util_dll_load().cwipc_remove_outliers(pc.as_cwipc_p(), kNeighbors, stdDesvMultThresh, perTile))


def cwipc_tilefilter(pc: cwipc_pointcloud_wrapper, tile: int) -> cwipc_pointcloud_wrapper:
    return cwipc_pointcloud_wrapper(cwipc_util_dll_load().cwipc_tilefilter(pc.as_cwipc_p(), tile))


def cwipc_tilefilter_masked(pc: cwipc_pointcloud_wrapper, mask: int) -> cwipc_pointcloud_wrapper:
    """(tile & mask) != 0 -- ref: python/cwipc/registration/util.py:98-112, here one kernel instead of a host round trip."""
    return cwipc_pointcloud_wrapper(cwipc_util_dll_load().cwipc_cuda_tilefilter_masked(pc.as_cwipc_p(), mask))


def cwipc_downsample_pertile(pc: cwipc_pointcloud_wrapper, voxelsize: float) -> cwipc_pointcloud_wrapper:
    """cwipc_downsample of every tile (camera) on its own, the results joined in first-appearance order of the tile values:
    python/cwipc/registration/util.py:170-182 (tilefilter -> downsample per tile, then join) as one library call."""
    return cwipc_pointcloud_wrapper(cwipc_util_dll_load().cwipc_cuda_downsample_pertile(pc.as_cwipc_p(), voxelsize))


def cwipc_transform(pc: cwipc_pointcloud_wrapper, matrices: Any) -> cwipc_pointcloud_wrapper:
    """Every point moved by a 4x4 matrix on the device (cwipc_cuda_transform in include/cwipc_util_cuda.h): `matrices` is
    one (4, 4) array-like for the whole cloud, or a mapping {tile value: (4, 4) array-like}, where tile 0 applies to every
    value without an entry of its own and the points of other values are copied unchanged.  This replaces the round trip
    get_numpy_matrix -> numpy -> cwipc_from_numpy_matrix.  A matrix of another shape raises ValueError before the library
    is called; the library checks the rest (NULL and one ERROR log)."""
    if isinstance(matrices, Mapping):
        tiles, ms = list(matrices.keys()), list(matrices.values())
    else:
        tiles, ms = [0], [matrices]
    table = numpy.zeros((len(ms), 4, 4), numpy.float64)
    for i, m in enumerate(ms):
        a = numpy.asarray(m, dtype=numpy.float64)
        if a.shape != (4, 4):
            raise ValueError(f"cwipc_transform: a matrix must have shape (4, 4), not {a.shape}")
        table[i] = a
    if not all(0 <= int(t) <= 255 for t in tiles):
        raise ValueError("cwipc_transform: tile values are 0..255")
    t = numpy.array([int(v) for v in tiles], numpy.uint8)
    return cwipc_pointcloud_wrapper(cwipc_util_dll_load().cwipc_cuda_transform(pc.as_cwipc_p(), table.ctypes.data, t.ctypes.data, len(ms)))


def cwipc_tilemap(pc: cwipc_pointcloud_wrapper, mapping: Union[List[int], dict, bytes]) -> cwipc_pointcloud_wrapper:
    if not isinstance(mapping, (bytes, bytearray, list)):
        m = [0] * 256
        for k in mapping:
            m[k] = mapping[k]
        mapping = m
    return cwipc_pointcloud_wrapper(cwipc_util_dll_load().cwipc_tilemap(pc.as_cwipc_p(), bytes(mapping)))


def cwipc_colormap(pc: cwipc_pointcloud_wrapper, clearBits: int, setBits: int) -> cwipc_pointcloud_wrapper:
    return cwipc_pointcloud_wrapper(cwipc_util_dll_load().cwipc_colormap(pc.as_cwipc_p(), clearBits, setBits))


def cwipc_crop(pc: cwipc_pointcloud_wrapper, bbox: Sequence[float]) -> cwipc_pointcloud_wrapper:
    return cwipc_pointcloud_wrapper(cwipc_util_dll_load().cwipc_crop(pc.as_cwipc_p(), (ctypes.c_float * 6)(*bbox)))


def cwipc_join(pc1: cwipc_pointcloud_wrapper, pc2: cwipc_pointcloud_wrapper) -> cwipc_pointcloud_wrapper:
    return cwipc_pointcloud_wrapper(cwipc_util_dll_load().cwipc_join(pc1.as_cwipc_p(), pc2.as_cwipc_p()))


def cwipc_join_multi(pcs: Iterable[cwipc_pointcloud_wrapper]) -> cwipc_pointcloud_wrapper:
    import functools
    return functools.reduce(cwipc_join, pcs)


# ---- extensions -----------------------------------------------------------------------------------
def cuda_device_count() -> int:
    return cwipc_util_dll_load().cwipc_cuda_device_count()


def cuda_set_device(device: int) -> None:
    if cwipc_util_dll_load().cwipc_cuda_set_device(device) != 0:
        raise CwipcError(f"no CUDA device {device}")


def cuda_synchronize() -> None:
    if cwipc_util_dll_load().cwipc_cuda_synchronize() != 0:
        raise CwipcError("cwipc_cuda_synchronize failed")


def cuda_kernel_launches() -> int:
    return cwipc_util_dll_load().cwipc_cuda_kernel_launches()


def knn_mean_distances(pc: cwipc_pointcloud_wrapper, kNeighbors: int) -> numpy.ndarray:
    """Diagnostic: first pass of cwipc_remove_outliers (mean distance to the k nearest neighbours per point)."""
    n = pc.count()
    out = numpy.zeros(n, numpy.float32)
    rv = cwipc_util_dll_load().cwipc_cuda_knn_mean_distances(pc.as_cwipc_p(), kNeighbors, out.ctypes.data, n)
    if rv < 0:
        raise CwipcError("cwipc_cuda_knn_mean_distances failed")
    return out


def downsample_keys(pc: cwipc_pointcloud_wrapper, voxelsize: float) -> numpy.ndarray:
    """Diagnostic: the 64-bit voxel sort key of every input point."""
    n = pc.count()
    out = numpy.zeros(n, numpy.uint64)
    rv = cwipc_util_dll_load().cwipc_cuda_downsample_keys(pc.as_cwipc_p(), voxelsize, out.ctypes.data, n)
    if rv < 0:
        raise CwipcError("cwipc_cuda_downsample_keys failed")
    return out


# ---- partitioned clouds (one cloud over several GPUs; see slab.py) ----------------------------------
class cwipc_cuda_octree_state(ctypes.Structure):
    """include/cwipc_util_cuda.h: struct cwipc_cuda_octree_state"""
    _fields_ = [("min", ctypes.c_double * 3), ("max", ctypes.c_double * 3), ("depth", ctypes.c_int32), ("valid", ctypes.c_int32), ("points", ctypes.c_uint64)]

    def to_array(self) -> numpy.ndarray:
        return numpy.array(list(self.min) + list(self.max) + [float(self.depth), float(self.valid), float(self.points)], numpy.float64)

    @classmethod
    def from_array(cls, a) -> "cwipc_cuda_octree_state":
        st = cls()
        for i in range(3):
            st.min[i] = float(a[i])
            st.max[i] = float(a[3 + i])
        st.depth = int(a[6])
        st.valid = int(a[7])
        st.points = int(a[8])
        return st


def octree_replay(pc: cwipc_pointcloud_wrapper, cellsize: float, state: cwipc_cuda_octree_state):
    """Insert pc's points into the octree box `state` (updated in place); returns pc's bounding box (6 floats)."""
    bounds = numpy.zeros(6, numpy.float32)
    rv = cwipc_util_dll_load().cwipc_cuda_octree_replay(pc.as_cwipc_p(), cellsize, ctypes.addressof(state), bounds.ctypes.data)
    if rv != 0:
        raise CwipcError("cwipc_cuda_octree_replay failed")
    return bounds


def downsample_planned(pc: cwipc_pointcloud_wrapper, voxelsize: float, state: cwipc_cuda_octree_state, bounds) -> cwipc_pointcloud_wrapper:
    b = numpy.ascontiguousarray(bounds, numpy.float32)
    rv = cwipc_util_dll_load().cwipc_cuda_downsample_planned(pc.as_cwipc_p(), voxelsize, ctypes.addressof(state), b.ctypes.data)
    if not rv:
        raise CwipcError("cwipc_cuda_downsample_planned failed")
    return cwipc_pointcloud_wrapper(rv)


def from_device_points(dev_ptr: int, npoint: int, timestamp: int) -> cwipc_pointcloud_wrapper:
    rv = cwipc_util_dll_load().cwipc_cuda_from_device_points(dev_ptr, npoint, timestamp)
    if not rv:
        raise CwipcError("cwipc_cuda_from_device_points failed")
    return cwipc_pointcloud_wrapper(rv)


def pointcloud_device_ptr(pc: cwipc_pointcloud_wrapper) -> int:
    return cwipc_util_dll_load().cwipc_cuda_pointcloud_device_ptr(pc.as_cwipc_p()) or 0


def knn_query(pc: cwipc_pointcloud_wrapper, kNeighbors: int, nquery: int):
    mean = numpy.zeros(nquery, numpy.float32)
    kth2 = numpy.zeros(nquery, numpy.float32)
    rv = cwipc_util_dll_load().cwipc_cuda_knn_query(pc.as_cwipc_p(), kNeighbors, nquery, mean.ctypes.data, kth2.ctypes.data)
    if rv < 0:
        raise CwipcError("cwipc_cuda_knn_query failed")
    return mean, kth2


def knn_lists(pc: cwipc_pointcloud_wrapper, queries: numpy.ndarray, kNeighbors: int, limits: Optional[numpy.ndarray] = None) -> numpy.ndarray:
    q = numpy.ascontiguousarray(queries)
    out = numpy.zeros((len(q), kNeighbors + 1), numpy.float32)
    lim = None if limits is None else numpy.ascontiguousarray(limits, numpy.float32)
    rv = cwipc_util_dll_load().cwipc_cuda_knn_lists(pc.as_cwipc_p(), q.ctypes.data, None if lim is None else lim.ctypes.data, len(q), kNeighbors, out.ctypes.data)
    if rv < 0:
        raise CwipcError("cwipc_cuda_knn_lists failed")
    return out


def knn_merge_lists(lists: numpy.ndarray, kNeighbors: int):
    """lists[nlists][nq][k+1] -> (mean[nq], kth2[nq])"""
    l = numpy.ascontiguousarray(lists, numpy.float32)
    nlists, nq = l.shape[0], l.shape[1]
    mean = numpy.zeros(nq, numpy.float32)
    kth2 = numpy.zeros(nq, numpy.float32)
    rv = cwipc_util_dll_load().cwipc_cuda_knn_merge_lists(l.ctypes.data, nlists, nq, kNeighbors, mean.ctypes.data, kth2.ctypes.data)
    if rv < 0:
        raise CwipcError("cwipc_cuda_knn_merge_lists failed")
    return mean, kth2


def distance_stats(dist: numpy.ndarray):
    d = numpy.ascontiguousarray(dist, numpy.float32)
    sums = numpy.zeros(2, numpy.float64)
    if cwipc_util_dll_load().cwipc_cuda_distance_stats(d.ctypes.data, len(d), sums.ctypes.data) != 0:
        raise CwipcError("cwipc_cuda_distance_stats failed")
    return float(sums[0]), float(sums[1])


def outlier_threshold(total: float, sq: float, n: float, mul: float) -> float:
    return cwipc_util_dll_load().cwipc_cuda_outlier_threshold(total, sq, n, mul)


def filter_by_distance(pc: cwipc_pointcloud_wrapper, dist: numpy.ndarray, threshold: float) -> cwipc_pointcloud_wrapper:
    d = numpy.ascontiguousarray(dist, numpy.float32)
    rv = cwipc_util_dll_load().cwipc_cuda_filter_by_distance(pc.as_cwipc_p(), d.ctypes.data, len(d), threshold)
    if not rv:
        raise CwipcError("cwipc_cuda_filter_by_distance failed")
    return cwipc_pointcloud_wrapper(rv)


def sort_u64(words: numpy.ndarray, begin_bit: int, end_bit: int) -> numpy.ndarray:
    """Diagnostic: the library's stable radix sort on bits [begin_bit, end_bit) of a uint64 array."""
    w = numpy.ascontiguousarray(words, numpy.uint64).copy()
    if cwipc_util_dll_load().cwipc_cuda_sort_u64(w.ctypes.data, len(w), begin_bit, end_bit) != 0:
        raise CwipcError("cwipc_cuda_sort_u64 failed")
    return w


class cuda_distances:
    """Device-resident mean kNN distances of a slab's points (include/cwipc_util_cuda.h: cwipc_cuda_distances)."""

    def __init__(self, pc: cwipc_pointcloud_wrapper, kNeighbors: int, nquery: int, x_lo: float, x_hi: float):
        nopen = ctypes.c_int(0)
        self._h = cwipc_util_dll_load().cwipc_cuda_knn_query_open(pc.as_cwipc_p(), kNeighbors, nquery, x_lo, x_hi, ctypes.byref(nopen))
        if not self._h:
            raise CwipcError("cwipc_cuda_knn_query_open failed")
        self.nopen = nopen.value
        self._pc = pc

    def __del__(self):
        self.free()

    def free(self) -> None:
        if getattr(self, "_h", None):
            cwipc_util_dll_load().cwipc_cuda_distances_free(self._h)
            self._h = None

    def open_queries(self):
        idx = numpy.zeros(self.nopen, numpy.uint32)
        pts = numpy.zeros(self.nopen, cwipc_point_numpy_dtype)
        kth2 = numpy.zeros(self.nopen, numpy.float32)
        if self.nopen and cwipc_util_dll_load().cwipc_cuda_distances_open(self._h, self._pc.as_cwipc_p(), idx.ctypes.data, pts.ctypes.data, kth2.ctypes.data) < 0:
            raise CwipcError("cwipc_cuda_distances_open failed")
        return idx, pts, kth2

    def patch(self, values: numpy.ndarray) -> None:
        v = numpy.ascontiguousarray(values, numpy.float32)
        if cwipc_util_dll_load().cwipc_cuda_distances_patch(self._h, v.ctypes.data, len(v)) < 0:
            raise CwipcError("cwipc_cuda_distances_patch failed")

    def stats(self):
        sums = numpy.zeros(2, numpy.float64)
        if cwipc_util_dll_load().cwipc_cuda_distances_stats(self._h, sums.ctypes.data) != 0:
            raise CwipcError("cwipc_cuda_distances_stats failed")
        return float(sums[0]), float(sums[1])

    def filter(self, pc: cwipc_pointcloud_wrapper, threshold: float) -> cwipc_pointcloud_wrapper:
        rv = cwipc_util_dll_load().cwipc_cuda_distances_filter(pc.as_cwipc_p(), self._h, threshold)
        if not rv:
            raise CwipcError("cwipc_cuda_distances_filter failed")
        return cwipc_pointcloud_wrapper(rv)


# ---- one cloud partitioned over several GPUs: the library's own NCCL protocol (csrc/slab.cpp) -----------------------
class cuda_comm:
    """cwipc_cuda_comm: one rank of a group of processes (or threads), one GPU each.  `unique_id` (128 bytes from
    cuda_comm.unique_id() on one rank) has to reach every rank by the caller's own means; size 1 needs none."""

    def __init__(self, unique_id: Optional[bytes], nranks: int, rank: int):
        buf = ctypes.create_string_buffer(unique_id, 128) if unique_id is not None else None
        self._c = cwipc_util_dll_load().cwipc_cuda_comm_create(buf, nranks, rank)
        if not self._c:
            raise CwipcError("cwipc_cuda_comm_create failed (NCCL not found, or ncclCommInitRank failed)")
        self.rank, self.size = rank, nranks

    @staticmethod
    def unique_id() -> bytes:
        buf = ctypes.create_string_buffer(128)
        if cwipc_util_dll_load().cwipc_cuda_comm_unique_id(buf) != 0:
            raise CwipcError("cwipc_cuda_comm_unique_id failed (libnccl.so.2 not found?)")
        return buf.raw

    def free(self) -> None:
        if self._c:
            cwipc_util_dll_load().cwipc_cuda_comm_free(self._c)
            self._c = None

    def downsample(self, pc: cwipc_pointcloud_wrapper, voxelsize: float) -> cwipc_pointcloud_wrapper:
        return cwipc_pointcloud_wrapper(cwipc_util_dll_load().cwipc_cuda_slab_downsample(pc.as_cwipc_p(), voxelsize, self._c))

    def remove_outliers(self, pc: cwipc_pointcloud_wrapper, kNeighbors: int, stddevMulThresh: float, perTile: bool = False, halo: float = 0.0) -> cwipc_pointcloud_wrapper:
        return cwipc_pointcloud_wrapper(cwipc_util_dll_load().cwipc_cuda_slab_remove_outliers(pc.as_cwipc_p(), kNeighbors, stddevMulThresh, perTile, halo, self._c))

    def tilefilter(self, pc: cwipc_pointcloud_wrapper, tile: int):
        off, tot = ctypes.c_uint64(0), ctypes.c_uint64(0)
        rv = cwipc_pointcloud_wrapper(cwipc_util_dll_load().cwipc_cuda_slab_tilefilter(pc.as_cwipc_p(), tile, self._c, ctypes.byref(off), ctypes.byref(tot)))
        return rv, off.value, tot.value
