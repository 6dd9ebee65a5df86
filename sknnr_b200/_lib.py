"""ctypes binding of libsknnr_b200.so (the C ABI declared in include/sknnr_b200.h).

The library must have been built (``python -m sknnr_b200._build`` or
``__graft_entry__.build()``); a missing library or a missing CUDA device is a loud error.
There is no CPU fallback and no other backend.
"""

from __future__ import annotations

import ctypes as C
import os

from ._build import lib_path

# mirrors include/sknnr_b200.h
ABI_VERSION = 1
F64, F32 = 0, 1
EXCLUDE_SELF, DETERMINISTIC, TRANSFORMED, DEVICE_PTRS, CHECK_FINITE = 1, 2, 4, 8, 16
W_NONE, W_UNIFORM, W_DISTANCE = 0, 1, 2
ENGINE_AUTO, ENGINE_SIMT, ENGINE_TENSOR, ENGINE_EXACT = 0, 1, 2, 3
METRICS = {"euclidean": 0, "manhattan": 1, "chebyshev": 2}   # SKNNR_METRIC_*
MAX_CODE = 31743

EXPORTS = [
    "sknnr_last_error", "sknnr_abi_version", "sknnr_device_count", "sknnr_set_option",
    "sknnr_index_create", "sknnr_index_destroy", "sknnr_kneighbors", "sknnr_transform",
    "sknnr_weighted_average", "sknnr_index_stats", "sknnr_index_cascade_counts", "sknnr_hamming_index_create",
    "sknnr_hamming_index_destroy", "sknnr_hamming_kneighbors",
    "sknnr_hamming_weighted_average", "sknnr_hamming_index_stats", "sknnr_host_alloc",
    "sknnr_host_free", "sknnr_measure_fp32_peak", "sknnr_forest_create", "sknnr_forest_destroy",
    "sknnr_forest_apply", "sknnr_hamming_kneighbors_forest", "sknnr_raster_kneighbors",
    "sknnr_hamming_raster_kneighbors_forest", "sknnr_device_alloc", "sknnr_device_free",
    "sknnr_ipc_export", "sknnr_ipc_open", "sknnr_ipc_close", "sknnr_device_copy", "sknnr_host_chunk_plan",
    "sknnr_index_create_metric",
]


class Stats(C.Structure):
    _fields_ = [
        ("n_queries", C.c_int64), ("n_fallback", C.c_int64), ("kernel_launches", C.c_int64),
        ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64), ("engine", C.c_int64),
        ("search_ms", C.c_double),
    ]

    def as_dict(self):
        return {f: getattr(self, f) for f, _ in self._fields_}


class SknnrError(RuntimeError):
    pass


class NonFiniteInput(ValueError):
    """SKNNR_ENONFINITE: the device found NaN / inf among the query values (SKNNR_CHECK_FINITE)."""


_lib = None


def load() -> C.CDLL:
    """Load the shared library (once) and declare every prototype."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise SknnrError(
            f"{path} is missing: build it with `python -m sknnr_b200._build` "
            "(sknnr_b200 has no CPU fallback)"
        )
    lib = C.CDLL(path)
    vp, i32, i64, u32 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32
    lib.sknnr_last_error.restype = C.c_char_p
    lib.sknnr_last_error.argtypes = []
    lib.sknnr_abi_version.restype = C.c_int
    lib.sknnr_device_count.argtypes = [C.POINTER(C.c_int)]
    lib.sknnr_set_option.argtypes = [C.c_char_p, i64]
    lib.sknnr_index_create.argtypes = [vp, i64, i32, vp, vp, vp, i32, vp, i32, i32, C.POINTER(vp)]
    lib.sknnr_index_create_metric.argtypes = [vp, i64, i32, vp, vp, vp, i32, vp, i32, i32, i32, C.POINTER(vp)]
    lib.sknnr_index_destroy.argtypes = [vp]
    lib.sknnr_kneighbors.argtypes = [vp, vp, i32, i64, i64, i64, i32, u32, i32, vp, vp, i32, vp, vp]
    lib.sknnr_transform.argtypes = [vp, vp, i32, i64, i64, vp]
    lib.sknnr_weighted_average.argtypes = [vp, vp, vp, i64, i32, vp]
    lib.sknnr_index_stats.argtypes = [vp, C.POINTER(Stats)]
    lib.sknnr_index_cascade_counts.argtypes = [vp, C.POINTER(C.c_int64)]
    lib.sknnr_hamming_index_create.argtypes = [vp, i64, i32, vp, vp, i32, i32, C.POINTER(vp)]
    lib.sknnr_hamming_index_destroy.argtypes = [vp]
    lib.sknnr_hamming_kneighbors.argtypes = [vp, vp, i64, i64, i64, i32, u32, i32, vp, vp, i32, vp, vp]
    lib.sknnr_hamming_weighted_average.argtypes = [vp, vp, vp, i64, i32, vp]
    lib.sknnr_hamming_index_stats.argtypes = [vp, C.POINTER(Stats)]
    lib.sknnr_host_alloc.argtypes = [C.POINTER(vp), i64]
    lib.sknnr_host_free.argtypes = [vp]
    lib.sknnr_measure_fp32_peak.argtypes = [i32, C.POINTER(C.c_double)]
    lib.sknnr_forest_create.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, C.POINTER(vp)]
    lib.sknnr_forest_destroy.argtypes = [vp]
    lib.sknnr_forest_apply.argtypes = [vp, vp, i32, i64, i64, vp]
    lib.sknnr_hamming_kneighbors_forest.argtypes = [vp, vp, vp, i32, i64, i64, i64, i32, u32, i32, vp, vp, i32,
                                                    vp, vp]
    lib.sknnr_raster_kneighbors.argtypes = [vp, vp, i32, i64, i64, i32, C.c_double, i32, u32, i32, vp, vp, i32,
                                            vp, C.c_double, i64, C.c_double, C.POINTER(i64)]
    lib.sknnr_hamming_raster_kneighbors_forest.argtypes = [vp] + lib.sknnr_raster_kneighbors.argtypes
    lib.sknnr_device_alloc.argtypes = [i32, C.POINTER(vp), i64]
    lib.sknnr_device_free.argtypes = [i32, vp]
    lib.sknnr_ipc_export.argtypes = [i32, vp, vp]
    lib.sknnr_ipc_open.argtypes = [i32, vp, C.POINTER(vp)]
    lib.sknnr_ipc_close.argtypes = [i32, vp]
    lib.sknnr_device_copy.argtypes = [i32, vp, vp, i64, i32, vp]
    for name in EXPORTS:
        if name != "sknnr_last_error":
            getattr(lib, name).restype = C.c_int
    if lib.sknnr_abi_version() != ABI_VERSION:
        raise SknnrError("libsknnr_b200.so ABI version mismatch; rebuild it")
    _lib = lib
    return lib


def check(rc: int) -> None:
    """Translate a status code into the exception the reference layer would raise."""
    if rc == 0:
        return
    msg = load().sknnr_last_error().decode("utf-8", "replace")
    if rc == -1:
        raise ValueError(msg)
    if rc == -5:
        raise NotImplementedError(msg)
    if rc == -6:
        raise NonFiniteInput(msg)
    raise SknnrError(msg)


def device_count() -> int:
    n = C.c_int(0)
    check(load().sknnr_device_count(C.byref(n)))
    return n.value


def set_option(name: str, value: int) -> None:
    check(load().sknnr_set_option(name.encode(), int(value)))


def host_chunk_plan(n_q: int, chunk_rows: int = 1 << 20) -> list[int]:
    """Rows per chunk of a host-buffer call (host code only: works without a device)."""
    n = C.c_int32(0)
    lib = load()
    check(lib.sknnr_host_chunk_plan(C.c_int64(n_q), C.c_int64(chunk_rows), None, 0, C.byref(n)))
    rows = (C.c_int64 * max(n.value, 1))()
    check(lib.sknnr_host_chunk_plan(C.c_int64(n_q), C.c_int64(chunk_rows), rows, n.value, C.byref(n)))
    return [int(rows[i]) for i in range(n.value)]


def measure_fp32_peak(device: int = 0) -> float:
    v = C.c_double(0.0)
    check(load().sknnr_measure_fp32_peak(device, C.byref(v)))
    return v.value
