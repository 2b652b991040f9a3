"""ctypes binding of libbmx.so (include/bmx.h).  Fails loudly when the library is missing."""
from __future__ import annotations

import ctypes
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_uint64, c_void_p
from pathlib import Path

import os

# BMX_LIB points the binding at another build of the same ABI (A/B runs in profiles/); default: in-tree
LIB_PATH = Path(os.environ.get("BMX_LIB") or Path(__file__).resolve().parent / "libbmx.so")

BMX_OK = 0
BMX_E_BADARG = -1
BMX_E_CUDA = -2
BMX_E_NOMEM = -3
BMX_E_NODEVICE = -4
BMX_E_TABLES = -5
BMX_E_EXCHANGE = -6

VARIANT_AUTO = 0
VARIANT_QGRAM = 1
VARIANT_WINDOW = 2
VARIANT_SHIFTAND = 3
VARIANT_NAMES = {0: "auto", 1: "qgram", 2: "window", 3: "shiftand"}
IGNORE_CASE = 0x100   # BMX_IGNORE_CASE: OR'ed into a variant, ASCII case-insensitive search

# every symbol include/bmx.h declares (tests/test_host_logic.py checks the header against this list)
EXPORTS = [
    "bmx_version", "bmx_last_error", "bmx_device_count", "bmx_build_tables", "bmx_search",
    "bmx_search_ex", "bmx_search_device", "bmx_search_device_ex", "bmx_search_partitions",
    "bmx_find_first", "bmx_find_first_device", "bmx_search_multi",
    "bmx_scanner_create", "bmx_scanner_destroy", "bmx_scanner_set_pattern", "bmx_scanner_begin",
    "bmx_scanner_scan", "bmx_scanner_finish", "bmx_scanner_export_result", "bmx_scanner_set_timing", "bmx_mg_create", "bmx_mg_destroy", "bmx_mg_device_count", "bmx_mg_search", "bmx_synth_fill_device", "bmx_partition_words",
    "bmx_mg_search_device", "bmx_exchange_create", "bmx_exchange_destroy", "bmx_exchange_handle", "bmx_exchange_connect",
    "bmx_exchange_connect_local", "bmx_exchange_post", "bmx_exchange_collect", "bmx_exchange_wait", "bmx_release_memory", "bmx_search_multi_device",
    "bmx_search_ranges", "bmx_search_ranges_device",
    "bmx_dict_create", "bmx_dict_destroy", "bmx_dict_search", "bmx_dict_search_device",
]


class BmxStats(ctypes.Structure):
    _fields_ = [
        ("device_ms", c_float),
        ("variant", c_int32),
        ("kernel_launches", c_int32),
        ("grid", c_int32),
        ("stages", c_int32),
        ("tile_bytes", c_int32),
        ("smem_bytes", c_int32),
        ("tiles", c_int64),
        ("scan_kernel_ms", c_float),
        ("reserved", c_int32),
    ]

    def as_dict(self) -> dict:
        d = {name: getattr(self, name) for name, _ in self._fields_}
        v = d["variant"]
        d["variant"] = VARIANT_NAMES.get(v & ~IGNORE_CASE, str(v))
        d["ignore_case"] = bool(v & IGNORE_CASE)   # the case-folding kernels ran
        return d


class BmxError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"bmx error {code}: {message}")
        self.code = code


_lib = None


def load() -> ctypes.CDLL:
    """Load libbmx.so.  There is no fallback: a missing library is an error."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  This package has no CPU or PyTorch fallback."
        )
    lib = ctypes.CDLL(str(LIB_PATH))
    lib.bmx_version.restype = c_int
    lib.bmx_last_error.restype = c_char_p
    lib.bmx_device_count.restype = c_int
    lib.bmx_build_tables.argtypes = [c_char_p, c_int32, POINTER(c_int32), POINTER(c_int32)]
    lib.bmx_search.argtypes = [c_void_p, c_int64, c_char_p, c_int32, c_void_p, c_int64, POINTER(c_uint64)]
    lib.bmx_search_ex.argtypes = [c_int, c_void_p, c_int64, c_char_p, c_int32, c_void_p, c_int64,
                                  POINTER(c_uint64), c_int32, POINTER(BmxStats)]
    lib.bmx_search_device.argtypes = [c_void_p, c_int64, c_char_p, c_int32, c_void_p, c_int64,
                                      POINTER(c_uint64), POINTER(c_float), c_void_p]
    lib.bmx_search_device_ex.argtypes = [c_void_p, c_int64, c_char_p, c_int32, c_int64, c_void_p, c_int64,
                                         POINTER(c_uint64), c_int32, POINTER(BmxStats), c_void_p]
    lib.bmx_search_multi.argtypes = [c_int, c_void_p, c_int64, c_int32, POINTER(c_char_p), POINTER(c_int32),
                                     POINTER(c_void_p), POINTER(c_int64), POINTER(c_uint64)]
    lib.bmx_search_multi_device.argtypes = [c_void_p, c_int64, c_int32, POINTER(c_char_p), POINTER(c_int32),
                                            POINTER(c_void_p), POINTER(c_int64), POINTER(c_uint64), c_void_p]
    lib.bmx_find_first.argtypes = [c_void_p, c_int64, c_char_p, c_int32, POINTER(c_int64)]
    lib.bmx_find_first_device.argtypes = [c_void_p, c_int64, c_char_p, c_int32, POINTER(c_int64), c_void_p]
    lib.bmx_search_partitions.argtypes = [c_void_p, c_char_p, POINTER(c_int32), POINTER(c_int32),
                                          POINTER(c_int32), POINTER(c_int32), c_int32, c_int32]
    lib.bmx_search_ranges.argtypes = [c_int, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_char_p, c_int32,
                                      c_void_p, c_int64, c_void_p, c_void_p]
    lib.bmx_search_ranges_device.argtypes = [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_char_p, c_int32,
                                             c_void_p, c_int64, c_void_p, c_void_p, POINTER(c_uint64), c_void_p]
    lib.bmx_dict_create.argtypes = [c_int, c_int32, POINTER(c_char_p), POINTER(c_int32), POINTER(c_void_p)]
    lib.bmx_dict_destroy.argtypes = [c_void_p]
    lib.bmx_dict_destroy.restype = None
    lib.bmx_dict_search.argtypes = [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p, POINTER(c_uint64)]
    lib.bmx_dict_search_device.argtypes = [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_void_p,
                                           POINTER(c_uint64), c_void_p]
    lib.bmx_scanner_create.argtypes = [c_int, POINTER(c_void_p)]
    lib.bmx_scanner_destroy.argtypes = [c_void_p]
    lib.bmx_scanner_destroy.restype = None
    lib.bmx_scanner_set_pattern.argtypes = [c_void_p, c_char_p, c_int32, c_int32, c_void_p]
    lib.bmx_scanner_begin.argtypes = [c_void_p, c_void_p, c_int64, c_void_p]
    lib.bmx_scanner_scan.argtypes = [c_void_p, c_void_p, c_int64, c_int64, c_void_p]
    lib.bmx_scanner_set_timing.argtypes = [c_void_p, c_int]
    lib.bmx_scanner_export_result.argtypes = [c_void_p, c_void_p, c_int64, c_void_p]
    lib.bmx_scanner_finish.argtypes = [c_void_p, POINTER(c_uint64), POINTER(BmxStats), c_void_p]
    lib.bmx_partition_words.argtypes = [c_void_p, c_int64, c_int32, POINTER(c_int32)]
    lib.bmx_mg_create.argtypes = [c_int, POINTER(c_void_p)]
    lib.bmx_mg_destroy.argtypes = [c_void_p]
    lib.bmx_mg_destroy.restype = None
    lib.bmx_mg_device_count.argtypes = [c_void_p]
    lib.bmx_mg_device_count.restype = c_int
    lib.bmx_mg_search.argtypes = [c_void_p, c_void_p, c_int64, c_char_p, c_int32, c_void_p, c_int64, POINTER(c_uint64), POINTER(c_uint64)]
    lib.bmx_mg_search_device.argtypes = [c_void_p, POINTER(c_void_p), POINTER(c_int64), POINTER(c_int64), c_char_p, c_int32,
                                         c_void_p, c_int64, POINTER(c_uint64), POINTER(c_uint64)]
    lib.bmx_exchange_create.argtypes = [c_int, c_int, c_int, c_int, c_int64, c_int64, c_int, POINTER(c_void_p)]
    lib.bmx_exchange_destroy.argtypes = [c_void_p]
    lib.bmx_exchange_destroy.restype = None
    lib.bmx_exchange_handle.argtypes = [c_void_p, c_void_p]
    lib.bmx_exchange_connect.argtypes = [c_void_p, c_void_p]
    lib.bmx_exchange_connect_local.argtypes = [POINTER(c_void_p), c_int]
    lib.bmx_exchange_post.argtypes = [c_void_p, c_void_p, c_void_p, POINTER(c_uint64)]
    lib.bmx_exchange_collect.argtypes = [c_void_p, c_void_p, c_int64, c_void_p, POINTER(c_uint64)]
    lib.bmx_exchange_wait.argtypes = [c_void_p, c_uint64, POINTER(c_uint64), POINTER(c_uint64), POINTER(c_int64)]
    lib.bmx_release_memory.argtypes = [c_int]
    lib.bmx_synth_fill_device.argtypes = [c_void_p, c_int64, c_int64, c_uint64, c_char_p, c_int32, c_void_p]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if fn.restype is c_int and name not in ("bmx_version", "bmx_device_count"):
            fn.restype = c_int
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != BMX_OK:
        raise BmxError(rc, load().bmx_last_error().decode("utf-8", "replace"))
