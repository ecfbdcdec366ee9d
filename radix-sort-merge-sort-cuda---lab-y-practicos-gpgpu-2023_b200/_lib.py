"""ctypes binding of libb200sort.so (include/b200sort.h).  Fails loudly if the library is absent."""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_NAME = os.environ.get("B200SORT_LIB", "libb200sort.so")     # libb200sort_checked.so: make checked

ALGO_RADIX = 0
ALGO_MERGE = 1
ALGO_LAB = 2
MAX_N = 1 << 30

_STATUS = {0: "ok", 1: "invalid argument", 2: "workspace", 3: "CUDA runtime error",
           4: "no sm_100 device", 5: "allocation failed"}


class B200SortError(RuntimeError):
    def __init__(self, status: int, detail: str = ""):
        self.status = status
        super().__init__(f"b200sort status {status} ({_STATUS.get(status, '?')}){': ' + detail if detail else ''}")


def lib_path() -> str:
    return os.path.join(_HERE, _LIB_NAME)


# name -> (restype, argtypes); every symbol include/b200sort.h declares
_vp, _sz, _i, _u64 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_ulonglong
SIGNATURES = {
    "b200sort_version": (ctypes.c_char_p, []),
    "b200sort_status_string": (ctypes.c_char_p, [_i]),
    "b200sort_last_cuda_error": (_i, []),
    "b200sort_last_cuda_error_string": (ctypes.c_char_p, []),
    "b200sort_device_check": (_i, []),
    "b200sort_workspace_bytes": (_sz, [_sz, _i]),
    "b200sort_radix_i32": (_i, [_vp, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_merge_i32": (_i, [_vp, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_radix_pairs_i32": (_i, [_vp, _vp, _vp, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_radix_pairs_copy_i32": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_lab_i32": (_i, [_vp, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_lab_tile_sort_i32": (_i, [_vp, _vp, _sz, _vp]),
    "b200sort_sort_i32": (_i, [_i, _vp, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_sort_copy_i32": (_i, [_i, _vp, _vp, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_sort_timed_i32": (_i, [_i, _vp, _vp, _vp, _sz, _vp, _sz, _vp, _vp]),
    "b200sort_sort_keys": (_i, [_i, _i, _i, _vp, _vp, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_radix_pairs_keys": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_keys64_workspace_bytes": (_sz, [_sz]),
    "b200sort_sort_keys64": (_i, [_i, _i, _vp, _vp, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_radix_pairs_keys64": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_keys16_workspace_bytes": (_sz, [_sz]),
    "b200sort_sort_keys16": (_i, [_i, _i, _vp, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_radix_pairs_keys16": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_segmented_workspace_bytes": (_sz, [_sz, _sz]),
    "b200sort_segmented_sort_keys": (_i, [_i, _i, _vp, _vp, _vp, _sz, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_segmented_pairs_keys": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_segmented_class_max": (_sz, [_i]),
    "b200sort_segmented16_workspace_bytes": (_sz, [_sz, _sz]),
    "b200sort_segmented16_class_max": (_sz, [_i]),
    "b200sort_segmented_sort_keys16": (_i, [_i, _i, _vp, _vp, _vp, _sz, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_segmented_pairs_keys16": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_segmented64_workspace_bytes": (_sz, [_sz, _sz]),
    "b200sort_segmented64_class_max": (_sz, [_i]),
    "b200sort_segmented_sort_keys64": (_i, [_i, _i, _vp, _vp, _vp, _sz, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_segmented_pairs_keys64": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_radix_sort_indices_keys": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_segmented_sort_indices_keys": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_radix_sort_indices_keys16": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_segmented_sort_indices_keys16": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _sz, _vp, _sz, _vp]),
    "b200sort_radix_histogram_i32": (_i, [_vp, _sz, _vp, _vp]),
    "b200sort_radix_pass_i32": (_i, [_vp, _vp, _sz, _i, _vp, _sz, _vp]),
    "b200sort_block_sort_tile": (_sz, []),
    "b200sort_block_sort_i32": (_i, [_vp, _vp, _sz, _vp]),
    "b200sort_merge_tile": (_sz, []),
    "b200sort_merge_partition_i32": (_i, [_vp, _sz, _sz, _vp, _vp]),
    "b200sort_merge_pass_i32": (_i, [_vp, _vp, _sz, _sz, _vp, _vp]),
    "b200sort_radix_set_variant": (_i, [_i]),
    "b200sort_radix_num_variants": (_i, []),
    "b200sort_radix_variant_name": (ctypes.c_char_p, [_i]),
    "b200sort_radix_tile": (_sz, []),
    "b200sort_merge_set_variant": (_i, [_i]),
    "b200sort_merge_num_variants": (_i, []),
    "b200sort_merge_variant_name": (ctypes.c_char_p, [_i]),
    "b200sort_radix_set_skip": (_i, [_i]),
    "b200sort_debug_set_phase_buffer": (_i, [_vp]),
    "b200sort_radix_atomic_order_ok": (_i, []),
    "b200sort_debug_checked_build": (_i, []),
    "b200sort_debug_check_failures": (_u64, []),
    "b200sort_debug_check_failures_by_site": (_u64, [_vp]),
    "b200sort_radix_effective_variant_name": (ctypes.c_char_p, []),
    "b200sort_launch_count": (_u64, []),
    "b200sort_launch_count_reset": (None, []),
    "b200sort_dist_histogram_i32": (_i, [_vp, _sz, _i, _vp, _vp]),
    "b200sort_dist_plan": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "b200sort_dist_workspace_bytes": (_sz, [_sz, _i]),
    "b200sort_dist_partition_i32": (_i, [_vp, _sz, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "b200sort_dist_plan_device": (_i, [_vp, _i, _i, _i, _u64, _vp, _vp, _vp, _sz, _vp]),
    "b200sort_dist_partition_planned_i32": (_i, [_vp, _sz, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "b200sort_radix_copy_devn_i32": (_i, [_vp, _vp, _vp, _sz, _vp, _vp, _vp, _sz, _vp]),
    "b200sort_device_malloc": (_i, [ctypes.POINTER(_vp), _sz]),
    "b200sort_device_free": (_i, [_vp]),
    "b200sort_ipc_export": (_i, [_vp, _vp]),
    "b200sort_ipc_open": (_i, [_vp, ctypes.POINTER(_vp)]),
    "b200sort_ipc_close": (_i, [_vp]),
    "b200sort_order_array_host": (_i, [_vp, _sz, _i]),
    "b200sort_host_set_streaming": (_i, [_i]),
    "b200sort_order_with_trust_host": (_i, [_vp, _sz]),
    "b200sort_host_release": (None, []),
    "b200sort_host_alloc_pinned": (_i, [ctypes.POINTER(_vp), _sz]),
    "b200sort_host_free_pinned": (_i, [_vp]),
}
# the C++ symbols of include/lab.h
LAB_SYMBOLS = {"_Z11order_arrayPii": (None, [_vp, _i]), "_Z16order_with_trustPii": (None, [_vp, _i])}

_lib = None


def lib() -> ctypes.CDLL:
    """The loaded library; raises if it has not been built (``make`` / ``__graft_entry__.build()``)."""
    global _lib
    if _lib is None:
        path = lib_path()
        if not os.path.exists(path):
            raise FileNotFoundError(
                f"{path} is missing: build it with `make` (there is no CPU fallback)")
        handle = ctypes.CDLL(path)
        for name, (res, args) in {**SIGNATURES, **LAB_SYMBOLS}.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(status: int) -> None:
    if status != 0:
        detail = ""
        if status == 3:
            detail = lib().b200sort_last_cuda_error_string().decode()
        raise B200SortError(status, detail)
