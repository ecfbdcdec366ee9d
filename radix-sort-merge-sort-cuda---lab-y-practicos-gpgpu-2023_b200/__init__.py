"""b200sort -- B200-native (sm_100a) radix sort and merge sort of 32-bit signed keys behind the
GPGPU-2023 lab's operator boundary (``order_array`` / ``order_with_trust``,
/root/reference/Sord Radix y Merge/include/lab.h:9-10).

The product is ``libb200sort.so`` (hand-written CUDA + a C-ABI, see include/b200sort.h); this
package is the thin host-side mirror of that interface used by the tests, the drivers and
bench.py.  ``sort`` / ``sort_by_key`` (keys.py) sort torch CUDA tensors of int32, uint32 or float32
keys, ascending or descending; ``sort64`` / ``sort64_by_key`` (keys64.py) the same for int64, uint64 or float64
keys; ``sort16`` / ``sort16_by_key`` (keys16.py) for int16, uint16, float16 or bfloat16 keys;
``segmented_sort`` / ``segmented_sort_by_key`` (segmented.py) sort every
segment (row, or offsets range) of one tensor on its own in one call; ``sort_with_indices`` (keys.py) and
``segmented_sort_with_indices`` (segmented.py) return the sorted 32-bit keys with their int64 positions, as
``torch.sort`` does, and ``sort16_with_indices`` (keys16.py) and ``segmented_sort16_with_indices`` (segmented16.py)
the sorted 16-bit keys with theirs; ``segmented_sort16`` /
``segmented_sort16_by_key`` (segmented16.py) and ``segmented_sort64`` / ``segmented_sort64_by_key`` (segmented64.py)
do the same for 16-bit and 64-bit keys.  There is no CPU fallback anywhere: every sort call fails loudly
without the CUDA library or without an sm_100 device.
"""
from ._lib import (ALGO_LAB, ALGO_MERGE, ALGO_RADIX, B200SortError, lib, lib_path, check)  # noqa: F401
from .lab import order_array, order_with_trust  # noqa: F401
from .keys import KEY_F32, KEY_I32, KEY_U32, sort, sort_by_key, sort_with_indices  # noqa: F401
from .keys64 import KEY_F64, KEY_I64, KEY_U64, sort64, sort64_by_key  # noqa: F401
from .keys16 import KEY_BF16, KEY_F16, KEY_I16, KEY_U16, sort16, sort16_by_key, sort16_with_indices  # noqa: F401
from .segmented import segmented_sort, segmented_sort_by_key, segmented_sort_with_indices  # noqa: F401
from .segmented16 import segmented_sort16, segmented_sort16_by_key, segmented_sort16_with_indices  # noqa: F401
from .segmented64 import segmented_sort64, segmented_sort64_by_key  # noqa: F401
from . import datagen  # noqa: F401

__all__ = ["order_array", "order_with_trust", "sort", "sort_by_key", "sort64", "sort64_by_key", "sort16",
           "sort16_by_key", "segmented_sort", "segmented_sort_by_key", "segmented_sort16", "segmented_sort16_by_key",
           "segmented_sort64", "segmented_sort64_by_key", "sort_with_indices", "segmented_sort_with_indices",
           "sort16_with_indices", "segmented_sort16_with_indices",
           "lib", "lib_path", "B200SortError", "ALGO_RADIX", "ALGO_MERGE", "ALGO_LAB", "KEY_I32", "KEY_U32", "KEY_F32", "KEY_I64", "KEY_U64", "KEY_F64", "KEY_I16",
           "KEY_U16", "KEY_F16", "KEY_BF16", "datagen"]
