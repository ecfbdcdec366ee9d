"""Sorting many independent segments of a torch tensor of 64-bit keys in one call (b200sort_segmented_sort_keys64,
b200sort_segmented_pairs_keys64 in include/b200sort.h).

Keys are int64, uint64 or float64, in the orders of ``b200sort.sort64`` (float64: IEEE-754 totalOrder on the bit
patterns, see ``keys64.py``).  Segments take the two forms of ``b200sort.segmented_sort``, and the number of kernel
launches depends neither on the number of segments nor on the data.  Digit passes in which every key of a segment
agrees are skipped on the device, so rows of int64 ids below 2^32 cost about half of what rows of full-width keys do.
"""
from __future__ import annotations

from ._lib import check, lib
from .keys64 import KEY_F64, KEY_I64, KEY_U64
from .segmented import _segments


def _key_type(torch, x) -> int:
    types = {torch.int64: KEY_I64, torch.uint64: KEY_U64, torch.float64: KEY_F64}
    if not isinstance(x, torch.Tensor):
        raise TypeError(f"expected a torch.Tensor, got {type(x).__name__}")
    if x.dtype not in types:
        raise TypeError(f"keys must be torch.int64, torch.uint64 or torch.float64, got {x.dtype} "
                        f"(32-bit keys: b200sort.segmented_sort; 16-bit keys: b200sort.segmented_sort16)")
    return types[x.dtype]


def _workspace(torch, n: int, segments: int, device):
    ws_bytes = lib().b200sort_segmented64_workspace_bytes(n, segments)
    ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=device)
    return ws, ws.data_ptr() + (-ws.data_ptr()) % 256, ws_bytes


def segmented_sort64(keys, offsets=None, *, descending: bool = False):
    """A copy of ``keys`` (int64, uint64 or float64) with every segment sorted on its own; ``keys`` is left untouched.

    ``keys`` 1-D with ``offsets``: segment i is ``keys[offsets[i]:offsets[i+1]]``; ``offsets`` is a 1-D int32 or int64
    CUDA tensor of num_segments + 1 entries on the same device, checked with one host synchronisation.  ``keys`` 2-D
    contiguous with ``offsets=None``: every row is a segment, with no check and no synchronisation.  The result has
    ``keys``' shape.  Runs on ``torch.cuda.current_stream(keys.device)``.
    """
    import torch

    key_type = _key_type(torch, keys)
    n, offs, segments = _segments(torch, keys, offsets)
    out = torch.empty_like(keys)
    if n == 0:
        return out
    with torch.cuda.device(keys.device):
        tmp = torch.empty_like(keys)
        ws, ws_ptr, ws_bytes = _workspace(torch, n, segments, keys.device)
        stream = torch.cuda.current_stream(keys.device).cuda_stream
        check(lib().b200sort_segmented_sort_keys64(key_type, int(bool(descending)), keys.data_ptr(), out.data_ptr(),
                                                   tmp.data_ptr(), n, offs.data_ptr(), segments, ws_ptr, ws_bytes,
                                                   stream))
    return out


def segmented_sort64_by_key(keys, values, offsets=None, *, descending: bool = False):
    """``(sorted keys, values in the same order)``: a STABLE sort by 64-bit key of every segment of (key, value) pairs.

    ``values``: int32 of ``keys``' shape on the same device.  Segments as in ``segmented_sort64``.  Equal keys keep
    their input order in both directions.  The neighbour ids of every node of a CSR graph, sorted with their edge
    numbers::

        e = torch.arange(ids.numel(), dtype=torch.int32, device=ids.device)
        sorted_ids, edges = segmented_sort64_by_key(ids, e, rowptr)

    Without NaN and -0.0 this equals ``torch.sort(x, dim=-1, stable=True, descending=...)`` in values and indices (as
    int32).
    """
    import torch

    key_type = _key_type(torch, keys)
    if not isinstance(values, torch.Tensor):
        raise TypeError(f"expected a torch.Tensor of values, got {type(values).__name__}")
    if values.dtype != torch.int32:
        raise TypeError(f"values must be torch.int32, got {values.dtype}")
    if values.shape != keys.shape or not values.is_contiguous():
        raise ValueError(f"values must be contiguous with keys' shape {tuple(keys.shape)}, got {tuple(values.shape)}")
    if values.device != keys.device:
        raise ValueError(f"keys and values are on different devices: {keys.device} and {values.device}")
    n, offs, segments = _segments(torch, keys, offsets)
    k_out, v_out = torch.empty_like(keys), torch.empty_like(values)
    if n == 0:
        return k_out, v_out
    with torch.cuda.device(keys.device):
        k_tmp, v_tmp = torch.empty_like(keys), torch.empty_like(values)
        ws, ws_ptr, ws_bytes = _workspace(torch, n, segments, keys.device)
        stream = torch.cuda.current_stream(keys.device).cuda_stream
        check(lib().b200sort_segmented_pairs_keys64(key_type, int(bool(descending)), keys.data_ptr(), values.data_ptr(),
                                                    k_out.data_ptr(), v_out.data_ptr(), k_tmp.data_ptr(),
                                                    v_tmp.data_ptr(), n, offs.data_ptr(), segments, ws_ptr, ws_bytes,
                                                    stream))
    return k_out, v_out
