"""Sorting many independent segments of a torch tensor of 16-bit keys in one call (b200sort_segmented_sort_keys16,
b200sort_segmented_pairs_keys16, b200sort_segmented_sort_indices_keys16 in include/b200sort.h).

Keys are int16, uint16, float16 or bfloat16, in the orders of ``b200sort.sort16`` (float16 and bfloat16: IEEE-754
totalOrder on the bit patterns, see ``keys16.py``).  Segments take the two forms of ``b200sort.segmented_sort``, and
the number of kernel launches does not depend on the number of segments.
"""
from __future__ import annotations

from ._lib import check, lib
from .keys16 import _key_type
from .segmented import _segments

_OTHERS = "32-bit keys: b200sort.segmented_sort"


def _workspace(torch, n: int, segments: int, device):
    ws_bytes = lib().b200sort_segmented16_workspace_bytes(n, segments)
    ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=device)
    return ws, ws.data_ptr() + (-ws.data_ptr()) % 256, ws_bytes


def segmented_sort16(keys, offsets=None, *, descending: bool = False):
    """A copy of ``keys`` (int16, uint16, float16 or bfloat16) with every segment sorted on its own; ``keys`` is left
    untouched.

    ``keys`` 1-D with ``offsets``: segment i is ``keys[offsets[i]:offsets[i+1]]``; ``offsets`` is a 1-D int32 or int64
    CUDA tensor of num_segments + 1 entries on the same device, checked with one host synchronisation.  ``keys`` 2-D
    contiguous with ``offsets=None``: every row is a segment, with no check and no synchronisation.  The result has
    ``keys``' shape.  Runs on ``torch.cuda.current_stream(keys.device)``.
    """
    import torch

    key_type = _key_type(torch, keys, _OTHERS)
    n, offs, segments = _segments(torch, keys, offsets)
    out = torch.empty_like(keys)
    if n == 0:
        return out
    with torch.cuda.device(keys.device):
        tmp = torch.empty_like(keys)
        ws, ws_ptr, ws_bytes = _workspace(torch, n, segments, keys.device)
        stream = torch.cuda.current_stream(keys.device).cuda_stream
        check(lib().b200sort_segmented_sort_keys16(key_type, int(bool(descending)), keys.data_ptr(), out.data_ptr(),
                                                   tmp.data_ptr(), n, offs.data_ptr(), segments, ws_ptr, ws_bytes,
                                                   stream))
    return out


def segmented_sort16_by_key(keys, values, offsets=None, *, descending: bool = False):
    """``(sorted keys, values in the same order)``: a STABLE sort by 16-bit key of every segment of (key, value) pairs.

    ``values``: int32 of ``keys``' shape on the same device.  Segments as in ``segmented_sort16``.  Equal keys keep
    their input order in both directions.  For every row's sorted keys with their int64 column indices (what
    ``torch.sort(logits, dim=-1, descending=True)`` returns for top-p sampling) call
    ``segmented_sort16_with_indices``: it makes the indices on the device.
    """
    import torch

    key_type = _key_type(torch, keys, _OTHERS)
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
        check(lib().b200sort_segmented_pairs_keys16(key_type, int(bool(descending)), keys.data_ptr(), values.data_ptr(),
                                                    k_out.data_ptr(), v_out.data_ptr(), k_tmp.data_ptr(),
                                                    v_tmp.data_ptr(), n, offs.data_ptr(), segments, ws_ptr, ws_bytes,
                                                    stream))
    return k_out, v_out


def segmented_sort16_with_indices(keys, offsets=None, *, descending: bool = False):
    """``(values, indices)``: every segment of ``keys`` (int16, uint16, float16 or bfloat16) sorted on its own, and the
    int64 position of every value inside its segment.

    Segments as in ``segmented_sort16``: the rows of a 2-D contiguous ``keys``, or the ``offsets`` ranges of a 1-D one.
    ``indices`` has ``keys``' shape; for rows it holds column indices, for offsets ``i - offsets[s]``.  ``keys`` is
    left untouched.  The sort is STABLE in both directions, so without NaN and -0.0 rows give exactly
    ``torch.sort(keys, dim=-1, stable=True, descending=descending)``, values and indices, dtype for dtype.  No index
    array is read: the kernels make the positions and store them as int64 the last time they move.  Runs on
    ``torch.cuda.current_stream(keys.device)``.
    """
    import torch

    key_type = _key_type(torch, keys, "32-bit keys: b200sort.segmented_sort_with_indices")
    n, offs, segments = _segments(torch, keys, offsets)
    values = torch.empty_like(keys)
    indices = torch.empty(keys.shape, dtype=torch.int64, device=keys.device)
    if n == 0:
        return values, indices
    with torch.cuda.device(keys.device):
        k_tmp = torch.empty_like(keys)
        i_tmp = torch.empty(n, dtype=torch.int32, device=keys.device)
        ws, ws_ptr, ws_bytes = _workspace(torch, n, segments, keys.device)
        stream = torch.cuda.current_stream(keys.device).cuda_stream
        check(lib().b200sort_segmented_sort_indices_keys16(key_type, int(bool(descending)), keys.data_ptr(),
                                                           values.data_ptr(), indices.data_ptr(), k_tmp.data_ptr(),
                                                           i_tmp.data_ptr(), n, offs.data_ptr(), segments, ws_ptr,
                                                           ws_bytes, stream))
    return values, indices
