"""Sorting many independent segments of a torch tensor in one call (b200sort_segmented_sort_keys,
b200sort_segmented_pairs_keys, b200sort_segmented_sort_indices_keys in include/b200sort.h).

Keys are int32, uint32 or float32, in the orders of ``b200sort.sort`` (float32: IEEE-754 totalOrder on the bit
patterns, see ``keys.py``).  The number of kernel launches does not depend on the number of segments.
"""
from __future__ import annotations

from ._lib import check, lib
from .keys import _check_layout, _key_type


def _segments(torch, keys, offsets):
    """(n, int32 offsets on keys' device, number of segments) for a 1-D ``keys`` with ``offsets`` or a 2-D ``keys``."""
    if offsets is None:
        if keys.dim() != 2 or not keys.is_contiguous():
            raise ValueError(f"without offsets keys must be a 2-D contiguous tensor (one segment per row), got shape "
                             f"{tuple(keys.shape)}, strides {tuple(keys.stride())}")
        if not keys.is_cuda:
            raise ValueError(f"keys must be a CUDA tensor (there is no CPU fallback), got device {keys.device}")
        rows, length = keys.shape
        if keys.numel() >= 1 << 31:
            raise ValueError(f"{keys.numel()} keys: segment offsets are int32")
        return keys.numel(), torch.arange(0, rows + 1, dtype=torch.int64, device=keys.device).mul_(length).to(torch.int32), rows
    _check_layout(keys, "keys (with offsets)")
    if not isinstance(offsets, torch.Tensor):
        raise TypeError(f"expected a torch.Tensor of offsets, got {type(offsets).__name__}")
    if offsets.dtype not in (torch.int32, torch.int64):
        raise TypeError(f"offsets must be torch.int32 or torch.int64, got {offsets.dtype}")
    if offsets.dim() != 1 or offsets.numel() < 1:
        raise ValueError(f"offsets must be a 1-D tensor of num_segments + 1 entries, got shape {tuple(offsets.shape)}")
    if offsets.device != keys.device:
        raise ValueError(f"keys and offsets are on different devices: {keys.device} and {offsets.device}")
    n = keys.numel()
    # first, last and "decreases somewhere", fetched in one copy: the one host synchronisation of the check
    first, last, bad = torch.stack([offsets[0], offsets[-1],
                                    (offsets[1:] < offsets[:-1]).any().to(offsets.dtype)]).tolist()
    if first != 0 or last != n or bad:
        raise ValueError(f"offsets must start at 0, end at n = {n} and never decrease (got first {first}, last {last}"
                         f"{', a decrease' if bad else ''})")
    return n, offsets.to(torch.int32).contiguous(), offsets.numel() - 1


def _workspace(torch, n: int, segments: int, device):
    ws_bytes = lib().b200sort_segmented_workspace_bytes(n, segments)
    ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=device)
    return ws, ws.data_ptr() + (-ws.data_ptr()) % 256, ws_bytes


def segmented_sort(keys, offsets=None, *, descending: bool = False):
    """A copy of ``keys`` with every segment sorted on its own; ``keys`` is left untouched.

    ``keys`` 1-D (int32, uint32 or float32) with ``offsets``: segment i is ``keys[offsets[i]:offsets[i+1]]``.
    ``offsets`` is a 1-D int32 or int64 CUDA tensor of num_segments + 1 entries on the same device; it is checked
    for ``offsets[0] == 0``, ``offsets[-1] == n`` and for never decreasing, which costs one host synchronisation.
    ``keys`` 2-D contiguous with ``offsets=None``: every row is a segment, like ``torch.sort(keys, dim=-1)``, with no
    check and no synchronisation.  The result has ``keys``' shape.  Runs on ``torch.cuda.current_stream(keys.device)``.
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
        check(lib().b200sort_segmented_sort_keys(key_type, int(bool(descending)), keys.data_ptr(), out.data_ptr(),
                                                 tmp.data_ptr(), n, offs.data_ptr(), segments, ws_ptr, ws_bytes, stream))
    return out


def segmented_sort_by_key(keys, values, offsets=None, *, descending: bool = False):
    """``(sorted keys, values in the same order)``: a STABLE sort by key of every segment of (key, value) pairs.

    ``values``: int32 of ``keys``' shape on the same device.  Segments as in ``segmented_sort``.  Equal keys keep
    their input order in both directions.  For every row's sorted keys with their int64 column indices (what
    ``torch.sort(x, dim=-1)`` returns) call ``segmented_sort_with_indices``: it makes the indices on the device.
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
        check(lib().b200sort_segmented_pairs_keys(key_type, int(bool(descending)), keys.data_ptr(), values.data_ptr(),
                                                  k_out.data_ptr(), v_out.data_ptr(), k_tmp.data_ptr(), v_tmp.data_ptr(),
                                                  n, offs.data_ptr(), segments, ws_ptr, ws_bytes, stream))
    return k_out, v_out


def segmented_sort_with_indices(keys, offsets=None, *, descending: bool = False):
    """``(values, indices)``: every segment of ``keys`` sorted on its own, and the int64 position of every value
    inside its segment.

    Segments as in ``segmented_sort``: the rows of a 2-D contiguous ``keys``, or the ``offsets`` ranges of a 1-D one.
    ``indices`` has ``keys``' shape; for rows it holds column indices, for offsets ``i - offsets[s]``.  ``keys`` is
    left untouched.  The sort is STABLE in both directions, so without NaN and -0.0 rows give exactly
    ``torch.sort(keys, dim=-1, stable=True, descending=descending)``, values and indices, dtype for dtype.  No index
    array is read: the kernels make the positions and store them as int64 the last time they move.  Runs on
    ``torch.cuda.current_stream(keys.device)``.
    """
    import torch

    key_type = _key_type(torch, keys, "16-bit keys: b200sort.segmented_sort16_with_indices")
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
        check(lib().b200sort_segmented_sort_indices_keys(key_type, int(bool(descending)), keys.data_ptr(),
                                                         values.data_ptr(), indices.data_ptr(), k_tmp.data_ptr(),
                                                         i_tmp.data_ptr(), n, offs.data_ptr(), segments, ws_ptr,
                                                         ws_bytes, stream))
    return values, indices
