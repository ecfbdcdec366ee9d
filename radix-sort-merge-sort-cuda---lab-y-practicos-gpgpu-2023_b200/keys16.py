"""Sorting torch tensors of int16, uint16, float16 or bfloat16 keys, ascending or descending (b200sort_sort_keys16,
b200sort_radix_pairs_keys16 in include/b200sort.h).

float16 and bfloat16 keys are ordered by IEEE-754 totalOrder on their bit patterns, as float32 keys are in
``b200sort.sort``: -NaN < -inf < negatives < -0.0 < +0.0 < positives < +inf < +NaN, NaNs of one sign by payload.
That is not what ``torch.sort`` does (it treats -0.0 == +0.0 and puts every NaN last); on inputs without NaN and -0.0
the two agree.  The output holds the input's bit patterns, permuted.
"""
from __future__ import annotations

from ._lib import check, lib
from .keys import _check_layout

KEY_I16 = 6
KEY_U16 = 7
KEY_F16 = 8
KEY_BF16 = 9


def _key_type(torch, x, others: str = "32-bit keys: b200sort.sort; 64-bit keys: b200sort.sort64") -> int:
    types = {torch.int16: KEY_I16, torch.uint16: KEY_U16, torch.float16: KEY_F16, torch.bfloat16: KEY_BF16}
    if not isinstance(x, torch.Tensor):
        raise TypeError(f"expected a torch.Tensor, got {type(x).__name__}")
    if x.dtype not in types:
        raise TypeError(f"keys must be torch.int16, torch.uint16, torch.float16 or torch.bfloat16, got {x.dtype} "
                        f"({others})")
    return types[x.dtype]


def _workspace(torch, n: int, device):
    ws_bytes = lib().b200sort_keys16_workspace_bytes(n)
    ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=device)
    return ws, ws.data_ptr() + (-ws.data_ptr()) % 256, ws_bytes


def sort16(x, *, descending: bool = False):
    """A sorted copy of the 1-D CUDA tensor ``x`` (int16, uint16, float16 or bfloat16); ``x`` is left untouched.

    A counting sort: one read of ``x`` counts each of the 65536 bit patterns, and the output is written pattern by
    pattern.  float16 and bfloat16 follow IEEE-754 totalOrder, not ``torch.sort`` (see the module docstring).  Runs
    on ``torch.cuda.current_stream(x.device)``.
    """
    import torch

    key_type = _key_type(torch, x)
    _check_layout(x, "keys")
    n = x.numel()
    out = torch.empty_like(x)
    if n == 0:
        return out
    with torch.cuda.device(x.device):
        ws, ws_ptr, ws_bytes = _workspace(torch, n, x.device)
        stream = torch.cuda.current_stream(x.device).cuda_stream
        check(lib().b200sort_sort_keys16(key_type, int(bool(descending)), x.data_ptr(), out.data_ptr(), n, ws_ptr,
                                         ws_bytes, stream))
    return out


def sort16_by_key(keys, values, *, descending: bool = False):
    """``(sorted keys, values in the same order)``: a STABLE sort of (16-bit key, int32 value) pairs by key.

    ``keys``: 1-D CUDA tensor of int16, uint16, float16 or bfloat16; ``values``: int32 of the same length on the
    same device.  Equal keys keep their input order in both directions.  The inputs are left untouched.  argsort::

        order = sort16_by_key(x, torch.arange(n, dtype=torch.int32, device=x.device))[1]

    On inputs without NaN and -0.0 this equals ``torch.sort(x, stable=True, descending=descending)``, values and
    indices (as int32).
    """
    import torch

    key_type = _key_type(torch, keys)
    if not isinstance(values, torch.Tensor):
        raise TypeError(f"expected a torch.Tensor of values, got {type(values).__name__}")
    if values.dtype != torch.int32:
        raise TypeError(f"values must be torch.int32, got {values.dtype}")
    _check_layout(keys, "keys")
    _check_layout(values, "values")
    if values.numel() != keys.numel():
        raise ValueError(f"keys and values differ in length: {keys.numel()} and {values.numel()}")
    if values.device != keys.device:
        raise ValueError(f"keys and values are on different devices: {keys.device} and {values.device}")
    n = keys.numel()
    k_out, v_out = torch.empty_like(keys), torch.empty_like(values)
    if n == 0:
        return k_out, v_out
    with torch.cuda.device(keys.device):
        k_tmp, v_tmp = torch.empty_like(keys), torch.empty_like(values)
        ws, ws_ptr, ws_bytes = _workspace(torch, n, keys.device)
        stream = torch.cuda.current_stream(keys.device).cuda_stream
        check(lib().b200sort_radix_pairs_keys16(key_type, int(bool(descending)), keys.data_ptr(), values.data_ptr(),
                                                k_out.data_ptr(), v_out.data_ptr(), k_tmp.data_ptr(), v_tmp.data_ptr(),
                                                n, ws_ptr, ws_bytes, stream))
    return k_out, v_out
