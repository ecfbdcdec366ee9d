"""Sorting torch tensors of int32, uint32 or float32 keys, ascending or descending (b200sort_sort_keys,
b200sort_radix_pairs_keys in include/b200sort.h).

float32 keys are ordered by IEEE-754 totalOrder on their bit patterns:
-NaN < -inf < negatives < -0.0 < +0.0 < positives < +inf < +NaN, NaNs of one sign by payload.  That is not what
``torch.sort`` does (it treats -0.0 == +0.0 and puts every NaN last); on inputs without NaN and -0.0 the two agree.
The output holds the input's bit patterns, permuted.
"""
from __future__ import annotations

from ._lib import ALGO_MERGE, ALGO_RADIX, check, lib

KEY_I32 = 0
KEY_U32 = 1
KEY_F32 = 2
_ALGOS = {"radix": ALGO_RADIX, "merge": ALGO_MERGE}


def _key_type(torch, x) -> int:
    types = {torch.int32: KEY_I32, torch.uint32: KEY_U32, torch.float32: KEY_F32}
    if not isinstance(x, torch.Tensor):
        raise TypeError(f"expected a torch.Tensor, got {type(x).__name__}")
    if x.dtype not in types:
        raise TypeError(f"keys must be torch.int32, torch.uint32 or torch.float32, got {x.dtype}")
    return types[x.dtype]


def _check_layout(x, what: str) -> None:
    if x.dim() != 1 or not x.is_contiguous():
        raise ValueError(f"{what} must be a 1-D contiguous tensor, got shape {tuple(x.shape)}, "
                         f"strides {tuple(x.stride())}")
    if not x.is_cuda:
        raise ValueError(f"{what} must be a CUDA tensor (there is no CPU fallback), got device {x.device}")


def _workspace(torch, n: int, algo: int, device):
    ws_bytes = lib().b200sort_workspace_bytes(n, algo)
    ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=device)
    return ws, ws.data_ptr() + (-ws.data_ptr()) % 256, ws_bytes


def sort(x, *, descending: bool = False, algo: str = "radix"):
    """A sorted copy of the 1-D CUDA tensor ``x`` (int32, uint32 or float32); ``x`` is left untouched.

    ``algo`` is ``"radix"`` (onesweep LSD radix sort) or ``"merge"`` (block sort + merge-path merges); both give
    the same, unique, result.  float32 follows IEEE-754 totalOrder, not ``torch.sort`` (see the module docstring).
    Runs on ``torch.cuda.current_stream(x.device)``.
    """
    import torch

    key_type = _key_type(torch, x)
    _check_layout(x, "keys")
    if algo not in _ALGOS:
        raise ValueError(f"algo must be one of {sorted(_ALGOS)}, got {algo!r}")
    n = x.numel()
    out = torch.empty_like(x)
    if n == 0:
        return out
    with torch.cuda.device(x.device):
        tmp = torch.empty_like(x)
        ws, ws_ptr, ws_bytes = _workspace(torch, n, _ALGOS[algo], x.device)
        stream = torch.cuda.current_stream(x.device).cuda_stream
        check(lib().b200sort_sort_keys(_ALGOS[algo], key_type, int(bool(descending)), x.data_ptr(), out.data_ptr(),
                                       tmp.data_ptr(), n, ws_ptr, ws_bytes, stream))
    return out


def sort_by_key(keys, values, *, descending: bool = False):
    """``(sorted keys, values in the same order)``: a STABLE sort of (key, value) pairs by key on the radix path.

    ``keys``: 1-D CUDA tensor of int32, uint32 or float32; ``values``: int32 of the same length on the same device.
    Equal keys keep their input order in both directions, so a descending result is not the reverse of the
    ascending one.  The inputs are left untouched.  argsort::

        order = sort_by_key(x, torch.arange(n, dtype=torch.int32, device=x.device))[1]

    On inputs without NaN and -0.0 this equals ``torch.sort(x, stable=True, descending=descending)``, values and
    indices; float32 keys otherwise follow IEEE-754 totalOrder (see the module docstring).
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
        ws, ws_ptr, ws_bytes = _workspace(torch, n, ALGO_RADIX, keys.device)
        stream = torch.cuda.current_stream(keys.device).cuda_stream
        check(lib().b200sort_radix_pairs_keys(key_type, int(bool(descending)), keys.data_ptr(), values.data_ptr(),
                                              k_out.data_ptr(), v_out.data_ptr(), k_tmp.data_ptr(), v_tmp.data_ptr(),
                                              n, ws_ptr, ws_bytes, stream))
    return k_out, v_out
