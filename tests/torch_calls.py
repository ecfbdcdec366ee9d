"""The torch-facing sorts as one table, with the inputs, data sets and numpy references that tests of their calling
contexts share (tests/test_torch_capture_gpu.py: capture as a process's first call, side streams; and
tests/test_torch_api_cpu.py: the table covers every function).  Test infrastructure only.

Every entry names one function of ``b200sort`` with one key type and order, its form (1-D or rows of a 2-D tensor)
and what it returns (sorted keys; keys and int32 values; keys and int64 indices).  References are stable numpy
argsorts of the key images (key_orders*.py), per row with np.lexsort, and for indices the references of
test_sort_indices*_cpu.py; results are compared byte for byte.  numpy and torch are imported here, the library is
not loaded: a child process can build its inputs before its first library call.
"""
from __future__ import annotations

from typing import NamedTuple

import numpy as np

import key_orders as ko
import key_orders16 as ko16
import key_orders64 as ko64
from test_sort_indices16_cpu import sort16_indices_ref
from test_sort_indices_cpu import sort_indices_ref

KO = {16: ko16, 32: ko, 64: ko64}
WORD = {16: np.uint16, 32: np.uint32, 64: np.uint64}
SIGNED = {16: np.int16, 32: np.int32, 64: np.int64}
# image masks whose zero bytes make the digit passes over them skippable (every key has the same digit there)
MASKED = {16: 0x00FF, 32: 0x00FF00FF, 64: 0x00FF00FF00FF00FF}
TORCH_DTYPES = {  # key type -> name of the torch dtype
    ko.KEY_I32: "int32", ko.KEY_U32: "uint32", ko.KEY_F32: "float32",
    ko16.KEY_I16: "int16", ko16.KEY_U16: "uint16", ko16.KEY_F16: "float16", ko16.KEY_BF16: "bfloat16",
    ko64.KEY_I64: "int64", ko64.KEY_U64: "uint64", ko64.KEY_F64: "float64",
}
FLOATS = (ko.KEY_F32, ko16.KEY_F16, ko16.KEY_BF16, ko64.KEY_F64)

# 1-D sizes: the one-CTA sort (n <= 8192) and the pass kernels
SIZES_1D = [(5000,), (300001,)]
# rows: the onesweep class (> 8192), both CTA capacities (<= 8192, <= 1024) and the warp class (<= 128)
SIZES_ROWS = [(64, 9000), (128, 3000), (300, 1000), (1000, 100)]


class Call(NamedTuple):
    fn: str              # attribute of b200sort
    width: int           # key bits
    kt: int              # key type (key_orders*.KEY_*)
    desc: int
    form: str            # "1d" or "rows" (a 2-D tensor, every row a segment, no offsets)
    out: str             # "keys", "pairs" (keys, int32 values) or "indices" (keys, int64 positions)
    algo: str = ""       # b200sort.sort's algo, where given

    def shapes(self):
        return SIZES_1D if self.form == "1d" else SIZES_ROWS

    def run(self, keys, values=None):
        """The call on torch tensors, as a user writes it."""
        import b200sort
        kw = {"descending": bool(self.desc)}
        if self.algo:
            kw["algo"] = self.algo
        f = getattr(b200sort, self.fn)
        return f(keys, values, **kw) if self.out == "pairs" else f(keys, **kw)


def C(fn, kt, desc, form, out, algo=""):
    width = 16 if kt in ko16.NAMES else 64 if kt in ko64.NAMES else 32
    return Call(fn, width, kt, desc, form, out, algo)


# name -> call: the 16 torch-facing functions, and b200sort.sort once more with the merge algorithm.  The segmented
# functions are called in their rows form; the offsets form checks the offsets with one host synchronisation.
CALLS = {
    "sort": C("sort", ko.KEY_F32, 1, "1d", "keys"),
    "sort_merge": C("sort", ko.KEY_U32, 0, "1d", "keys", algo="merge"),
    "sort_by_key": C("sort_by_key", ko.KEY_F32, 0, "1d", "pairs"),
    "sort_with_indices": C("sort_with_indices", ko.KEY_I32, 1, "1d", "indices"),
    "sort16": C("sort16", ko16.KEY_BF16, 0, "1d", "keys"),
    "sort16_by_key": C("sort16_by_key", ko16.KEY_F16, 1, "1d", "pairs"),
    "sort16_with_indices": C("sort16_with_indices", ko16.KEY_BF16, 1, "1d", "indices"),
    "sort64": C("sort64", ko64.KEY_F64, 0, "1d", "keys"),
    "sort64_by_key": C("sort64_by_key", ko64.KEY_I64, 1, "1d", "pairs"),
    "segmented_sort": C("segmented_sort", ko.KEY_F32, 0, "rows", "keys"),
    "segmented_sort_by_key": C("segmented_sort_by_key", ko.KEY_U32, 1, "rows", "pairs"),
    "segmented_sort_with_indices": C("segmented_sort_with_indices", ko.KEY_F32, 1, "rows", "indices"),
    "segmented_sort16": C("segmented_sort16", ko16.KEY_I16, 0, "rows", "keys"),
    "segmented_sort16_by_key": C("segmented_sort16_by_key", ko16.KEY_U16, 1, "rows", "pairs"),
    "segmented_sort16_with_indices": C("segmented_sort16_with_indices", ko16.KEY_BF16, 1, "rows", "indices"),
    "segmented_sort64": C("segmented_sort64", ko64.KEY_F64, 1, "rows", "keys"),
    "segmented_sort64_by_key": C("segmented_sort64_by_key", ko64.KEY_U64, 0, "rows", "pairs"),
}


# ---- data sets -----------------------------------------------------------------------------------------------------
def dataset(c: Call, shape, kind: str, seed: int):
    """(key words of the key width, int32 values or None), flattened.  kind: "random" (bit patterns, float specials
    scattered through them), "all_equal" (every pass skippable) or "masked" (images with MASKED's zero bytes)."""
    n = int(np.prod(shape))
    rng = np.random.default_rng(seed)
    k = KO[c.width]
    w = WORD[c.width]
    if kind == "all_equal":
        words = np.full(n, rng.integers(0, 1 << c.width, dtype=np.uint64), np.uint64).astype(w)
    else:
        words = rng.integers(0, 1 << c.width, n, dtype=np.uint64).astype(w) if c.width < 64 else \
            rng.integers(0, 1 << 64, n, dtype=np.uint64)
        if kind == "masked":
            words = k.bits(k.inverse(words & w(MASKED[c.width]), c.kt, c.desc))
        elif c.kt in FLOATS:
            spec = k.float_specials(c.kt) if c.width == 16 else k.float_specials()
            pos = rng.integers(0, n, min(n, 4 * spec.size))
            words[pos] = np.resize(spec, pos.size)
    vals = rng.integers(-(1 << 31), 1 << 31, n, dtype=np.int64).astype(np.int32) if c.out == "pairs" else None
    return np.ascontiguousarray(words, w), vals


class Inputs:
    """The device inputs of one call at one shape: views that start `offset` elements into larger tensors (what
    slicing gives users), in the call's dtype and shape.  load() copies a data set in on the current stream."""

    def __init__(self, c: Call, shape, device="cuda", offset: int = 0):
        import torch
        self.c, self.shape = c, tuple(shape)
        n = int(np.prod(shape))
        self.key_base = torch.zeros(n + offset, dtype=getattr(torch, SIGNED[c.width].__name__), device=device)
        self.keys = self.key_base[offset:].view(getattr(torch, TORCH_DTYPES[c.kt])).view(self.shape)
        self.val_base = self.values = None
        if c.out == "pairs":
            self.val_base = torch.zeros(n + offset, dtype=torch.int32, device=device)
            self.values = self.val_base[offset:].view(self.shape)

    def args(self):
        return (self.keys, self.values) if self.c.out == "pairs" else (self.keys,)

    def load(self, data=None, src=None):
        """Copy `data` (dataset()) in, or device to device from `src` (staged())."""
        off = self.key_base.numel() - self.keys.numel()
        if src is None:
            src = staged(self, data)
        self.key_base[off:].copy_(src[0])
        if self.values is not None:
            self.val_base[off:].copy_(src[1])


def staged(inp: Inputs, data):
    """`data` as flat device tensors of the input's storage dtypes."""
    import torch
    words, vals = data
    dev = inp.key_base.device
    k = torch.from_numpy(words.view(SIGNED[inp.c.width])).to(dev)
    return k, (torch.from_numpy(vals).to(dev) if vals is not None else None)


# ---- references ------------------------------------------------------------------------------------------------------
def expected(c: Call, shape, data):
    """(sorted key words, values or int64 positions or None) of `data` sorted as `c` sorts it."""
    words, vals = data
    n = words.size
    row = shape[-1] if c.form == "rows" else n
    offsets = np.arange(0, n + 1, row, dtype=np.int64)
    if c.out == "indices":
        ref = sort16_indices_ref if c.width == 16 else sort_indices_ref
        return ref(words, offsets, c.kt, c.desc)
    img = KO[c.width].image(words, c.kt, c.desc)
    perm = np.lexsort((img, np.arange(n) // row))                       # lexsort is stable
    return words[perm], (vals[perm] if vals is not None else None)


def result_words(c: Call, out):
    """(key words, second output as numpy or None) of what the call returned, flattened."""
    import torch
    keys, second = (out, None) if c.out == "keys" else out
    kw = keys.reshape(-1).view(getattr(torch, SIGNED[c.width].__name__)).cpu().numpy().view(WORD[c.width])
    return kw, (second.reshape(-1).cpu().numpy() if second is not None else None)


def compare(c: Call, shape, data, out, what: str):
    """Assert that `out` (the call's result) is `data` sorted, byte for byte."""
    want_k, want_2 = expected(c, shape, data)
    got_k, got_2 = result_words(c, out)
    keys = out if c.out == "keys" else out[0]
    assert tuple(keys.shape) == tuple(shape), f"{what}: keys of shape {tuple(keys.shape)}"
    if got_k.tobytes() != want_k.tobytes():
        bad = np.flatnonzero(got_k != want_k)
        raise AssertionError(f"{what}: {bad.size} of {got_k.size} keys differ, first at {bad[0]}: "
                             f"got {int(got_k[bad[0]]):#x}, want {int(want_k[bad[0]]):#x}")
    if want_2 is not None:
        assert got_2.dtype == want_2.dtype, f"{what}: second output of dtype {got_2.dtype}"
        if got_2.tobytes() != want_2.tobytes():
            bad = np.flatnonzero(got_2 != want_2)
            raise AssertionError(f"{what}: {bad.size} of {got_2.size} {'values' if c.out == 'pairs' else 'indices'} "
                                 f"differ, first at {bad[0]}: got {got_2[bad[0]]}, want {want_2[bad[0]]}")
