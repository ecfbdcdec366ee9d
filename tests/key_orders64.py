"""Numpy reference of the 64-bit key orders of b200sort_sort_keys64 (test infrastructure only).

Every order is image(k) = k ^ (bit 63 of k set ? neg : pos) on the 64-bit pattern, sorted as uint64 ascending;
the reference sort is a stable argsort of the images.
"""
from __future__ import annotations

import numpy as np

KEY_I64, KEY_U64, KEY_F64 = 3, 4, 5
DTYPES = {KEY_I64: np.int64, KEY_U64: np.uint64, KEY_F64: np.float64}
NAMES = {KEY_I64: "i64", KEY_U64: "u64", KEY_F64: "f64"}
TOP, ALL = 1 << 63, (1 << 64) - 1
MASKS = {   # (key type, descending) -> (neg, pos)
    (KEY_I64, 0): (TOP, TOP), (KEY_I64, 1): (ALL ^ TOP, ALL ^ TOP),
    (KEY_U64, 0): (0, 0), (KEY_U64, 1): (ALL, ALL),
    (KEY_F64, 0): (ALL, TOP), (KEY_F64, 1): (0, ALL ^ TOP),
}
ORDERS = sorted(MASKS)


def bits(a: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(a).view(np.uint64)


def image(keys: np.ndarray, key_type: int, descending: int) -> np.ndarray:
    neg, pos = MASKS[(key_type, descending)]
    b = bits(keys)
    return b ^ np.where(b >> np.uint64(63), np.uint64(neg), np.uint64(pos))


def inverse(img: np.ndarray, key_type: int, descending: int) -> np.ndarray:
    """The keys (as their dtype) whose images are ``img``: keyed on the image's top bit."""
    neg, pos = MASKS[(key_type, descending)]
    set_mask, clear_mask = (neg, pos) if not neg & TOP else (pos, neg)
    img = np.ascontiguousarray(img, dtype=np.uint64)
    k = img ^ np.where(img >> np.uint64(63), np.uint64(set_mask), np.uint64(clear_mask))
    return k.view(DTYPES[key_type])


def sort_keys(keys: np.ndarray, key_type: int, descending: int) -> np.ndarray:
    return keys[np.argsort(image(keys, key_type, descending), kind="stable")]


def sort_pairs(keys: np.ndarray, vals: np.ndarray, key_type: int, descending: int):
    p = np.argsort(image(keys, key_type, descending), kind="stable")
    return keys[p], vals[p]


def float_specials() -> np.ndarray:
    """Bit patterns of the float64 values whose order the header spells out, in that (ascending) order."""
    f = np.float64

    def b(x):
        return int(np.array(x, f).view(np.uint64))
    pats = [
        0xFFFFFFFFFFFFFFFF, 0xFFF8000000000001, 0xFFF8000000000000,   # -NaN: quiet and signalling, by payload
        0xFFF7FFFFFFFFFFFF, 0xFFF0000000000001,
        0xFFF0000000000000,                                             # -inf
        b(-np.finfo(f).max), b(-1.0), b(-np.finfo(f).tiny),             # -DBL_MAX, -1, -DBL_MIN
        0x800FFFFFFFFFFFFF, 0x8000000000000001,                         # negative denormals
        0x8000000000000000,                                             # -0.0
        0x0000000000000000,                                             # +0.0
        0x0000000000000001, 0x000FFFFFFFFFFFFF,                         # positive denormals
        b(np.finfo(f).tiny), b(1.0), b(np.finfo(f).max),                # DBL_MIN, 1, DBL_MAX
        0x7FF0000000000000,                                             # +inf
        0x7FF0000000000001, 0x7FF7FFFFFFFFFFFF,                         # +NaN: signalling, then quiet, by payload
        0x7FF8000000000000, 0x7FF8000000000001, 0x7FFFFFFFFFFFFFFF,
    ]
    return np.array(pats, dtype=np.uint64)
