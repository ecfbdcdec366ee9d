"""Numpy reference of the key orders of b200sort_sort_keys (test infrastructure only).

Every order is image(k) = k ^ (top bit of k set ? neg : pos) on the 32-bit pattern, sorted as uint32 ascending;
the reference sort is a stable argsort of the images.
"""
from __future__ import annotations

import numpy as np

KEY_I32, KEY_U32, KEY_F32 = 0, 1, 2
DTYPES = {KEY_I32: np.int32, KEY_U32: np.uint32, KEY_F32: np.float32}
NAMES = {KEY_I32: "i32", KEY_U32: "u32", KEY_F32: "f32"}
MASKS = {   # (key type, descending) -> (neg, pos)
    (KEY_I32, 0): (0x80000000, 0x80000000), (KEY_I32, 1): (0x7FFFFFFF, 0x7FFFFFFF),
    (KEY_U32, 0): (0x00000000, 0x00000000), (KEY_U32, 1): (0xFFFFFFFF, 0xFFFFFFFF),
    (KEY_F32, 0): (0xFFFFFFFF, 0x80000000), (KEY_F32, 1): (0x00000000, 0x7FFFFFFF),
}
ORDERS = sorted(MASKS)


def bits(a: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(a).view(np.uint32)


def image(keys: np.ndarray, key_type: int, descending: int) -> np.ndarray:
    neg, pos = MASKS[(key_type, descending)]
    b = bits(keys)
    return b ^ np.where(b >> np.uint32(31), np.uint32(neg), np.uint32(pos))


def inverse(img: np.ndarray, key_type: int, descending: int) -> np.ndarray:
    """The keys (as their dtype) whose images are ``img``: keyed on the image's top bit."""
    neg, pos = MASKS[(key_type, descending)]
    set_mask, clear_mask = (neg, pos) if not neg & 0x80000000 else (pos, neg)
    img = np.ascontiguousarray(img, dtype=np.uint32)
    k = img ^ np.where(img >> np.uint32(31), np.uint32(set_mask), np.uint32(clear_mask))
    return k.view(DTYPES[key_type])


def sort_keys(keys: np.ndarray, key_type: int, descending: int) -> np.ndarray:
    return keys[np.argsort(image(keys, key_type, descending), kind="stable")]


def sort_pairs(keys: np.ndarray, vals: np.ndarray, key_type: int, descending: int):
    p = np.argsort(image(keys, key_type, descending), kind="stable")
    return keys[p], vals[p]


def float_specials() -> np.ndarray:
    """Bit patterns of the float32 values whose order the header spells out, in that (ascending) order."""
    f = np.float32
    pats = [
        0xFFFFFFFF, 0xFFC00001, 0xFFC00000, 0xFFBFFFFF, 0xFF800001,   # -NaN: quiet and signalling, by payload
        0xFF800000,                                                    # -inf
        int(np.array(-np.finfo(f).max, f).view(np.uint32)),           # -FLT_MAX
        int(np.array(-1.0, f).view(np.uint32)),
        int(np.array(-np.finfo(f).tiny, f).view(np.uint32)),          # -FLT_MIN
        0x807FFFFF, 0x80000001,                                        # negative denormals
        0x80000000,                                                    # -0.0
        0x00000000,                                                    # +0.0
        0x00000001, 0x007FFFFF,                                        # positive denormals
        int(np.array(np.finfo(f).tiny, f).view(np.uint32)),           # FLT_MIN
        int(np.array(1.0, f).view(np.uint32)),
        int(np.array(np.finfo(f).max, f).view(np.uint32)),            # FLT_MAX
        0x7F800000,                                                    # +inf
        0x7F800001, 0x7FBFFFFF, 0x7FC00000, 0x7FC00001, 0x7FFFFFFF,   # +NaN: signalling, then quiet, by payload
    ]
    return np.array(pats, dtype=np.uint32)
