"""Numpy reference of the 16-bit key orders of b200sort_sort_keys16 (test infrastructure only).

Every order is image(k) = k ^ (bit 15 of k set ? neg : pos) on the 16-bit pattern, sorted as uint16 ascending; the
reference sort is a stable argsort of the images.  numpy has no bfloat16, so bfloat16 keys are held as their uint16
bit patterns.
"""
from __future__ import annotations

import numpy as np

KEY_I16, KEY_U16, KEY_F16, KEY_BF16 = 6, 7, 8, 9
DTYPES = {KEY_I16: np.int16, KEY_U16: np.uint16, KEY_F16: np.float16, KEY_BF16: np.uint16}
NAMES = {KEY_I16: "i16", KEY_U16: "u16", KEY_F16: "f16", KEY_BF16: "bf16"}
TOP, ALL = 1 << 15, (1 << 16) - 1
MASKS = {   # (key type, descending) -> (neg, pos)
    (KEY_I16, 0): (TOP, TOP), (KEY_I16, 1): (ALL ^ TOP, ALL ^ TOP),
    (KEY_U16, 0): (0, 0), (KEY_U16, 1): (ALL, ALL),
    (KEY_F16, 0): (ALL, TOP), (KEY_F16, 1): (0, ALL ^ TOP),
    (KEY_BF16, 0): (ALL, TOP), (KEY_BF16, 1): (0, ALL ^ TOP),
}
ORDERS = sorted(MASKS)


def bits(a: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(a).view(np.uint16)


def image(keys: np.ndarray, key_type: int, descending: int) -> np.ndarray:
    neg, pos = MASKS[(key_type, descending)]
    b = bits(keys)
    return b ^ np.where(b >> np.uint16(15), np.uint16(neg), np.uint16(pos)).astype(np.uint16)


def inverse(img: np.ndarray, key_type: int, descending: int) -> np.ndarray:
    """The keys (as their dtype) whose images are ``img``: keyed on the image's top bit."""
    neg, pos = MASKS[(key_type, descending)]
    set_mask, clear_mask = (neg, pos) if not neg & TOP else (pos, neg)
    img = np.ascontiguousarray(img, dtype=np.uint16)
    k = img ^ np.where(img >> np.uint16(15), np.uint16(set_mask), np.uint16(clear_mask)).astype(np.uint16)
    return k.view(DTYPES[key_type])


def sort_keys(keys: np.ndarray, key_type: int, descending: int) -> np.ndarray:
    return keys[np.argsort(image(keys, key_type, descending), kind="stable")]


def sort_pairs(keys: np.ndarray, vals: np.ndarray, key_type: int, descending: int):
    p = np.argsort(image(keys, key_type, descending), kind="stable")
    return keys[p], vals[p]


def bf16_bits(x) -> np.ndarray:
    """bfloat16 patterns of float32 values, rounded to nearest even (as torch rounds)."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    r = (u + np.uint64(0x7FFF) + ((u >> np.uint64(16)) & np.uint64(1))) >> np.uint64(16)
    return r.astype(np.uint16)


def float_specials(key_type: int) -> np.ndarray:
    """Bit patterns of the float16 or bfloat16 values whose order the header spells out, in that (ascending) order."""
    if key_type == KEY_F16:
        f = np.float16

        def b(x):
            return int(np.array(x, f).view(np.uint16))
        pats = [0xFFFF, 0xFE01, 0xFE00,                 # -NaN: quiet, by payload
                0xFDFF, 0xFC01,                         # -NaN: signalling
                0xFC00,                                 # -inf
                b(-np.finfo(f).max), b(-1.0), b(-np.finfo(f).tiny),
                0x83FF, 0x8001,                         # negative denormals
                0x8000, 0x0000,                         # -0.0, +0.0
                0x0001, 0x03FF,                         # positive denormals
                b(np.finfo(f).tiny), b(1.0), b(np.finfo(f).max),
                0x7C00,                                 # +inf
                0x7C01, 0x7DFF, 0x7E00, 0x7E01, 0x7FFF]  # +NaN: signalling, then quiet, by payload
    else:
        pats = [0xFFFF, 0xFFC1, 0xFFC0,                 # -NaN: quiet, by payload
                0xFFBF, 0xFF81,                         # -NaN: signalling
                0xFF80,                                 # -inf
                0xFF7F, 0xBF80, 0x8080,                 # -max, -1, -min normal
                0x807F, 0x8001,                         # negative denormals
                0x8000, 0x0000,                         # -0.0, +0.0
                0x0001, 0x007F,                         # positive denormals
                0x0080, 0x3F80, 0x7F7F,                 # min normal, 1, max
                0x7F80,                                 # +inf
                0x7F81, 0x7FBF, 0x7FC0, 0x7FC1, 0x7FFF]  # +NaN: signalling, then quiet, by payload
    return np.array(pats, dtype=np.uint16)
