"""int16 / uint16 / float16 / bfloat16 keys without a GPU: argument validation of b200sort_sort_keys16 and
b200sort_radix_pairs_keys16, the cross-rejection of key types between the 16-bit and the other entry points, the
workspace query, the Python calls' input checks, and the numpy reference of the 16-bit key orders."""
import numpy as np
import pytest

import b200sort
from b200sort._lib import ALGO_MERGE, ALGO_RADIX, MAX_N, lib

import key_orders16 as ko

INVALID, WORKSPACE = 1, 2
P = 256          # a non-NULL, 256-byte aligned pointer value: never dereferenced, validation fails first
WS = 1 << 24


def test_sort_keys16_validation_before_any_device_work():
    L = lib()
    for kt in (-1, 0, 1, 2, 3, 4, 5, 10, 99):                   # the 32- and 64-bit key types included
        assert L.b200sort_sort_keys16(kt, 0, P, P, 10, P, WS, None) == INVALID, kt
    for desc in (-1, 2):
        assert L.b200sort_sort_keys16(ko.KEY_BF16, desc, P, P, 10, P, WS, None) == INVALID
    for kt, desc in ko.ORDERS:
        assert L.b200sort_sort_keys16(kt, desc, None, P, 10, P, WS, None) == INVALID          # NULL d_in
        assert L.b200sort_sort_keys16(kt, desc, P, None, 10, P, WS, None) == INVALID          # NULL d_out
        assert L.b200sort_sort_keys16(kt, desc, None, P, 1, P, WS, None) == INVALID           # NULL with n = 1
        assert L.b200sort_sort_keys16(kt, desc, P, P, MAX_N + 1, P, 1 << 40, None) == INVALID
        for a in ((P + 1, P), (P, P + 1), (P + 3, P + 3)):         # odd key pointers
            assert L.b200sort_sort_keys16(kt, desc, *a, 10, P, WS, None) == INVALID, a
        assert L.b200sort_sort_keys16(kt, desc, P, P, 10, None, 0, None) == WORKSPACE         # no workspace
        assert L.b200sort_sort_keys16(kt, desc, P, P, 10, P, 8, None) == WORKSPACE           # too small
        assert L.b200sort_sort_keys16(kt, desc, P, P, 10, P + 8, WS, None) == WORKSPACE      # misaligned
        assert L.b200sort_sort_keys16(kt, desc, None, None, 0, None, 0, None) == 0           # empty input
        assert L.b200sort_sort_keys16(kt, desc, P, P, 1, None, 0, None) == 0                 # in place, 1 key


def test_pairs_keys16_validation_before_any_device_work():
    L = lib()
    args = lambda: [P, P, P, P, P, P, 10, P, WS, None]         # keys in, vals in, keys out, vals out, tmps, n, ws, stream
    for kt in (-1, 0, 1, 2, 3, 4, 5, 10):
        assert L.b200sort_radix_pairs_keys16(kt, 0, *args()) == INVALID, kt
    assert L.b200sort_radix_pairs_keys16(ko.KEY_U16, 2, *args()) == INVALID
    for kt, desc in ko.ORDERS:
        for i in range(6):                                      # every pointer NULL in turn
            a = args(); a[i] = None
            assert L.b200sort_radix_pairs_keys16(kt, desc, *a) == INVALID, (kt, desc, i)
        for i in (0, 2, 4):                                     # odd key pointers
            a = args(); a[i] = P + 1
            assert L.b200sort_radix_pairs_keys16(kt, desc, *a) == INVALID, (kt, desc, i)
        a = args(); a[6] = MAX_N + 1
        assert L.b200sort_radix_pairs_keys16(kt, desc, *a) == INVALID
        a = args(); a[7] = None
        assert L.b200sort_radix_pairs_keys16(kt, desc, *a) == WORKSPACE
        a = args(); a[8] = 16
        assert L.b200sort_radix_pairs_keys16(kt, desc, *a) == WORKSPACE
        a = args(); a[7] = P + 64
        assert L.b200sort_radix_pairs_keys16(kt, desc, *a) == WORKSPACE
        # keys in place but values copied, and the other way round: the plan is shared by keys and values
        assert L.b200sort_radix_pairs_keys16(kt, desc, P, P, P, 2 * P, P, P, 10, P, WS, None) == INVALID
        assert L.b200sort_radix_pairs_keys16(kt, desc, P, P, 2 * P, P, P, P, 10, P, WS, None) == INVALID
        assert L.b200sort_radix_pairs_keys16(kt, desc, None, None, None, None, None, None, 0, None, 0, None) == 0
        assert L.b200sort_radix_pairs_keys16(kt, desc, P, P, P, P, P, P, 1, None, 0, None) == 0


def test_pairs_keys16_refuse_2_30_keys_with_skipping_off():
    L = lib()
    n = 1 << 30
    ws = L.b200sort_keys16_workspace_bytes(n)
    try:
        L.b200sort_radix_set_skip(0)
        assert L.b200sort_radix_pairs_keys16(ko.KEY_I16, 0, P, P, P, P, P, P, n, P, ws, None) == INVALID
    finally:
        L.b200sort_radix_set_skip(1)


def test_other_entry_points_reject_the_16_bit_key_types():
    L = lib()
    for kt in (ko.KEY_I16, ko.KEY_U16, ko.KEY_F16, ko.KEY_BF16):
        for algo in (ALGO_RADIX, ALGO_MERGE):
            assert L.b200sort_sort_keys(algo, kt, 0, P, P, P, 10, P, WS, None) == INVALID
        assert L.b200sort_radix_pairs_keys(kt, 0, P, P, P, P, P, P, 10, P, WS, None) == INVALID
        assert L.b200sort_sort_keys64(kt, 0, P, P, P, 10, P, WS, None) == INVALID
        assert L.b200sort_radix_pairs_keys64(kt, 0, P, P, P, P, P, P, 10, P, WS, None) == INVALID
        assert L.b200sort_segmented_sort_keys(kt, 0, P, P, P, 10, P, 1, P, WS, None) == INVALID


def test_workspace_query():
    L = lib()
    sizes = [0, 1, 2, 8191, 8192, 8193, 1 << 16, (1 << 20) + 3, 1 << 28, MAX_N]
    ws = [L.b200sort_keys16_workspace_bytes(n) for n in sizes]
    assert all(w > 0 for w in ws)
    assert all(a <= b for a, b in zip(ws, ws[1:])), ws
    assert b200sort.KEY_I16 == ko.KEY_I16 and b200sort.KEY_U16 == ko.KEY_U16
    assert b200sort.KEY_F16 == ko.KEY_F16 and b200sort.KEY_BF16 == ko.KEY_BF16


def test_python_calls_reject_bad_inputs():
    import torch
    for dt in (torch.int32, torch.float32, torch.int64, torch.int8, torch.uint8):
        with pytest.raises(TypeError, match="b200sort.sort"):
            b200sort.sort16(torch.zeros(8, dtype=dt))
    with pytest.raises(TypeError):
        b200sort.sort16(np.zeros(8, dtype=np.int16))
    with pytest.raises(ValueError, match="CUDA"):
        b200sort.sort16(torch.zeros(8, dtype=torch.bfloat16))                   # a CPU tensor
    with pytest.raises(ValueError, match="contiguous"):
        b200sort.sort16(torch.zeros(16, dtype=torch.float16)[::2])
    with pytest.raises(ValueError, match="1-D"):
        b200sort.sort16(torch.zeros(4, 4, dtype=torch.int16))
    with pytest.raises(TypeError):
        b200sort.sort16_by_key(torch.zeros(8, dtype=torch.int32), torch.zeros(8, dtype=torch.int32))
    with pytest.raises(TypeError):
        b200sort.sort16_by_key(torch.zeros(8, dtype=torch.int16), torch.zeros(8, dtype=torch.int64))
    with pytest.raises(TypeError):
        b200sort.sort16_by_key(torch.zeros(8, dtype=torch.int16), np.zeros(8, dtype=np.int32))
    with pytest.raises(ValueError):
        b200sort.sort16_by_key(torch.zeros(8, dtype=torch.float16), torch.zeros(8, dtype=torch.int32))   # CPU
    with pytest.raises(ValueError):
        b200sort.sort16_by_key(torch.zeros(16, dtype=torch.uint16)[::2], torch.zeros(8, dtype=torch.int32))
    # the 32- and 64-bit calls keep refusing 16-bit keys
    for dt in (torch.int16, torch.uint16, torch.float16, torch.bfloat16):
        with pytest.raises(TypeError):
            b200sort.sort(torch.zeros(8, dtype=dt))
        with pytest.raises(TypeError, match="b200sort.sort16"):
            b200sort.sort64(torch.zeros(8, dtype=dt))


def test_reference_image_is_a_bijection_on_all_patterns():
    every = np.arange(1 << 16, dtype=np.uint16)
    for kt, desc in ko.ORDERS:
        img = ko.image(every.view(ko.DTYPES[kt]), kt, desc)
        assert np.unique(img).size == every.size, (kt, desc)
        assert ko.bits(ko.inverse(img, kt, desc)).tobytes() == every.tobytes(), (kt, desc)
        assert ko.bits(ko.image(ko.inverse(every, kt, desc), kt, desc)).tobytes() == every.tobytes(), (kt, desc)


@pytest.mark.parametrize("kt", [ko.KEY_F16, ko.KEY_BF16])
def test_reference_orders_the_float_specials_in_total_order(kt):
    spec = ko.float_specials(kt)
    for desc in (0, 1):
        img = ko.image(spec, kt, desc)
        assert (img[1:] > img[:-1]).all() if desc == 0 else (img[1:] < img[:-1]).all(), desc
    if kt == ko.KEY_F16:
        f = spec.view(np.float16)
        plain = spec[~np.isnan(f) & (spec != np.uint16(ko.TOP))]    # without NaN and -0.0 the order is numpy's
        vals = np.concatenate([plain, np.random.default_rng(5).standard_normal(10000).astype(np.float16).view(np.uint16)])
        got = ko.sort_keys(vals.view(np.float16), kt, 0)
        assert got.tobytes() == np.sort(vals.view(np.float16), kind="stable").tobytes()
    else:
        x = np.random.default_rng(6).standard_normal(10000).astype(np.float32)
        b = ko.bf16_bits(x)
        as_f32 = (b.astype(np.uint32) << np.uint32(16)).view(np.float32)
        b = b[as_f32 != 0]                                      # no -0.0
        as_f32 = as_f32[as_f32 != 0]
        assert ko.sort_keys(b, kt, 0).tobytes() == b[np.argsort(as_f32, kind="stable")].tobytes()
        assert ko.sort_keys(b, kt, 1).tobytes() == b[np.argsort(-as_f32, kind="stable")].tobytes()


def test_reference_integer_orders_are_numeric():
    u = np.random.default_rng(7).integers(0, 1 << 16, 100000).astype(np.uint16)
    assert ko.sort_keys(u, ko.KEY_U16, 0).tobytes() == np.sort(u).tobytes()
    assert ko.sort_keys(u, ko.KEY_U16, 1).tobytes() == np.sort(u)[::-1].tobytes()
    i = u.view(np.int16)
    assert ko.sort_keys(i, ko.KEY_I16, 0).tobytes() == np.sort(i).tobytes()
    assert ko.sort_keys(i, ko.KEY_I16, 1).tobytes() == np.sort(i)[::-1].tobytes()
