"""int64 / uint64 / float64 keys without a GPU: argument validation of b200sort_sort_keys64 and
b200sort_radix_pairs_keys64, the workspace query, the Python calls' input checks, and the numpy reference of the
64-bit key orders."""
import numpy as np
import pytest

import b200sort
from b200sort._lib import ALGO_MERGE, ALGO_RADIX, MAX_N, lib

import key_orders64 as ko

INVALID, WORKSPACE = 1, 2
P = 256          # a non-NULL, 256-byte aligned pointer value: never dereferenced, validation fails first
WS = 1 << 20


def test_sort_keys64_validation_before_any_device_work():
    L = lib()
    for kt in (-1, 0, 1, 2, 6, 99):                             # the 32-bit key types included
        assert L.b200sort_sort_keys64(kt, 0, P, P, P, 10, P, WS, None) == INVALID, kt
    for desc in (-1, 2):
        assert L.b200sort_sort_keys64(ko.KEY_F64, desc, P, P, P, 10, P, WS, None) == INVALID
    for kt, desc in ko.ORDERS:
        assert L.b200sort_sort_keys64(kt, desc, None, P, P, 10, P, WS, None) == INVALID       # NULL d_in
        assert L.b200sort_sort_keys64(kt, desc, P, None, P, 10, P, WS, None) == INVALID       # NULL d_out
        assert L.b200sort_sort_keys64(kt, desc, P, P, None, 10, P, WS, None) == INVALID       # NULL d_tmp
        assert L.b200sort_sort_keys64(kt, desc, None, P, P, 1, P, WS, None) == INVALID        # NULL with n = 1
        assert L.b200sort_sort_keys64(kt, desc, P, P, P, MAX_N + 1, P, 1 << 40, None) == INVALID
        for i in range(3):                                      # 4-byte (not 8-byte) aligned key pointers
            a = [P, P, P]; a[i] = P + 4
            assert L.b200sort_sort_keys64(kt, desc, *a, 10, P, WS, None) == INVALID, i
        assert L.b200sort_sort_keys64(kt, desc, P, P, P, 10, None, 0, None) == WORKSPACE      # no workspace
        assert L.b200sort_sort_keys64(kt, desc, P, P, P, 10, P, 8, None) == WORKSPACE        # too small
        assert L.b200sort_sort_keys64(kt, desc, P, P, P, 10, P + 8, WS, None) == WORKSPACE   # misaligned
        assert L.b200sort_sort_keys64(kt, desc, None, None, None, 0, None, 0, None) == 0      # empty input
        assert L.b200sort_sort_keys64(kt, desc, P, P, P, 1, None, 0, None) == 0               # in place, 1 key


def test_pairs_keys64_validation_before_any_device_work():
    L = lib()
    args = lambda: [P, P, P, P, P, P, 10, P, WS, None]         # keys in, vals in, keys out, vals out, tmps, n, ws, stream
    for kt in (-1, 0, 1, 2, 6):
        assert L.b200sort_radix_pairs_keys64(kt, 0, *args()) == INVALID, kt
    assert L.b200sort_radix_pairs_keys64(ko.KEY_U64, 2, *args()) == INVALID
    for kt, desc in ko.ORDERS:
        for i in range(6):                                      # every pointer NULL in turn
            a = args(); a[i] = None
            assert L.b200sort_radix_pairs_keys64(kt, desc, *a) == INVALID, (kt, desc, i)
        for i in (0, 2, 4):                                     # key pointers 4-byte aligned
            a = args(); a[i] = P + 4
            assert L.b200sort_radix_pairs_keys64(kt, desc, *a) == INVALID, (kt, desc, i)
        a = args(); a[6] = MAX_N + 1
        assert L.b200sort_radix_pairs_keys64(kt, desc, *a) == INVALID
        a = args(); a[7] = None
        assert L.b200sort_radix_pairs_keys64(kt, desc, *a) == WORKSPACE
        a = args(); a[8] = 16
        assert L.b200sort_radix_pairs_keys64(kt, desc, *a) == WORKSPACE
        # keys in place but values copied: the plan is shared by keys and values
        assert L.b200sort_radix_pairs_keys64(kt, desc, P, P, P, 2 * P, P, P, 10, P, WS, None) == INVALID
        assert L.b200sort_radix_pairs_keys64(kt, desc, None, None, None, None, None, None, 0, None, 0, None) == 0
        assert L.b200sort_radix_pairs_keys64(kt, desc, P, P, P, P, P, P, 1, None, 0, None) == 0


def test_32_bit_entry_points_still_reject_the_64_bit_key_types():
    L = lib()
    for kt in (ko.KEY_I64, ko.KEY_U64, ko.KEY_F64):
        for algo in (ALGO_RADIX, ALGO_MERGE):
            assert L.b200sort_sort_keys(algo, kt, 0, P, P, P, 10, P, WS, None) == INVALID
        assert L.b200sort_radix_pairs_keys(kt, 0, P, P, P, P, P, P, 10, P, WS, None) == INVALID


def test_workspace_query():
    L = lib()
    sizes = [0, 1, 2, 4095, 4096, 4097, 1 << 16, (1 << 20) + 3, 1 << 28, MAX_N]
    ws = [L.b200sort_keys64_workspace_bytes(n) for n in sizes]
    assert all(w > 0 for w in ws)
    assert all(a <= b for a, b in zip(ws, ws[1:])), ws
    # one query for every key type: an n-sized workspace serves keys and pairs in any order (checked on the GPU)
    assert b200sort.KEY_I64 == ko.KEY_I64 and b200sort.KEY_U64 == ko.KEY_U64 and b200sort.KEY_F64 == ko.KEY_F64


def test_python_calls_reject_bad_inputs():
    import torch
    for dt in (torch.int32, torch.float32, torch.uint32, torch.int16):
        with pytest.raises(TypeError, match="b200sort.sort"):
            b200sort.sort64(torch.zeros(8, dtype=dt))
    with pytest.raises(TypeError):
        b200sort.sort64(np.zeros(8, dtype=np.int64))
    with pytest.raises(ValueError, match="CUDA"):
        b200sort.sort64(torch.zeros(8, dtype=torch.int64))                     # a CPU tensor
    with pytest.raises(ValueError, match="contiguous"):
        b200sort.sort64(torch.zeros(16, dtype=torch.float64)[::2])
    with pytest.raises(ValueError, match="1-D"):
        b200sort.sort64(torch.zeros(4, 4, dtype=torch.int64))
    with pytest.raises(TypeError):
        b200sort.sort64_by_key(torch.zeros(8, dtype=torch.int32), torch.zeros(8, dtype=torch.int32))
    with pytest.raises(TypeError):
        b200sort.sort64_by_key(torch.zeros(8, dtype=torch.int64), torch.zeros(8, dtype=torch.int64))
    with pytest.raises(TypeError):
        b200sort.sort64_by_key(torch.zeros(8, dtype=torch.int64), np.zeros(8, dtype=np.int32))
    with pytest.raises(ValueError):
        b200sort.sort64_by_key(torch.zeros(8, dtype=torch.float64), torch.zeros(8, dtype=torch.int32))   # CPU tensors
    with pytest.raises(ValueError):
        b200sort.sort64_by_key(torch.zeros(16, dtype=torch.int64)[::2], torch.zeros(8, dtype=torch.int32))


def test_reference_image_is_a_bijection():
    rng = np.random.default_rng(3)
    top = np.arange(1 << 16, dtype=np.uint64) >> np.uint64(8)
    bottom = np.arange(1 << 16, dtype=np.uint64) & np.uint64(0xFF)
    grid = (top << np.uint64(56)) | bottom                       # all 2^16 combinations of the top and bottom bytes
    sample = np.concatenate([rng.integers(0, 1 << 63, 1 << 18, dtype=np.uint64) * np.uint64(2) + np.uint64(1),
                             grid, ko.float_specials(),
                             np.array([0, 1, ko.TOP - 1, ko.TOP, ko.TOP + 1, ko.ALL], dtype=np.uint64)])
    sample = np.unique(sample)
    for kt, desc in ko.ORDERS:
        keys = sample.view(ko.DTYPES[kt])
        img = ko.image(keys, kt, desc)
        assert np.unique(img).size == sample.size, (kt, desc)
        assert ko.bits(ko.inverse(img, kt, desc)).tobytes() == sample.tobytes(), (kt, desc)
        assert ko.bits(ko.image(ko.inverse(sample, kt, desc), kt, desc)).tobytes() == sample.tobytes(), (kt, desc)
        assert np.unique(ko.image(grid, kt, desc)).size == grid.size, (kt, desc)


def test_reference_orders_the_float_specials_as_specified():
    spec = ko.float_specials()
    for desc in (0, 1):
        img = ko.image(spec, ko.KEY_F64, desc)
        assert (img[1:] > img[:-1]).all() if desc == 0 else (img[1:] < img[:-1]).all(), desc
    f = spec.view(np.float64)
    plain = spec[~np.isnan(f) & (spec != np.uint64(ko.TOP))]       # without NaN and -0.0 the order is numpy's
    rng = np.random.default_rng(5)
    vals = np.concatenate([plain, rng.standard_normal(10000).view(np.uint64)])
    got = ko.sort_keys(vals.view(np.float64), ko.KEY_F64, 0)
    assert got.tobytes() == np.sort(vals.view(np.float64), kind="stable").tobytes()


def test_reference_integer_orders_are_numeric():
    rng = np.random.default_rng(7)
    u = rng.integers(0, 1 << 64, 100000, dtype=np.uint64)
    assert ko.sort_keys(u, ko.KEY_U64, 0).tobytes() == np.sort(u).tobytes()
    assert ko.sort_keys(u, ko.KEY_U64, 1).tobytes() == np.sort(u)[::-1].tobytes()
    i = u.view(np.int64)
    assert ko.sort_keys(i, ko.KEY_I64, 0).tobytes() == np.sort(i).tobytes()
    assert ko.sort_keys(i, ko.KEY_I64, 1).tobytes() == np.sort(i)[::-1].tobytes()
