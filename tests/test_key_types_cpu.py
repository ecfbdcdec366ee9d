"""uint32 / float32 keys and descending order without a GPU: argument validation of b200sort_sort_keys and
b200sort_radix_pairs_keys, the Python call's input checks, and the numpy reference of the key orders."""
import numpy as np
import pytest

import b200sort
from b200sort._lib import ALGO_LAB, ALGO_MERGE, ALGO_RADIX, MAX_N, lib

import key_orders as ko

INVALID, WORKSPACE = 1, 2
P = 256          # a non-NULL, 256-byte aligned pointer value: never dereferenced, validation fails first


@pytest.mark.parametrize("algo", [ALGO_RADIX, ALGO_MERGE])
def test_sort_keys_validation_before_any_device_work(algo):
    L = lib()
    for kt in (-1, 3, 99):
        assert L.b200sort_sort_keys(algo, kt, 0, P, P, P, 10, P, 1 << 20, None) == INVALID
    for desc in (-1, 2):
        assert L.b200sort_sort_keys(algo, ko.KEY_F32, desc, P, P, P, 10, P, 1 << 20, None) == INVALID
    for kt, desc in ko.ORDERS:
        assert L.b200sort_sort_keys(algo, kt, desc, None, P, P, 10, P, 1 << 20, None) == INVALID      # NULL d_in
        assert L.b200sort_sort_keys(algo, kt, desc, P, None, P, 10, P, 1 << 20, None) == INVALID      # NULL d_out
        assert L.b200sort_sort_keys(algo, kt, desc, P, P, None, 10, P, 1 << 20, None) == INVALID      # NULL d_tmp
        assert L.b200sort_sort_keys(algo, kt, desc, P, P, P, MAX_N + 1, P, 1 << 40, None) == INVALID  # n too large
        assert L.b200sort_sort_keys(algo, kt, desc, P, P, P, 10, None, 0, None) == WORKSPACE          # no workspace
        assert L.b200sort_sort_keys(algo, kt, desc, P, P, P, 10, P, 8, None) == WORKSPACE             # too small
        if algo == ALGO_RADIX:                                  # as b200sort_radix_i32 (the merge sort takes any)
            assert L.b200sort_sort_keys(algo, kt, desc, P, P, P, 10, P + 4, 1 << 20, None) == WORKSPACE
        assert L.b200sort_sort_keys(algo, kt, desc, None, None, None, 0, None, 0, None) == 0          # empty input
        assert L.b200sort_sort_keys(algo, kt, desc, P, P, P, 1, None, 0, None) == 0                   # in place, 1 key
    assert L.b200sort_sort_keys(7, ko.KEY_U32, 0, P, P, P, 10, P, 1 << 20, None) == INVALID           # unknown algorithm


def test_lab_pipeline_takes_int32_ascending_only():
    L = lib()
    for kt, desc in ko.ORDERS:
        if (kt, desc) != (ko.KEY_I32, 0):
            assert L.b200sort_sort_keys(ALGO_LAB, kt, desc, P, P, P, 10, P, 1 << 20, None) == INVALID
    assert L.b200sort_sort_keys(ALGO_LAB, ko.KEY_I32, 0, P, P, P, 10, None, 0, None) == WORKSPACE     # = b200sort_lab_i32


def test_pairs_keys_validation_before_any_device_work():
    L = lib()
    args = lambda: [P, P, P, P, P, P, 10, P, 1 << 20, None]    # keys in, vals in, keys out, vals out, tmps, n, ws, stream
    for kt in (-1, 3):
        assert L.b200sort_radix_pairs_keys(kt, 0, *args()) == INVALID
    assert L.b200sort_radix_pairs_keys(ko.KEY_U32, 2, *args()) == INVALID
    for kt, desc in ko.ORDERS:
        for i in range(6):                                      # every pointer NULL in turn
            a = args(); a[i] = None
            assert L.b200sort_radix_pairs_keys(kt, desc, *a) == INVALID, (kt, desc, i)
        a = args(); a[6] = MAX_N + 1
        assert L.b200sort_radix_pairs_keys(kt, desc, *a) == INVALID
        a = args(); a[7] = None
        assert L.b200sort_radix_pairs_keys(kt, desc, *a) == WORKSPACE
        a = args(); a[8] = 16
        assert L.b200sort_radix_pairs_keys(kt, desc, *a) == WORKSPACE
        # keys in place but values copied: the plan is shared by keys and values
        assert L.b200sort_radix_pairs_keys(kt, desc, P, P, P, 2 * P, P, P, 10, P, 1 << 20, None) == INVALID
        assert L.b200sort_radix_pairs_keys(kt, desc, None, None, None, None, None, None, 0, None, 0, None) == 0


def test_python_sort_rejects_bad_inputs():
    import torch
    with pytest.raises(TypeError):
        b200sort.sort(torch.zeros(8, dtype=torch.float64))
    with pytest.raises(TypeError):
        b200sort.sort(torch.zeros(8, dtype=torch.int64))
    with pytest.raises(TypeError):
        b200sort.sort(np.zeros(8, dtype=np.float32))
    with pytest.raises(ValueError, match="CUDA"):
        b200sort.sort(torch.zeros(8, dtype=torch.float32))                     # a CPU tensor
    with pytest.raises(ValueError, match="contiguous"):
        b200sort.sort(torch.zeros(16, dtype=torch.float32)[::2])
    with pytest.raises(ValueError, match="1-D"):
        b200sort.sort(torch.zeros(4, 4, dtype=torch.uint32))
    with pytest.raises(TypeError):
        b200sort.sort_by_key(torch.zeros(8, dtype=torch.float64), torch.zeros(8, dtype=torch.int32))
    with pytest.raises(TypeError):
        b200sort.sort_by_key(torch.zeros(8, dtype=torch.int32), torch.zeros(8, dtype=torch.int64))
    with pytest.raises(ValueError):
        b200sort.sort_by_key(torch.zeros(8, dtype=torch.uint32), torch.zeros(8, dtype=torch.int32))   # CPU tensors
    with pytest.raises(ValueError):
        b200sort.sort_by_key(torch.zeros(16, dtype=torch.float32)[::2], torch.zeros(8, dtype=torch.int32))


def test_reference_image_is_a_bijection():
    rng = np.random.default_rng(3)
    sample = np.concatenate([rng.integers(0, 1 << 32, 1 << 20, dtype=np.uint64).astype(np.uint32),
                             ko.float_specials(),
                             np.array([0, 1, 0x7FFFFFFF, 0x80000000, 0x80000001, 0xFFFFFFFF], dtype=np.uint32)])
    sample = np.unique(sample)
    for kt, desc in ko.ORDERS:
        keys = sample.view(ko.DTYPES[kt])
        img = ko.image(keys, kt, desc)
        assert np.unique(img).size == sample.size, (kt, desc)                  # injective on the sample
        assert ko.bits(ko.inverse(img, kt, desc)).tobytes() == sample.tobytes(), (kt, desc)
        assert ko.bits(ko.image(ko.inverse(sample, kt, desc), kt, desc)).tobytes() == sample.tobytes(), (kt, desc)
    # every one of the 2^16 combinations of the top and bottom bytes maps back and forth
    grid = ((np.arange(1 << 16, dtype=np.uint32) >> 8) << 24) | (np.arange(1 << 16, dtype=np.uint32) & 0xFF)
    for kt, desc in ko.ORDERS:
        assert np.unique(ko.image(grid, kt, desc)).size == grid.size


def test_reference_orders_the_float_specials_as_specified():
    spec = ko.float_specials()
    for desc in (0, 1):
        img = ko.image(spec, ko.KEY_F32, desc).astype(np.int64)
        steps = np.diff(img)
        assert (steps > 0).all() if desc == 0 else (steps < 0).all(), desc
    # without NaN and -0.0 the order is numpy's
    f = spec.view(np.float32)
    plain = spec[~np.isnan(f) & (spec != 0x80000000)]
    rng = np.random.default_rng(5)
    vals = np.concatenate([plain, rng.standard_normal(10000).astype(np.float32).view(np.uint32)])
    got = ko.sort_keys(vals.view(np.float32), ko.KEY_F32, 0)
    assert got.tobytes() == np.sort(vals.view(np.float32), kind="stable").tobytes()


def test_reference_integer_orders_are_numeric():
    rng = np.random.default_rng(7)
    u = rng.integers(0, 1 << 32, 100000, dtype=np.uint64).astype(np.uint32)
    assert ko.sort_keys(u, ko.KEY_U32, 0).tobytes() == np.sort(u).tobytes()
    assert ko.sort_keys(u, ko.KEY_U32, 1).tobytes() == np.sort(u)[::-1].tobytes()
    i = u.view(np.int32)
    assert ko.sort_keys(i, ko.KEY_I32, 0).tobytes() == np.sort(i).tobytes()
    assert ko.sort_keys(i, ko.KEY_I32, 1).tobytes() == np.sort(i)[::-1].tobytes()
