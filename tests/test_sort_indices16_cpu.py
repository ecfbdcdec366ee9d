"""Sort with indices of 16-bit keys without a GPU: argument validation of b200sort_radix_sort_indices_keys16 and
b200sort_segmented_sort_indices_keys16 before any device work, the Python calls' input checks, and the numpy
reference (a stable argsort of the key images, positions made segment-local) used by
tests/test_sort_indices16_gpu.py."""
import numpy as np
import pytest

import b200sort
from b200sort._lib import MAX_N, lib

import key_orders16 as ko

INVALID, WORKSPACE = 1, 2
P = 256          # a non-NULL, 256-byte aligned pointer value: never dereferenced, validation fails first
WS = 1 << 40     # a workspace size no call needs
OTHER_TYPES = (-1, 0, 1, 2, 3, 4, 5, 10, 99)   # 32-bit, 64-bit and unknown key types


def sort16_indices_ref(keys: np.ndarray, offsets, key_type: int, desc: int):
    """(keys with every segment sorted, int64 position of each inside its segment): the stable sort of
    (key, position) pairs in the order (key_type, desc), segment by segment."""
    offsets = np.asarray(offsets, dtype=np.int64)
    seg = np.repeat(np.arange(offsets.size - 1), np.diff(offsets))
    p = np.lexsort((ko.image(keys, key_type, desc), seg))          # lexsort is stable
    local = np.arange(keys.size, dtype=np.int64) - offsets[:-1][seg]
    return keys[p], local[p]


def test_1d_validation_before_any_device_work():
    L = lib()
    f = L.b200sort_radix_sort_indices_keys16
    args = lambda: [P, P, P, P, P, 10, P, WS, None]   # keys in, out, idx out, tmp keys, tmp idx, n, ws, ws bytes, stream
    for kt in OTHER_TYPES:
        assert f(kt, 0, *args()) == INVALID, kt
    for desc in (-1, 2):
        assert f(ko.KEY_BF16, desc, *args()) == INVALID
    for kt, desc in ko.ORDERS:
        for i in range(5):                                          # every pointer NULL in turn
            for n in (1, 10):
                a = args(); a[i] = None; a[5] = n
                assert f(kt, desc, *a) == INVALID, (kt, desc, i, n)
        for i in (0, 1, 3):                                         # odd key pointers
            a = args(); a[i] = P + 1
            assert f(kt, desc, *a) == INVALID, (kt, desc, i)
        for off in (2, 4, 6):                                       # index output not 8-byte aligned
            a = args(); a[2] = P + off
            assert f(kt, desc, *a) == INVALID, off
        a = args(); a[0] = a[1] = a[3] = P + 2                      # keys need only 2-byte alignment
        a[6] = None
        assert f(kt, desc, *a) == WORKSPACE
        a = args(); a[5] = MAX_N + 1
        assert f(kt, desc, *a) == INVALID                           # n too large
        for i, v in ((6, None), (7, 16), (6, P + 4)):               # no, small, misaligned workspace
            a = args(); a[i] = v
            assert f(kt, desc, *a) == WORKSPACE, (i, v)
        assert f(kt, desc, None, None, None, None, None, 0, None, 0, None) == 0      # n == 0: no device work
    try:                                                            # skipping off: 2^30 keys would overflow a count
        L.b200sort_radix_set_skip(0)
        a = args(); a[5] = MAX_N
        assert f(ko.KEY_I16, 0, *a) == INVALID
    finally:
        L.b200sort_radix_set_skip(1)


def test_segmented_validation_before_any_device_work():
    L = lib()
    f = L.b200sort_segmented_sort_indices_keys16
    args = lambda: [P, P, P, P, P, 10, P, 3, P, WS, None]   # ..., n, offsets, segments, ws, ws bytes, stream
    for kt in OTHER_TYPES:
        assert f(kt, 0, *args()) == INVALID, kt
    assert f(ko.KEY_U16, 2, *args()) == INVALID
    for kt, desc in ko.ORDERS:
        for i in range(5):
            a = args(); a[i] = None
            assert f(kt, desc, *a) == INVALID, (kt, desc, i)
        for i, v, want in ((0, P + 1, INVALID), (1, P + 1, INVALID), (3, P + 1, INVALID), (2, P + 4, INVALID),
                           (5, MAX_N + 1, INVALID), (7, MAX_N + 1, INVALID), (6, None, INVALID),
                           (8, None, WORKSPACE), (9, 16, WORKSPACE), (8, P + 4, WORKSPACE)):
            a = args(); a[i] = v
            assert f(kt, desc, *a) == want, (kt, desc, i, v)
        assert f(kt, desc, *([None] * 5), 0, None, 0, None, 0, None) == 0
        assert f(kt, desc, *([None] * 5), 0, P, 5, None, 0, None) == 0             # n == 0, five empty segments


def test_32_bit_entry_points_still_reject_16_bit_types():
    L = lib()
    for kt, desc in ko.ORDERS:
        assert L.b200sort_radix_sort_indices_keys(kt, desc, P, P, P, P, P, 10, P, WS, None) == INVALID
        assert L.b200sort_segmented_sort_indices_keys(kt, desc, P, P, P, P, P, 10, P, 3, P, WS, None) == INVALID


def test_python_calls_reject_bad_inputs():
    torch = pytest.importorskip("torch")
    for dt in (torch.int32, torch.float32, torch.int64, torch.float64, torch.uint8):
        with pytest.raises(TypeError, match="int16.*uint16.*float16.*bfloat16"):
            b200sort.sort16_with_indices(torch.zeros(8, dtype=dt))
        with pytest.raises(TypeError, match="int16.*uint16.*float16.*bfloat16"):
            b200sort.segmented_sort16_with_indices(torch.zeros((2, 4), dtype=dt))
    with pytest.raises(TypeError, match="b200sort.sort_with_indices"):
        b200sort.sort16_with_indices(torch.zeros(8, dtype=torch.float32))
    with pytest.raises(TypeError, match="b200sort.segmented_sort_with_indices"):
        b200sort.segmented_sort16_with_indices(torch.zeros((2, 4), dtype=torch.float32))
    for dt in (torch.int16, torch.uint16, torch.float16, torch.bfloat16):   # the 32-bit calls name the 16-bit ones
        with pytest.raises(TypeError, match="b200sort.sort16_with_indices"):
            b200sort.sort_with_indices(torch.zeros(8, dtype=dt))
        with pytest.raises(TypeError, match="b200sort.segmented_sort16_with_indices"):
            b200sort.segmented_sort_with_indices(torch.zeros((2, 4), dtype=dt))
    h = torch.bfloat16
    with pytest.raises(TypeError):
        b200sort.sort16_with_indices(np.zeros(8, np.float16))
    with pytest.raises(ValueError):
        b200sort.sort16_with_indices(torch.zeros((2, 4), dtype=h))                     # 2-D
    with pytest.raises(ValueError):
        b200sort.sort16_with_indices(torch.zeros(8, dtype=h)[::2])                     # not contiguous
    with pytest.raises(ValueError):
        b200sort.sort16_with_indices(torch.zeros(8, dtype=h))                          # a CPU tensor
    offs = torch.tensor([0, 8], dtype=torch.int32)
    with pytest.raises(ValueError):
        b200sort.segmented_sort16_with_indices(torch.zeros(8, dtype=h))                # 1-D needs offsets
    with pytest.raises(ValueError):
        b200sort.segmented_sort16_with_indices(torch.zeros((2, 4, 2), dtype=h))        # 3-D
    with pytest.raises(ValueError):
        b200sort.segmented_sort16_with_indices(torch.zeros((4, 4), dtype=h).t())       # not contiguous
    with pytest.raises(ValueError):
        b200sort.segmented_sort16_with_indices(torch.zeros((2, 4), dtype=h))           # a CPU tensor
    with pytest.raises(ValueError):
        b200sort.segmented_sort16_with_indices(torch.zeros(8, dtype=h), offs)          # a CPU tensor
    with pytest.raises(ValueError):
        b200sort.segmented_sort16_with_indices(torch.zeros((2, 4), dtype=h), offs)     # 2-D with offsets


@pytest.mark.parametrize("order", ko.ORDERS, ids=[f"{ko.NAMES[k]}_{'desc' if d else 'asc'}" for k, d in ko.ORDERS])
def test_reference_matches_a_loop_over_segments(order):
    kt, desc = order
    rng = np.random.default_rng(19 + kt * 2 + desc)
    lens = rng.choice([0, 1, 2, 7, 50, 300], size=40)
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    n = int(offsets[-1])
    keys = (rng.integers(0, 40, n).astype(np.uint16) * np.uint16(0x0101)).view(ko.DTYPES[kt])   # duplicates
    gk, gi = sort16_indices_ref(keys, offsets, kt, desc)
    assert gi.dtype == np.int64
    for i in range(len(lens)):
        a, b = offsets[i], offsets[i + 1]
        wk, wi = ko.sort_pairs(keys[a:b], np.arange(b - a, dtype=np.int64), kt, desc)
        assert ko.bits(gk[a:b]).tobytes() == ko.bits(wk).tobytes() and gi[a:b].tobytes() == wi.tobytes()
    k1, i1 = sort16_indices_ref(keys, [0, n], kt, desc)                          # 1-D: positions in the array
    assert i1.tobytes() == np.argsort(ko.image(keys, kt, desc), kind="stable").astype(np.int64).tobytes()
