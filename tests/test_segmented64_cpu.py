"""Segmented sort of 64-bit keys without a GPU: argument validation of b200sort_segmented_sort_keys64 /
_pairs_keys64 before any device work, key types rejected in both directions, the workspace and size-class queries,
the Python calls' input checks, and the numpy reference of a segmented 64-bit sort (used by
tests/test_segmented64_gpu.py)."""
import numpy as np
import pytest

import b200sort
from b200sort._lib import MAX_N, lib

import key_orders64 as ko

INVALID, WORKSPACE = 1, 2
P = 256          # a non-NULL, 256-byte aligned pointer value: never dereferenced, validation fails first
WS = 1 << 40     # a workspace size no call needs


def segment_ids(offsets: np.ndarray) -> np.ndarray:
    """Segment index of every key."""
    offsets = np.asarray(offsets, dtype=np.int64)
    return np.repeat(np.arange(offsets.size - 1), np.diff(offsets))


def seg_sort_keys(keys: np.ndarray, offsets: np.ndarray, key_type: int, desc: int) -> np.ndarray:
    return keys[np.lexsort((ko.image(keys, key_type, desc), segment_ids(offsets)))]


def seg_sort_pairs(keys: np.ndarray, vals: np.ndarray, offsets: np.ndarray, key_type: int, desc: int):
    p = np.lexsort((ko.image(keys, key_type, desc), segment_ids(offsets)))     # lexsort is stable
    return keys[p], vals[p]


def test_keys_validation_before_any_device_work():
    f = lib().b200sort_segmented_sort_keys64
    args = lambda: [P, P, P, 10, P, 3, P, WS, None]    # in, out, tmp, n, offsets, segments, ws, ws bytes, stream
    for kt in (-1, 0, 1, 2, 6, 7, 8, 9, 10, 99):       # the 32- and 16-bit key types included
        assert f(kt, 0, *args()) == INVALID, kt
    for desc in (-1, 2):
        assert f(ko.KEY_F64, desc, *args()) == INVALID
    for kt, desc in ko.ORDERS:
        for i in range(3):                                          # NULL in, out, tmp
            a = args(); a[i] = None
            assert f(kt, desc, *a) == INVALID, i
        for i in range(3):                                          # key pointers off an 8-byte boundary
            for off in (1, 2, 4):
                a = args(); a[i] = P + off
                assert f(kt, desc, *a) == INVALID, ("misaligned", i, off)
            a = args(); a[i] = P + 8; a[7] = 16                     # 8-byte aligned: past validation
            assert f(kt, desc, *a) == WORKSPACE, ("aligned", i)
        a = args(); a[3] = MAX_N + 1
        assert f(kt, desc, *a) == INVALID                           # n too large
        a = args(); a[5] = MAX_N + 1
        assert f(kt, desc, *a) == INVALID                           # too many segments
        a = args(); a[4] = None
        assert f(kt, desc, *a) == INVALID                           # NULL offsets
        a = args(); a[6] = None
        assert f(kt, desc, *a) == WORKSPACE                         # no workspace
        a = args(); a[7] = 16
        assert f(kt, desc, *a) == WORKSPACE                         # too small
        a = args(); a[6] = P + 8
        assert f(kt, desc, *a) == WORKSPACE                         # misaligned
        for i in range(2):                                          # n == 1 copies a key: NULL in or out
            a = args(); a[3] = 1; a[i] = None
            assert f(kt, desc, *a) == INVALID, ("n == 1", i)
        a = args(); a[3] = MAX_N; a[7] = 16
        assert f(kt, desc, *a) == WORKSPACE                         # n = 2^30 passes the key checks
        # the order of the checks: key type, then data pointers, then offsets, then the workspace
        assert f(kt, 2, None, None, None, 10, None, 3, None, 0, None) == INVALID
        assert f(kt, desc, P + 4, P, P, 10, P, 3, None, 0, None) == INVALID
        assert f(kt, desc, P, P, P, 10, None, 3, None, 0, None) == INVALID
        assert f(kt, desc, None, None, None, 0, None, 0, None, 0, None) == 0      # n == 0: no device work
        assert f(kt, desc, None, None, None, 0, P, 5, None, 0, None) == 0         # n == 0, five empty segments


def test_pairs_validation_before_any_device_work():
    f = lib().b200sort_segmented_pairs_keys64
    args = lambda: [P, P, P, P, P, P, 10, P, 3, P, WS, None]   # keys/vals in, out, tmp, n, offsets, segs, ws, bytes
    for kt in (-1, 0, 1, 2, 6, 7, 8, 9, 10, 99):
        assert f(kt, 0, *args()) == INVALID, kt
    assert f(ko.KEY_I64, 2, *args()) == INVALID
    assert f(ko.KEY_I64, -1, *args()) == INVALID
    for kt, desc in ko.ORDERS:
        for i in range(6):                                          # every data pointer NULL in turn
            a = args(); a[i] = None
            assert f(kt, desc, *a) == INVALID, (kt, desc, i)
        for i in (0, 2, 4):                                         # key pointers off an 8-byte boundary
            a = args(); a[i] = P + 4
            assert f(kt, desc, *a) == INVALID, ("misaligned", i)
        a = args(); a[0] = a[2] = P + 8; a[4] = P + 24; a[10] = 16  # 8-byte aligned: past validation
        assert f(kt, desc, *a) == WORKSPACE
        for i, v, want in ((6, MAX_N + 1, INVALID), (8, MAX_N + 1, INVALID), (7, None, INVALID),
                           (9, None, WORKSPACE), (10, 16, WORKSPACE), (9, P + 8, WORKSPACE)):
            a = args(); a[i] = v
            assert f(kt, desc, *a) == want, (kt, desc, i)
        for i in range(4):                                          # n == 1 copies a pair: NULL in or out
            a = args(); a[6] = 1; a[i] = None
            assert f(kt, desc, *a) == INVALID, ("n == 1", kt, desc, i)
        a = args(); a[2] = 512                                      # keys copied, values in place
        assert f(kt, desc, *a) == INVALID
        a = args(); a[3] = 512                                      # keys in place, values copied
        assert f(kt, desc, *a) == INVALID
        a = args(); a[2] = 512; a[7] = None                         # the mix is found before the offsets
        assert f(kt, desc, *a) == INVALID
        assert f(kt, desc, *([None] * 6), 0, None, 0, None, 0, None) == 0
        assert f(kt, desc, *([None] * 6), 0, P, 4, None, 0, None) == 0


def test_other_segmented_entry_points_still_reject_64_bit_keys():
    L = lib()
    for kt in (ko.KEY_I64, ko.KEY_U64, ko.KEY_F64):
        for f in (L.b200sort_segmented_sort_keys, L.b200sort_segmented_sort_keys16):
            assert f(kt, 0, P, P, P, 10, P, 3, P, WS, None) == INVALID, (f, kt)
        for f in (L.b200sort_segmented_pairs_keys, L.b200sort_segmented_pairs_keys16):
            assert f(kt, 0, P, P, P, P, P, P, 10, P, 3, P, WS, None) == INVALID, (f, kt)


def test_workspace_depends_on_n_and_segments_only():
    L = lib()
    ns = [0, 1, 2, 100, 129, 1025, 4096, 8192, 8193, 4096 * 3 + 1, 1 << 20, (1 << 28) + 3, MAX_N]
    ss = [0, 1, 2, 7, 1000, 1 << 20, MAX_N]
    for s in ss:
        w = [L.b200sort_segmented64_workspace_bytes(n, s) for n in ns]
        assert w == sorted(w), (s, w)
    for n in ns:
        w = [L.b200sort_segmented64_workspace_bytes(n, s) for s in ss]
        assert w == sorted(w), (n, w)
    # the same (n, S) always gives the same size, and a small fraction of the keys' bytes at scale
    assert L.b200sort_segmented64_workspace_bytes(12345, 17) == L.b200sort_segmented64_workspace_bytes(12345, 17)
    assert L.b200sort_segmented64_workspace_bytes(1 << 28, 2048) < (1 << 28)
    # with a segment per key the class lists dominate; still below the 8 bytes of the keys themselves
    assert L.b200sort_segmented64_workspace_bytes(1 << 28, 1 << 28) < 8 * (1 << 28)


def test_class_max_is_increasing_and_ends_with_zero():
    L = lib()
    c = [L.b200sort_segmented64_class_max(i) for i in range(8)]
    k = c.index(0)
    assert k >= 3 and all(v == 0 for v in c[k:])
    assert c[0] == 1 and all(a < b for a, b in zip(c[:k - 1], c[1:k]))
    assert L.b200sort_segmented64_class_max(-1) == 0
    assert c[:4] == [1, 128, 1024, 8192]


def test_python_calls_reject_bad_inputs():
    torch = pytest.importorskip("torch")
    x = torch.zeros(8, dtype=torch.int64)
    offs = torch.tensor([0, 8], dtype=torch.int32)
    for dt in (torch.float32, torch.int32, torch.int16, torch.bfloat16, torch.uint8):
        with pytest.raises(TypeError, match="b200sort.segmented_sort;.*b200sort.segmented_sort16"):
            b200sort.segmented_sort64(torch.zeros((2, 4), dtype=dt))
        with pytest.raises(TypeError, match="b200sort.segmented_sort16"):
            b200sort.segmented_sort64_by_key(torch.zeros((2, 4), dtype=dt), torch.zeros((2, 4), dtype=torch.int32))
    with pytest.raises(TypeError):
        b200sort.segmented_sort64(np.zeros(8, np.int64), offs)
    with pytest.raises(ValueError):
        b200sort.segmented_sort64(x)                                 # 1-D needs offsets
    with pytest.raises(ValueError):
        b200sort.segmented_sort64(torch.zeros((2, 4, 2), dtype=torch.float64))   # 3-D
    with pytest.raises(ValueError):
        b200sort.segmented_sort64(torch.zeros((4, 4), dtype=torch.int64).t())    # not contiguous
    with pytest.raises(ValueError):
        b200sort.segmented_sort64(torch.zeros((2, 4), dtype=torch.uint64))       # a CPU tensor
    with pytest.raises(ValueError):
        b200sort.segmented_sort64(x, offs)                           # a CPU tensor
    with pytest.raises(ValueError):
        b200sort.segmented_sort64(torch.zeros((2, 4), dtype=torch.int64), offs)  # 2-D with offsets
    k = torch.zeros((2, 4), dtype=torch.int64)
    with pytest.raises(TypeError):
        b200sort.segmented_sort64_by_key(k, torch.zeros((2, 4), dtype=torch.int64))   # 64-bit values
    with pytest.raises(TypeError):
        b200sort.segmented_sort64_by_key(k, np.zeros((2, 4), np.int32))
    with pytest.raises(ValueError):
        b200sort.segmented_sort64_by_key(k, torch.zeros((2, 3), dtype=torch.int32))
    with pytest.raises(ValueError):
        b200sort.segmented_sort64_by_key(k, torch.zeros((4, 2), dtype=torch.int32).t())


@pytest.mark.parametrize("order", ko.ORDERS, ids=[f"{ko.NAMES[k]}_{'desc' if d else 'asc'}" for k, d in ko.ORDERS])
def test_reference_matches_a_loop_over_segments(order):
    kt, desc = order
    rng = np.random.default_rng(5 + kt * 2 + desc)
    lens = rng.choice([0, 1, 2, 7, 50, 300, 2000], size=60)
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    n = int(offsets[-1])
    pool = np.concatenate([ko.float_specials(), rng.integers(0, 1 << 63, 30, dtype=np.uint64)])
    keys = pool[rng.integers(0, pool.size, n)].view(ko.DTYPES[kt])          # heavy duplicates, every sign
    vals = np.arange(n, dtype=np.int32)
    got = seg_sort_keys(keys, offsets, kt, desc)
    gk, gv = seg_sort_pairs(keys, vals, offsets, kt, desc)
    for i in range(len(lens)):
        a, b = offsets[i], offsets[i + 1]
        assert ko.bits(got[a:b]).tobytes() == ko.bits(ko.sort_keys(keys[a:b], kt, desc)).tobytes()
        wk, wv = ko.sort_pairs(keys[a:b], vals[a:b], kt, desc)
        assert ko.bits(gk[a:b]).tobytes() == ko.bits(wk).tobytes() and gv[a:b].tobytes() == wv.tobytes()
