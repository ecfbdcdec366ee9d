"""The streamed host-array path's schedule (order_host_streamed in csrc/api.cu), run on real keys by the numpy model
in tests/host_stream_model.py, and the operator's argument checks, which come before any device work.  No GPU."""
import numpy as np
import pytest

import b200sort
import host_stream_model as hsm
from b200sort._lib import ALGO_LAB, ALGO_MERGE, ALGO_RADIX, MAX_N

C, T = hsm.STREAM_CHUNKS, hsm.SORT_TILE


def test_constants_come_from_the_sources():
    assert C >= 2 and C & (C - 1) == 0
    assert T == b200sort.lib().b200sort_merge_tile()
    assert hsm.MAX_N == MAX_N
    assert hsm.DIRECT_BYTES == (1 << 20) * 4 and hsm.STAGE_BYTES == 8 << 20
    # every n that streams has a valid schedule: (C - 1) chunk < n once n > C (C - 1) 2T (see below)
    assert hsm.STREAM_MIN_KEYS > C * (C - 1) * 2 * T


def _check_run(keys: np.ndarray, tile: int, what: str) -> None:
    tr = hsm.run(keys, tile)
    assert not tr.unready_reads, f"{what}: merges read incomplete runs {tr.unready_reads[:4]}"
    assert tr.covered.min() == 1 and tr.covered.max() == 1, f"{what}: copy-back ranges do not tile [0, n) once each"
    assert tr.host.tobytes() == np.sort(keys).tobytes(), what


def test_every_n_with_a_small_tile():
    """Every n up to 4000 with a 4-key merge tile.  Where the last chunk starts inside the array the schedule sorts;
    that fails only below C (C - 1) 2T, which at the real tile is far below the switch to streaming."""
    rng = np.random.default_rng(5)
    tile = 4
    bound = C * (C - 1) * 2 * tile
    valid = 0
    for n in range(1, 4001):
        s = hsm.schedule(n, tile)
        if not s.valid:
            assert n <= bound, n
            continue
        valid += 1
        keys = rng.integers(-40, 40, n).astype(np.int32) if n % 3 else rng.integers(-2**31, 2**31, n).astype(np.int32)
        _check_run(keys, tile, f"n={n}")
    assert valid > 4000 - bound


@pytest.mark.parametrize("tile", [4, 8, 16, 64])
def test_random_n_and_every_stress_input(tile):
    rng = np.random.default_rng(tile)
    lo = C * (C - 1) * 2 * tile + 1
    for n in sorted(set(int(x) for x in rng.integers(lo, 60 * lo, 12))) + [lo]:
        s = hsm.schedule(n, tile)
        edges = [e0 for e0, _ in s.copies[1:]]
        for kind in hsm.STRESS:
            _check_run(hsm.stress_keys(kind, n, s.chunk, edges, tile, seed=n), tile, f"tile={tile} n={n} {kind}")


def test_stress_inputs_have_their_shape():
    tile, n = 16, 20011
    s = hsm.schedule(n, tile)
    chunk, edges = s.chunk, [e0 for e0, _ in s.copies[1:]]
    starts = [off for off, _ in s.pieces]
    k = {kind: hsm.stress_keys(kind, n, chunk, edges, tile) for kind in hsm.STRESS}
    for kind, keys in k.items():
        assert keys.dtype == np.int32 and keys.size == n, kind
    for i, off in enumerate(starts):
        assert np.all(k["mod8"][off:off + chunk] % 8 == i % 8)
    last = starts[-1]
    assert k["smallest_in_one_chunk"][last:].max() <= k["smallest_in_one_chunk"][:last].min()
    srt = np.sort(k["straddle"])
    w = 3 * tile // 2
    for e in edges:
        assert np.all(srt[e - w:e + w] == srt[e - w]), e
    for b in starts[1:]:
        assert np.all(k["straddle"][b - w:b + w] == k["straddle"][b - w]), b
    ex = k["extremes"]
    assert (ex == hsm.INT_MAX).mean() > 0.25 and (ex == hsm.INT_MIN).mean() > 0.1
    assert set(np.unique(k["lab_rand100"])) <= set(range(100))
    assert np.all(np.diff(k["ascending"]) == 1) and np.all(np.diff(k["descending"]) == -1)


def _real_sizes() -> list:
    lo, hi = hsm.STREAM_MIN_KEYS, hsm.MAX_N
    edges = [lo, lo + 1, lo + 2, lo + T - 1, lo + T, lo + 2 * T * C - 1, lo + 2 * T * C, lo + 12345,
             3 * (1 << 24) + 77, (1 << 26) - 1, 1 << 26, (1 << 28) - 1, 1 << 28, hi - 1, hi,
             hsm.shortest_last_chunk(5 << 20), hsm.shortest_last_chunk(hsm.align_up(lo // C, 2 * T) + 2 * T)]
    sweep = np.unique(np.geomspace(lo, hi, 3000).astype(np.int64))
    rng = np.random.default_rng(3)
    return sorted(set(edges) | set(int(x) for x in sweep) | set(int(x) for x in rng.integers(lo, hi, 500)))


def test_schedule_at_the_real_constants():
    """From kStreamMinKeys to B200SORT_MAX_N: every chunk starts inside the array, so `len` never wraps; the
    chunks tile [0, n); every run is a multiple of the merge tile and every merge has both its runs; offsets and
    split points fit in 32 bits; the tile ranges of the last merge tile [0, tiles) and their copies [0, n), and the
    `e0 >= n` break is reached exactly when a range starts past the last tile (never, at these sizes)."""
    for n in _real_sizes():
        s = hsm.schedule(n)
        assert s.valid, n
        assert [off for off, _ in s.pieces] == [i * s.chunk for i in range(C)]
        assert sum(ln for _, ln in s.pieces) == n and all(0 < ln <= s.chunk for _, ln in s.pieces), n
        assert s.chunk - s.pieces[-1][1] < 2 * C * T, n
        assert s.chunk % (2 * T) == 0 and s.run % T == 0, n
        for i, l, start, sub, run in s.merges:
            assert run % T == 0 and start % (2 * run) == 0 and run < sub <= 2 * run and start + sub <= n, (n, i, l)
        if C == 8:
            assert [(i, l) for i, l, *_ in s.merges] == [(1, 0), (3, 0), (3, 1), (5, 0), (7, 0), (7, 1)]
        assert s.run < n <= 2 * s.run, n                      # the last level is one pair of runs
        assert n + T < 2**32 and s.tiles + 1 < 2**32, n       # 32-bit offsets and split points
        ranges = [(t0, t1) for t0, t1 in s.ranges if t0 < t1]
        assert ranges[0][0] == 0 and ranges[-1][1] == s.tiles and all(a[1] == b[0] for a, b in zip(ranges, ranges[1:]))
        assert s.copies[0][0] == 0 and s.copies[-1][1] == n, n
        assert all(a[1] == b[0] for a, b in zip(s.copies, s.copies[1:])), n
        assert (s.break_at is not None) == ((C - 1) * s.per >= s.tiles), n
        assert s.break_at is None, n


def test_break_is_reached_where_the_model_says():
    """The copy-back loop ends at `e0 >= n` exactly when a tile range starts past the last tile, which takes fewer
    than about C (C - 1) tiles: with a 4-key tile it happens for small n only, never once the schedule is valid.
    Wherever it happens the ranges after it are empty and the copies still tile [0, n)."""
    reached_valid = reached_small = 0
    for n in range(2, 3000):
        s = hsm.schedule(n, 4)
        assert (s.break_at is not None) == ((C - 1) * s.per >= s.tiles), n
        if s.break_at is not None:
            assert all(t0 >= s.tiles for t0, _ in s.ranges[s.break_at:]), n
            reached_valid += s.valid
            reached_small += 1
        assert s.copies[0][0] == 0 and s.copies[-1][1] == n, n
        assert all(a[1] == b[0] for a, b in zip(s.copies, s.copies[1:])), n
    assert reached_small > 0 and reached_valid == 0


def test_shortest_last_chunk():
    for chunk in (hsm.align_up(hsm.STREAM_MIN_KEYS // C, 2 * T) + 2 * T, 5 << 20, 1 << 27):
        n = hsm.shortest_last_chunk(chunk)
        s = hsm.schedule(n)
        assert s.chunk == chunk and s.pieces[-1][1] == chunk - 2 * C * T + 1
        assert hsm.schedule(n - 1).chunk != chunk                    # one key fewer and the chunks shrink
    assert hsm.shortest_last_chunk(5 << 20) >= hsm.STREAM_MIN_KEYS


def test_staged_copy_sizes_hit_the_chunk_edges():
    """The pageable sizes the GPU tests use: the direct-copy limit, and whole staging chunks of kStageBytes +- 1 key
    for 1, 3 and 16 copy threads."""
    assert (hsm.DIRECT_BYTES // 4) in hsm.STAGED_SIZES and (hsm.DIRECT_BYTES // 4 + 1) in hsm.STAGED_SIZES
    for threads in hsm.COPY_THREADS:
        rems = set()
        for n in hsm.STAGED_SIZES:
            if 4 * n <= hsm.DIRECT_BYTES:
                continue
            used, chunk_bytes, chunks = hsm.staged_geometry(4 * n, threads)
            assert 1 <= used <= threads and chunks >= 1
            if chunk_bytes == hsm.STAGE_BYTES:
                rems.add((4 * n) % hsm.STAGE_BYTES)
        assert {0, 4, hsm.STAGE_BYTES - 4} <= rems, (threads, rems)


@pytest.mark.parametrize("algo", [ALGO_RADIX, ALGO_MERGE, ALGO_LAB])
def test_host_operator_rejects_before_any_work(algo):
    """Checks that return before the device is touched, so they hold with or without a GPU: n > B200SORT_MAX_N,
    an unknown algorithm and NULL with n > 1 are invalid; n = 0 and n = 1 are a no-op, NULL included."""
    L = b200sort.lib()
    keys = np.array([5, -3, 9, 1], np.int32)
    before = keys.copy()
    count = L.b200sort_launch_count()
    p = keys.ctypes.data
    assert L.b200sort_order_array_host(p, hsm.MAX_N + 1, algo) == 1
    assert L.b200sort_order_array_host(p, 2**64 - 1, algo) == 1
    for bad in (-1, 3, 7):
        assert L.b200sort_order_array_host(p, 4, bad) == 1
        assert L.b200sort_order_array_host(p, 0, bad) == 1           # the algorithm is checked first
    assert L.b200sort_order_array_host(None, 2, algo) == 1
    assert L.b200sort_order_array_host(None, hsm.STREAM_MIN_KEYS, algo) == 1
    for n in (0, 1):
        assert L.b200sort_order_array_host(p, n, algo) == 0
        assert L.b200sort_order_array_host(None, n, algo) == 0
    assert L.b200sort_order_with_trust_host(p, hsm.MAX_N + 1) == 1
    assert L.b200sort_order_with_trust_host(None, 5) == 1
    assert L.b200sort_order_with_trust_host(p, 1) == 0 and L.b200sort_order_with_trust_host(None, 0) == 0
    assert L.b200sort_launch_count() == count
    assert keys.tobytes() == before.tobytes()
