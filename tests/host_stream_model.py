"""numpy model of the host-array operator's streamed path (order_host_streamed in csrc/api.cu).  Test
infrastructure only, numpy only.

The constants are read from the sources, so a change there reaches the model:
  kStreamChunks, kStreamMinKeys, kDirectBytes, kStageBytes  csrc/api.cu
  kSortTile (the merge tile)                                 csrc/merge.cu
  B200SORT_MAX_N                                             include/b200sort.h

`schedule` restates the arithmetic of order_host_streamed in C's size_t semantics (an offset past n
makes `n - off` wrap, as it would there).  `run` executes that schedule on real keys, with the two device
buffers prefilled with a sentinel: chunk sorts in place (their scratch range of the other buffer clobbered),
the intermediate merges on the chunk that
completes their pair, each level reading the buffer its parity selects, the last level range by range,
then the copy-back ranges.  The merge tile is a parameter, so a small tile makes the schedule cheap.

`stress_keys` builds the inputs that stress the chunk merges; the GPU tests use it too.
"""
from __future__ import annotations

import os
import re
from dataclasses import dataclass, field

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "radix-sort-merge-sort-cuda---lab-y-practicos-gpgpu-2023_b200", "csrc")
_U64 = 1 << 64
INT_MIN, INT_MAX = -2**31, 2**31 - 1


def constant(source: str, name: str) -> int:
    """The value of `constexpr <type> name = <integer expression>;` in csrc/<source>; the expression may use
    casts, integer literals, + - * << and other such constants of the same file."""
    text = open(os.path.join(CSRC, source)).read()
    m = re.search(r"constexpr\s+[\w:]+\s+" + name + r"\s*=\s*([^;]+);", text)
    assert m, f"{name} not found in {source}"
    expr = re.sub(r"\((?:size_t|int|unsigned|uint32_t)\)", "", m.group(1))
    expr = re.sub(r"\b(\d+)[uU]?[lL]*\b", r"\1", expr)
    expr = re.sub(r"\bk\w+\b", lambda k: str(constant(source, k.group(0))), expr)
    assert re.fullmatch(r"[\d\s()+\-*<]+", expr), (name, m.group(1))
    return int(eval(expr))      # digits, parentheses, + - * << only (asserted above)


STREAM_CHUNKS = constant("api.cu", "kStreamChunks")
STREAM_MIN_KEYS = constant("api.cu", "kStreamMinKeys")
DIRECT_BYTES = constant("api.cu", "kDirectBytes")
STAGE_BYTES = constant("api.cu", "kStageBytes")
SORT_TILE = constant("merge.cu", "kSortTile")
MAX_N = int(eval(re.search(r"#define\s+B200SORT_MAX_N\s+\(\(size_t\)(\d+\s*<<\s*\d+)\)",
                           open(os.path.join(ROOT, "include", "b200sort.h")).read()).group(1)))


def div_up(a: int, b: int) -> int:
    return (a + b - 1) // b


def align_up(a: int, b: int) -> int:
    return div_up(a, b) * b


def _sub(a: int, b: int) -> int:
    """a - b in size_t."""
    return (a - b) % _U64


@dataclass
class Schedule:
    n: int
    tile: int
    chunks: int
    chunk: int
    levels: int
    pieces: list = field(default_factory=list)     # (off, len) of chunk i, as order_host_streamed computes them
    merges: list = field(default_factory=list)     # (after chunk i, level l, start, sub, run)
    run: int = 0                                   # the last level's run
    tiles: int = 0
    per: int = 0
    ranges: list = field(default_factory=list)     # (tile_begin, tile_end) of the last level, clamped to tiles
    copies: list = field(default_factory=list)     # (e0, e1) copied back
    break_at: int | None = None                    # k at which `e0 >= n` ends the copy-back loop

    @property
    def valid(self) -> bool:
        """Every chunk starts inside the array (else `n - off` wraps and the chunk copy runs past n)."""
        return all(off < self.n for off, _ in self.pieces)


def schedule(n: int, tile: int = SORT_TILE, chunks: int = STREAM_CHUNKS) -> Schedule:
    """The arithmetic of order_host_streamed for n keys."""
    levels = 0
    while (1 << levels) < chunks:
        levels += 1
    chunk = align_up(div_up(n, chunks), 2 * tile)
    s = Schedule(n, tile, chunks, chunk, levels)
    for i in range(chunks):
        off = i * chunk
        s.pieces.append((off, _sub(n, off) if _sub(n, off) < chunk else chunk))
        l = 0
        while l + 1 < levels and ((i + 1) & ((2 << l) - 1)) == 0:
            run = chunk << l
            start = (i + 1 - (2 << l)) * chunk
            sub = _sub(n, start) if _sub(n, start) < 2 * run else 2 * run
            s.merges.append((i, l, start, sub, run))
            l += 1
    s.run = chunk << (levels - 1)
    s.tiles = div_up(n, tile)
    s.per = div_up(s.tiles, chunks)
    for k in range(chunks):
        s.ranges.append((k * s.per, min((k + 1) * s.per, s.tiles)))
    for k in range(chunks):
        e0 = k * s.per * tile
        if e0 >= n:
            s.break_at = k
            break
        s.copies.append((e0, min((k + 1) * s.per * tile, n)))
    return s


def shortest_last_chunk(chunk: int, tile: int = SORT_TILE, chunks: int = STREAM_CHUNKS) -> int:
    """The n whose schedule has chunks of `chunk` keys (a multiple of 2 * tile) and the shortest last chunk the
    rounding allows.  chunk < n / chunks + 2 tile, so the last chunk, n - (chunks - 1) chunk, is longer than
    chunk - 2 chunks tile: it is never much shorter than the others."""
    return chunks * chunk - 2 * chunks * tile + 1


# pageable sizes for the staged copy: the direct-copy limit and one key over it, a ragged size, and whole
# kStageBytes staging chunks +- 1 key (at 2^28 bytes every thread count up to 16 uses full chunks)
STAGED_SIZES = (DIRECT_BYTES // 4, DIRECT_BYTES // 4 + 1, (3 << 21) + 1, (1 << 26) - 1, 1 << 26, (1 << 26) + 1)
COPY_THREADS = (1, 3, 16)


def staged_geometry(nbytes: int, threads: int) -> tuple:
    """(threads used, staging chunk bytes, chunks) of staged_copy in csrc/api.cu for a pageable transfer."""
    used = threads
    want = nbytes // (4 << 20)
    if used > want:
        used = max(want, 1)
    chunk_bytes = max(min(align_up(div_up(nbytes, 2 * used), 4096), STAGE_BYTES), 256 << 10)
    return used, chunk_bytes, div_up(nbytes, chunk_bytes)


def merge_runs(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """merge(a, b), a's keys before equal b's, assuming both sorted (unsorted input gives a wrong result, as the
    merge-path kernels would)."""
    out = np.empty(a.size + b.size, dtype=a.dtype)
    out[np.arange(a.size) + np.searchsorted(b, a, "left")] = a
    out[np.arange(b.size) + np.searchsorted(a, b, "right")] = b
    return out


def merge_pass(src: np.ndarray, n: int, run: int) -> np.ndarray:
    """One merge pass over src[0, n): every pair of runs [base, base + run), [base + run, base + 2 run) merged."""
    out = np.empty(n, dtype=src.dtype)
    for base in range(0, n, 2 * run):
        mid, end = min(base + run, n), min(base + 2 * run, n)
        out[base:end] = merge_runs(src[base:mid], src[mid:end])
    return out


def _is_sorted(a: np.ndarray) -> bool:
    return bool(np.all(a[1:] >= a[:-1]))


@dataclass
class Trace:
    host: np.ndarray            # the host array after the copy back
    covered: np.ndarray         # how many copy-back ranges wrote each host element
    unready_reads: list         # (level, run index) of every merge input that was not a complete sorted run


def run(keys: np.ndarray, tile: int, chunks: int = STREAM_CHUNKS, sentinel: int = INT_MIN + 12345) -> Trace:
    """Execute schedule(len(keys), tile, chunks) on keys."""
    n = keys.size
    s = schedule(n, tile, chunks)
    assert s.valid, f"n={n}: a chunk starts past the end"
    buf = [np.full(n, sentinel, np.int32), np.full(n, sentinel, np.int32)]       # d_keys, d_tmp
    ready: set = set()                      # (level, run index) complete and sorted in buf[level & 1]
    unready: list = []

    def read_runs(l: int, start: int, sub: int, run_len: int) -> tuple:
        src = buf[l & 1]
        a, b = src[start:start + min(run_len, sub)], src[start + min(run_len, sub):start + sub]
        for j, piece in ((start // run_len, a), (start // run_len + 1, b)):
            if piece.size and ((l, j) not in ready or not _is_sorted(piece)):
                unready.append((l, j))
        return a, b

    def written(which: int, lo: int, hi: int) -> None:
        """buf[which][lo, hi) was overwritten: the runs kept there are gone."""
        for l, j in list(ready):
            r0 = j * (s.chunk << l)
            if (l & 1) == which and r0 < hi and lo < r0 + (s.chunk << l):
                ready.discard((l, j))

    merges = iter(s.merges)
    pending = next(merges, None)
    for i, (off, ln) in enumerate(s.pieces):
        written(0, off, off + ln)
        buf[0][off:off + ln] = np.sort(keys[off:off + ln])          # H2D of chunk i, then its sort in place ...
        written(1, off, off + ln)
        buf[1][off:off + ln] = sentinel                             # ... with d_tmp's range as its scratch
        ready.add((0, i))
        while pending is not None and pending[0] == i:
            _, l, start, sub, run_len = pending
            a, b = read_runs(l, start, sub, run_len)
            written((l + 1) & 1, start, start + sub)
            buf[(l + 1) & 1][start:start + sub] = merge_runs(a, b)
            ready.add((l + 1, start // (2 * run_len)))
            pending = next(merges, None)
    # last level: the whole array is one pair of runs; each range writes its output tiles
    src_l = s.levels - 1
    for base in range(0, n, 2 * s.run):
        read_runs(src_l, base, min(2 * s.run, n - base), s.run)
    merged = merge_pass(buf[src_l & 1], n, s.run)
    dst = buf[s.levels & 1]
    for t0, t1 in s.ranges:
        if t0 < t1:
            dst[t0 * tile:min(t1 * tile, n)] = merged[t0 * tile:min(t1 * tile, n)]
    host = keys.copy()
    covered = np.zeros(n, np.int32)
    for e0, e1 in s.copies:
        host[e0:e1] = dst[e0:e1]
        covered[e0:e1] += 1
    return Trace(host, covered, unready)


# ---- inputs that stress the chunk merges ----------------------------------------------------------------------------
STRESS = ("ascending", "descending", "all_equal", "mod8", "smallest_in_one_chunk", "straddle", "extremes",
          "lab_rand100")


def _lab_rand100(n: int, seed: int) -> np.ndarray:
    """glibc rand() % 100 (the reference driver's keys): 2^20 of them, repeated to n."""
    from b200sort import datagen
    return np.resize(datagen.lab_rand(min(n, 1 << 20), 100, seed), n)


def stress_keys(kind: str, n: int, chunk: int, out_edges, tile: int, seed: int = 1) -> np.ndarray:
    """n keys of `kind`, laid out against input chunks of `chunk` keys and output boundaries `out_edges`:
      ascending / descending / all_equal   the merge-path splits at both extremes, and every key tied;
      mod8                  chunk i holds only keys = i (mod 8), so every merge interleaves key by key;
      smallest_in_one_chunk the last chunk holds the smallest keys of the array;
      straddle              a run of equal keys (3/2 tiles each side) around every chunk boundary in the input,
                            and in the output around every boundary of out_edges;
      extremes              a quarter INT_MAX (the merge kernels' padding value), an eighth INT_MIN, and the
                            last two tiles of every chunk INT_MAX;
      lab_rand100           glibc rand() % 100."""
    rng = np.random.default_rng(seed)
    if kind == "ascending":
        return (np.arange(n, dtype=np.int64) - n // 2).astype(np.int32)
    if kind == "descending":
        return (n // 2 - np.arange(n, dtype=np.int64)).astype(np.int32)
    if kind == "all_equal":
        return np.full(n, -5, np.int32)
    if kind == "lab_rand100":
        return _lab_rand100(n, seed)
    uni = rng.integers(INT_MIN, INT_MAX, n, dtype=np.int64, endpoint=True)
    starts = list(range(0, n, chunk))
    if kind == "mod8":
        out = np.empty(n, np.int64)
        for i, off in enumerate(starts):
            piece = uni[off:off + chunk]
            out[off:off + chunk] = (piece // 8) * 8 + (i % 8)
        return np.clip(out, INT_MIN, INT_MAX).astype(np.int32)
    if kind == "smallest_in_one_chunk":
        srt = np.sort(uni)
        last = starts[-1]
        out = np.empty(n, np.int64)
        out[last:] = rng.permutation(srt[:n - last])
        out[:last] = rng.permutation(srt[n - last:])
        return out.astype(np.int32)
    if kind == "extremes":
        out = uni.copy()
        pick = rng.random(n)
        out[pick < 0.25] = INT_MAX
        out[(pick >= 0.25) & (pick < 0.375)] = INT_MIN
        for off in starts:
            end = min(off + chunk, n)
            out[max(off, end - 2 * tile):end] = INT_MAX
        return out.astype(np.int32)
    assert kind == "straddle", kind
    w = 3 * tile // 2
    srt = np.sort(uni)
    runs = []
    for e in out_edges:                                         # equal runs around the output boundaries
        lo, hi = max(e - w, 0), min(e + w, n)
        srt[lo:hi] = srt[lo]
        runs.append((lo, hi))
    # place run j around input chunk boundary j (cycling), the other keys shuffled into the rest
    out = np.empty(n, np.int64)
    taken = np.zeros(n, bool)
    used = np.zeros(n, bool)
    bounds = starts[1:] or [n // 2]
    for j, (lo, hi) in enumerate(runs):
        b = bounds[j % len(bounds)]
        left = (hi - lo) // 2
        p0 = max(b - left, 0)
        p1 = min(p0 + (hi - lo), n)
        free = ~taken[p0:p1]
        cnt = int(free.sum())
        out[p0:p1][free] = srt[lo:lo + cnt]
        taken[p0:p1] |= free
        used[lo:lo + cnt] = True
    rest = rng.permutation(srt[~used])
    out[~taken] = rest
    return out.astype(np.int32)
