"""Segmented sort of 64-bit keys on the GPU (b200sort_segmented_sort_keys64, b200sort_segmented_pairs_keys64 and the
torch-facing b200sort.segmented_sort64 / segmented_sort64_by_key), byte for byte against the numpy reference of
tests/test_segmented64_cpu.py.  Every C-ABI call here runs on one workspace that is reused and never cleared, with
guard words around keys, values and scratch and past ws_bytes, all checked after each call."""
import os
import subprocess
import sys

import numpy as np
import pytest

import b200sort
from b200sort._lib import check, lib
from helpers import stream_ptr

import key_orders64 as ko
from test_segmented64_cpu import seg_sort_keys, seg_sort_pairs
from test_segmented_gpu import ragged_offsets

pytestmark = pytest.mark.gpu

ORDER_IDS = [f"{ko.NAMES[k]}_{'desc' if d else 'asc'}" for k, d in ko.ORDERS]
TILE = 4096                      # keys per tile of the segmented onesweep (kSeg64Tile, csrc/segmented64.cuh)
G = 48                           # guard words on each side of every buffer
GUARD64 = 0x5A5A5A5A5A5A5A5A
GUARD32 = 0x5A5A5A5A
WS_TAIL = 4096                   # guarded workspace bytes past ws_bytes

_ws_state = {}


def _class_bounds():
    L = lib()
    out, c = [], 0
    while L.b200sort_segmented64_class_max(c):
        out.append(L.b200sort_segmented64_class_max(c))
        c += 1
    return out


def row_lengths():
    ls = {1, 2, 31, 32, 33, 2 * TILE + 1, 3 * TILE - 1, 3 * TILE, 3 * TILE + 1, 4 * TILE, 65537, (1 << 20) + 3}
    for m in _class_bounds():
        ls |= {m - 1, m, m + 1}
    return sorted(x for x in ls if x >= 1)


def _workspace(nbytes: int):
    """The module's workspace: grown when a call needs more, never cleared.  Returns (pointer, guard snapshot)."""
    import torch
    ws = _ws_state.get("ws")
    if ws is None or ws.numel() < nbytes + WS_TAIL + 256:
        ws = torch.randint(0, 256, (max(nbytes, 1 << 20) * 2 + WS_TAIL + 256,), dtype=torch.uint8, device="cuda")
        _ws_state["ws"] = ws
    ptr = ws.data_ptr() + (-ws.data_ptr()) % 256
    at = ptr - ws.data_ptr()
    return ptr, ws[at + nbytes:at + nbytes + WS_TAIL].clone(), (at, nbytes)


def _check_ws_tail(snapshot, where, what):
    ws = _ws_state["ws"]
    at, nbytes = where
    assert __import__("torch").equal(ws[at + nbytes:at + nbytes + WS_TAIL], snapshot), f"{what}: past ws_bytes written"


class _Buf:
    """Device words holding ``a`` at word G + offset of a guarded buffer."""

    def __init__(self, a: np.ndarray, offset: int = 0, itemsize: int = 8):
        import torch
        self.n, self.at = a.size, G + offset
        dt, fill = (torch.int64, GUARD64) if itemsize == 8 else (torch.int32, GUARD32)
        self.t = torch.full((a.size + 2 * G + offset,), fill, dtype=dt, device="cuda")
        self.fill = fill
        if a.size:
            self.t[self.at:self.at + a.size] = torch.from_numpy(np.ascontiguousarray(a).view(
                np.int64 if itemsize == 8 else np.int32).copy()).cuda()
        self.ptr = self.t.data_ptr() + itemsize * self.at

    def body(self) -> np.ndarray:
        return self.t[self.at:self.at + self.n].cpu().numpy()

    def guards_ok(self) -> bool:
        return bool((self.t[:self.at] == self.fill).all()) and bool((self.t[self.at + self.n:] == self.fill).all())


def run(keys, offsets, kt, desc, vals=None, in_place=False, offset=0, stream=None):
    """The library's result: uint64 words (and int32 values for pairs).  Checks every guard and that the copy form
    leaves its input alone."""
    import torch
    n = keys.size
    offsets = np.asarray(offsets, np.int64)
    S = offsets.size - 1
    kin = _Buf(ko.bits(keys), offset)
    kout = kin if in_place else _Buf(np.full(n, 0xA5A5A5A5A5A5A5A5, np.uint64), offset)
    ktmp = _Buf(np.full(n, 0x3C3C3C3C3C3C3C3C, np.uint64), offset)
    d_off = torch.from_numpy(offsets.astype(np.int32)).cuda()
    nbytes = lib().b200sort_segmented64_workspace_bytes(n, S)
    ptr, snap, where = _workspace(nbytes)
    st = stream if stream is not None else stream_ptr()
    bufs = [kin, kout, ktmp]
    if vals is None:
        check(lib().b200sort_segmented_sort_keys64(kt, desc, kin.ptr, kout.ptr, ktmp.ptr, n, d_off.data_ptr(), S, ptr,
                                                   nbytes, st))
    else:
        vin = _Buf(vals, 0, 4)
        vout = vin if in_place else _Buf(np.full(n, -1, np.int32), 0, 4)
        vtmp = _Buf(np.full(n, -2, np.int32), 0, 4)
        bufs += [vin, vout, vtmp]
        check(lib().b200sort_segmented_pairs_keys64(kt, desc, kin.ptr, vin.ptr, kout.ptr, vout.ptr, ktmp.ptr, vtmp.ptr,
                                                    n, d_off.data_ptr(), S, ptr, nbytes, st))
    torch.cuda.synchronize()
    what = f"n={n} S={S} order={kt},{desc} pairs={vals is not None} in_place={in_place} offset={offset}"
    assert all(b.guards_ok() for b in bufs), f"{what}: a guard word changed"
    _check_ws_tail(snap, where, what)
    if not in_place:
        assert kin.body().view(np.uint64).tobytes() == ko.bits(keys).tobytes(), f"{what}: the copy form wrote its keys"
        if vals is not None:
            assert bufs[3].body().tobytes() == np.ascontiguousarray(vals, np.int32).tobytes(), f"{what}: ... values"
    got = kout.body().view(np.uint64)
    return got if vals is None else (got, bufs[4].body())


def assert_words(got: np.ndarray, want: np.ndarray, what):
    want = ko.bits(want)
    if got.tobytes() != want.tobytes():
        bad = np.flatnonzero(got != want)
        raise AssertionError(f"{what}: {bad.size} of {got.size} words differ, first at {bad[0]}: "
                             f"got {int(got[bad[0]]):#018x}, want {int(want[bad[0]]):#018x}")


def check_all(keys, offsets, kt, desc, what, modes=((False, False), (False, True), (True, False), (True, True)),
              offset=0):
    """Keys and pairs, copied and in place, against the reference."""
    want = seg_sort_keys(keys, offsets, kt, desc)
    vals = np.arange(keys.size, dtype=np.int32)
    wk, wv = seg_sort_pairs(keys, vals, offsets, kt, desc)
    for pairs, in_place in modes:
        w = f"{what} pairs={pairs} in_place={in_place}"
        if pairs:
            gk, gv = run(keys, offsets, kt, desc, vals, in_place, offset)
            assert_words(gk, wk, w)
            assert gv.tobytes() == wv.tobytes(), f"{w}: values"
        else:
            assert_words(run(keys, offsets, kt, desc, None, in_place, offset), want, w)


def random_keys(n: int, kt: int, seed: int) -> np.ndarray:
    rng = np.random.default_rng(seed)
    w = rng.integers(0, 1 << 64, n, dtype=np.uint64) if n else np.zeros(0, np.uint64)
    if kt == ko.KEY_F64 and n:
        spec = ko.float_specials()
        pos = rng.integers(0, n, min(n, 4 * spec.size))
        w[pos] = np.resize(spec, pos.size)
    return w.view(ko.DTYPES[kt])


def every_class_layout(seed: int, big=(9000, 20000)) -> np.ndarray:
    """A few segments of every class: empty, one key, warp, both CTA capacities and the onesweep."""
    rng = np.random.default_rng(seed)
    lens = np.concatenate([[0, 0, 1, 1], rng.integers(2, 129, 6), rng.integers(129, 1025, 4),
                           rng.integers(1025, 8193, 3), [8192, 1024, 128, 8193], list(big)])
    rng.shuffle(lens)
    return np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)


# ---- sizes, orders and layouts ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_equal_rows_every_class_boundary(order):
    kt, desc = order
    for L_ in row_lengths():
        B = max(1, min(2048, (1 << 20) // L_))
        keys = random_keys(B * L_, kt, 100 + L_ % 97)
        check_all(keys, np.arange(B + 1, dtype=np.int64) * L_, kt, desc, f"L={L_} B={B}")


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_ragged_segments_with_empty_ones(order):
    kt, desc = order
    offsets = ragged_offsets(7 + kt * 2 + desc, total_segments=2000, big=1)
    check_all(random_keys(int(offsets[-1]), kt, 3), offsets, kt, desc, "ragged")


def test_more_segments_than_keys():
    rng = np.random.default_rng(3)
    n, S = 20000, 200000
    offsets = np.concatenate([[0], np.sort(rng.integers(0, n + 1, S - 1)), [n]]).astype(np.int64)
    for kt, desc in ko.ORDERS:
        check_all(random_keys(n, kt, 9), offsets, kt, desc, f"S > n {kt},{desc}", modes=((False, False), (True, True)))


def test_segments_start_at_every_element_offset():
    """The buffers start 0..7 words past a 64-byte boundary, and the segments at every element offset."""
    offsets = every_class_layout(4)
    n = int(offsets[-1])
    keys = random_keys(n, ko.KEY_I64, 5)
    for offset in range(8):
        check_all(keys, offsets, ko.KEY_I64, offset & 1, f"offset={offset}", offset=offset)
    shift = np.concatenate([[0], np.minimum(offsets[1:-1] + 3, n), [n]])   # every boundary moved by 3 keys
    check_all(keys, shift, ko.KEY_U64, 1, "shifted boundaries")


def test_a_key_pointer_off_8_bytes_is_rejected():
    import torch
    n = 1000
    k = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    v = torch.zeros(n, dtype=torch.int32, device="cuda")
    offs = torch.tensor([0, n], dtype=torch.int32, device="cuda")
    nbytes = lib().b200sort_segmented64_workspace_bytes(n, 1)
    ptr, _, _ = _workspace(nbytes)
    L = lib()
    L.b200sort_launch_count_reset()
    for i in range(3):
        p = [k.data_ptr()] * 3
        p[i] += 4
        assert L.b200sort_segmented_sort_keys64(ko.KEY_I64, 0, *p, n, offs.data_ptr(), 1, ptr, nbytes, stream_ptr()) == 1
        assert L.b200sort_segmented_pairs_keys64(ko.KEY_I64, 0, p[0], v.data_ptr(), p[1], v.data_ptr(), p[2],
                                                 v.data_ptr(), n, offs.data_ptr(), 1, ptr, nbytes, stream_ptr()) == 1
    assert L.b200sort_launch_count() == 0


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_float64_specials(order):
    kt, desc = order
    offsets = every_class_layout(11)
    n = int(offsets[-1])
    spec = ko.float_specials()
    keys = np.resize(spec, n).copy()                 # NaN payloads of both signs, +-0, +-inf, subnormals
    keys[::3] = random_keys(keys[::3].size, ko.KEY_U64, n)
    check_all(keys.view(ko.DTYPES[kt]), offsets, kt, desc, "specials")


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_pairs_are_stable_in_every_class(order):
    kt, desc = order
    offsets = ragged_offsets(21 + kt, total_segments=2000, big=1)
    n = int(offsets[-1])
    pool = random_keys(40, kt, 23)
    keys = pool[np.random.default_rng(24).integers(0, 40, n)]            # every key 40-fold or more
    check_all(keys, offsets, kt, desc, "ties", modes=((True, False), (True, True)))


def test_pairs_keys_in_place_values_copied_is_rejected():
    import torch
    n = 1000
    k = torch.zeros(n, dtype=torch.int64, device="cuda"); t = torch.zeros_like(k)
    v = torch.zeros(n, dtype=torch.int32, device="cuda"); v2 = torch.zeros_like(v); tv = torch.zeros_like(v)
    offs = torch.tensor([0, n], dtype=torch.int32, device="cuda")
    nbytes = lib().b200sort_segmented64_workspace_bytes(n, 1)
    ptr, _, _ = _workspace(nbytes)
    L = lib()
    L.b200sort_launch_count_reset()
    st = L.b200sort_segmented_pairs_keys64(ko.KEY_I64, 0, k.data_ptr(), v.data_ptr(), k.data_ptr(), v2.data_ptr(),
                                           t.data_ptr(), tv.data_ptr(), n, offs.data_ptr(), 1, ptr, nbytes, stream_ptr())
    assert st == 1 and L.b200sort_launch_count() == 0


# ---- pass skipping ---------------------------------------------------------------------------------------------------
def varying_bytes(n: int, mask: int, seed: int, base=None) -> np.ndarray:
    """Keys equal to `base` except in the bytes named by the bits of `mask`, which are random."""
    rng = np.random.default_rng(seed)
    base = np.uint64(rng.integers(0, 1 << 64, dtype=np.uint64) if base is None else base)
    bm = np.uint64(sum(0xFF << (8 * b) for b in range(8) if mask >> b & 1))
    return (base & ~bm) | (rng.integers(0, 1 << 64, n, dtype=np.uint64) & bm)


def test_every_subset_of_varying_bytes():
    """All 256 subsets of varying bytes on a layout that reaches every class, keys and pairs, copied and in place:
    every pattern of executed and skipped passes, each order in turn."""
    offsets = every_class_layout(12)
    n = int(offsets[-1])
    for mask in range(256):
        kt, desc = ko.ORDERS[mask % len(ko.ORDERS)]
        keys = varying_bytes(n, mask, mask).view(ko.DTYPES[kt])
        check_all(keys, offsets, kt, desc, f"mask={mask:#04x}")


@pytest.mark.parametrize("kind", ["ids_below_2_32", "constant_low_word", "all_equal"])
def test_skippable_rows(kind):
    rng = np.random.default_rng(7)
    for L_ in (16, 700, 5000, 40001):
        B = max(1, (1 << 20) // L_)
        n = B * L_
        if kind == "ids_below_2_32":
            w = rng.integers(0, 1 << 32, n, dtype=np.uint64)
        elif kind == "constant_low_word":
            w = (rng.integers(0, 1 << 32, n, dtype=np.uint64) << np.uint64(32)) | np.uint64(0x9E3779B9)
        else:
            w = np.full(n, 0x400921FB54442D18, np.uint64)
        for kt, desc in ((ko.KEY_I64, 0), (ko.KEY_I64, 1), (ko.KEY_F64, 1), (ko.KEY_U64, 0)):
            check_all(w.view(ko.DTYPES[kt]), np.arange(B + 1) * L_, kt, desc, f"{kind} L={L_}")


def _mixed_layout(cta: bool):
    """Segments of ids below 2^32, except one that also varies in byte 7: large segments, or (cta) CTA-class ones."""
    lens = [3000, 7000, 1025, 900, 8192] * 4 if cta else [9000, 30000, 8193, 70000, 12288]
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    n = int(offsets[-1])
    rng = np.random.default_rng(8)
    w = rng.integers(0, 1 << 32, n, dtype=np.uint64)
    s = 2 if not cta else 7
    w[offsets[s]:offsets[s + 1]] ^= rng.integers(0, 2, offsets[s + 1] - offsets[s], dtype=np.uint64) << np.uint64(61)
    return w, offsets


@pytest.mark.parametrize("cta", [False, True], ids=["onesweep", "cta_classes"])
def test_one_segment_varying_in_byte_7_runs_that_pass(cta):
    w, offsets = _mixed_layout(cta)
    for kt, desc in ko.ORDERS:
        check_all(w.view(ko.DTYPES[kt]), offsets, kt, desc, f"mixed {kt},{desc}")


# ---- fallbacks and invariants ----------------------------------------------------------------------------------------
def test_rank_safe_fallback_gives_the_same_bytes():
    """With B200SORT_RANK_SAFE=1 the ballot-ranked forms run, in every class, for keys and for pairs."""
    code = (
        "import sys; sys.path.insert(0, '.'); sys.path.insert(0, 'tests')\n"
        "import numpy as np\n"
        "from b200sort._lib import lib\n"
        "import key_orders64 as ko\n"
        "import test_segmented64_gpu as t\n"
        "assert lib().b200sort_radix_atomic_order_ok() == 0\n"
        "offsets = t.ragged_offsets(41, total_segments=2000, big=1)\n"
        "n = int(offsets[-1])\n"
        "for kt, desc in ko.ORDERS:\n"
        "    k = t.random_keys(n, kt, kt + desc)\n"
        "    t.check_all(k, offsets, kt, desc, ('safe', kt, desc), modes=((False, False), (True, True)))\n"
        "    k = (k.view(np.uint64) % np.uint64(100)).view(ko.DTYPES[kt])\n"
        "    t.check_all(k, offsets, kt, desc, ('safe ties', kt, desc), modes=((True, False),))\n"
        "print('ok')\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", code], cwd=root, env={**os.environ, "B200SORT_RANK_SAFE": "1"},
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


def _counted(keys, offsets, kt, desc, pairs):
    L = lib()
    vals = np.arange(keys.size, dtype=np.int32) if pairs else None
    L.b200sort_launch_count_reset()
    got = run(keys, offsets, kt, desc, vals)
    return got, L.b200sort_launch_count()


def test_independent_of_the_1d_variant_and_skip_switches():
    L = lib()
    offsets = ragged_offsets(31, total_segments=1000, big=1)
    keys = varying_bytes(int(offsets[-1]), 0x0F, 3).view(np.int64)        # upper passes skipped
    base = [_counted(keys, offsets, ko.KEY_I64, 1, p) for p in (False, True)]
    try:
        assert L.b200sort_radix_set_variant(2) == 0
        L.b200sort_radix_set_skip(0)
        other = [_counted(keys, offsets, ko.KEY_I64, 1, p) for p in (False, True)]
    finally:
        L.b200sort_radix_set_variant(0)
        L.b200sort_radix_set_skip(1)
    assert base[0][0].tobytes() == other[0][0].tobytes() and base[0][1] == other[0][1]
    assert all(a.tobytes() == b.tobytes() for a, b in zip(base[1][0], other[1][0])) and base[1][1] == other[1][1]
    assert_words(base[0][0], seg_sort_keys(keys, offsets, ko.KEY_I64, 1), "reference")


def test_launch_count_does_not_depend_on_segments_or_skip_pattern():
    n = 1 << 20
    counts = set()
    for S in (1, 7, 1000, 10 ** 6):
        offsets = (np.arange(S + 1, dtype=np.int64) * n // S)
        for mask in (0x00, 0x0F, 0xF0, 0x55, 0xAA, 0xFF):
            keys = varying_bytes(n, mask, S + mask).view(np.int64)
            for pairs in (False, True):
                got, c = _counted(keys, offsets, ko.KEY_I64, 0, pairs)
                counts.add((pairs, c))
                if mask in (0x55, 0xFF):
                    want = seg_sort_keys(keys, offsets, ko.KEY_I64, 0)
                    assert_words(got[0] if pairs else got, want, f"S={S} mask={mask:#x}")
    assert len(counts) == 2, counts


def test_cuda_graph_capture_and_replay():
    import torch
    L = lib()
    check(L.b200sort_device_check())
    B, Lr = 64, 9000
    x = torch.empty((B, Lr), dtype=torch.int64, device="cuda")
    v = torch.arange(Lr, dtype=torch.int32, device="cuda").repeat(B).view(B, Lr)
    ko_, vo = torch.empty_like(x), torch.empty_like(v)
    kt_, vt = torch.empty_like(x), torch.empty_like(v)
    offs = torch.tensor([0, 100, 1000, 1000, 50000] + [Lr * i for i in range(6, B + 1)], dtype=torch.int32,
                        device="cuda")
    S = offs.numel() - 1
    nbytes = L.b200sort_segmented64_workspace_bytes(B * Lr, S)
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
    ptr = ws.data_ptr() + (-ws.data_ptr()) % 256
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        check(L.b200sort_segmented_pairs_keys64(ko.KEY_I64, 1, x.data_ptr(), v.data_ptr(), ko_.data_ptr(),
                                                vo.data_ptr(), kt_.data_ptr(), vt.data_ptr(), B * Lr, offs.data_ptr(), S,
                                                ptr, nbytes, s.cuda_stream))
    o = offs.cpu().numpy()
    for seed, mask in ((1, 0xFF), (2, 0x0F), (3, 0x81), (4, 0x00)):       # the replays skip different passes
        keys = varying_bytes(B * Lr, mask, seed).view(np.int64)
        x.copy_(torch.from_numpy(keys).view(B, Lr))
        g.replay()
        torch.cuda.synchronize()
        wk, wv = seg_sort_pairs(keys, np.tile(np.arange(Lr, dtype=np.int32), B), o, ko.KEY_I64, 1)
        assert_words(ko_.view(-1).cpu().numpy().view(np.uint64), wk, f"replay {seed}")
        assert vo.view(-1).cpu().numpy().tobytes() == wv.tobytes(), seed


def test_malformed_offsets_stay_in_bounds():
    """Malformed offsets give an undefined order, but every key and value written lies in the output: the guard
    words around out and tmp are untouched (run() checks them)."""
    n = 50000
    keys = random_keys(n, ko.KEY_U64, 77)
    cases = ([0, 30000, 10000, 50000], [0, 60000, -5, 20000, 99999], [5, 4, 3, 2, 1, 0], [0, 40000, 9000, 45000, 50000],
             [0, 9000, 3, 20000, 19000, 50000], [0, 20000, 0, 20000, 50000])
    for offs in cases:
        for pairs in (False, True):
            for in_place in (False, True):
                run(keys, offs, ko.KEY_U64, int(pairs), np.arange(n, dtype=np.int32) if pairs else None, in_place)


def _rows(torch, B, L_, dtype, seed):
    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    if dtype == torch.float64:
        x = torch.randn((B, L_), device="cuda", generator=g, dtype=torch.float64)
        return torch.where(x == 0, torch.ones_like(x), x)                 # no +-0.0: torch.sort treats them as equal
    return torch.randint(-2 ** 62, 2 ** 62, (B, L_), device="cuda", generator=g, dtype=torch.int64) // (
        1 if seed % 2 else 2 ** 40)


@pytest.mark.parametrize("L_", [8, 64, 256, 1024, 8192, 32000, 128256])
def test_python_calls_match_torch_sort(L_):
    import torch
    B = max(1, (1 << 21) // L_)
    idx = torch.arange(L_, dtype=torch.int32, device="cuda").repeat(B).view(B, L_)
    for dtype, seed in ((torch.float64, 1), (torch.int64, 2), (torch.int64, 3)):
        x = _rows(torch, B, L_, dtype, L_ + seed)
        pristine = x.clone()
        for desc in (True, False):
            tv, ti = torch.sort(x, dim=-1, stable=True, descending=desc)
            k = b200sort.segmented_sort64(x, descending=desc)
            assert k.shape == x.shape and k.dtype == dtype and torch.equal(k, tv), (dtype, desc)
            k, v = b200sort.segmented_sort64_by_key(x, idx, descending=desc)
            assert torch.equal(k, tv) and torch.equal(v, ti.to(torch.int32)), (dtype, desc)
            offs = torch.arange(B + 1, device="cuda") * L_                   # the same rows as 1-D keys and offsets
            for o in (offs, offs.to(torch.int32)):
                k1, v1 = b200sort.segmented_sort64_by_key(x.view(-1), idx.view(-1), o, descending=desc)
                assert torch.equal(k1.view(B, L_), tv) and torch.equal(v1.view(B, L_), ti.to(torch.int32))
        assert torch.equal(x.view(torch.int64), pristine.view(torch.int64))


def test_python_call_on_a_slice_starting_at_element_1():
    import torch
    n = 30001
    base = torch.from_numpy(random_keys(n + 1, ko.KEY_I64, 6)).cuda()
    x = base[1:]                                                        # 8 bytes past the allocation's start
    offs = torch.tensor([0, 5, 200, 3000, 12000, n], device="cuda")
    got = b200sort.segmented_sort64(x, offs, descending=True)
    want = seg_sort_keys(x.cpu().numpy(), offs.cpu().numpy(), ko.KEY_I64, 1)
    assert_words(got.cpu().numpy().view(np.uint64), want, "slice")
    k, v = b200sort.segmented_sort64_by_key(x, torch.arange(n, dtype=torch.int32, device="cuda"), offs)
    wk, wv = seg_sort_pairs(x.cpu().numpy(), np.arange(n, dtype=np.int32), offs.cpu().numpy(), ko.KEY_I64, 0)
    assert_words(k.cpu().numpy().view(np.uint64), wk, "slice pairs")
    assert v.cpu().numpy().tobytes() == wv.tobytes()


def test_python_call_rejects_invalid_offsets_before_any_launch():
    import torch
    L = lib()
    x = torch.zeros(100, dtype=torch.int64, device="cuda")
    for b in ([1, 100], [0, 99], [0, 101], [0, 60, 40, 100], [-1, 50, 100]):
        for dt in (torch.int32, torch.int64):
            L.b200sort_launch_count_reset()
            with pytest.raises(ValueError):
                b200sort.segmented_sort64(x, torch.tensor(b, dtype=dt, device="cuda"))
            with pytest.raises(ValueError):
                b200sort.segmented_sort64_by_key(x, torch.zeros(100, dtype=torch.int32, device="cuda"),
                                                 torch.tensor(b, dtype=dt, device="cuda"))
            assert L.b200sort_launch_count() == 0, b


def test_python_call_on_a_non_default_device():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible")
    dev = torch.device("cuda", torch.cuda.device_count() - 1)
    B, L_ = 30, 30001
    w = random_keys(B * L_, ko.KEY_F64, 5)
    x = torch.from_numpy(w).to(dev).view(B, L_)
    assert torch.cuda.current_device() != dev.index
    offsets = np.arange(B + 1) * L_
    got = b200sort.segmented_sort64(x, descending=True)
    assert got.device == dev
    assert_words(got.cpu().numpy().reshape(-1).view(np.uint64), seg_sort_keys(w, offsets, ko.KEY_F64, 1), "keys")
    v = torch.arange(L_, dtype=torch.int32, device=dev).repeat(B).view(B, L_)
    k, vv = b200sort.segmented_sort64_by_key(x, v)
    wk, wv = seg_sort_pairs(w, np.tile(np.arange(L_, dtype=np.int32), B), offsets, ko.KEY_F64, 0)
    assert_words(k.cpu().numpy().reshape(-1).view(np.uint64), wk, "pairs keys")
    assert vv.cpu().numpy().reshape(-1).tobytes() == wv.tobytes()


# ---- full size -------------------------------------------------------------------------------------------------------
def _image_i64(torch, k, desc):
    """image(k) - 2^63 as int64, so that torch's signed compare is the uint64 order of the images."""
    neg, pos = ko.MASKS[(ko.KEY_I64, desc)]
    m = torch.where(k < 0, torch.tensor(neg - (1 << 64) if neg >= 1 << 63 else neg, device=k.device),
                    torch.tensor(pos - (1 << 64) if pos >= 1 << 63 else pos, device=k.device))
    return (k ^ m) ^ torch.tensor(-(1 << 63), device=k.device)


@pytest.mark.parametrize("L_", [1 << 12, 1 << 17])
def test_full_size_2_28_rows(L_):
    """2^28 int64 keys in rows, descending pairs: every row sorted, a permutation of its row, stable."""
    import torch
    n = 1 << 28
    B = n // L_
    g = torch.Generator(device="cuda"); g.manual_seed(12)
    x = torch.randint(0, 1 << 20, (n,), dtype=torch.int64, device="cuda", generator=g) * 0x100000001 - (1 << 40)
    v = torch.arange(L_, dtype=torch.int32, device="cuda").repeat(B)
    k, vo = b200sort.segmented_sort64_by_key(x.view(B, L_), v.view(B, L_), descending=True)
    torch.cuda.synchronize()
    img = _image_i64(torch, k, 1)
    assert not bool((img[:, 1:] < img[:, :-1]).any()), "a row is not sorted"
    ties = img[:, 1:] == img[:, :-1]
    assert not bool((ties & (vo[:, 1:] <= vo[:, :-1])).any()), "equal keys out of input order"
    del img, ties
    assert torch.equal(torch.sort(vo, dim=-1)[0], v.view(B, L_)), "values are not a permutation of each row"
    assert torch.equal(torch.gather(x.view(B, L_), 1, vo.to(torch.int64)), k)


def test_n_2_30_in_one_segment():
    """n = 2^30 is accepted: one segment of int64 ids below 2^32, where the 4 upper digits hold all 2^30 keys (those
    passes are skipped).  Checked by order and by a fingerprint of the multiset."""
    import torch
    n = 1 << 30
    g = torch.Generator(device="cuda"); g.manual_seed(30)
    x = torch.randint(0, 1 << 32, (n,), dtype=torch.int64, device="cuda", generator=g)
    fp = lambda t: (int(t.sum()), int((t * 0x1E3779B97F4A7C15).bitwise_xor(t >> 7).sum()))
    want = fp(x)
    y = b200sort.segmented_sort64(x, torch.tensor([0, n], dtype=torch.int64, device="cuda"))
    torch.cuda.synchronize()
    del x
    assert not bool((y[1:] < y[:-1]).any()), "not sorted"
    assert fp(y) == want, "not a permutation of the input"
