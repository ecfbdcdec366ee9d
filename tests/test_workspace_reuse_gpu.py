"""A reused, never-cleared workspace and guarded buffers for the 16-bit, segmented, merge and lab sorts, stale state
left by one entry point for another (the 64-bit and the indices sorts among them), and CUDA graph replay of the 32-bit
1-D sorts.

Every device-array entry point takes a caller-owned workspace and must rewrite whatever it reads there before reading
it: real callers (torch's caching allocator, a benchmark loop, a replayed graph) hand it back holding the previous
call's bytes, often in another entry point's layout.  A status row that a call forgot to clear reads as a wrong prefix
and puts keys in the wrong place; a write past ws_bytes, tmp[n] or out[n] lands in a neighbouring allocation.  Neither
crashes, so this module looks for both:
  * one workspace for the whole module (digit_patterns.Workspace), filled with 0xFF once and never cleared, sized for
    the largest call of any family; the bytes past each call's ws_bytes must not change;
  * every key and value array inside canary words (digit_patterns.DevBuf): nothing may be written past n in out or
    tmp, and the copy forms must leave their inputs alone;
  * explicit pairs of calls (A, then B) on that workspace, where A leaves flags and plausible counts where B reads;
  * the 32-bit entry points captured once in a CUDA graph and replayed on data that takes other device-side plans.

Everything goes through the C-ABI; torch only owns the memory.  References are stable numpy argsorts of the key
images (tests/key_orders.py, key_orders16.py, key_orders64.py), per segment for the segmented sorts (np.lexsort), with
the argsort itself (made segment-local) as the reference of the int64 indices, and oracle.radix_sort for the lab
pipeline; results are compared byte for byte.
"""
import functools

import numpy as np
import pytest

import digit_patterns as dp
import key_orders as ko
import key_orders16 as ko16
import key_orders64 as ko64
import oracle
from b200sort import datagen
from b200sort._lib import ALGO_LAB, ALGO_MERGE, ALGO_RADIX, check, lib
from helpers import stream_ptr
from test_keys16_gpu import random_keys as keys16_of
from test_keys64_gpu import random_keys as keys64_of
from test_segmented_cpu import segment_ids
from test_segmented_gpu import mixed_keys as keys32_of, ragged_offsets

pytestmark = pytest.mark.gpu

N16 = [1, 2, 8191, 8193, 65537, (1 << 20) + 3, (1 << 23) + 5]
N16_BIG = (1 << 23) + 5
N32_BIG = (1 << 23) + 4099                  # the default configuration runs tma3 (group rows in the status area)
MERGE_N = [4097, 100001, (1 << 20) + 4099]
LAB_N = [1, 2, 4095, 4096, 4097, 100001, (1 << 20) + 4099]
ORDERS16_IDS = [f"{ko16.NAMES[k]}_{'desc' if d else 'asc'}" for k, d in ko16.ORDERS]
MERGE_ORDERS = [(ko.KEY_U32, 0), (ko.KEY_U32, 1), (ko.KEY_F32, 0), (ko.KEY_F32, 1)]
I32 = (ko.KEY_I32, 0)
# word offsets of (keys in, keys out, keys tmp, values in, values out, values tmp) past a 16-byte boundary; 2-byte keys
# count 2-byte words, so 1, 3 and 7 are 2, 6 and 14 bytes
OFFS16 = [(0, 0, 0, 0, 0, 0), (1, 3, 7, 1, 2, 3), (3, 7, 1, 2, 3, 0), (7, 1, 3, 3, 0, 1)]
OFFS32 = [(0, 0, 0, 0, 0, 0), (1, 2, 3, 1, 2, 3), (2, 3, 1, 2, 3, 0), (3, 1, 2, 3, 0, 1)]
# 8-byte keys and int64 indices need 8-byte alignment: even word offsets
OFFS64 = [(0, 0, 0, 0, 0, 0), (2, 0, 2, 1, 2, 3)]
# image masks whose zero bytes make the digit passes over them skippable: 16-bit pass 1, 32-bit passes 1 and 3,
# 64-bit passes 1, 3, 5 and 7
MASKED = {16: 0x00FF, 32: 0x00FF00FF, 64: 0x00FF00FF00FF00FF}

# family: (key bits, pairs, scratch keys); the C-ABI entry points beside each
FAMILIES = {
    "keys16": (16, False, False),       # b200sort_sort_keys16
    "pairs16": (16, True, True),        # b200sort_radix_pairs_keys16
    "seg16": (16, False, True),         # b200sort_segmented_sort_keys16
    "seg16_pairs": (16, True, True),    # b200sort_segmented_pairs_keys16
    "seg": (32, False, True),           # b200sort_segmented_sort_keys
    "seg_pairs": (32, True, True),      # b200sort_segmented_pairs_keys
    "i32": (32, False, True),           # b200sort_sort_i32 (in place) / b200sort_sort_copy_i32, with `algo`
    "keys": (32, False, True),          # b200sort_sort_keys, with `algo`
    "pairs_i32": (32, True, True),      # b200sort_radix_pairs_i32 / b200sort_radix_pairs_copy_i32
    "pairs": (32, True, True),          # b200sort_radix_pairs_keys
    "keys64": (64, False, True),        # b200sort_sort_keys64
    "pairs64": (64, True, True),        # b200sort_radix_pairs_keys64
    "seg64": (64, False, True),         # b200sort_segmented_sort_keys64
    "seg64_pairs": (64, True, True),    # b200sort_segmented_pairs_keys64
    "idx": (32, False, True),           # b200sort_radix_sort_indices_keys
    "seg_idx": (32, False, True),       # b200sort_segmented_sort_indices_keys
    "idx16": (16, False, True),         # b200sort_radix_sort_indices_keys16
    "seg_idx16": (16, False, True),     # b200sort_segmented_sort_indices_keys16
}
# the families that return int64 indices (into an 8-byte buffer) and take n int32 of index scratch
INDICES = {"idx", "seg_idx", "idx16", "seg_idx16"}


def _ko(width: int):
    return {16: ko16, 32: ko, 64: ko64}[width]


# ---- segment layouts ---------------------------------------------------------------------------------------------
def _class_bounds(width: int):
    L = lib()
    f = {16: L.b200sort_segmented16_class_max, 32: L.b200sort_segmented_class_max,
         64: L.b200sort_segmented64_class_max}[width]
    out, c = [], 0
    while f(c):
        out.append(f(c))
        c += 1
    return out


def row_lengths(width: int):
    """Every class boundary +-1."""
    return sorted({x for m in _class_bounds(width) for x in (m - 1, m, m + 1) if x >= 1})


@functools.lru_cache(maxsize=None)
def layout(name) -> np.ndarray:
    """int32 offsets of a named layout; the last one is n."""
    kind = name[0]
    if kind == "rows":                                           # B equal rows of L keys
        _, L_, B = name
        return (np.arange(B + 1, dtype=np.int64) * L_).astype(np.int32)
    if kind == "ragged":                                         # empty, one-key, every class, > 2^20
        _, seed, total, big = name
        return ragged_offsets(seed, total_segments=total, big=big)
    if kind == "one":
        return np.array([0, name[1]], np.int32)
    if kind == "long_ragged":                                    # one long segment, then a ragged tail
        tail = ragged_offsets(name[1], total_segments=2000, big=0)
        return np.concatenate([[0], tail + (1 << 22)]).astype(np.int32)
    if kind in ("many_large", "few_large"):
        # the same n and number of segments, so the same workspace layout: 200 segments of 40000 keys and 3896 empty
        # ones, or 3 large segments among 4093 of 2..1024 keys (or S segments, `large` of them of 40000 keys)
        S, large = name[1:] if len(name) > 1 else (4096, 200)
        n = large * 40000
        if kind == "many_large":
            lens = np.concatenate([np.full(large, 40000), np.zeros(S - large, np.int64)])
        else:
            small = np.random.default_rng(5).integers(2, 1025, S - 3)
            rest = n - int(small.sum())
            lens = np.concatenate([small[:1000], [rest // 3], small[1000:2000], [rest // 3], small[2000:],
                                   [rest - 2 * (rest // 3)]])
        return np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    raise ValueError(name)


def class_rows(width: int):
    return [("rows", L_, max(1, min(1024, (1 << 20) // L_))) for L_ in row_lengths(width)]


RAGGED = ("ragged", 17, 3000, 2)
ONE = ("one", (1 << 21) + 7)
ROWS_2_17 = ("rows", 1 << 17, 64)
LONG_RAGGED = ("long_ragged", 9)
RAGGED_SMALL = ("ragged", 23, 3000, 0)                          # 1.75M keys: 12 onesweep-class segments
MANY_LARGE_2M, FEW_LARGE_2M = ("many_large", 1024, 48), ("few_large", 1024, 48)     # 1.92M keys
ROWS_9000 = ("rows", 9000, 232)                                  # 2.09M keys in onesweep-class rows


def seg_ws_bytes(width: int, n: int, S: int) -> int:
    L = lib()
    return {16: L.b200sort_segmented16_workspace_bytes, 32: L.b200sort_segmented_workspace_bytes,
            64: L.b200sort_segmented64_workspace_bytes}[width](n, S)


def ws_need(fam: str, n: int, seg=None, algo: int = ALGO_RADIX) -> int:
    """The workspace bytes of one call.  The indices sorts take those of the pairs sorts of their width."""
    L = lib()
    width = FAMILIES[fam][0]
    if seg is not None:
        offs = layout(seg)
        return seg_ws_bytes(width, int(offs[-1]), offs.size - 1)
    if width == 16:
        return L.b200sort_keys16_workspace_bytes(n)
    if width == 64:
        return L.b200sort_keys64_workspace_bytes(n)
    return L.b200sort_workspace_bytes(n, algo)


# ---- the module's workspace and buffers ----------------------------------------------------------------------------
_ws = None


def workspace() -> dp.Workspace:
    global _ws
    if _ws is None:
        L = lib()
        needs = [L.b200sort_keys16_workspace_bytes(N16_BIG), L.b200sort_workspace_bytes(N32_BIG, ALGO_RADIX),
                 L.b200sort_workspace_bytes(N32_BIG, ALGO_MERGE)]
        seg = [(w, name) for w in (16, 32) for name in class_rows(w) + [RAGGED, ONE]]
        for width, name in seg:
            offs = layout(name)
            needs.append(seg_ws_bytes(width, int(offs[-1]), offs.size - 1))
        needs += [ws_need(job[0], job[1], job[4], job[5]) for pair in STALE.values() for job in pair]
        _ws = dp.Workspace(max(needs))
    return _ws


@pytest.fixture(scope="module", autouse=True)
def _workspace_tail_and_check_failures():
    yield
    L = lib()
    if _ws is not None:
        _ws.check_tail()
    if L.b200sort_debug_checked_build() == 1:
        assert L.b200sort_debug_check_failures() == 0


_bufs = {}


def _buf(role: str, n: int, word_offset: int, itemsize: int) -> dp.DevBuf:
    key = (role, n, word_offset, itemsize)
    if key not in _bufs:
        _bufs[key] = dp.DevBuf(n, word_offset, itemsize, salt=len(_bufs) + 1)
    return _bufs[key]


@functools.lru_cache(maxsize=None)
def _device_offsets(name):
    import torch
    return torch.from_numpy(layout(name)).cuda()


# ---- one guarded call --------------------------------------------------------------------------------------------
def run(fam: str, keys: np.ndarray, order, in_place: bool = False, offs=OFFS32[0], seg=None, algo: int = ALGO_RADIX,
        what: str = ""):
    """Sort `keys` by family `fam` (FAMILIES) with every array guarded, on the module workspace.  Pairs carry the
    values arange(n).  seg: the layout name of the segmented families.  Returns (key words, values, int64 indices or
    None)."""
    import torch
    L = lib()
    width, pairs, has_tmp = FAMILIES[fam]
    kt, desc = order
    item = width // 8
    n = keys.size
    words = _ko(width).bits(keys)
    kin = _buf("kin", n, offs[0], item).load(words)
    kout = kin if in_place else _buf("kout", n, offs[1], item).load()
    ktmp = _buf("ktmp", n, offs[2], item).load() if has_tmp else None
    if pairs:
        vals = np.arange(n, dtype=np.int32)
        vin = _buf("vin", n, offs[3], 4).load(vals)
        vout = vin if in_place else _buf("vout", n, offs[4], 4).load()
        vtmp = _buf("vtmp", n, offs[5], 4).load()
    if fam in INDICES:
        iout = _buf("iout", n, 2 * (offs[4] & 1), 8).load()
        itmp = _buf("itmp", n, offs[5], 4).load()
    if seg is not None:
        d_off = _device_offsets(seg)
        S = d_off.numel() - 1
        assert int(layout(seg)[-1]) == n
    need = ws_need(fam, n, seg, algo)
    ws = workspace()
    assert need + ws.GUARD <= ws.cap, f"{what}: the module workspace is sized without this call"
    before = ws.guard(need).cpu()
    s = stream_ptr()
    if fam == "keys16":
        st = L.b200sort_sort_keys16(kt, desc, kin.ptr, kout.ptr, n, ws.ptr, need, s)
    elif fam == "pairs16":
        st = L.b200sort_radix_pairs_keys16(kt, desc, kin.ptr, vin.ptr, kout.ptr, vout.ptr, ktmp.ptr, vtmp.ptr, n,
                                           ws.ptr, need, s)
    elif fam in ("seg16", "seg", "seg64"):
        f = {16: L.b200sort_segmented_sort_keys16, 32: L.b200sort_segmented_sort_keys,
             64: L.b200sort_segmented_sort_keys64}[width]
        st = f(kt, desc, kin.ptr, kout.ptr, ktmp.ptr, n, d_off.data_ptr(), S, ws.ptr, need, s)
    elif fam in ("seg16_pairs", "seg_pairs", "seg64_pairs"):
        f = {16: L.b200sort_segmented_pairs_keys16, 32: L.b200sort_segmented_pairs_keys,
             64: L.b200sort_segmented_pairs_keys64}[width]
        st = f(kt, desc, kin.ptr, vin.ptr, kout.ptr, vout.ptr, ktmp.ptr, vtmp.ptr, n, d_off.data_ptr(), S, ws.ptr,
               need, s)
    elif fam == "keys64":
        st = L.b200sort_sort_keys64(kt, desc, kin.ptr, kout.ptr, ktmp.ptr, n, ws.ptr, need, s)
    elif fam == "pairs64":
        st = L.b200sort_radix_pairs_keys64(kt, desc, kin.ptr, vin.ptr, kout.ptr, vout.ptr, ktmp.ptr, vtmp.ptr, n,
                                           ws.ptr, need, s)
    elif fam in ("idx", "idx16"):
        f = L.b200sort_radix_sort_indices_keys16 if width == 16 else L.b200sort_radix_sort_indices_keys
        st = f(kt, desc, kin.ptr, kout.ptr, iout.ptr, ktmp.ptr, itmp.ptr, n, ws.ptr, need, s)
    elif fam in ("seg_idx", "seg_idx16"):
        f = L.b200sort_segmented_sort_indices_keys16 if width == 16 else L.b200sort_segmented_sort_indices_keys
        st = f(kt, desc, kin.ptr, kout.ptr, iout.ptr, ktmp.ptr, itmp.ptr, n, d_off.data_ptr(), S, ws.ptr, need, s)
    elif fam == "i32":
        assert order == I32
        st = (L.b200sort_sort_i32(algo, kin.ptr, ktmp.ptr, n, ws.ptr, need, s) if in_place else
              L.b200sort_sort_copy_i32(algo, kin.ptr, kout.ptr, ktmp.ptr, n, ws.ptr, need, s))
    elif fam == "keys":
        st = L.b200sort_sort_keys(algo, kt, desc, kin.ptr, kout.ptr, ktmp.ptr, n, ws.ptr, need, s)
    elif fam == "pairs_i32":
        assert order == I32
        st = (L.b200sort_radix_pairs_i32(kin.ptr, vin.ptr, ktmp.ptr, vtmp.ptr, n, ws.ptr, need, s) if in_place else
              L.b200sort_radix_pairs_copy_i32(kin.ptr, vin.ptr, kout.ptr, vout.ptr, ktmp.ptr, vtmp.ptr, n, ws.ptr,
                                              need, s))
    elif fam == "pairs":
        st = L.b200sort_radix_pairs_keys(kt, desc, kin.ptr, vin.ptr, kout.ptr, vout.ptr, ktmp.ptr, vtmp.ptr, n,
                                         ws.ptr, need, s)
    else:
        raise ValueError(fam)
    check(st)
    torch.cuda.synchronize()
    got = kout.read(f"{what} keys out").view(words.dtype)
    if has_tmp:
        ktmp.read(f"{what} keys tmp")
    if not in_place:
        assert kin.read(f"{what} keys in").tobytes() == words.tobytes(), f"{what}: the copy form modified its keys"
    got_vals = None
    if pairs:
        got_vals = vout.read(f"{what} values out")
        vtmp.read(f"{what} values tmp")
        if not in_place:
            assert vin.read(f"{what} values in").tobytes() == vals.tobytes(), f"{what}: the copy form modified its values"
    if fam in INDICES:
        got_vals = iout.read(f"{what} indices out").view(np.int64)
        itmp.read(f"{what} indices tmp")
    assert torch.equal(ws.guard(need).cpu(), before), f"{what}: workspace written past ws_bytes = {need}"
    return got, got_vals


def assert_words(got: np.ndarray, want: np.ndarray, what: str):
    if got.tobytes() != want.tobytes():
        bad = np.flatnonzero(got != want)
        w = 2 + 2 * got.dtype.itemsize
        raise AssertionError(f"{what}: {bad.size} of {got.size} words differ, first at {bad[0]}: "
                             f"got {int(got[bad[0]]):#0{w}x}, want {int(want[bad[0]]):#0{w}x}")


@functools.lru_cache(maxsize=8)
def case(width: int, n: int, order, seed: int, seg=None, data: str = "random"):
    """(keys, reference permutation) of random bit patterns with float specials, or (data "masked") of random images
    with the zero bytes of MASKED: a stable argsort of the images, segment by segment if `seg` names a layout (then n
    is the layout's)."""
    kt, desc = order
    if seg is not None:
        n = int(layout(seg)[-1])
    keys = {16: keys16_of, 32: keys32_of, 64: keys64_of}[width](n, kt, seed)
    k = _ko(width)
    if data == "masked":
        w = k.bits(keys)
        keys = k.inverse(w & w.dtype.type(MASKED[width]), kt, desc)
    img = k.image(keys, kt, desc)
    perm = (np.argsort(img, kind="stable") if seg is None else np.lexsort((img, segment_ids(layout(seg)))))
    return keys, perm


def expect(fam: str, n: int, order, seed: int, what: str, seg=None, algo: int = ALGO_RADIX, data: str = "random",
           **kw):
    """run() on the keys of case() and compare with the reference, byte for byte."""
    width = FAMILIES[fam][0]
    keys, perm = case(width, n, order, seed, seg, data)
    got, got_vals = run(fam, keys, order, seg=seg, algo=algo, what=what, **kw)
    if algo == ALGO_LAB:
        want = oracle.radix_sort(keys).view(np.uint32)
        assert want.tobytes() == _ko(width).bits(keys)[perm].tobytes()      # the oracle and the argsort agree
    else:
        want = _ko(width).bits(keys)[perm]
    assert_words(got, want, what)
    if fam in INDICES:
        pos = np.arange(keys.size, dtype=np.int64)
        if seg is not None:                                              # positions inside the segment
            offs = layout(seg).astype(np.int64)
            pos -= offs[:-1][segment_ids(offs)]
        assert_words(got_vals, pos[perm], what + " indices")
    elif got_vals is not None:
        assert_words(got_vals, perm.astype(np.uint32), what + " values")


def _n_of(seg) -> int:
    return int(layout(seg)[-1])


# ---- 2. guarded single calls -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("order", ko16.ORDERS, ids=ORDERS16_IDS)
def test_keys16_and_pairs16_guarded(order):
    j = ko16.ORDERS.index(order)
    for i, n in enumerate(N16):
        for in_place in (False, True):
            o = OFFS16[(i + j + in_place) % len(OFFS16)]
            if in_place:
                o = (o[0], o[0], o[2], o[3], o[3], o[5])
            for fam in ("keys16", "pairs16"):
                expect(fam, n, order, n + j, f"{fam} {order} n={n} in_place={in_place} offsets {o}", in_place=in_place,
                       offs=o)


@pytest.mark.parametrize("width", [32, 16])
@pytest.mark.parametrize("kind", ["class_rows", "ragged", "one_segment"])
def test_segmented_guarded(kind, width):
    """Equal rows at every class boundary +-1 (the orders take turns), a ragged mix with empty, one-key and > 2^20-key
    segments, and one segment of all n keys, in every order, keys and pairs, in place and copied."""
    orders = ko16.ORDERS if width == 16 else ko.ORDERS
    fams = ("seg16", "seg16_pairs") if width == 16 else ("seg", "seg_pairs")
    offsets = OFFS16 if width == 16 else OFFS32
    if kind == "class_rows":
        runs = [(name, orders[i % len(orders)], i) for i, name in enumerate(class_rows(width))]
    else:
        name = RAGGED if kind == "ragged" else ONE
        runs = [(name, order, i) for i, order in enumerate(orders)]
    for name, order, i in runs:
        for in_place in (False, True):
            o = offsets[(i + in_place) % len(offsets)]
            if in_place:
                o = (o[0], o[0], o[2], o[3], o[3], o[5])
            for fam in fams:
                expect(fam, _n_of(name), order, i, f"{fam} {name} {order} in_place={in_place} offsets {o}", seg=name,
                       in_place=in_place, offs=o)


@pytest.mark.parametrize("order", MERGE_ORDERS, ids=["u32_asc", "u32_desc", "f32_asc", "f32_desc"])
def test_merge_sort_keys_guarded(order):
    """b200sort_sort_keys with the merge algorithm: the non-default orders keep their split points in the workspace."""
    for n in MERGE_N:
        for o in OFFS32:
            expect("keys", n, order, n, f"merge {order} n={n} offsets {o}", algo=ALGO_MERGE, offs=o)
        expect("keys", n, order, n, f"merge {order} n={n} in place", algo=ALGO_MERGE, in_place=True,
               offs=(1, 1, 3, 0, 0, 0))


def test_lab_pipeline_guarded():
    """b200sort_sort_i32 / b200sort_sort_copy_i32 with the lab algorithm, against oracle.radix_sort."""
    for i, n in enumerate(LAB_N):
        for in_place in (False, True):
            o = OFFS32[(i + in_place) % len(OFFS32)]
            if in_place:
                o = (o[0], o[0], o[2], 0, 0, 0)
            expect("i32", n, I32, n, f"lab n={n} in_place={in_place} offsets {o}", algo=ALGO_LAB, in_place=in_place,
                   offs=o)


# ---- 3. stale state from another call ------------------------------------------------------------------------------
# A job: (family, n or None, order, seed, segment layout or None, algo, in place, data).  Each case runs A, then B
# twice on the shared workspace without clearing it, and names the region of state B must rewrite before it reads it.
def J(fam, n=None, order=I32, seed=0, seg=None, algo=ALGO_RADIX, in_place=False, data="random"):
    return (fam, n if seg is None else _n_of(seg), order, seed, seg, algo, in_place, data)


BF16_D, U16_A, F32_D, U32_D = (ko16.KEY_BF16, 1), (ko16.KEY_U16, 0), (ko.KEY_F32, 1), (ko.KEY_U32, 1)
F32_A, I32_D, F16_A = (ko.KEY_F32, 0), (ko.KEY_I32, 1), (ko16.KEY_F16, 0)
F64_D, F64_A, U64_A, I64_D = (ko64.KEY_F64, 1), (ko64.KEY_F64, 0), (ko64.KEY_U64, 0), (ko64.KEY_I64, 1)
STALE = {
    # the segmented sort's lists, histograms and status rows (flags and counts of 1024 full tiles) lie where the
    # 16-bit sort keeps the not-zeroed half of its control block (incl, digit bases, skip flags, buffer plan) and its
    # per-CTA count rows: the scan kernel and the passes must write them before they read them
    "seg16_rows_then_pairs16": (J("seg16_pairs", order=BF16_D, seg=ROWS_2_17), J("pairs16", (1 << 20) + 3, U16_A, 1)),
    # 148 per-CTA count rows and 2 x 1025 status rows with flags, then a segmented call whose segment histograms and
    # status rows lie on them: classify must zero each large segment's histogram, the histogram kernel the first
    # pass's rows of every tile, pass 0 the second pass's rows
    "pairs16_big_then_seg16_long_ragged": (J("pairs16", N16_BIG, BF16_D, 2, in_place=True),
                                           J("seg16_pairs", order=U16_A, seg=LONG_RAGGED, seed=3)),
    # the same layout (n, number of segments): 200 large segments leave list entries, histograms, prefix and status
    # rows; B has 3 large segments, so list entries past its device count, and rows past its tiles, are stale
    "seg_many_large_then_few_large": (J("seg_pairs", order=F32_D, seg=("many_large",)),
                                      J("seg_pairs", order=U32_D, seg=("few_large",), seed=1)),
    # tma3's look-back group rows and tile rows (flags, counts) where the segmented sort keeps its lists, histograms and
    # status rows
    "radix_tma3_then_seg_pairs": (J("i32", N32_BIG, I32, 4), J("seg_pairs", order=F32_D, seg=RAGGED, seed=5)),
    # the segmented sort's control, lists and prefix where the merge sort keeps its split points
    "seg_then_merge": (J("seg", order=F32_D, seg=RAGGED, seed=6), J("keys", (1 << 20) + 4099, U32_D, 7, algo=ALGO_MERGE)),
    # a large call then a small one of the same family: the small call's rows are a prefix of the large call's, all
    # holding flags and counts, and its control block holds the large call's tickets, plan and scan results
    "keys16_big_then_small": (J("keys16", N16_BIG, BF16_D, 8), J("keys16", 8193, U16_A, 9)),
    "pairs16_big_then_small": (J("pairs16", N16_BIG, U16_A, 10), J("pairs16", 65537, BF16_D, 11)),
    "seg16_big_then_small": (J("seg16_pairs", order=BF16_D, seg=ROWS_2_17, seed=12),
                             J("seg16_pairs", order=U16_A, seg=("rows", 3 * 8192 + 1, 40), seed=13)),
    "seg_big_then_small": (J("seg_pairs", order=F32_D, seg=("many_large",), seed=14),
                           J("seg_pairs", order=U32_D, seg=("rows", 8193, 127), seed=15)),
    "radix_big_then_small": (J("keys", N32_BIG, F32_D, 16), J("keys", 300001, U32_D, 17)),
    "pairs_big_then_small": (J("pairs", N32_BIG, F32_D, 18), J("pairs", 300001, U32_D, 19)),
    "merge_big_then_small": (J("keys", (1 << 20) + 4099, F32_D, 20, algo=ALGO_MERGE),
                             J("keys", 100001, U32_D, 21, algo=ALGO_MERGE)),
    "lab_big_then_small": (J("i32", (1 << 20) + 4099, I32, 22, algo=ALGO_LAB), J("i32", 100001, I32, 23, algo=ALGO_LAB)),
    # The 64-bit and the indices sorts.  The indices sorts use the pairs sorts' workspace layout, and which of their
    # passes runs last, and so stores the int64 indices, is read on the device from the plan in the control block.
    # A runs all four passes and leaves their skip flags (clear), buffer selectors, final-copy word, digit bases and
    # status rows with flags; B's images have bytes 1 and 3 constant: its histogram's last block must rewrite
    # every skip flag and selector, so that pass 2, not A's pass 3, stores the int64 indices
    "pairs_then_idx_masked": (J("pairs", 300001, F32_D, 30), J("idx", 300001, U32_D, 31, data="masked")),
    # the other way round: A leaves passes 1 and 3 flagged as skipped and a plan that ends in pass 2; B runs all four,
    # so its histogram's last block must clear those flags and rewrite the plan before any pass reads them
    "idx_masked_then_pairs": (J("idx", 300001, F32_A, 32, data="masked"), J("pairs", 300001, U32_D, 33)),
    # 8 passes of tickets and digit counts, then 8 x 256 digit bases and the 64-bit plan over the 32-bit control
    # block and its status rows: B's memset must cover its own zeroed half, its histogram the rest, its passes the rows
    "keys64_big_then_idx": (J("keys64", (1 << 21) + 5, F64_D, 34), J("idx", (1 << 20) + 7, I32_D, 35)),
    # the same layout (the 16-bit sorts' workspace): A leaves the block scans, high-byte counts, bases and a plan of
    # two executed passes in the not-zeroed half of the control block; B's high image byte is constant, so pass 1 is
    # skipped and pass 0 must store the int64 indices
    "pairs16_then_idx16_masked": (J("pairs16", 65537, BF16_D, 36), J("idx16", 65537, F16_A, 37, data="masked")),
    # the two passes' status rows with flags and the indices plan, then a counting sort whose per-CTA count rows and scan
    # results lie on them
    "idx16_big_then_keys16_small": (J("idx16", (1 << 21) + 3, BF16_D, 38), J("keys16", 8193, U16_A, 39)),
    # the same layout: 48 large segments leave list entries, first keys, 8-pass histograms, prefix and status rows; B
    # has 3 large segments, so list entries past its device count, and rows past its tiles, are stale
    "seg64_many_large_then_few_large": (J("seg64_pairs", order=F64_D, seg=MANY_LARGE_2M, seed=40),
                                        J("seg64_pairs", order=U64_A, seg=FEW_LARGE_2M, seed=41)),
    # 232 onesweep-class rows leave the indices sort's lists, histograms and status rows; the 64-bit segmented
    # sort keeps its control (the vary words among it), lists, first keys and histograms there
    "seg_idx_rows_then_seg64_ragged": (J("seg_idx", order=F32_D, seg=ROWS_9000, seed=42),
                                       J("seg64", order=I64_D, seg=RAGGED_SMALL, seed=43)),
    # the 64-bit lists, first keys and 8-pass histograms where the 16-bit indices sort keeps its lists, histograms and
    # status rows (rows of 128256 bf16 keys: top-p sampling over a vocabulary)
    "seg64_then_seg_idx16": (J("seg64_pairs", order=U64_A, seg=RAGGED_SMALL, seed=44),
                             J("seg_idx16", order=BF16_D, seg=("rows", 128256, 16), seed=45)),
    # the same layout as the pairs sort: A executes all four passes, B (bytes 1 and 3 constant in every row) two,
    # so its per-segment skip decisions and its last pass must be its own
    "seg_pairs_then_seg_idx_masked": (J("seg_pairs", order=U32_D, seg=ROWS_9000, seed=50),
                                      J("seg_idx", order=F32_D, seg=ROWS_9000, seed=51, data="masked")),
    "keys64_big_then_small": (J("keys64", (1 << 21) + 5, U64_A, 46), J("keys64", 65537, F64_A, 47)),
    "seg_idx_big_then_small": (J("seg_idx", order=U32_D, seg=ROWS_9000, seed=48),
                               J("seg_idx", order=F32_A, seg=("rows", 8193, 127), seed=49)),
}


def do(job, what: str):
    fam, n, order, seed, seg, algo, in_place, data = job
    width = FAMILIES[fam][0]
    if in_place:
        offs = (2, 2, 0, 3, 3, 0) if width == 64 else (1, 1, 2, 3, 3, 0)
    else:
        offs = {16: OFFS16, 32: OFFS32, 64: OFFS64}[width][1]
    expect(fam, n, order, seed, what, seg=seg, algo=algo, in_place=in_place, data=data, offs=offs)


@pytest.mark.parametrize("name", list(STALE))
def test_stale_state_from_another_call(name):
    a, b = STALE[name]
    do(a, f"{name}: A")
    do(b, f"{name}: B after A")
    do(b, f"{name}: B again")


def test_segment_layouts_target_what_they_name():
    """The stale-state layouts are what their comments say (no GPU work)."""
    many, few = layout(("many_large",)), layout(("few_large",))
    assert many[-1] == few[-1] and many.size == few.size
    big = lib().b200sort_segmented_class_max(3)
    assert int((np.diff(many) > big).sum()) == 200 and int((np.diff(few) > big).sum()) == 3
    r = np.diff(layout(RAGGED))
    assert (r == 0).any() and (r == 1).any() and (r > (1 << 20)).sum() == 2
    lr = np.diff(layout(LONG_RAGGED))
    assert lr[0] == 1 << 22 and lr.size > 1000
    many, few = layout(MANY_LARGE_2M), layout(FEW_LARGE_2M)
    assert many[-1] == few[-1] == 48 * 40000 and many.size == few.size == 1025
    big64 = lib().b200sort_segmented64_class_max(3)
    assert int((np.diff(many) > big64).sum()) == 48 and int((np.diff(few) > big64).sum()) == 3
    r = np.diff(layout(RAGGED_SMALL))
    assert (r == 0).any() and (r == 1).any() and (r > big64).sum() >= 10
    for name in ("pairs_then_idx_masked", "idx_masked_then_pairs", "pairs16_then_idx16_masked",
                 "seg_pairs_then_seg_idx_masked"):                      # A and B execute different pass sets
        assert [job[7] for job in STALE[name]].count("masked") == 1, name
        for fam, n, order, seed, seg, _, _, data in STALE[name]:
            width = FAMILIES[fam][0]
            img = _ko(width).image(case(width, n, order, seed, seg, data)[0], *order)
            assert (data == "masked") == (not (img & ~img.dtype.type(MASKED[width])).any()), (name, fam)


# ---- 4. graph capture and replay of the 32-bit 1-D entry points ---------------------------------------------------
GRAPH_ENTRIES = {   # name: (family, order, algo, in place)
    "radix_i32": ("i32", I32, ALGO_RADIX, True),
    "sort_copy_i32": ("i32", I32, ALGO_RADIX, False),
    "sort_keys_radix": ("keys", F32_D, ALGO_RADIX, False),
    "sort_keys_merge": ("keys", U32_D, ALGO_MERGE, False),
    "radix_pairs_i32": ("pairs_i32", I32, ALGO_RADIX, True),
    "radix_pairs_keys": ("pairs", (ko.KEY_F32, 0), ALGO_RADIX, False),
    "lab": ("i32", I32, ALGO_LAB, False),
}
GRAPH_N = [5000, 300001, (1 << 23) + 5]           # the one-CTA sort, the pass kernels, tma3


def graph_keys(kind: str, n: int, order) -> np.ndarray:
    """Uniform images, all equal (every pass skipped), or masked with 0x00FF00FF (passes 1 and 3 skipped)."""
    img = datagen.uniform_u32(n, n)
    if kind == "all_equal":
        img = np.full(n, 0x9E3779B1, np.uint32)
    elif kind == "masked":
        img = img & np.uint32(0x00FF00FF)
    return ko.inverse(img, *order)


@pytest.mark.parametrize("entry", list(GRAPH_ENTRIES))
def test_graph_capture_and_replay_32(entry):
    import torch
    L = lib()
    check(L.b200sort_device_check())          # the lazy lane-order self-test blocks: run it before capturing
    fam, order, algo, in_place = GRAPH_ENTRIES[entry]
    kt, desc = order
    pairs = FAMILIES[fam][1]
    ws = workspace()
    for n in GRAPH_N:
        need = L.b200sort_workspace_bytes(n, algo)
        kin = _buf("g_kin", n, 0, 4)
        kout = kin if in_place else _buf("g_kout", n, 1, 4)
        ktmp = _buf("g_ktmp", n, 2, 4)
        if pairs:
            vin = _buf("g_vin", n, 3, 4)
            vout = vin if in_place else _buf("g_vout", n, 0, 4)
            vtmp = _buf("g_vtmp", n, 1, 4)

        def load(kind: str):
            keys = graph_keys(kind, n, order)
            kin.load(ko.bits(keys))
            if not in_place:
                kout.load()
            ktmp.load()
            if pairs:
                vin.load(np.arange(n, dtype=np.int32))
                if not in_place:
                    vout.load()
                vtmp.load()
            return keys

        def call(s):
            if entry == "radix_i32":
                return L.b200sort_radix_i32(kin.ptr, ktmp.ptr, n, ws.ptr, need, s)
            if fam == "i32":
                return L.b200sort_sort_copy_i32(algo, kin.ptr, kout.ptr, ktmp.ptr, n, ws.ptr, need, s)
            if fam == "keys":
                return L.b200sort_sort_keys(algo, kt, desc, kin.ptr, kout.ptr, ktmp.ptr, n, ws.ptr, need, s)
            if fam == "pairs_i32":
                return L.b200sort_radix_pairs_i32(kin.ptr, vin.ptr, ktmp.ptr, vtmp.ptr, n, ws.ptr, need, s)
            return L.b200sort_radix_pairs_keys(kt, desc, kin.ptr, vin.ptr, kout.ptr, vout.ptr, ktmp.ptr, vtmp.ptr, n,
                                               ws.ptr, need, s)

        def verify(keys, what):
            torch.cuda.synchronize()
            perm = np.argsort(ko.image(keys, kt, desc), kind="stable")
            assert_words(kout.read(what + " keys out"), ko.bits(keys)[perm], what)
            ktmp.read(what + " keys tmp")
            if not in_place:
                assert kin.read(what + " keys in").tobytes() == ko.bits(keys).tobytes(), what + ": input modified"
            if pairs:
                assert_words(vout.read(what + " values out"), perm.astype(np.uint32), what + " values")
                vtmp.read(what + " values tmp")
            assert torch.equal(ws.guard(need).cpu(), before), what + ": workspace written past ws_bytes"

        before = ws.guard(need).cpu()
        counts = {}
        for kind in ("uniform", "all_equal", "masked"):             # eager: the launch count does not depend on data
            keys = load(kind)
            L.b200sort_launch_count_reset()
            check(call(stream_ptr()))
            counts[f"eager {kind}"] = L.b200sort_launch_count()
            verify(keys, f"{entry} n={n} eager {kind}")
        load("uniform")
        torch.cuda.synchronize()
        s = torch.cuda.Stream()
        g = torch.cuda.CUDAGraph()
        L.b200sort_launch_count_reset()
        with torch.cuda.graph(g, stream=s):
            check(call(s.cuda_stream))
        counts["capture"] = L.b200sort_launch_count()
        assert len(set(counts.values())) == 1, (entry, n, counts)
        for kind in ("all_equal", "masked", "uniform", "all_equal"):
            keys = load(kind)                                       # new data into the captured buffers
            g.replay()
            verify(keys, f"{entry} n={n} replay {kind}")
        del g
