"""A reused, never-cleared workspace and guarded buffers for the 16-bit, segmented, merge and lab sorts, stale state
left by one entry point for another, and CUDA graph replay of the 32-bit 1-D sorts.

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
images (tests/key_orders.py, tests/key_orders16.py), per segment for the segmented sorts (np.lexsort), and
oracle.radix_sort for the lab pipeline; results are compared byte for byte.
"""
import functools

import numpy as np
import pytest

import digit_patterns as dp
import key_orders as ko
import key_orders16 as ko16
import oracle
from b200sort import datagen
from b200sort._lib import ALGO_LAB, ALGO_MERGE, ALGO_RADIX, check, lib
from helpers import stream_ptr
from test_keys16_gpu import random_keys as keys16_of
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
}


def _ko(width: int):
    return ko16 if width == 16 else ko


# ---- segment layouts ---------------------------------------------------------------------------------------------
def _class_bounds(width: int):
    L = lib()
    f = L.b200sort_segmented16_class_max if width == 16 else L.b200sort_segmented_class_max
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
        # ones, or 3 large segments among 4093 of 2..1024 keys
        S, n = 4096, 200 * 40000
        if kind == "many_large":
            lens = np.concatenate([np.full(200, 40000), np.zeros(S - 200, np.int64)])
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


def seg_ws_bytes(width: int, n: int, S: int) -> int:
    L = lib()
    return (L.b200sort_segmented16_workspace_bytes if width == 16 else L.b200sort_segmented_workspace_bytes)(n, S)


# ---- the module's workspace and buffers ----------------------------------------------------------------------------
_ws = None


def workspace() -> dp.Workspace:
    global _ws
    if _ws is None:
        L = lib()
        needs = [L.b200sort_keys16_workspace_bytes(N16_BIG), L.b200sort_workspace_bytes(N32_BIG, ALGO_RADIX),
                 L.b200sort_workspace_bytes(N32_BIG, ALGO_MERGE)]
        seg = [(w, name) for w in (16, 32) for name in class_rows(w) + [RAGGED, ONE]]
        seg += [(FAMILIES[job[0]][0], job[4]) for pair in STALE.values() for job in pair if job[4] is not None]
        for width, name in seg:
            offs = layout(name)
            needs.append(seg_ws_bytes(width, int(offs[-1]), offs.size - 1))
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
    values arange(n).  seg: the layout name of the segmented families.  Returns (key words, values or None)."""
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
    if seg is not None:
        d_off = _device_offsets(seg)
        S = d_off.numel() - 1
        assert int(layout(seg)[-1]) == n
        need = seg_ws_bytes(width, n, S)
    elif width == 16:
        need = L.b200sort_keys16_workspace_bytes(n)
    else:
        need = L.b200sort_workspace_bytes(n, algo)
    ws = workspace()
    assert need + ws.GUARD <= ws.cap, f"{what}: the module workspace is sized without this call"
    before = ws.guard(need).cpu()
    s = stream_ptr()
    if fam == "keys16":
        st = L.b200sort_sort_keys16(kt, desc, kin.ptr, kout.ptr, n, ws.ptr, need, s)
    elif fam == "pairs16":
        st = L.b200sort_radix_pairs_keys16(kt, desc, kin.ptr, vin.ptr, kout.ptr, vout.ptr, ktmp.ptr, vtmp.ptr, n,
                                           ws.ptr, need, s)
    elif fam in ("seg16", "seg"):
        f = L.b200sort_segmented_sort_keys16 if width == 16 else L.b200sort_segmented_sort_keys
        st = f(kt, desc, kin.ptr, kout.ptr, ktmp.ptr, n, d_off.data_ptr(), S, ws.ptr, need, s)
    elif fam in ("seg16_pairs", "seg_pairs"):
        f = L.b200sort_segmented_pairs_keys16 if width == 16 else L.b200sort_segmented_pairs_keys
        st = f(kt, desc, kin.ptr, vin.ptr, kout.ptr, vout.ptr, ktmp.ptr, vtmp.ptr, n, d_off.data_ptr(), S, ws.ptr,
               need, s)
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
    got = kout.read(f"{what} keys out")
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
    assert torch.equal(ws.guard(need).cpu(), before), f"{what}: workspace written past ws_bytes = {need}"
    return got, got_vals


def assert_words(got: np.ndarray, want: np.ndarray, what: str):
    if got.tobytes() != want.tobytes():
        bad = np.flatnonzero(got != want)
        w = 2 + 2 * got.dtype.itemsize
        raise AssertionError(f"{what}: {bad.size} of {got.size} words differ, first at {bad[0]}: "
                             f"got {int(got[bad[0]]):#0{w}x}, want {int(want[bad[0]]):#0{w}x}")


@functools.lru_cache(maxsize=8)
def case(width: int, n: int, order, seed: int, seg=None):
    """(keys, reference permutation) of random bit patterns with float specials: a stable argsort of the images,
    segment by segment if `seg` names a layout (then n is the layout's)."""
    kt, desc = order
    if seg is not None:
        n = int(layout(seg)[-1])
    keys = keys16_of(n, kt, seed) if width == 16 else keys32_of(n, kt, seed)
    img = _ko(width).image(keys, kt, desc)
    perm = (np.argsort(img, kind="stable") if seg is None else np.lexsort((img, segment_ids(layout(seg)))))
    return keys, perm


def expect(fam: str, n: int, order, seed: int, what: str, seg=None, algo: int = ALGO_RADIX, **kw):
    """run() on the keys of case() and compare with the reference, byte for byte."""
    width = FAMILIES[fam][0]
    keys, perm = case(width, n, order, seed, seg)
    got, got_vals = run(fam, keys, order, seg=seg, algo=algo, what=what, **kw)
    if algo == ALGO_LAB:
        want = oracle.radix_sort(keys).view(np.uint32)
        assert want.tobytes() == _ko(width).bits(keys)[perm].tobytes()      # the oracle and the argsort agree
    else:
        want = _ko(width).bits(keys)[perm]
    assert_words(got, want, what)
    if got_vals is not None:
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
# A job: (family, n or None, order, seed, segment layout or None, algo, in place).  Each case runs A, then B twice on
# the shared workspace without clearing it, and names the region of state B must rewrite before it reads it.
def J(fam, n=None, order=I32, seed=0, seg=None, algo=ALGO_RADIX, in_place=False):
    return (fam, n if seg is None else _n_of(seg), order, seed, seg, algo, in_place)


BF16_D, U16_A, F32_D, U32_D = (ko16.KEY_BF16, 1), (ko16.KEY_U16, 0), (ko.KEY_F32, 1), (ko.KEY_U32, 1)
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
}


def do(job, what: str):
    fam, n, order, seed, seg, algo, in_place = job
    expect(fam, n, order, seed, what, seg=seg, algo=algo, in_place=in_place,
           offs=(1, 1, 2, 3, 3, 0) if in_place else OFFS32[1] if FAMILIES[fam][0] == 32 else OFFS16[1])


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
