"""The radix sorts' device-side pass plan on the GPU: every set of skipped passes, near-constant and hot digits,
misaligned buffers with canary guards around every array, a reused never-cleared workspace, the device key count of
b200sort_radix_copy_devn_i32 and the timed entry point.

Everything goes through the C-ABI; torch only owns device memory.  The reference is a stable numpy argsort of the key
images (tests/key_orders.py, tests/key_orders64.py); results are compared byte for byte.  The keys come from
tests/digit_patterns.py, whose generators are checked on the CPU by tests/test_pass_plan_cpu.py.
"""
import contextlib
import ctypes
import functools
import itertools
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import digit_patterns as dp
import key_orders as ko
import key_orders64 as ko64
import oracle
from b200sort._lib import ALGO_MERGE, ALGO_RADIX, check, lib
from helpers import stream_ptr

pytestmark = pytest.mark.gpu

# 32-bit: at least two look-back groups of 32 tiles for every shape (tma3 16384-key tiles, shape 1 10240, pairs 5120),
# and a ragged last tile
N = 33 * 16384 + 4099
N_BIG = (1 << 23) + 4099          # the default configuration runs tma3 from 2^23 keys on
N64 = 3 * 4096 + 17               # 64-bit: 4096-key tiles, ragged last tile
N64_BIG = (1 << 20) + 3
TILE = {1: 10240, 2: 10240, 3: 16384, "pairs": 5120, 64: 4096}
SHAPES = [1, 2, 3]                # b200sort_radix_set_variant: pipelined2, its ballot-ranked form, tma3 at any size
SETS32 = [frozenset(s) for r in range(5) for s in itertools.combinations(range(4), r)]
SETS64 = [frozenset(s) for r in range(9) for s in itertools.combinations(range(8), r)]
I32, U32, F32 = (ko.KEY_I32, 0), (ko.KEY_U32, 0), (ko.KEY_F32, 1)
KEY_ORDERS32 = {"i32_desc": (ko.KEY_I32, 1), "u32_asc": (ko.KEY_U32, 0), "f32_desc": (ko.KEY_F32, 1)}
ORDER64_IDS = [f"{ko64.NAMES[k]}_{'desc' if d else 'asc'}" for k, d in ko64.ORDERS]


def _label(S) -> str:
    return "{" + ",".join(map(str, sorted(S))) + "}"


@contextlib.contextmanager
def plan_config(variant: int = 0, skip: int = 1):
    """Radix shape and pass skipping for the block; the defaults come back whatever happens."""
    L = lib()
    try:
        check(L.b200sort_radix_set_variant(variant))
        L.b200sort_radix_set_skip(skip)
        yield
    finally:
        L.b200sort_radix_set_variant(0)
        L.b200sort_radix_set_skip(1)


# ---- guarded device buffers and the shared workspace (digit_patterns.DevBuf, digit_patterns.Workspace) -----------
_bufs = {}


def _buf(role: str, n: int, word_offset: int, itemsize: int = 4) -> dp.DevBuf:
    key = (role, n, word_offset, itemsize)
    if key not in _bufs:
        _bufs[key] = dp.DevBuf(n, word_offset, itemsize, salt=len(_bufs) + 1)
    return _bufs[key]


_ws = None


def workspace() -> dp.Workspace:
    global _ws
    if _ws is None:
        L = lib()
        _ws = dp.Workspace(max(L.b200sort_workspace_bytes(N_BIG, ALGO_RADIX), L.b200sort_workspace_bytes(N_BIG, ALGO_MERGE),
                               L.b200sort_keys64_workspace_bytes(N64_BIG)))
    return _ws


@pytest.fixture(scope="module", autouse=True)
def _no_check_failures():
    yield
    L = lib()
    if _ws is not None:
        _ws.check_tail()
    if L.b200sort_debug_checked_build() == 1:
        assert L.b200sort_debug_check_failures() == 0


# ---- one call of an entry point -----------------------------------------------------------------------------------
WIDE = {"keys64", "pairs64"}
PAIRS = {"pairs_i32", "pairs", "pairs64"}


def run(entry: str, keys: np.ndarray, order=I32, in_place: bool = False, offs=(0, 0, 0, 0, 0, 0),
        algo: int = ALGO_RADIX, what: str = ""):
    """Sort `keys` by one entry point with every buffer guarded.  Returns (key words, values or None, ms or None).

    entry: "i32" (b200sort_radix_i32 / b200sort_sort_copy_i32), "keys" (b200sort_sort_keys), "pairs_i32"
    (b200sort_radix_pairs_i32 / _pairs_copy_i32), "pairs" (b200sort_radix_pairs_keys), "keys64", "pairs64" and
    "timed" (b200sort_sort_timed_i32 with `algo`).  Pairs carry the values arange(n).  offs: word offsets of
    (keys in, keys out, keys tmp, values in, values out, values tmp); in place, out is in."""
    import torch
    L = lib()
    kt, desc = order
    n = keys.size
    item = 8 if entry in WIDE else 4
    words = dp.orders_module(kt).bits(keys)
    kin = _buf("kin", n, offs[0], item).load(words)
    kout = kin if in_place else _buf("kout", n, offs[1], item).load()
    ktmp = _buf("ktmp", n, offs[2], item).load()
    pairs = entry in PAIRS
    if pairs:
        vals = np.arange(n, dtype=np.int32)
        vin = _buf("vin", n, offs[3]).load(vals)
        vout = vin if in_place else _buf("vout", n, offs[4]).load()
        vtmp = _buf("vtmp", n, offs[5]).load()
    ws = workspace()
    need = (L.b200sort_keys64_workspace_bytes(n) if entry in WIDE else L.b200sort_workspace_bytes(n, algo))
    before = ws.guard(need).cpu()
    s = stream_ptr()
    ms = None
    if entry == "i32":
        st = (L.b200sort_radix_i32(kin.ptr, ktmp.ptr, n, ws.ptr, need, s) if in_place else
              L.b200sort_sort_copy_i32(ALGO_RADIX, kin.ptr, kout.ptr, ktmp.ptr, n, ws.ptr, need, s))
    elif entry == "keys":
        st = L.b200sort_sort_keys(ALGO_RADIX, kt, desc, kin.ptr, kout.ptr, ktmp.ptr, n, ws.ptr, need, s)
    elif entry == "timed":
        ms = (ctypes.c_float * 6)(*([-1.0] * 6))
        st = L.b200sort_sort_timed_i32(algo, kin.ptr, kout.ptr, ktmp.ptr, n, ws.ptr, need, s, ms)
    elif entry == "pairs_i32":
        st = (L.b200sort_radix_pairs_i32(kin.ptr, vin.ptr, ktmp.ptr, vtmp.ptr, n, ws.ptr, need, s) if in_place else
              L.b200sort_radix_pairs_copy_i32(kin.ptr, vin.ptr, kout.ptr, vout.ptr, ktmp.ptr, vtmp.ptr, n, ws.ptr, need, s))
    elif entry == "pairs":
        st = L.b200sort_radix_pairs_keys(kt, desc, kin.ptr, vin.ptr, kout.ptr, vout.ptr, ktmp.ptr, vtmp.ptr, n, ws.ptr,
                                         need, s)
    elif entry == "keys64":
        st = L.b200sort_sort_keys64(kt, desc, kin.ptr, kout.ptr, ktmp.ptr, n, ws.ptr, need, s)
    elif entry == "pairs64":
        st = L.b200sort_radix_pairs_keys64(kt, desc, kin.ptr, vin.ptr, kout.ptr, vout.ptr, ktmp.ptr, vtmp.ptr, n,
                                           ws.ptr, need, s)
    else:
        raise ValueError(entry)
    check(st)
    torch.cuda.synchronize()
    got = kout.read(f"{what} keys out")
    ktmp.read(f"{what} keys tmp")
    if not in_place:
        assert kin.read(f"{what} keys in").tobytes() == words.tobytes(), f"{what}: the copy form modified its keys"
    got_vals = None
    if pairs:
        got_vals = vout.read(f"{what} values out").view(np.int32)
        vtmp.read(f"{what} values tmp")
        if not in_place:
            assert vin.read(f"{what} values in").tobytes() == vals.tobytes(), f"{what}: the copy form modified its values"
    assert torch.equal(ws.guard(need).cpu(), before), f"{what}: workspace written past ws_bytes = {need}"
    if item == 8:
        got = got.view(np.uint64)
    return got, got_vals, (list(ms) if ms is not None else None)


def assert_words(got: np.ndarray, want: np.ndarray, what: str):
    if got.tobytes() != want.tobytes():
        bad = np.flatnonzero(got != want)
        w = 18 if got.dtype.itemsize == 8 else 10
        raise AssertionError(f"{what}: {bad.size} of {got.size} words differ, first at {bad[0]}: "
                             f"got {int(got[bad[0]]):#0{w}x}, want {int(want[bad[0]]):#0{w}x}")


def expect(entry, keys, order, perm, what, **kw):
    """run() and compare with keys[perm] (and values perm for pairs)."""
    got, got_vals, ms = run(entry, keys, order, what=what, **kw)
    assert_words(got, dp.orders_module(order[0]).bits(keys)[perm], what)
    if got_vals is not None:
        assert_words(got_vals.view(np.uint32), perm.astype(np.uint32), what + " values")
    return ms


@functools.lru_cache(maxsize=24)
def pattern(width: int, n: int, S: frozenset, seed: int, consts=None):
    """(images, stable argsort of the images) of with_constant_digits; the images do not depend on the order."""
    plain = (ko.KEY_U32, 0) if width == 32 else (ko64.KEY_U64, 0)      # image == key
    img = dp.with_constant_digits(n, S, plain, seed, consts)
    return img, np.argsort(img, kind="stable")


def _consts(i: int):
    return (None, 0, 255)[i % 3]


# ---- 1. 32-bit, every set of skipped passes -----------------------------------------------------------------------
KEYS_ENTRIES = [("i32", I32)] + [("keys", o) for o in KEY_ORDERS32.values()]
KEYS_IDS = ["i32"] + list(KEY_ORDERS32)


@pytest.mark.parametrize("entry,order", KEYS_ENTRIES, ids=KEYS_IDS)
@pytest.mark.parametrize("shape", SHAPES)
def test_every_skip_set_32(shape, entry, order):
    with plan_config(shape):
        for i, S in enumerate(SETS32):
            img, perm = pattern(32, N, S, i, _consts(i))
            keys = dp.keys_of(img, order)
            for skip in (1, 0):
                lib().b200sort_radix_set_skip(skip)
                for in_place in (False, True):
                    expect(entry, keys, order, perm, f"shape {shape} {entry} S={_label(S)} skip={skip} "
                           f"in_place={in_place}", in_place=in_place)


@pytest.mark.parametrize("entry,order", [("pairs_i32", I32), ("pairs", F32), ("pairs", (ko.KEY_U32, 1))],
                         ids=["pairs_i32", "pairs_f32_desc", "pairs_u32_desc"])
def test_every_skip_set_32_pairs(entry, order):
    with plan_config():
        for i, S in enumerate(SETS32):
            img, perm = pattern(32, N, S, i, _consts(i))
            keys = dp.keys_of(img, order)
            for skip in (1, 0):
                lib().b200sort_radix_set_skip(skip)
                for in_place in (False, True):
                    expect(entry, keys, order, perm, f"{entry} S={_label(S)} skip={skip} in_place={in_place}",
                           in_place=in_place)


# executed passes 4, 3 (twice), 2, 1, 0
BIG_SETS = [frozenset(), frozenset({0}), frozenset({2}), frozenset({1, 2}), frozenset({0, 1, 3}), frozenset(range(4))]


@pytest.mark.parametrize("entry,order", [("i32", I32), ("keys", F32), ("pairs_i32", I32)], ids=["i32", "f32_desc", "pairs_i32"])
def test_skip_sets_in_the_default_configuration_at_2_23(entry, order):
    """From 2^23 keys on the default configuration runs tma3 (keys) and the pairs kernel on the same plan."""
    with plan_config():
        for i, S in enumerate(BIG_SETS):
            img, perm = pattern(32, N_BIG, S, 50 + i, _consts(i))
            keys = dp.keys_of(img, order)
            for in_place in (False, True):
                expect(entry, keys, order, perm, f"n=2^23+4099 {entry} S={_label(S)} in_place={in_place}",
                       in_place=in_place)


# ---- 2. 32-bit misalignment -----------------------------------------------------------------------------------------
MIS_SETS = [frozenset(), frozenset({0}), frozenset({1, 2, 3}), frozenset(range(4))]


@pytest.mark.parametrize("entry,order", [("i32", I32), ("keys", F32)], ids=["i32", "f32_desc"])
@pytest.mark.parametrize("shape", [1, 3])
def test_misaligned_keys_32(shape, entry, order):
    """in, out and tmp each at word offset 0..3 (all 64 combinations; in place 16), guards intact everywhere."""
    with plan_config(shape):
        for i, S in enumerate(MIS_SETS):
            img, perm = pattern(32, N, S, 100 + i, _consts(i))
            keys = dp.keys_of(img, order)
            for a, b, c in itertools.product(range(4), repeat=3):
                expect(entry, keys, order, perm, f"shape {shape} {entry} S={_label(S)} offsets in={a} out={b} tmp={c}",
                       offs=(a, b, c, 0, 0, 0))
                if b == 0:
                    expect(entry, keys, order, perm, f"shape {shape} {entry} S={_label(S)} in place at {a} tmp={c}",
                           in_place=True, offs=(a, a, c, 0, 0, 0))


def _pair_offsets():
    rng = np.random.default_rng(2024)
    return [tuple(int(x) for x in rng.integers(0, 4, 6)) for _ in range(32)] + [(k,) * 6 for k in range(4)]


@pytest.mark.parametrize("entry,order", [("pairs_i32", I32), ("pairs", F32)], ids=["pairs_i32", "pairs_f32_desc"])
def test_misaligned_pairs_32(entry, order):
    with plan_config():
        for i, S in enumerate(MIS_SETS):
            img, perm = pattern(32, N, S, 100 + i, _consts(i))
            keys = dp.keys_of(img, order)
            for offs in _pair_offsets():
                expect(entry, keys, order, perm, f"{entry} S={_label(S)} offsets {offs}", offs=offs)
                ip = (offs[0], offs[0], offs[2], offs[3], offs[3], offs[5])
                expect(entry, keys, order, perm, f"{entry} S={_label(S)} in place offsets {ip}", in_place=True, offs=ip)


# ---- 3. 64-bit, every set of skipped passes ----------------------------------------------------------------------
def matrix64(sets, orders, n=N64, skip=1, offsets=((0,) * 6,), seed0=0):
    """Keys and pairs, copy and in place, for every set, order and offset tuple."""
    with plan_config(skip=skip):
        for i, S in enumerate(sets):
            img, perm = pattern(64, n, S, seed0 + i, _consts(i))
            for j, order in enumerate(orders):
                keys = dp.keys_of(img, order)
                offs = offsets[(i + j) % len(offsets)]
                for entry in ("keys64", "pairs64"):
                    for in_place in (False, True):
                        o = (offs[0], offs[0], offs[2], offs[3], offs[3], offs[5]) if in_place else offs
                        expect(entry, keys, order, perm, f"n={n} {entry} {order} S={_label(S)} skip={skip} "
                               f"in_place={in_place} offsets {o}", in_place=in_place, offs=o)


@pytest.mark.parametrize("order", ko64.ORDERS, ids=ORDER64_IDS)
def test_every_skip_set_64(order):
    matrix64(SETS64, [order])


ONE_OFF64 = [frozenset({p}) for p in range(8)] + [frozenset(set(range(8)) - {p}) for p in range(8)]


def test_one_pass_skipped_or_one_executed_at_2_20():
    matrix64(ONE_OFF64, [(ko64.KEY_I64, 0), (ko64.KEY_F64, 1)], n=N64_BIG, seed0=300)


# executed passes 8 down to 0, odd and even, including gaps
SOME64 = [frozenset(s) for s in ((), (0,), (7,), (0, 7), (1, 2, 3), (0, 1, 2, 3), (4, 5, 6, 7), (0, 2, 4, 6),
                                 (1, 2, 3, 4, 5), (0, 1, 2, 3, 4, 5), (1, 2, 3, 4, 5, 6, 7), tuple(range(8)))]
# in, out, tmp 0 or 8 bytes past a 16-byte boundary (all 8 combinations), values at word offsets 0..3
OFFS64 = [(a, b, c, k % 4, (k + 1) % 4, (k + 2) % 4)
          for k, (a, b, c) in enumerate(itertools.product((0, 2), repeat=3))]


def test_misaligned_64():
    matrix64(SOME64, ko64.ORDERS, offsets=OFFS64, seed0=400)


def test_skipping_off_64():
    matrix64(SOME64, [(ko64.KEY_I64, 1), (ko64.KEY_U64, 0)], skip=0, offsets=OFFS64[::3], seed0=500)


def _subprocess(code: str, env: dict):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    prog = ("import sys; sys.path.insert(0, '.'); sys.path.insert(0, 'tests')\n"
            "from b200sort._lib import lib\n"
            "import test_pass_plan_gpu as t\n" + code +
            "\nassert lib().b200sort_debug_checked_build() == 0 or lib().b200sort_debug_check_failures() == 0\n"
            "t.workspace().check_tail()\nprint('ok')\n")
    r = subprocess.run([sys.executable, "-c", prog], cwd=root, env={**os.environ, **env}, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


def test_rank_safe_fallback():
    """B200SORT_RANK_SAFE=1: the ballot-ranked pass kernels of every path on the same plans."""
    _subprocess("assert lib().b200sort_radix_atomic_order_ok() == 0\n"
                "t.matrix64(t.SOME64[::2], [(t.ko64.KEY_F64, 0)], offsets=t.OFFS64[::2], seed0=600)\n"
                "t.matrix32_pairs(t.MIS_SETS, seed0=600)\n",
                {"B200SORT_RANK_SAFE": "1"})


def matrix32_pairs(sets, seed0):
    with plan_config():
        for i, S in enumerate(sets):
            img, perm = pattern(32, N, S, seed0 + i, _consts(i))
            for entry, order in (("pairs_i32", I32), ("pairs", F32), ("keys", F32), ("i32", I32)):
                keys = dp.keys_of(img, order)
                for in_place in (False, True):
                    expect(entry, keys, order, perm, f"{entry} S={_label(S)} in_place={in_place}", in_place=in_place)


# ---- 4. near-constant digits ---------------------------------------------------------------------------------------
NEAR32 = [("i32", I32, 1, TILE[1]), ("i32", I32, 3, TILE[3]), ("keys", F32, 1, TILE[1]), ("keys", F32, 3, TILE[3]),
          ("pairs_i32", I32, 0, TILE["pairs"]), ("pairs", (ko.KEY_U32, 1), 0, TILE["pairs"])]


@pytest.mark.parametrize("p", range(4))
def test_near_constant_digit_32(p):
    """Digit p is one value in all keys but one: the pass must run (a skipped pass leaves the odd key misplaced)."""
    for entry, order, shape, tile in NEAR32:
        with plan_config(shape):
            for where in dp.WHERE:
                img, _, _ = dp.near_constant(N, p, where, U32, tile=tile, seed=p)
                perm = np.argsort(img, kind="stable")
                keys = dp.keys_of(img, order)
                for in_place in (False, True):
                    expect(entry, keys, order, perm, f"shape {shape} {entry} pass {p} odd key {where} "
                           f"in_place={in_place}", in_place=in_place)


@pytest.mark.parametrize("p", range(8))
def test_near_constant_digit_64(p):
    for where in dp.WHERE:
        img, _, _ = dp.near_constant(N64, p, where, (ko64.KEY_U64, 0), tile=TILE[64], seed=p)
        perm = np.argsort(img, kind="stable")
        for order in ((ko64.KEY_I64, 0), (ko64.KEY_F64, 1)):
            keys = dp.keys_of(img, order)
            for entry in ("keys64", "pairs64"):
                for in_place in (False, True):
                    expect(entry, keys, order, perm, f"{entry} {order} pass {p} odd key {where} in_place={in_place}",
                           in_place=in_place)


# ---- 5. hot digits and locally hot runs ---------------------------------------------------------------------------
# (entry, order, shape): shapes 1-3 by variant; variant 0 below 8193 keys is the one-CTA kernel, above it shape 1
HOT_ENTRIES = [("i32", I32, 1), ("i32", I32, 2), ("i32", I32, 3), ("pairs_i32", I32, 0), ("keys", F32, 0),
               ("i32", I32, 0)]


def hot_matrix(n, entries=HOT_ENTRIES):
    for p in range(4):
        for value in (0, 0x80, 255):
            for fraction in dp.HOT_FRACTIONS:
                img = dp.hot_digit(n, p, value, fraction, U32, seed=p * 7 + value)
                perm = np.argsort(img, kind="stable")
                for entry, order, shape in entries:
                    with plan_config(shape):
                        expect(entry, dp.keys_of(img, order), order, perm,
                               f"n={n} shape {shape} {entry} pass {p} digit {value:#x} on {fraction}")
        img = dp.locally_hot(n, p, U32, seed=p)
        perm = np.argsort(img, kind="stable")
        for entry, order, shape in entries:
            with plan_config(shape):
                expect(entry, dp.keys_of(img, order), order, perm, f"n={n} shape {shape} {entry} pass {p} locally hot")


@pytest.mark.parametrize("n", [N, 8191, 8193])
def test_hot_digits(n):
    hot_matrix(n)


def test_hot_digits_without_the_one_cta_kernel():
    """B200SORT_RADIX_SMALL=0: the pass kernels, not the one-CTA sort, see the small sizes in the default shape."""
    _subprocess("for n in (8191, 8193):\n"
                "    t.hot_matrix(n, [e for e in t.HOT_ENTRIES if e[2] == 0])\n",
                {"B200SORT_RADIX_SMALL": "0"})


# ---- 6. the key count in device memory -----------------------------------------------------------------------------
DEVN_SETS = [frozenset(), frozenset({0}), frozenset({3}), frozenset({1, 2}), frozenset({0, 1, 3}), frozenset(range(4))]


@pytest.mark.parametrize("shape", [0, 3])
def test_copy_devn(shape):
    """b200sort_radix_copy_devn_i32 sorts the first *d_n of n_max keys; out[m:n_max] and every guard stay."""
    import torch
    L = lib()
    d_n = torch.zeros(1, dtype=torch.int32, device="cuda")
    d_hist = torch.zeros(4 * 256, dtype=torch.int32, device="cuda")
    ws = workspace()
    need = L.b200sort_workspace_bytes(N, ALGO_RADIX)
    with plan_config(shape):
        for i, S in enumerate(DEVN_SETS):
            img, _ = pattern(32, N, S, 700 + i, _consts(i))
            keys = dp.keys_of(img, I32)
            for m in (0, 1, 2, 4099, N - 1, N):
                perm = np.argsort(img[:m], kind="stable")
                for with_hist in (False, True):
                    what = f"devn shape {shape} S={_label(S)} m={m} hist={with_hist}"
                    kin = _buf("kin", N, 1).load(keys)
                    kout = _buf("kout", N, 2).load()
                    ktmp = _buf("ktmp", N, 3).load()
                    d_n.fill_(m)
                    if with_hist:
                        h = oracle.digit_histograms(keys[:m]).astype(np.uint32)
                        d_hist.copy_(torch.from_numpy(h.reshape(-1).view(np.int32)))
                    before = ws.guard(need).cpu()
                    check(L.b200sort_radix_copy_devn_i32(kin.ptr, kout.ptr, ktmp.ptr, N, d_n.data_ptr(),
                                                         d_hist.data_ptr() if with_hist else None, ws.ptr, need,
                                                         stream_ptr()))
                    torch.cuda.synchronize()
                    got = kout.read(what + " out")
                    ktmp.read(what + " tmp")
                    assert kin.read(what + " in").tobytes() == ko.bits(keys).tobytes(), what + ": input modified"
                    assert_words(got[:m], ko.bits(keys[:m])[perm], what)
                    assert_words(got[m:], kout.g.fill[kout.g.start + m:kout.g.end], what + ": out past m written")
                    assert torch.equal(ws.guard(need).cpu(), before), what + ": workspace written past ws_bytes"


# ---- 7. the timed entry point ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("algo", [ALGO_RADIX, ALGO_MERGE], ids=["radix", "merge"])
def test_timed_entry_point(algo):
    """b200sort_sort_timed_i32 runs the same plan (radix without the one-CTA path) with events around it."""
    with plan_config():
        for i, S in enumerate(SETS32):
            img, perm = pattern(32, N, S, i, _consts(i))
            keys = dp.keys_of(img, I32)
            for in_place in (False, True):
                ms = expect("timed", keys, I32, perm, f"timed algo {algo} S={_label(S)} in_place={in_place}",
                            in_place=in_place, algo=algo)
                used = ms[:6] if algo == ALGO_RADIX else ms[:3]
                assert all(math.isfinite(x) and x >= 0 for x in used), ms
                if algo == ALGO_MERGE:
                    assert ms[2] == float(int(ms[2])) and ms[2] >= 1, ms     # the number of merge passes
        # and the one-CTA-sized input, which the timed form sends through the pass kernels
        keys = dp.with_constant_digits(8191, {1}, I32, 5)
        perm = np.argsort(ko.image(keys, *I32), kind="stable")
        expect("timed", keys, I32, perm, f"timed algo {algo} n=8191", algo=algo)
