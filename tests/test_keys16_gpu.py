"""16-bit keys on the GPU (b200sort_sort_keys16, b200sort_radix_pairs_keys16 and the torch-facing b200sort.sort16 /
sort16_by_key), byte for byte against the numpy reference of tests/key_orders16.py."""
import os
import subprocess
import sys

import numpy as np
import pytest

import b200sort
from b200sort._lib import check, lib
from helpers import stream_ptr

import key_orders16 as ko

pytestmark = pytest.mark.gpu

ORDER_IDS = [f"{ko.NAMES[k]}_{'desc' if d else 'asc'}" for k, d in ko.ORDERS]
TILE = 8192          # keys per onesweep tile of the pairs passes (csrc/radix16.cu)
SIZES = [0, 1, 2, 31, 33, TILE - 1, TILE, TILE + 1, 65535, 65536, 65537, (1 << 20) + 3, (1 << 23) + 5]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ws(n: int):
    import torch
    nbytes = lib().b200sort_keys16_workspace_bytes(n)
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
    return ws, ws.data_ptr() + (-ws.data_ptr()) % 256, nbytes


def _placed(a: np.ndarray, byte_offset: int, fill: int):
    """(tensor, pointer) of 16-bit words placed byte_offset bytes past a 16-byte boundary, guarded by `fill` words."""
    import torch
    k = byte_offset // 2
    t = torch.full((a.size + 16,), fill, dtype=torch.int16, device="cuda")
    if a.size:
        t[k:k + a.size] = torch.from_numpy(ko.bits(a).view(np.int16).copy()).cuda()
    return t, t.data_ptr() + byte_offset


def _read(t, byte_offset: int, n: int) -> np.ndarray:
    return t.cpu().numpy().view(np.uint16)[byte_offset // 2:byte_offset // 2 + n]


def _guards_intact(t, byte_offset: int, n: int, fill: int, what: str):
    w = t.cpu().numpy().view(np.uint16)
    k = byte_offset // 2
    g = np.concatenate([w[:k], w[k + n:]])
    assert (g == np.uint16(fill & 0xFFFF)).all(), f"{what}: a write outside the array"


def sort16_keys(keys, kt, desc, in_place, offs=(0, 0)):
    """The library's keys-only result as uint16 words; checks that the copy form leaves its input alone and that
    nothing is written past either end of the output."""
    import torch
    n = keys.size
    src, p_in = _placed(keys, offs[0], 0x5A5A)
    if in_place:
        out, p_out, o_out = src, p_in, offs[0]
    else:
        out, p_out = _placed(np.zeros(n, np.uint16), offs[1], 0x3C3C)
        o_out = offs[1]
    ws, ptr, nbytes = _ws(n)
    check(lib().b200sort_sort_keys16(kt, desc, p_in, p_out, n, ptr, nbytes, stream_ptr()))
    torch.cuda.synchronize()
    if not in_place:
        assert _read(src, offs[0], n).tobytes() == ko.bits(keys).tobytes(), "the copy form modified its input"
    _guards_intact(out, o_out, n, 0x5A5A if in_place else 0x3C3C, "keys")
    return _read(out, o_out, n)


def sort16_pairs(keys, vals, kt, desc, in_place, offs=(0, 0, 0)):
    import torch
    n = keys.size
    dk, p_k = _placed(keys, offs[0], 0x5A5A)
    dv = torch.from_numpy(np.ascontiguousarray(vals, np.int32)).cuda()
    if in_place:
        ok, p_ok, o_ok, ov = dk, p_k, offs[0], dv
    else:
        ok, p_ok = _placed(np.zeros(n, np.uint16), offs[1], 0x3C3C)
        o_ok = offs[1]
        ov = torch.zeros(max(n, 1), dtype=torch.int32, device="cuda")
    tk, p_tk = _placed(np.zeros(n, np.uint16), offs[2], 0)
    tv = torch.empty(max(n, 1), dtype=torch.int32, device="cuda")
    ws, ptr, nbytes = _ws(n)
    check(lib().b200sort_radix_pairs_keys16(kt, desc, p_k, dv.data_ptr(), p_ok, ov.data_ptr(), p_tk, tv.data_ptr(),
                                            n, ptr, nbytes, stream_ptr()))
    torch.cuda.synchronize()
    if not in_place:
        assert _read(dk, offs[0], n).tobytes() == ko.bits(keys).tobytes() and dv.cpu().numpy()[:n].tobytes() == vals.tobytes()
    _guards_intact(ok, o_ok, n, 0x5A5A if in_place else 0x3C3C, "pairs keys")
    return _read(ok, o_ok, n), ov.cpu().numpy()[:n]


def random_keys(n: int, kt: int, seed: int) -> np.ndarray:
    rng = np.random.default_rng(seed)
    w = rng.integers(0, 1 << 16, n).astype(np.uint16)
    if kt in (ko.KEY_F16, ko.KEY_BF16) and n:
        spec = ko.float_specials(kt)
        pos = rng.integers(0, n, min(n, 4 * spec.size))
        w[pos] = np.resize(spec, pos.size)
    return w.view(ko.DTYPES[kt])


def assert_words(got: np.ndarray, want: np.ndarray, what: str):
    want = ko.bits(want)
    if got.tobytes() != want.tobytes():
        bad = np.flatnonzero(got != want)
        raise AssertionError(f"{what}: {bad.size} of {got.size} keys differ, first at {bad[0]}: "
                             f"got {int(got[bad[0]]):#06x}, want {int(want[bad[0]]):#06x}")


def check_both(keys, kt, desc, what, in_place_set=(False, True), offs_k=(0, 0), offs_p=(0, 0, 0)):
    vals = np.arange(keys.size, dtype=np.int32)[::-1].copy()
    p = np.argsort(ko.image(keys, kt, desc), kind="stable")
    for in_place in in_place_set:
        w = f"{what} in_place={in_place}"
        assert_words(sort16_keys(keys, kt, desc, in_place, offs_k), keys[p], "keys " + w)
        gk, gv = sort16_pairs(keys, vals, kt, desc, in_place, offs_p)
        assert_words(gk, keys[p], "pairs keys " + w)
        assert gv.tobytes() == vals[p].tobytes(), "pairs values " + w


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_keys_and_pairs_match_the_reference(order):
    kt, desc = order
    for n in SIZES:
        check_both(random_keys(n, kt, n + 11 * kt + desc), kt, desc, f"n={n}")


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_every_bit_pattern_shuffled_and_repeated(order):
    kt, desc = order
    rng = np.random.default_rng(kt * 2 + desc)
    keys = np.tile(np.arange(1 << 16, dtype=np.uint16), 3)
    rng.shuffle(keys)
    keys = keys.view(ko.DTYPES[kt])
    check_both(keys, kt, desc, "all 65536 patterns x3")
    got = sort16_keys(keys, kt, desc, False)
    want = np.repeat(ko.bits(ko.inverse(np.arange(1 << 16, dtype=np.uint16), kt, desc)), 3)
    assert got.tobytes() == want.tobytes()                     # each pattern three times, in image order


@pytest.mark.parametrize("offset", [2, 6, 14])
def test_key_pointers_off_a_16_byte_boundary(offset):
    for n in (1, 7, 9, 33, 65537, (1 << 20) + 3):
        for kt, desc in ((ko.KEY_I16, 0), (ko.KEY_BF16, 1), (ko.KEY_F16, 0)):
            keys = random_keys(n, kt, n + offset)
            for offs_k, offs_p in (((offset, 0), (offset, 0, 0)), ((0, offset), (0, offset, offset)),
                                   ((offset, 16 - offset), (offset, 16 - offset, offset))):
                check_both(keys, kt, desc, f"n={n} offsets={offs_k}", offs_k=offs_k, offs_p=offs_p)


def low_entropy(kind: str, n: int) -> np.ndarray:
    rng = np.random.default_rng(9)
    r = rng.integers(0, 1 << 16, n).astype(np.uint16)
    if kind == "all_equal":
        return np.full(n, 0xC123, np.uint16)
    if kind == "constant_low_byte":                             # pass 0 skippable
        return (r & np.uint16(0xFF00)) | np.uint16(0x5A)
    if kind == "constant_high_byte":                            # pass 1 skippable
        return (r & np.uint16(0x00FF)) | np.uint16(0x3C00)
    if kind == "small_signed":
        return rng.integers(-100, 101, n).astype(np.int16).view(np.uint16)
    if kind == "ties":
        return (r % np.uint16(37)) * np.uint16(0x0101)
    raise ValueError(kind)


@pytest.mark.parametrize("kind", ["all_equal", "constant_low_byte", "constant_high_byte", "small_signed", "ties"])
def test_low_entropy_with_and_without_pass_skipping(kind):
    L = lib()
    try:
        for skip in (1, 0):
            L.b200sort_radix_set_skip(skip)
            for n in (TILE * 3 + 17, (1 << 20) + 3):
                w = low_entropy(kind, n)
                for kt, desc in ((ko.KEY_I16, 0), (ko.KEY_I16, 1), (ko.KEY_U16, 1), (ko.KEY_BF16, 0)):
                    check_both(w.view(ko.DTYPES[kt]), kt, desc, f"{kind} skip={skip} n={n} order={kt},{desc}")
    finally:
        L.b200sort_radix_set_skip(1)


def test_many_copies_of_one_key():
    """Copies of one pattern fill a 16-bit shared counter past 0xFFFF in every histogram CTA once there are more
    than 65535 per CTA: the wrap repairs for the low and the high half of a counter word, and a carry from the low
    half that wraps the high half too (two neighbouring patterns, both heavy)."""
    for n in (65535, 65536, 65537, (1 << 20) + 3, (1 << 24) + 5, 1 << 25):
        for kt, desc, pat in ((ko.KEY_I16, 0, 0x1234), (ko.KEY_U16, 1, 0x1235), (ko.KEY_BF16, 0, 0xBF80)):
            keys = np.full(n, pat, np.uint16).view(ko.DTYPES[kt])
            assert_words(sort16_keys(keys, kt, desc, False), keys, f"keys n={n} pattern {pat:#x}")
            if n <= (1 << 24) + 5:
                gk, gv = sort16_pairs(keys, np.arange(n, dtype=np.int32), kt, desc, True)
                assert_words(gk, keys, f"pairs n={n}"); assert (gv == np.arange(n, dtype=np.int32)).all()
    rng = np.random.default_rng(1)
    for n in ((1 << 24) + 5, 1 << 25):
        keys = np.where(rng.random(n) < 0.5, np.uint16(0x4000), np.uint16(0x4001))   # images 2m and 2m + 1 (uint16)
        keys[:3] = 0xFFFF
        assert_words(sort16_keys(keys, ko.KEY_U16, 0, True), np.sort(keys), f"two neighbours n={n}")


def test_rank_safe_fallback_for_pairs():
    """With B200SORT_RANK_SAFE=1 the ballot-ranked pass kernels run."""
    code = (
        "import sys; sys.path.insert(0, '.'); sys.path.insert(0, 'tests')\n"
        "import numpy as np\n"
        "from b200sort._lib import lib\n"
        "import key_orders16 as ko\n"
        "import test_keys16_gpu as t\n"
        "assert lib().b200sort_radix_atomic_order_ok() == 0\n"
        "for kt, desc in ko.ORDERS:\n"
        "    for n in (t.TILE + 1, (1 << 20) + 3):\n"
        "        k = t.random_keys(n, kt, n + kt)\n"
        "        t.check_both(k, kt, desc, ('safe', kt, desc, n), in_place_set=(False,))\n"
        "        k = (k.view(np.uint16) % np.uint16(100)).view(ko.DTYPES[kt])\n"
        "        t.check_both(k, kt, desc, ('safe ties', kt, desc, n), in_place_set=(True,))\n"
        "print('ok')\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env={**os.environ, "B200SORT_RANK_SAFE": "1"},
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


def test_launch_count_does_not_depend_on_size_or_data():
    L = lib()
    check(L.b200sort_device_check())                             # the lane-order self-test launches a kernel once
    counts = set()
    for n in (2, 100, TILE + 1, (1 << 20) + 3):
        for kind in ("all_equal", "constant_low_byte", "small_signed"):
            keys = low_entropy(kind, n).view(np.int16)
            L.b200sort_launch_count_reset()
            got = sort16_keys(keys, ko.KEY_I16, 0, False)
            counts.add(("keys", L.b200sort_launch_count()))
            L.b200sort_launch_count_reset()
            sort16_pairs(keys, np.arange(n, dtype=np.int32), ko.KEY_I16, 1, False)
            counts.add(("pairs", L.b200sort_launch_count()))
            assert_words(got, ko.sort_keys(keys, ko.KEY_I16, 0), f"{kind} n={n}")
    assert counts == {("keys", 3), ("pairs", 5)}, counts


def test_cuda_graph_capture_and_replay():
    import torch
    L = lib()
    check(L.b200sort_device_check())
    n = (1 << 20) + 3
    x = torch.empty(n, dtype=torch.bfloat16, device="cuda")
    v = torch.arange(n, dtype=torch.int32, device="cuda")
    ko_, vo = torch.empty_like(x), torch.empty_like(v)
    kt_, vt = torch.empty_like(x), torch.empty_like(v)
    so = torch.empty_like(x)
    ws, ptr, nbytes = _ws(n)
    ws2, ptr2, _ = _ws(n)
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        check(L.b200sort_radix_pairs_keys16(ko.KEY_BF16, 1, x.data_ptr(), v.data_ptr(), ko_.data_ptr(), vo.data_ptr(),
                                            kt_.data_ptr(), vt.data_ptr(), n, ptr, nbytes, s.cuda_stream))
        check(L.b200sort_sort_keys16(ko.KEY_BF16, 0, x.data_ptr(), so.data_ptr(), n, ptr2, nbytes, s.cuda_stream))
    for seed in (1, 2, 3):
        rng = np.random.default_rng(seed)
        a = rng.integers(-5000, 5000, n).astype(np.float32) / 8 if seed != 3 else np.full(n, 2.5, np.float32)
        a[a == 0] = 0.5
        x.copy_(torch.from_numpy(a).to(torch.bfloat16))
        g.replay()
        torch.cuda.synchronize()
        tv, ti = torch.sort(x, stable=True, descending=True)
        assert torch.equal(ko_, tv) and torch.equal(vo, ti.to(torch.int32)), seed
        assert torch.equal(so, torch.sort(x).values), seed


@pytest.mark.parametrize("dtype", ["int16", "float16", "bfloat16"])
def test_python_calls_match_torch_sort(dtype):
    import torch
    for n in (1000, 300001, (1 << 22) + 1):
        g = torch.Generator(device="cuda"); g.manual_seed(n)
        if dtype == "int16":
            x = torch.randint(-2**15, 2**15, (n,), dtype=torch.int32, device="cuda", generator=g).to(torch.int16)
        else:
            x = (torch.randn(n, device="cuda", generator=g) * 100).to(getattr(torch, dtype))
            x[x == 0] = 0.5                                      # no -0.0
        before = x.clone()
        idx = torch.arange(n, dtype=torch.int32, device="cuda")
        for desc in (False, True):
            tv, ti = torch.sort(x, stable=True, descending=desc)
            k = b200sort.sort16(x, descending=desc)
            assert torch.equal(k, tv), (dtype, n, desc)
            k, v = b200sort.sort16_by_key(x, idx, descending=desc)
            assert torch.equal(k, tv) and torch.equal(v, ti.to(torch.int32)), (dtype, n, desc)
        assert torch.equal(x.view(torch.int16), before.view(torch.int16))
    u = np.random.default_rng(4).integers(0, 1 << 16, 5000).astype(np.uint16)    # uint16 against the reference
    got = b200sort.sort16(torch.from_numpy(u.view(np.int16)).cuda().view(torch.uint16), descending=True)
    assert got.view(torch.int16).cpu().numpy().view(np.uint16).tobytes() == np.sort(u)[::-1].tobytes()


def test_where_total_order_and_torch_sort_differ():
    """-0.0 sorts before +0.0 and NaNs go by sign and payload; torch.sort keeps zeros in input order, NaNs last."""
    import torch
    a = np.array([0.0, np.nan, -0.0, 1.0, -np.nan, -1.0], dtype=np.float16)
    x = torch.from_numpy(a).cuda()
    got = b200sort.sort16(x).cpu().numpy()
    assert got.tobytes() == ko.sort_keys(a, ko.KEY_F16, 0).tobytes()
    assert np.signbit(got[0]) and np.isnan(got[0])               # -NaN first
    assert np.signbit(got[2]) and got[2] == 0 and not np.signbit(got[3])
    tv = torch.sort(x).values.cpu().numpy()
    assert np.isnan(tv[-1]) and np.isnan(tv[-2]) and tv.tobytes() != got.tobytes()


def _images(torch, t, kt, desc):
    """image(k) as int32: the order of these is the order of the keys."""
    neg, pos = ko.MASKS[(kt, desc)]
    w = t.view(torch.int16).to(torch.int32) & 0xFFFF
    return w ^ torch.where(w >= 0x8000, torch.tensor(neg, device=t.device), torch.tensor(pos, device=t.device))


@pytest.mark.parametrize("case", ["bf16_asc_keys", "f16_desc_keys", "i16_asc_pairs", "bf16_desc_pairs"])
def test_full_size_2_28(case):
    import torch
    n = 1 << 28
    g = torch.Generator(device="cuda"); g.manual_seed(12)
    kt = {"bf16": ko.KEY_BF16, "f16": ko.KEY_F16, "i16": ko.KEY_I16}[case.split("_")[0]]
    desc = 1 if "_desc_" in case else 0
    if kt == ko.KEY_I16:
        x = torch.randint(-2**15, 2**15, (n,), dtype=torch.int32, device="cuda", generator=g).to(torch.int16)
    else:
        x = torch.randint(-2**15, 2**15, (n,), dtype=torch.int32, device="cuda", generator=g).to(torch.int16)
        x = x.view(torch.bfloat16 if kt == ko.KEY_BF16 else torch.float16)          # uniform bit patterns
    out = torch.empty_like(x)
    ws, ptr, nbytes = _ws(n)
    pairs = case.endswith("pairs")
    if not pairs:
        check(lib().b200sort_sort_keys16(kt, desc, x.data_ptr(), out.data_ptr(), n, ptr, nbytes, stream_ptr()))
    else:
        tmp = torch.empty_like(x)
        v = torch.arange(n, dtype=torch.int32, device="cuda")
        vo = torch.empty_like(v); vt = torch.empty_like(v)
        check(lib().b200sort_radix_pairs_keys16(kt, desc, x.data_ptr(), v.data_ptr(), out.data_ptr(), vo.data_ptr(),
                                                tmp.data_ptr(), vt.data_ptr(), n, ptr, nbytes, stream_ptr()))
    torch.cuda.synchronize()
    img = _images(torch, out, kt, desc)
    assert not bool((img[1:] < img[:-1]).any()), "not sorted"
    want = torch.bincount(_images(torch, x, kt, desc), minlength=1 << 16)
    assert torch.equal(torch.bincount(img, minlength=1 << 16), want), "not a permutation of the input"
    if pairs:
        assert torch.equal(x.view(torch.int16)[vo.to(torch.int64)], out.view(torch.int16)), "values do not follow keys"
        same = img[1:] == img[:-1]
        assert not bool((same & (vo[1:] <= vo[:-1])).any()), "pairs not stable"


@pytest.mark.parametrize("case", ["two_halves", "all_equal"])
def test_keys_only_at_2_30(case):
    import torch
    n = 1 << 30
    x = torch.full((n,), 0x1234, dtype=torch.int16, device="cuda")
    if case == "two_halves":
        x[::2] = -7                                              # 2^29 each of two values, interleaved
    out = torch.empty_like(x)
    ws, ptr, nbytes = _ws(n)
    check(lib().b200sort_sort_keys16(ko.KEY_I16, 0, x.data_ptr(), out.data_ptr(), n, ptr, nbytes, stream_ptr()))
    torch.cuda.synchronize()
    if case == "two_halves":
        half = n // 2
        assert bool((out[:half] == -7).all()) and bool((out[half:] == 0x1234).all())
    else:
        assert bool((out == 0x1234).all())


def test_python_call_on_a_non_default_device():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible")
    dev = torch.device("cuda", torch.cuda.device_count() - 1)
    n = 100003
    keys = random_keys(n, ko.KEY_F16, 5)
    x = torch.from_numpy(keys).to(dev)
    assert torch.cuda.current_device() != dev.index
    got = b200sort.sort16(x, descending=True)
    assert got.device == dev
    assert_words(got.cpu().numpy().view(np.uint16), ko.sort_keys(keys, ko.KEY_F16, 1), "keys")
    v = torch.arange(n, dtype=torch.int32, device=dev)
    k, vv = b200sort.sort16_by_key(x, v)
    wk, wv = ko.sort_pairs(keys, np.arange(n, dtype=np.int32), ko.KEY_F16, 0)
    assert_words(k.cpu().numpy().view(np.uint16), wk, "pairs keys")
    assert vv.cpu().numpy().tobytes() == wv.tobytes()


def test_checked_library_counts_no_violations():
    """The self-asserting build (make checked) runs the 16-bit part of tools/sanitize_target.py: fill and scatter
    destinations below n, marks and staged positions inside their tile."""
    lib_path = os.path.join(ROOT, os.path.basename(os.path.dirname(b200sort.__file__)), "libb200sort_checked.so")
    if not os.path.exists(lib_path):
        pytest.skip("checked library not built (make checked)")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "sanitize_target.py"), "keys16"], cwd=ROOT,
                       env={**os.environ, "B200SORT_LIB": "libb200sort_checked.so"},
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "CHECKED BUILD: 0 violated" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
