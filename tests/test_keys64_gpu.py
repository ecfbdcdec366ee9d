"""64-bit keys on the GPU (b200sort_sort_keys64, b200sort_radix_pairs_keys64 and the torch-facing b200sort.sort64 /
sort64_by_key), byte for byte against the numpy reference of tests/key_orders64.py."""
import os
import subprocess
import sys

import numpy as np
import pytest

import b200sort
from b200sort._lib import check, lib
from helpers import stream_ptr

import key_orders64 as ko

pytestmark = pytest.mark.gpu

ORDER_IDS = [f"{ko.NAMES[k]}_{'desc' if d else 'asc'}" for k, d in ko.ORDERS]
TILE = 4096          # keys per onesweep tile (kR64Tile, csrc/radix64.cu)
SIZES = [0, 1, 2, 31, 33, TILE - 1, TILE, TILE + 1, 65537, (1 << 20) + 3, (1 << 23) + 5]


def _dev(a: np.ndarray):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int64).copy()).cuda()


def _words(t) -> np.ndarray:
    return t.cpu().numpy().view(np.uint64)


def _ws(n: int):
    import torch
    nbytes = lib().b200sort_keys64_workspace_bytes(n)
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
    return ws, ws.data_ptr() + (-ws.data_ptr()) % 256, nbytes


def sort64_keys(keys, kt, desc, in_place):
    """The library's keys-only result as uint64 words; checks that the copy form leaves its input alone."""
    import torch
    n = keys.size
    src = _dev(keys)
    out = src if in_place else torch.full((max(n, 1),), 0x5A5A5A5A, dtype=torch.int64, device="cuda")
    tmp = torch.empty(max(n, 1), dtype=torch.int64, device="cuda")
    ws, ptr, nbytes = _ws(n)
    check(lib().b200sort_sort_keys64(kt, desc, src.data_ptr(), out.data_ptr(), tmp.data_ptr(), n, ptr, nbytes,
                                     stream_ptr()))
    torch.cuda.synchronize()
    if not in_place:
        assert _words(src)[:n].tobytes() == ko.bits(keys).tobytes(), "the copy form modified its input"
    return _words(out)[:n]


def sort64_pairs(keys, vals, kt, desc, in_place):
    import torch
    n = keys.size
    dk, dv = _dev(keys), torch.from_numpy(np.ascontiguousarray(vals, np.int32)).cuda()
    if in_place:
        ok, ov = dk, dv
    else:
        ok = torch.zeros(max(n, 1), dtype=torch.int64, device="cuda")
        ov = torch.zeros(max(n, 1), dtype=torch.int32, device="cuda")
    tk = torch.empty(max(n, 1), dtype=torch.int64, device="cuda"); tv = torch.empty(max(n, 1), dtype=torch.int32, device="cuda")
    ws, ptr, nbytes = _ws(n)
    check(lib().b200sort_radix_pairs_keys64(kt, desc, dk.data_ptr(), dv.data_ptr(), ok.data_ptr(), ov.data_ptr(),
                                            tk.data_ptr(), tv.data_ptr(), n, ptr, nbytes, stream_ptr()))
    torch.cuda.synchronize()
    if not in_place:
        assert _words(dk)[:n].tobytes() == ko.bits(keys).tobytes() and dv.cpu().numpy()[:n].tobytes() == vals.tobytes()
    return _words(ok)[:n], ov.cpu().numpy()[:n]


def random_keys(n: int, kt: int, seed: int) -> np.ndarray:
    rng = np.random.default_rng(seed)
    w = rng.integers(0, 1 << 64, n, dtype=np.uint64, endpoint=False) if n else np.zeros(0, np.uint64)
    if kt == ko.KEY_F64 and n:
        spec = ko.float_specials()
        pos = rng.integers(0, n, min(n, 4 * spec.size))
        w[pos] = np.resize(spec, pos.size)
    return w.view(ko.DTYPES[kt])


def assert_words(got: np.ndarray, want: np.ndarray, what: str):
    want = ko.bits(want)
    if got.tobytes() != want.tobytes():
        bad = np.flatnonzero(got != want)
        raise AssertionError(f"{what}: {bad.size} of {got.size} keys differ, first at {bad[0]}: "
                             f"got {int(got[bad[0]]):#018x}, want {int(want[bad[0]]):#018x}")


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_keys_and_pairs_match_the_reference(order):
    kt, desc = order
    for n in SIZES:
        keys = random_keys(n, kt, n + 11 * kt + desc)
        vals = np.arange(n, dtype=np.int32)[::-1].copy()
        p = np.argsort(ko.image(keys, kt, desc), kind="stable")
        for in_place in (False, True):
            assert_words(sort64_keys(keys, kt, desc, in_place), keys[p], f"keys n={n} in_place={in_place}")
            gk, gv = sort64_pairs(keys, vals, kt, desc, in_place)
            assert_words(gk, keys[p], f"pairs keys n={n} in_place={in_place}")
            assert gv.tobytes() == vals[p].tobytes(), f"pairs values n={n} in_place={in_place}"


@pytest.mark.parametrize("desc", [0, 1])
def test_float_specials_scattered_through_random_data(desc):
    n = 300001
    rng = np.random.default_rng(desc)
    w = rng.standard_normal(n).view(np.uint64).copy()
    spec = ko.float_specials()
    w[rng.integers(0, n, 5000)] = np.resize(spec, 5000)
    keys = w.view(np.float64)
    assert_words(sort64_keys(keys, ko.KEY_F64, desc, False), ko.sort_keys(keys, ko.KEY_F64, desc), "specials")
    vals = np.arange(n, dtype=np.int32)
    wk, wv = ko.sort_pairs(keys, vals, ko.KEY_F64, desc)
    gk, gv = sort64_pairs(keys, vals, ko.KEY_F64, desc, True)
    assert_words(gk, wk, "specials pairs"); assert gv.tobytes() == wv.tobytes()


def low_entropy(kind: str, n: int) -> np.ndarray:
    rng = np.random.default_rng(9)
    r = rng.integers(0, 1 << 64, n, dtype=np.uint64)
    if kind == "all_equal":
        return np.full(n, 0xC01234567890ABCD, np.uint64)
    if kind == "below_2_32":                                     # four upper passes skippable
        return r >> np.uint64(32)
    if kind == "constant_low_word":                              # four lower passes skippable
        return (r & np.uint64(0xFFFFFFFF00000000)) | np.uint64(0x9ABCDEF0)
    if kind == "small_signed":                                   # two bins hold every key in the upper passes
        return rng.integers(-1000, 1001, n).astype(np.int64).view(np.uint64)
    if kind == "ties":
        return (r % np.uint64(37)) * np.uint64(0x0101010101010101)
    raise ValueError(kind)


@pytest.mark.parametrize("kind", ["all_equal", "below_2_32", "constant_low_word", "small_signed", "ties"])
def test_low_entropy_with_and_without_pass_skipping(kind):
    L = lib()
    try:
        for skip in (1, 0):
            L.b200sort_radix_set_skip(skip)
            for n in (TILE * 3 + 17, (1 << 20) + 3):
                w = low_entropy(kind, n)
                vals = np.arange(n, dtype=np.int32)
                for kt, desc in ((ko.KEY_I64, 0), (ko.KEY_I64, 1), (ko.KEY_U64, 1), (ko.KEY_F64, 0)):
                    keys = w.view(ko.DTYPES[kt])
                    p = np.argsort(ko.image(keys, kt, desc), kind="stable")
                    for in_place in (False, True):
                        what = f"{kind} skip={skip} n={n} order={kt},{desc} in_place={in_place}"
                        assert_words(sort64_keys(keys, kt, desc, in_place), keys[p], what)
                        gk, gv = sort64_pairs(keys, vals, kt, desc, in_place)
                        assert_words(gk, keys[p], "pairs " + what)
                        assert gv.tobytes() == vals[p].tobytes(), "pairs values " + what
    finally:
        L.b200sort_radix_set_skip(1)


def test_rank_safe_fallback_for_keys_and_pairs():
    """With B200SORT_RANK_SAFE=1 the ballot-ranked pass kernels run, for keys and for pairs."""
    code = (
        "import sys; sys.path.insert(0, '.'); sys.path.insert(0, 'tests')\n"
        "import numpy as np\n"
        "from b200sort._lib import lib\n"
        "import key_orders64 as ko\n"
        "import test_keys64_gpu as t\n"
        "assert lib().b200sort_radix_atomic_order_ok() == 0\n"
        "for kt, desc in ko.ORDERS:\n"
        "    for n in (t.TILE + 1, (1 << 20) + 3):\n"
        "        k = t.random_keys(n, kt, n + kt)\n"
        "        t.assert_words(t.sort64_keys(k, kt, desc, False), ko.sort_keys(k, kt, desc), (kt, desc, n))\n"
        "        k = (k.view(np.uint64) % np.uint64(100)).view(ko.DTYPES[kt])\n"
        "        v = np.arange(n, dtype=np.int32)\n"
        "        wk, wv = ko.sort_pairs(k, v, kt, desc)\n"
        "        gk, gv = t.sort64_pairs(k, v, kt, desc, True)\n"
        "        t.assert_words(gk, wk, ('pairs', kt, desc)); assert gv.tobytes() == wv.tobytes(), ('pairs', kt, desc)\n"
        "print('ok')\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", code], cwd=root, env={**os.environ, "B200SORT_RANK_SAFE": "1"},
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


def test_launch_count_does_not_depend_on_size_or_data():
    L = lib()
    check(L.b200sort_device_check())                             # the lane-order self-test launches a kernel once
    counts = set()
    for n in (2, 100, TILE + 1, (1 << 20) + 3):
        for kind in ("all_equal", "below_2_32", "small_signed"):
            keys = low_entropy(kind, n).view(np.int64)
            L.b200sort_launch_count_reset()
            got = sort64_keys(keys, ko.KEY_I64, 0, False)
            counts.add(("keys", L.b200sort_launch_count()))
            L.b200sort_launch_count_reset()
            sort64_pairs(keys, np.arange(n, dtype=np.int32), ko.KEY_I64, 1, False)
            counts.add(("pairs", L.b200sort_launch_count()))
            assert_words(got, ko.sort_keys(keys, ko.KEY_I64, 0), f"{kind} n={n}")
    assert counts == {("keys", 10), ("pairs", 10)}, counts


def test_cuda_graph_capture_and_replay():
    import torch
    L = lib()
    check(L.b200sort_device_check())
    n = (1 << 20) + 3
    x = torch.empty(n, dtype=torch.float64, device="cuda")
    v = torch.arange(n, dtype=torch.int32, device="cuda")
    ko_, vo = torch.empty_like(x), torch.empty_like(v)
    kt_, vt = torch.empty_like(x), torch.empty_like(v)
    ws, ptr, nbytes = _ws(n)
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        check(L.b200sort_radix_pairs_keys64(ko.KEY_F64, 1, x.data_ptr(), v.data_ptr(), ko_.data_ptr(), vo.data_ptr(),
                                            kt_.data_ptr(), vt.data_ptr(), n, ptr, nbytes, s.cuda_stream))
    for seed in (1, 2, 3):
        rng = np.random.default_rng(seed)
        a = rng.integers(-5000, 5000, n).astype(np.float64) / 8 if seed != 3 else np.full(n, 2.5)
        x.copy_(torch.from_numpy(a))
        g.replay()
        torch.cuda.synchronize()
        tv, ti = torch.sort(x, stable=True, descending=True)
        assert torch.equal(ko_, tv) and torch.equal(vo, ti.to(torch.int32)), seed


@pytest.mark.parametrize("dtype", ["int64", "float64"])
def test_python_calls_match_torch_sort(dtype):
    import torch
    for n in (1000, 300001):
        rng = np.random.default_rng(n)
        if dtype == "int64":
            a = rng.integers(-(1 << 62), 1 << 62, n)
            a[::7] = a[:: 7 * 5].repeat(5)[: a[::7].size]                  # duplicates
        else:
            a = np.round(rng.standard_normal(n) * 100, 1)
            a[a == 0] = 0.5                                      # no -0.0
        x = torch.from_numpy(a).cuda()
        idx = torch.arange(n, dtype=torch.int32, device="cuda")
        for desc in (False, True):
            tv, ti = torch.sort(x, stable=True, descending=desc)
            k = b200sort.sort64(x, descending=desc)
            assert torch.equal(k, tv), (dtype, n, desc)
            k, v = b200sort.sort64_by_key(x, idx, descending=desc)
            assert torch.equal(k, tv) and torch.equal(v, ti.to(torch.int32)), (dtype, n, desc)
        assert x.cpu().numpy().tobytes() == a.tobytes()
    # uint64 against the reference
    u = np.random.default_rng(4).integers(0, 1 << 64, 5000, dtype=np.uint64)
    got = b200sort.sort64(torch.from_numpy(u).cuda(), descending=True)
    assert got.cpu().numpy().tobytes() == np.sort(u)[::-1].tobytes()


def test_where_total_order_and_torch_sort_differ():
    """-0.0 sorts before +0.0 and NaNs go by sign and payload; torch.sort keeps zeros in input order, NaNs last."""
    import torch
    a = np.array([0.0, np.nan, -0.0, 1.0, -np.nan, -1.0], dtype=np.float64)
    x = torch.from_numpy(a).cuda()
    got = b200sort.sort64(x).cpu().numpy()
    want = ko.sort_keys(a, ko.KEY_F64, 0)
    assert got.tobytes() == want.tobytes()
    assert np.signbit(got[0]) and np.isnan(got[0])                # -NaN first
    assert np.signbit(got[2]) and got[2] == 0 and not np.signbit(got[3])   # -0.0 then +0.0
    tv = torch.sort(x).values.cpu().numpy()
    assert np.isnan(tv[-1]) and np.isnan(tv[-2]) and tv.tobytes() != got.tobytes()


def _images_i64(torch, t, kt, desc):
    """image(k) ^ (1 << 63) as int64: signed order of these = unsigned order of the images."""
    neg, pos = ko.MASKS[(kt, desc)]
    as_i64 = lambda m: m - (1 << 64) if m >= 1 << 63 else m
    w = t.view(torch.int64)
    img = w ^ torch.where(w < 0, torch.tensor(as_i64(neg), device=t.device), torch.tensor(as_i64(pos), device=t.device))
    return img ^ torch.tensor(as_i64(1 << 63), device=t.device)


@pytest.mark.parametrize("case", ["i64_asc_keys", "f64_desc_pairs"])
def test_full_size_2_28(case):
    import torch
    n = 1 << 28
    g = torch.Generator(device="cuda"); g.manual_seed(12)
    if case == "i64_asc_keys":
        kt, desc = ko.KEY_I64, 0
        x = torch.randint(-2**31, 2**31, (n, 2), dtype=torch.int64, device="cuda", generator=g).to(torch.int32)
        x = x.view(torch.int64).view(-1)                         # uniform 64-bit patterns
    else:
        kt, desc = ko.KEY_F64, 1
        x = torch.randint(-4000, 4000, (n,), dtype=torch.int64, device="cuda", generator=g).to(torch.float64) / 4
    out = torch.empty_like(x); tmp = torch.empty_like(x)
    ws, ptr, nbytes = _ws(n)
    if case == "i64_asc_keys":
        check(lib().b200sort_sort_keys64(kt, desc, x.data_ptr(), out.data_ptr(), tmp.data_ptr(), n, ptr, nbytes,
                                         stream_ptr()))
    else:
        v = torch.arange(n, dtype=torch.int32, device="cuda")
        vo = torch.empty_like(v); vt = torch.empty_like(v)
        check(lib().b200sort_radix_pairs_keys64(kt, desc, x.data_ptr(), v.data_ptr(), out.data_ptr(), vo.data_ptr(),
                                                tmp.data_ptr(), vt.data_ptr(), n, ptr, nbytes, stream_ptr()))
    torch.cuda.synchronize()
    del tmp
    img = _images_i64(torch, out, kt, desc)
    assert not bool((img[1:] < img[:-1]).any()), "not sorted"
    want = torch.sort(_images_i64(torch, x, kt, desc)).values
    assert torch.equal(img, want), "not a permutation of the input"
    del want
    if case == "f64_desc_pairs":
        assert torch.equal(x[vo.to(torch.int64)], out), "values do not follow their keys"
        same = img[1:] == img[:-1]
        assert not bool((same & (vo[1:] <= vo[:-1])).any()), "pairs not stable"


def test_python_call_on_a_non_default_device():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible")
    dev = torch.device("cuda", torch.cuda.device_count() - 1)
    n = 100003
    keys = random_keys(n, ko.KEY_F64, 5)
    x = torch.from_numpy(keys).to(dev)
    assert torch.cuda.current_device() != dev.index
    got = b200sort.sort64(x, descending=True)
    assert got.device == dev
    assert_words(got.cpu().numpy().view(np.uint64), ko.sort_keys(keys, ko.KEY_F64, 1), "keys")
    v = torch.arange(n, dtype=torch.int32, device=dev)
    k, vv = b200sort.sort64_by_key(x, v)
    wk, wv = ko.sort_pairs(keys, np.arange(n, dtype=np.int32), ko.KEY_F64, 0)
    assert_words(k.cpu().numpy().view(np.uint64), wk, "pairs keys")
    assert vv.cpu().numpy().tobytes() == wv.tobytes()
