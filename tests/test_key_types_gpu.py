"""uint32 / float32 keys and descending order on the GPU (b200sort_sort_keys, b200sort_radix_pairs_keys and the
torch-facing b200sort.sort / sort_by_key), byte for byte against the numpy reference of the key orders."""
import os
import subprocess
import sys

import numpy as np
import pytest

import b200sort
import oracle
from b200sort import datagen
from b200sort._lib import ALGO_MERGE, ALGO_RADIX, check, lib
from helpers import stream_ptr, workspace

import key_orders as ko

pytestmark = pytest.mark.gpu

NEW_ORDERS = [o for o in ko.ORDERS if o != (ko.KEY_I32, 0)]
ORDER_IDS = [f"{ko.NAMES[k]}_{'desc' if d else 'asc'}" for k, d in NEW_ORDERS]
ALGOS = {"radix": ALGO_RADIX, "merge": ALGO_MERGE}
SIZES = [0, 1, 2, 31, 33, 4096, 8191, 8192, 8193, 65537, (1 << 20) + 3, (1 << 23) + 5]


def _dev(a: np.ndarray, offset: int = 0):
    """Device copy of the 32-bit words of ``a`` starting `offset` elements into a larger buffer (unaligned pointers)."""
    import torch
    buf = torch.empty(a.size + offset + 1, dtype=torch.int32, device="cuda")
    buf[offset:offset + a.size] = torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).cuda()
    return buf, buf.data_ptr() + 4 * offset


def _words(buf, offset: int, n: int) -> np.ndarray:
    return buf[offset:offset + n].cpu().numpy().view(np.uint32)


def sort_keys(keys: np.ndarray, key_type: int, desc: int, algo: int, in_place: bool, offset: int = 0) -> np.ndarray:
    """The library's result as uint32 words; checks the copy form leaves its input alone."""
    import torch
    n = keys.size
    src, p_in = _dev(keys, offset)
    out, p_out = (src, p_in) if in_place else _dev(np.full(n, 0x5A5A5A5A, np.uint32), offset)
    tmp = torch.empty(max(n, 1), dtype=torch.int32, device="cuda")
    ws, ptr, nbytes = workspace(n, algo)
    check(lib().b200sort_sort_keys(algo, key_type, desc, p_in, p_out, tmp.data_ptr(), n, ptr, nbytes, stream_ptr()))
    torch.cuda.synchronize()
    if not in_place:
        assert _words(src, offset, n).tobytes() == ko.bits(keys).tobytes(), "the copy form modified its input"
    return _words(out, offset, n)


def sort_pairs(keys: np.ndarray, vals: np.ndarray, key_type: int, desc: int, in_place: bool):
    import torch
    n = keys.size
    dk, pk = _dev(keys)
    dv, pv = _dev(vals)
    (ok, pok), (ov, pov) = ((dk, pk), (dv, pv)) if in_place else (_dev(np.zeros(n, np.uint32)), _dev(np.zeros(n, np.int32)))
    tk = torch.empty(max(n, 1), dtype=torch.int32, device="cuda"); tv = torch.empty_like(tk)
    ws, ptr, nbytes = workspace(n, ALGO_RADIX)
    check(lib().b200sort_radix_pairs_keys(key_type, desc, pk, pv, pok, pov, tk.data_ptr(), tv.data_ptr(), n, ptr, nbytes,
                                          stream_ptr()))
    torch.cuda.synchronize()
    if not in_place:
        assert _words(dk, 0, n).tobytes() == ko.bits(keys).tobytes() and _words(dv, 0, n).tobytes() == ko.bits(vals).tobytes()
    return _words(ok, 0, n), _words(ov, 0, n).view(np.int32)


def mixed_keys(n: int, key_type: int, seed: int) -> np.ndarray:
    """Uniform random bit patterns, and for float32 the specials of the header sprinkled through them."""
    w = datagen.uniform_u32(n, seed)
    if key_type == ko.KEY_F32 and n:
        spec = ko.float_specials()
        pos = datagen.uniform_u32(min(n, 4 * spec.size), seed + 1) % np.uint32(n)
        w[pos] = np.resize(spec, pos.size)
    return w.view(ko.DTYPES[key_type])


def assert_words(got: np.ndarray, want: np.ndarray, what: str):
    want = ko.bits(want)
    if got.tobytes() != want.tobytes():
        bad = np.flatnonzero(got != want)
        raise AssertionError(f"{what}: {bad.size} of {got.size} words differ, first at {bad[0]}: "
                             f"got {got[bad[0]]:#010x}, want {want[bad[0]]:#010x}")


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("order", NEW_ORDERS, ids=ORDER_IDS)
def test_byte_exact_parity(order, n):
    kt, desc = order
    keys = mixed_keys(n, kt, 100 + n % 97)
    want = ko.sort_keys(keys, kt, desc)
    for name, algo in ALGOS.items():
        for in_place in (False, True):
            assert_words(sort_keys(keys, kt, desc, algo, in_place), want, f"{name} in_place={in_place}")


@pytest.mark.parametrize("order", NEW_ORDERS, ids=ORDER_IDS)
def test_float_specials_and_unaligned_pointers(order):
    kt, desc = order
    spec = ko.float_specials()
    for n in (spec.size, 5000, 70001):
        keys = np.resize(spec, n).copy()
        keys[::3] = datagen.uniform_u32(keys[::3].size, n)
        keys = keys.view(ko.DTYPES[kt])
        want = ko.sort_keys(keys, kt, desc)
        for name, algo in ALGOS.items():
            for offset in (0, 1, 2, 3):
                assert_words(sort_keys(keys, kt, desc, algo, False, offset), want, f"{name} n={n} offset={offset}")


def _low_entropy(kind: str, n: int) -> np.ndarray:
    if kind == "all_equal_f32":
        return np.full(n, -2.5, np.float32)
    if kind == "small_ints_f32":
        return (datagen.uniform_u32(n, 4) % np.uint32(100)).astype(np.float32) - np.float32(50)
    if kind == "masked_u32":
        return datagen.uniform_u32(n, 6) & np.uint32(0x00FF00FF)
    if kind == "top_byte_u32":
        return (datagen.uniform_u32(n, 8) & np.uint32(0xFF000000)) | np.uint32(0x00ABCDEF)
    raise KeyError(kind)


@pytest.mark.parametrize("kind", ["all_equal_f32", "small_ints_f32", "masked_u32", "top_byte_u32"])
def test_low_entropy_with_pass_skipping_on_and_off(kind):
    L = lib()
    try:
        for n in (5000, 300001, (1 << 20) + 12345):
            keys = _low_entropy(kind, n)
            kt = ko.KEY_F32 if keys.dtype == np.float32 else ko.KEY_U32
            for desc in (0, 1):
                want = ko.sort_keys(keys, kt, desc)
                for skip in (1, 0):
                    L.b200sort_radix_set_skip(skip)
                    for name, algo in ALGOS.items():
                        assert_words(sort_keys(keys, kt, desc, algo, False), want, f"{kind} n={n} desc={desc} skip={skip} {name}")
                    assert_words(sort_keys(keys, kt, desc, ALGO_RADIX, True), want, f"{kind} n={n} desc={desc} skip={skip} in place")
    finally:
        L.b200sort_radix_set_skip(1)


def test_every_shipped_shape():
    L = lib()
    n = (1 << 20) + 12345
    try:
        for v in range(4):
            assert L.b200sort_radix_set_variant(v) == 0
            name = L.b200sort_radix_variant_name(v).decode()
            for kt, desc in NEW_ORDERS:
                keys = mixed_keys(n, kt, 7 + v)
                assert_words(sort_keys(keys, kt, desc, ALGO_RADIX, False), ko.sort_keys(keys, kt, desc), f"{name} {kt},{desc}")
        L.b200sort_radix_set_variant(0)
        for mv in range(2):
            assert L.b200sort_merge_set_variant(mv) == 0
            for kt, desc in NEW_ORDERS:
                keys = mixed_keys(n, kt, 17 + mv)
                assert_words(sort_keys(keys, kt, desc, ALGO_MERGE, False), ko.sort_keys(keys, kt, desc),
                             f"merge variant {mv} {kt},{desc}")
    finally:
        L.b200sort_radix_set_variant(0)
        L.b200sort_merge_set_variant(0)


def test_rank_safe_fallback_for_keys_and_pairs():
    """With B200SORT_RANK_SAFE=1 the generic ballot-ranked shapes run, for keys and for pairs."""
    code = (
        "import sys; sys.path.insert(0, '.'); sys.path.insert(0, 'tests')\n"
        "import numpy as np\n"
        "from b200sort._lib import lib, ALGO_RADIX\n"
        "import key_orders as ko\n"
        "import test_key_types_gpu as t\n"
        "assert lib().b200sort_radix_atomic_order_ok() == 0\n"
        "for kt, desc in t.NEW_ORDERS:\n"
        "    for n in (5000, 300001, (1 << 20) + 12345):\n"
        "        k = t.mixed_keys(n, kt, n)\n"
        "        t.assert_words(t.sort_keys(k, kt, desc, ALGO_RADIX, False), ko.sort_keys(k, kt, desc), (kt, desc, n))\n"
        "        k = (k.view(np.uint32) % np.uint32(100)).astype(np.float32) if kt == ko.KEY_F32 else k\n"
        "        v = np.arange(n, dtype=np.int32)\n"
        "        wk, wv = ko.sort_pairs(k, v, kt, desc)\n"
        "        gk, gv = t.sort_pairs(k, v, kt, desc, False)\n"
        "        t.assert_words(gk, wk, ('pairs', kt, desc, n)); assert gv.tobytes() == wv.tobytes(), ('pairs', kt, desc, n)\n"
        "print('ok')\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", code], cwd=root, env={**os.environ, "B200SORT_RANK_SAFE": "1"},
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


@pytest.mark.parametrize("n", [0, 1, 2, 33, 5119, 5120, 5121, 100003, (1 << 20) + 17])
@pytest.mark.parametrize("order", NEW_ORDERS, ids=ORDER_IDS)
def test_sort_by_key_is_stable(order, n):
    kt, desc = order
    r = datagen.uniform_u32(n, 23 + n % 13) % np.uint32(100)           # many duplicates
    keys = r.astype(np.float32) if kt == ko.KEY_F32 else (r.view(np.int32) - 50 if kt == ko.KEY_I32 else r)
    vals = np.arange(n, dtype=np.int32)
    want_k, want_v = ko.sort_pairs(keys, vals, kt, desc)
    for in_place in (False, True):
        got_k, got_v = sort_pairs(keys, vals, kt, desc, in_place)
        assert_words(got_k, want_k, f"keys in_place={in_place}")
        assert got_v.tobytes() == want_v.tobytes(), f"values in_place={in_place}"


@pytest.mark.parametrize("dtype", ["int32", "uint32", "float32"])
def test_python_call_matches_torch_sort_without_nan_or_negative_zero(dtype):
    import torch
    n = 300001
    r = datagen.uniform_u32(n, 31)
    if dtype == "float32":
        a = (r % np.uint32(1000)).astype(np.float32) / np.float32(8) - np.float32(60)
    elif dtype == "uint32":
        a = r % np.uint32(5000) + np.uint32(0x7FFFF000)           # crosses the sign bit of int32
    else:
        a = r.view(np.int32) % 5000
    x = torch.from_numpy(a).cuda()
    # torch.sort on the same values (uint32 compared as int64, which torch.sort takes)
    cmp = torch.from_numpy(a.astype(np.int64) if dtype == "uint32" else a).cuda()
    idx = torch.arange(n, dtype=torch.int32, device="cuda")
    for desc in (False, True):
        tv, ti = torch.sort(cmp, stable=True, descending=desc)
        tv, ti = tv.cpu().numpy(), ti.cpu().numpy()
        k, v = b200sort.sort_by_key(x, idx, descending=desc)
        assert np.array_equal(k.cpu().numpy().astype(tv.dtype), tv) and np.array_equal(v.cpu().numpy(), ti), desc
        for algo in ("radix", "merge"):
            got = b200sort.sort(x, descending=desc, algo=algo).cpu().numpy()
            assert np.array_equal(got.astype(tv.dtype), tv), (desc, algo)
    assert x.cpu().numpy().tobytes() == a.tobytes()
    with pytest.raises(ValueError):
        b200sort.sort_by_key(x, idx[:-1])


def test_float_total_order_differs_from_torch_on_nan_and_negative_zero():
    import torch
    spec = ko.float_specials()
    x = torch.from_numpy(spec.view(np.float32)[::-1].copy()).cuda()
    got = b200sort.sort(x).cpu().numpy().view(np.uint32)
    assert got.tobytes() == spec.tobytes()                        # exactly the header's order, bits untouched
    got_d = b200sort.sort(x, descending=True).cpu().numpy().view(np.uint32)
    assert got_d.tobytes() == spec[::-1].tobytes()


def test_int32_ascending_is_the_i32_path():
    import torch
    L = lib()
    for n in (5000, 300001, (1 << 23) + 5):
        keys = datagen.uniform(n, 3)
        for name, algo in ALGOS.items():
            src, p = _dev(keys)
            a = torch.empty_like(src); b = torch.empty_like(src); tmp = torch.empty_like(src)
            ws, ptr, nbytes = workspace(n, algo)
            L.b200sort_launch_count_reset()
            check(L.b200sort_sort_copy_i32(algo, p, a.data_ptr(), tmp.data_ptr(), n, ptr, nbytes, stream_ptr()))
            c1 = L.b200sort_launch_count()
            L.b200sort_launch_count_reset()
            check(L.b200sort_sort_keys(algo, ko.KEY_I32, 0, p, b.data_ptr(), tmp.data_ptr(), n, ptr, nbytes, stream_ptr()))
            c2 = L.b200sort_launch_count()
            torch.cuda.synchronize()
            assert c1 == c2, (name, n, c1, c2)
            assert torch.equal(a[:n], b[:n]), (name, n)


@pytest.mark.parametrize("order", [(ko.KEY_F32, 0), (ko.KEY_F32, 1), (ko.KEY_U32, 0), (ko.KEY_U32, 1)],
                         ids=["f32_asc", "f32_desc", "u32_asc", "u32_desc"])
def test_full_size_2_28(order):
    """n = 2^28: sorted in the image domain, same multiset of bit patterns as the input, both algorithms."""
    import torch
    kt, desc = order
    n = 1 << 28
    neg, pos = ko.MASKS[order]
    g = torch.Generator(device="cuda"); g.manual_seed(11 + kt * 2 + desc)
    x = torch.randint(-2**31, 2**31, (n,), dtype=torch.int64, device="cuda", generator=g).to(torch.int32)
    fp_in = oracle.multiset_fingerprint(x.cpu().numpy())
    out = torch.empty_like(x); tmp = torch.empty_like(x)
    for algo in (ALGO_RADIX, ALGO_MERGE):
        ws, ptr, nbytes = workspace(n, algo)
        check(lib().b200sort_sort_keys(algo, kt, desc, x.data_ptr(), out.data_ptr(), tmp.data_ptr(), n, ptr, nbytes,
                                       stream_ptr()))
        torch.cuda.synchronize()
        del ws
        # image as a signed-comparable int32: out ^ mask(out) ^ 0x80000000
        m = torch.where(out < 0, torch.tensor(neg ^ 0x80000000, dtype=torch.int64, device="cuda"),
                        torch.tensor(pos ^ 0x80000000, dtype=torch.int64, device="cuda"))
        s = (out.to(torch.int64) & 0xFFFFFFFF) ^ m
        s = torch.where(s >= 2**31, s - 2**32, s)
        assert bool((s[1:] >= s[:-1]).all().item()), f"algo {algo}: not sorted in the image domain"
        del m, s
        assert oracle.multiset_fingerprint(out.cpu().numpy()) == fp_in, f"algo {algo}: multiset changed"


def test_python_call_on_a_non_default_device():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible")
    dev = torch.device("cuda", torch.cuda.device_count() - 1)
    n = 100003
    w = datagen.uniform_u32(n, 5)
    x = torch.from_numpy(w.view(np.float32)).to(dev)
    assert torch.cuda.current_device() != dev.index
    got = b200sort.sort(x, descending=True)
    assert got.device == dev
    assert_words(got.cpu().numpy().view(np.uint32), ko.sort_keys(w.view(np.float32), ko.KEY_F32, 1), "sort")
    k, v = b200sort.sort_by_key(x, torch.arange(n, dtype=torch.int32, device=dev))
    wk, wv = ko.sort_pairs(w.view(np.float32), np.arange(n, dtype=np.int32), ko.KEY_F32, 0)
    assert_words(k.cpu().numpy().view(np.uint32), wk, "sort_by_key keys")
    assert v.cpu().numpy().tobytes() == wv.tobytes()
