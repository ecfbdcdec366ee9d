"""Segmented sort on the GPU (b200sort_segmented_sort_keys, b200sort_segmented_pairs_keys and the torch-facing
b200sort.segmented_sort / segmented_sort_by_key), byte for byte against the numpy reference of
tests/test_segmented_cpu.py."""
import os
import subprocess
import sys

import numpy as np
import pytest

import b200sort
import oracle
from b200sort import datagen
from b200sort._lib import ALGO_RADIX, check, lib
from helpers import stream_ptr, workspace

import key_orders as ko
from test_segmented_cpu import seg_sort_keys, seg_sort_pairs

pytestmark = pytest.mark.gpu

ORDER_IDS = [f"{ko.NAMES[k]}_{'desc' if d else 'asc'}" for k, d in ko.ORDERS]
TILE = 6144          # keys per tile of the segmented onesweep (kSegTile, csrc/segmented.cuh)


def _class_bounds():
    L = lib()
    out, c = [], 0
    while L.b200sort_segmented_class_max(c):
        out.append(L.b200sort_segmented_class_max(c))
        c += 1
    return out


def row_lengths():
    ls = {1, 2, 31, 32, 33, 8191, 8192, 8193, TILE - 1, TILE, TILE + 1, 2 * TILE + 1, 65537, (1 << 20) + 3}
    for m in _class_bounds():
        ls |= {m - 1, m, m + 1}
    return sorted(x for x in ls if x >= 1)


def _dev(a: np.ndarray, offset: int = 0):
    import torch
    buf = torch.empty(a.size + offset + 1, dtype=torch.int32, device="cuda")
    buf[offset:offset + a.size] = torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).cuda()
    return buf, buf.data_ptr() + 4 * offset


def _words(buf, offset: int, n: int) -> np.ndarray:
    return buf[offset:offset + n].cpu().numpy().view(np.uint32)


def _ws(n: int, segments: int):
    import torch
    nbytes = lib().b200sort_segmented_workspace_bytes(n, segments)
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
    return ws, ws.data_ptr() + (-ws.data_ptr()) % 256, nbytes


def seg_keys(keys, offsets, kt, desc, in_place, offset=0):
    """The library's result as uint32 words; checks the copy form leaves its input alone."""
    import torch
    n = keys.size
    src, p_in = _dev(keys, offset)
    out, p_out = (src, p_in) if in_place else _dev(np.full(n, 0x5A5A5A5A, np.uint32), offset)
    tmp = torch.empty(max(n, 1), dtype=torch.int32, device="cuda")
    d_off = torch.from_numpy(np.asarray(offsets, np.int32)).cuda()
    ws, ptr, nbytes = _ws(n, d_off.numel() - 1)
    check(lib().b200sort_segmented_sort_keys(kt, desc, p_in, p_out, tmp.data_ptr(), n, d_off.data_ptr(),
                                             d_off.numel() - 1, ptr, nbytes, stream_ptr()))
    torch.cuda.synchronize()
    if not in_place:
        assert _words(src, offset, n).tobytes() == ko.bits(keys).tobytes(), "the copy form modified its input"
    return _words(out, offset, n)


def seg_pairs(keys, vals, offsets, kt, desc, in_place):
    import torch
    n = keys.size
    dk, pk = _dev(keys)
    dv, pv = _dev(vals)
    (ok, pok), (ov, pov) = ((dk, pk), (dv, pv)) if in_place else (_dev(np.zeros(n, np.uint32)), _dev(np.zeros(n, np.int32)))
    tk = torch.empty(max(n, 1), dtype=torch.int32, device="cuda"); tv = torch.empty_like(tk)
    d_off = torch.from_numpy(np.asarray(offsets, np.int32)).cuda()
    ws, ptr, nbytes = _ws(n, d_off.numel() - 1)
    check(lib().b200sort_segmented_pairs_keys(kt, desc, pk, pv, pok, pov, tk.data_ptr(), tv.data_ptr(), n,
                                              d_off.data_ptr(), d_off.numel() - 1, ptr, nbytes, stream_ptr()))
    torch.cuda.synchronize()
    if not in_place:
        assert _words(dk, 0, n).tobytes() == ko.bits(keys).tobytes() and _words(dv, 0, n).tobytes() == ko.bits(vals).tobytes()
    return _words(ok, 0, n), _words(ov, 0, n).view(np.int32)


def mixed_keys(n: int, key_type: int, seed: int) -> np.ndarray:
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


def ragged_offsets(seed: int, total_segments: int = 3000, big: int = 2) -> np.ndarray:
    """Seeded length mix covering every class at once: many empty and one-key segments, a long tail, a few > 2^20."""
    rng = np.random.default_rng(seed)
    lens = np.concatenate([
        np.zeros(total_segments // 4, np.int64), np.ones(total_segments // 4, np.int64),
        rng.integers(2, 129, total_segments // 4), rng.integers(129, 1025, total_segments // 8),
        rng.integers(1025, 8193, total_segments // 16), rng.integers(8193, 70000, 12),
        rng.integers((1 << 20) + 1, (1 << 20) + 50000, big),
        (rng.pareto(1.2, total_segments // 16) * 50).astype(np.int64)])
    rng.shuffle(lens)
    return np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_equal_rows_every_class_boundary(order):
    kt, desc = order
    for L_ in row_lengths():
        B = max(1, min(4096, (1 << 23) // L_))
        n = B * L_
        keys = mixed_keys(n, kt, 100 + L_ % 97)
        offsets = np.arange(B + 1, dtype=np.int64) * L_
        want = seg_sort_keys(keys, offsets, kt, desc)
        for in_place in (False, True):
            assert_words(seg_keys(keys, offsets, kt, desc, in_place), want, f"L={L_} B={B} in_place={in_place}")


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_ragged_segments(order):
    kt, desc = order
    offsets = ragged_offsets(7 + kt * 2 + desc)
    n = int(offsets[-1])
    keys = mixed_keys(n, kt, 3)
    want = seg_sort_keys(keys, offsets, kt, desc)
    for in_place in (False, True):
        assert_words(seg_keys(keys, offsets, kt, desc, in_place), want, f"ragged n={n} in_place={in_place}")


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_one_segment_equals_the_1d_sort(order):
    import torch
    kt, desc = order
    for n in (5000, 300001, (1 << 21) + 7):
        keys = mixed_keys(n, kt, n)
        got = seg_keys(keys, np.array([0, n]), kt, desc, False)
        src, p = _dev(keys)
        out = torch.empty_like(src); tmp = torch.empty_like(src)
        ws, ptr, nbytes = workspace(n, ALGO_RADIX)
        check(lib().b200sort_sort_keys(ALGO_RADIX, kt, desc, p, out.data_ptr(), tmp.data_ptr(), n, ptr, nbytes, stream_ptr()))
        torch.cuda.synchronize()
        assert got.tobytes() == _words(out, 0, n).tobytes(), n


def test_more_segments_than_keys():
    rng = np.random.default_rng(3)
    n, S = 20000, 200000
    cuts = np.sort(rng.integers(0, n + 1, S - 1))
    offsets = np.concatenate([[0], cuts, [n]]).astype(np.int32)
    for kt, desc in ko.ORDERS:
        keys = mixed_keys(n, kt, 9)
        assert_words(seg_keys(keys, offsets, kt, desc, False), seg_sort_keys(keys, offsets, kt, desc), (kt, desc))


def _low_entropy(kind: str, n: int) -> np.ndarray:
    r = datagen.uniform_u32(n, 4)
    return {"all_equal": np.full(n, 0x40200000, np.uint32), "two_valued": np.where(r & 1, 0xC0000000, 0x3F800000).astype(np.uint32),
            "sorted": np.sort(r), "reverse": np.sort(r)[::-1].copy()}[kind]


@pytest.mark.parametrize("kind", ["all_equal", "two_valued", "sorted", "reverse"])
def test_low_entropy_rows(kind):
    for L_ in (16, 700, 5000, 70001):
        B = max(1, (1 << 21) // L_)
        keys = _low_entropy(kind, B * L_)
        offsets = np.arange(B + 1) * L_
        for kt, desc in ((ko.KEY_F32, 1), (ko.KEY_U32, 0), (ko.KEY_I32, 0)):
            k = keys.view(ko.DTYPES[kt])
            assert_words(seg_keys(k, offsets, kt, desc, False), seg_sort_keys(k, offsets, kt, desc), f"{kind} L={L_} {kt},{desc}")
            v = np.arange(k.size, dtype=np.int32)
            wk, wv = seg_sort_pairs(k, v, offsets, kt, desc)
            gk, gv = seg_pairs(k, v, offsets, kt, desc, False)
            assert_words(gk, wk, f"pairs {kind} L={L_}")
            assert gv.tobytes() == wv.tobytes(), f"pairs {kind} L={L_}"


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_float_specials_and_unaligned_pointers(order):
    kt, desc = order
    spec = ko.float_specials()
    offsets = ragged_offsets(11, total_segments=400, big=0)
    n = int(offsets[-1])
    keys = np.resize(spec, n).copy()
    keys[::3] = datagen.uniform_u32(keys[::3].size, n)
    keys = keys.view(ko.DTYPES[kt])
    want = seg_sort_keys(keys, offsets, kt, desc)
    for offset in (0, 1, 2, 3):
        assert_words(seg_keys(keys, offsets, kt, desc, False, offset), want, f"offset={offset}")


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_pairs_are_stable_in_every_class(order):
    kt, desc = order
    offsets = ragged_offsets(21 + kt, total_segments=2000, big=1)
    n = int(offsets[-1])
    r = datagen.uniform_u32(n, 23) % np.uint32(100)                 # many duplicates
    keys = r.astype(np.float32) if kt == ko.KEY_F32 else (r.view(np.int32) - 50 if kt == ko.KEY_I32 else r)
    vals = np.arange(n, dtype=np.int32)
    want_k, want_v = seg_sort_pairs(keys, vals, offsets, kt, desc)
    for in_place in (False, True):
        got_k, got_v = seg_pairs(keys, vals, offsets, kt, desc, in_place)
        assert_words(got_k, want_k, f"keys in_place={in_place}")
        assert got_v.tobytes() == want_v.tobytes(), f"values in_place={in_place}"


def test_pairs_keys_in_place_values_copied_is_rejected():
    import torch
    n = 1000
    k = torch.zeros(n, dtype=torch.int32, device="cuda"); v = torch.zeros_like(k); v2 = torch.zeros_like(k)
    t = torch.zeros_like(k); tv = torch.zeros_like(k)
    offs = torch.tensor([0, n], dtype=torch.int32, device="cuda")
    ws, ptr, nbytes = _ws(n, 1)
    st = lib().b200sort_segmented_pairs_keys(ko.KEY_I32, 0, k.data_ptr(), v.data_ptr(), k.data_ptr(), v2.data_ptr(),
                                             t.data_ptr(), tv.data_ptr(), n, offs.data_ptr(), 1, ptr, nbytes, stream_ptr())
    assert st == 1


def test_independent_of_the_1d_variant_and_skip_switches():
    L = lib()
    offsets = ragged_offsets(31, total_segments=1000, big=1)
    keys = mixed_keys(int(offsets[-1]), ko.KEY_F32, 2)
    base = seg_keys(keys, offsets, ko.KEY_F32, 1, False)
    try:
        assert L.b200sort_radix_set_variant(2) == 0
        L.b200sort_radix_set_skip(0)
        assert seg_keys(keys, offsets, ko.KEY_F32, 1, False).tobytes() == base.tobytes()
    finally:
        L.b200sort_radix_set_variant(0)
        L.b200sort_radix_set_skip(1)
    assert_words(base, seg_sort_keys(keys, offsets, ko.KEY_F32, 1), "reference")


def test_rank_safe_fallback_for_keys_and_pairs():
    """With B200SORT_RANK_SAFE=1 the ballot-ranked forms run, in every class, for keys and for pairs."""
    code = (
        "import sys; sys.path.insert(0, '.'); sys.path.insert(0, 'tests')\n"
        "import numpy as np\n"
        "from b200sort._lib import lib\n"
        "import key_orders as ko\n"
        "import test_segmented_gpu as t\n"
        "assert lib().b200sort_radix_atomic_order_ok() == 0\n"
        "offsets = t.ragged_offsets(41, total_segments=2000, big=1)\n"
        "n = int(offsets[-1])\n"
        "for kt, desc in ko.ORDERS:\n"
        "    k = t.mixed_keys(n, kt, kt + desc)\n"
        "    t.assert_words(t.seg_keys(k, offsets, kt, desc, False), t.seg_sort_keys(k, offsets, kt, desc), (kt, desc))\n"
        "    k = (k.view(np.uint32) % np.uint32(100)).astype(np.float32) if kt == ko.KEY_F32 else k.view(np.uint32) % np.uint32(100)\n"
        "    k = k.view(ko.DTYPES[kt])\n"
        "    v = np.arange(n, dtype=np.int32)\n"
        "    wk, wv = t.seg_sort_pairs(k, v, offsets, kt, desc)\n"
        "    gk, gv = t.seg_pairs(k, v, offsets, kt, desc, False)\n"
        "    t.assert_words(gk, wk, ('pairs', kt, desc)); assert gv.tobytes() == wv.tobytes(), ('pairs', kt, desc)\n"
        "print('ok')\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", code], cwd=root, env={**os.environ, "B200SORT_RANK_SAFE": "1"},
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


def test_launch_count_does_not_depend_on_the_number_of_segments():
    import torch
    L = lib()
    n = 1 << 20
    keys = mixed_keys(n, ko.KEY_U32, 1)
    counts = []
    for S in (1, 10 ** 6):
        offsets = (np.arange(S + 1, dtype=np.int64) * n // S).astype(np.int32)
        L.b200sort_launch_count_reset()
        got = seg_keys(keys, offsets, ko.KEY_U32, 0, False)
        counts.append(L.b200sort_launch_count())
        assert_words(got, seg_sort_keys(keys, offsets, ko.KEY_U32, 0), f"S={S}")
    torch.cuda.synchronize()
    assert counts[0] == counts[1], counts


def test_cuda_graph_capture_and_replay():
    import torch
    L = lib()
    check(L.b200sort_device_check())
    B, Lr = 64, 3000
    x = torch.empty((B, Lr), dtype=torch.float32, device="cuda")
    v = torch.arange(Lr, dtype=torch.int32, device="cuda").repeat(B).view(B, Lr)
    ko_, vo = torch.empty_like(x), torch.empty_like(v)
    kt_, vt = torch.empty_like(x), torch.empty_like(v)
    offs = (torch.arange(B + 1, dtype=torch.int32, device="cuda") * Lr)
    ws, ptr, nbytes = _ws(B * Lr, B)
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        check(L.b200sort_segmented_pairs_keys(ko.KEY_F32, 1, x.data_ptr(), v.data_ptr(), ko_.data_ptr(), vo.data_ptr(),
                                              kt_.data_ptr(), vt.data_ptr(), B * Lr, offs.data_ptr(), B, ptr, nbytes,
                                              s.cuda_stream))
    for seed in (1, 2):
        a = (datagen.uniform_u32(B * Lr, seed) % np.uint32(5000)).astype(np.float32) - np.float32(2500)
        x.copy_(torch.from_numpy(a).view(B, Lr))
        g.replay()
        torch.cuda.synchronize()
        tv, ti = torch.sort(x, dim=-1, stable=True, descending=True)
        assert torch.equal(ko_, tv) and torch.equal(vo, ti.to(torch.int32)), seed


@pytest.mark.parametrize("L_", [16, 1000, 8000, 70001])
def test_python_calls_match_torch_sort(L_):
    import torch
    B = max(1, (1 << 20) // L_)
    r = datagen.uniform_u32(B * L_, L_)
    cases = {"float32": (r % np.uint32(3000)).astype(np.float32) / np.float32(4) - np.float32(300),
             "int32": r.view(np.int32) % 5000, "uint32": r % np.uint32(5000) + np.uint32(0x7FFFF000)}
    for dtype, a in cases.items():
        x = torch.from_numpy(a).cuda().view(B, L_)
        cmp = torch.from_numpy(a.astype(np.int64) if dtype == "uint32" else a).cuda().view(B, L_)
        idx = torch.arange(L_, dtype=torch.int32, device="cuda").repeat(B).view(B, L_)
        for desc in (False, True):
            tv, ti = torch.sort(cmp, dim=-1, stable=True, descending=desc)
            k = b200sort.segmented_sort(x, descending=desc)
            assert k.shape == x.shape and torch.equal(k.to(tv.dtype), tv), (dtype, desc)
            k, v = b200sort.segmented_sort_by_key(x, idx, descending=desc)
            assert torch.equal(k.to(tv.dtype), tv) and torch.equal(v.to(torch.int64), ti), (dtype, desc)
            # the same rows through 1-D keys and offsets (int64 and int32)
            offs = torch.arange(B + 1, device="cuda") * L_
            for o in (offs, offs.to(torch.int32)):
                k1 = b200sort.segmented_sort(x.view(-1), o, descending=desc)
                assert torch.equal(k1.view(B, L_).to(tv.dtype), tv), (dtype, desc, o.dtype)
    assert x.view(-1).cpu().numpy().tobytes() == cases["uint32"].tobytes()


def test_python_call_rejects_invalid_offsets_before_any_launch():
    import torch
    L = lib()
    x = torch.zeros(100, dtype=torch.float32, device="cuda")
    bad = [[1, 100], [0, 99], [0, 101], [0, 60, 40, 100], [-1, 50, 100]]
    for b in bad:
        for dt in (torch.int32, torch.int64):
            L.b200sort_launch_count_reset()
            with pytest.raises(ValueError):
                b200sort.segmented_sort(x, torch.tensor(b, dtype=dt, device="cuda"))
            with pytest.raises(ValueError):
                b200sort.segmented_sort_by_key(x, torch.zeros(100, dtype=torch.int32, device="cuda"),
                                               torch.tensor(b, dtype=dt, device="cuda"))
            assert L.b200sort_launch_count() == 0, b
    with pytest.raises(ValueError):
        b200sort.segmented_sort(x, torch.tensor([0, 100], dtype=torch.int32))            # offsets on the CPU


def test_malformed_offsets_stay_in_bounds():
    """Through the C-ABI malformed offsets give an undefined order, but every key written lies in the output."""
    import torch
    n = 50000
    keys = mixed_keys(n, ko.KEY_U32, 77)
    for offs in ([0, 30000, 10000, 50000], [0, 60000, -5, 20000, 99999], [5, 4, 3, 2, 1, 0], [0, 40000, 9000, 45000, 50000]):
        guard = 64
        buf = torch.full((n + 2 * guard,), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
        src, p_in = _dev(keys)
        tmp = torch.full((n + 2 * guard,), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
        d_off = torch.tensor(offs, dtype=torch.int32, device="cuda")
        ws, ptr, nbytes = _ws(n, len(offs) - 1)
        check(lib().b200sort_segmented_sort_keys(ko.KEY_U32, 0, p_in, buf.data_ptr() + 4 * guard, tmp.data_ptr() + 4 * guard,
                                                 n, d_off.data_ptr(), len(offs) - 1, ptr, nbytes, stream_ptr()))
        torch.cuda.synchronize()
        for b in (buf, tmp):
            assert bool((b[:guard] == 0x5A5A5A5A).all()) and bool((b[-guard:] == 0x5A5A5A5A).all()), offs


def test_python_call_on_a_non_default_device():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible")
    dev = torch.device("cuda", torch.cuda.device_count() - 1)
    B, L_ = 300, 3001
    w = datagen.uniform_u32(B * L_, 5)
    x = torch.from_numpy(w.view(np.float32)).to(dev).view(B, L_)
    assert torch.cuda.current_device() != dev.index
    offsets = np.arange(B + 1) * L_
    got = b200sort.segmented_sort(x, descending=True)
    assert got.device == dev
    assert_words(got.cpu().numpy().reshape(-1).view(np.uint32), seg_sort_keys(w.view(np.float32), offsets, ko.KEY_F32, 1), "keys")
    v = torch.arange(L_, dtype=torch.int32, device=dev).repeat(B).view(B, L_)
    k, vv = b200sort.segmented_sort_by_key(x, v)
    wk, wv = seg_sort_pairs(w.view(np.float32), np.tile(np.arange(L_, dtype=np.int32), B), offsets, ko.KEY_F32, 0)
    assert_words(k.cpu().numpy().reshape(-1).view(np.uint32), wk, "pairs keys")
    assert vv.cpu().numpy().reshape(-1).tobytes() == wv.tobytes()


def _check_sorted_segments(out, offs, kt, desc):
    """Every segment sorted in the image domain, with torch ops: no descent inside a segment."""
    import torch
    neg, pos = ko.MASKS[(kt, desc)]
    o64 = out.to(torch.int64) & 0xFFFFFFFF
    img = o64 ^ torch.where(o64 >= 2 ** 31, torch.tensor(neg, device="cuda"), torch.tensor(pos, device="cuda"))
    descent = img[1:] < img[:-1]
    del img, o64
    starts = torch.zeros(out.numel(), dtype=torch.bool, device="cuda")
    starts[offs[1:-1].to(torch.int64)] = True
    return not bool((descent & ~starts[1:]).any().item())


@pytest.mark.parametrize("layout", ["rows_2_17", "ragged"])
def test_full_size_2_28(layout):
    import torch
    n = 1 << 28
    if layout == "rows_2_17":
        offs = torch.arange(0, n + 1, 1 << 17, dtype=torch.int32, device="cuda")
    else:
        o = ragged_offsets(99, total_segments=200000, big=8)
        o = o[o < n]
        offs = torch.from_numpy(np.concatenate([o, [n]]).astype(np.int32)).cuda()
    S = offs.numel() - 1
    g = torch.Generator(device="cuda"); g.manual_seed(12)
    x = torch.randint(-2**31, 2**31, (n,), dtype=torch.int64, device="cuda", generator=g).to(torch.int32)
    fp_in = oracle.multiset_fingerprint(x.cpu().numpy())
    out = torch.empty_like(x); tmp = torch.empty_like(x)
    ws, ptr, nbytes = _ws(n, S)
    for kt, desc in ((ko.KEY_F32, 1), (ko.KEY_U32, 0)):
        check(lib().b200sort_segmented_sort_keys(kt, desc, x.data_ptr(), out.data_ptr(), tmp.data_ptr(), n,
                                                 offs.data_ptr(), S, ptr, nbytes, stream_ptr()))
        torch.cuda.synchronize()
        assert _check_sorted_segments(out, offs, kt, desc), (layout, kt, desc)
        assert oracle.multiset_fingerprint(out.cpu().numpy()) == fp_in, (layout, kt, desc)
    # each segment's multiset is its own: a segment-wise sum of the keys is unchanged
    seg = torch.repeat_interleave(torch.arange(S, device="cuda"), (offs[1:] - offs[:-1]).to(torch.int64))
    a = torch.zeros(S, dtype=torch.int64, device="cuda").index_add_(0, seg, x.to(torch.int64))
    b = torch.zeros(S, dtype=torch.int64, device="cuda").index_add_(0, seg, out.to(torch.int64))
    assert torch.equal(a, b)
