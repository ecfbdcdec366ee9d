"""Segmented sort of 16-bit keys on the GPU (b200sort_segmented_sort_keys16, b200sort_segmented_pairs_keys16 and the
torch-facing b200sort.segmented_sort16 / segmented_sort16_by_key), byte for byte against the numpy reference of
tests/test_segmented16_cpu.py."""
import os
import subprocess
import sys

import numpy as np
import pytest

import b200sort
from b200sort import datagen
from b200sort._lib import check, lib
from helpers import stream_ptr

import key_orders16 as ko
from test_segmented16_cpu import seg_sort_keys, seg_sort_pairs
from test_segmented_gpu import ragged_offsets

pytestmark = pytest.mark.gpu

ORDER_IDS = [f"{ko.NAMES[k]}_{'desc' if d else 'asc'}" for k, d in ko.ORDERS]
TILE = 8192          # keys per tile of the segmented onesweep (kSeg16Tile, csrc/segmented16.cuh)
GUARD = 0x5A5A


def _class_bounds():
    L = lib()
    out, c = [], 0
    while L.b200sort_segmented16_class_max(c):
        out.append(L.b200sort_segmented16_class_max(c))
        c += 1
    return out


def row_lengths():
    ls = {1, 2, 31, 32, 33, TILE - 1, TILE, TILE + 1, 2 * TILE + 1, 65537, (1 << 20) + 3}
    for m in _class_bounds():
        ls |= {m - 1, m, m + 1}
    return sorted(x for x in ls if x >= 1)


def _dev(a: np.ndarray, offset: int = 0, guard: int = 0):
    """A device buffer of 2-byte words holding ``a`` at word ``offset`` + ``guard``, GUARD words around it."""
    import torch
    words = ko.bits(a) if a.dtype.itemsize == 2 else np.ascontiguousarray(a).view(np.uint16)
    buf = torch.full((words.size + offset + 2 * guard + 2,), GUARD, dtype=torch.int16, device="cuda")
    at = offset + guard
    buf[at:at + words.size] = torch.from_numpy(words.view(np.int16)).cuda()
    return buf, buf.data_ptr() + 2 * at


def _words(buf, offset: int, n: int) -> np.ndarray:
    return buf[offset:offset + n].cpu().numpy().view(np.uint16)


def _ws(n: int, segments: int):
    import torch
    nbytes = lib().b200sort_segmented16_workspace_bytes(n, segments)
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
    return ws, ws.data_ptr() + (-ws.data_ptr()) % 256, nbytes


def seg_keys(keys, offsets, kt, desc, in_place, offset=0):
    """The library's result as uint16 words; checks the copy form leaves its input alone."""
    import torch
    n = keys.size
    src, p_in = _dev(keys, offset)
    out, p_out = (src, p_in) if in_place else _dev(np.full(n, 0xA5A5, np.uint16), offset)
    tmp, p_tmp = _dev(np.zeros(max(n, 1), np.uint16), offset)
    d_off = torch.from_numpy(np.asarray(offsets, np.int32)).cuda()
    ws, ptr, nbytes = _ws(n, d_off.numel() - 1)
    check(lib().b200sort_segmented_sort_keys16(kt, desc, p_in, p_out, p_tmp, n, d_off.data_ptr(), d_off.numel() - 1,
                                               ptr, nbytes, stream_ptr()))
    torch.cuda.synchronize()
    if not in_place:
        assert _words(src, offset, n).tobytes() == ko.bits(keys).tobytes(), "the copy form modified its input"
    return _words(out, offset, n)


def seg_pairs(keys, vals, offsets, kt, desc, in_place, offset=0):
    import torch
    n = keys.size
    dk, pk = _dev(keys, offset)
    dv = torch.from_numpy(np.ascontiguousarray(vals, np.int32)).cuda()
    if in_place:
        ok_, pok, ov = dk, pk, dv
    else:
        (ok_, pok), ov = _dev(np.zeros(n, np.uint16), offset), torch.zeros_like(dv)
    tk, ptk = _dev(np.zeros(max(n, 1), np.uint16), offset)
    tv = torch.empty(max(n, 1), dtype=torch.int32, device="cuda")
    d_off = torch.from_numpy(np.asarray(offsets, np.int32)).cuda()
    ws, ptr, nbytes = _ws(n, d_off.numel() - 1)
    check(lib().b200sort_segmented_pairs_keys16(kt, desc, pk, dv.data_ptr(), pok, ov.data_ptr(), ptk, tv.data_ptr(), n,
                                                d_off.data_ptr(), d_off.numel() - 1, ptr, nbytes, stream_ptr()))
    torch.cuda.synchronize()
    if not in_place:
        assert _words(dk, offset, n).tobytes() == ko.bits(keys).tobytes(), "the copy form modified its keys"
        assert dv.cpu().numpy().tobytes() == np.ascontiguousarray(vals, np.int32).tobytes(), "... its values"
    return _words(ok_, offset, n), ov.cpu().numpy()


def mixed_keys(n: int, key_type: int, seed: int) -> np.ndarray:
    w = datagen.uniform_u32(n, seed).astype(np.uint16)
    if key_type in (ko.KEY_F16, ko.KEY_BF16) and n:
        spec = ko.float_specials(key_type)
        pos = datagen.uniform_u32(min(n, 4 * spec.size), seed + 1) % np.uint32(n)
        w[pos] = np.resize(spec, pos.size)
    return w.view(ko.DTYPES[key_type])


def assert_words(got: np.ndarray, want: np.ndarray, what):
    want = ko.bits(want)
    if got.tobytes() != want.tobytes():
        bad = np.flatnonzero(got != want)
        raise AssertionError(f"{what}: {bad.size} of {got.size} words differ, first at {bad[0]}: "
                             f"got {got[bad[0]]:#06x}, want {want[bad[0]]:#06x}")


def check_pairs(keys, offsets, kt, desc, in_place, what, offset=0):
    vals = np.arange(keys.size, dtype=np.int32)
    wk, wv = seg_sort_pairs(keys, vals, offsets, kt, desc)
    gk, gv = seg_pairs(keys, vals, offsets, kt, desc, in_place, offset)
    assert_words(gk, wk, f"pairs keys {what}")
    assert gv.tobytes() == wv.tobytes(), f"pairs values {what}"


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_equal_rows_every_class_boundary(order):
    kt, desc = order
    for L_ in row_lengths():
        B = max(1, min(4096, (1 << 22) // L_))
        n = B * L_
        keys = mixed_keys(n, kt, 100 + L_ % 97)
        offsets = np.arange(B + 1, dtype=np.int64) * L_
        want = seg_sort_keys(keys, offsets, kt, desc)
        for in_place in (False, True):
            assert_words(seg_keys(keys, offsets, kt, desc, in_place), want, f"L={L_} B={B} in_place={in_place}")
            check_pairs(keys, offsets, kt, desc, in_place, f"L={L_} B={B} in_place={in_place}")


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_ragged_segments(order):
    kt, desc = order
    offsets = ragged_offsets(7 + kt * 2 + desc)
    n = int(offsets[-1])
    keys = mixed_keys(n, kt, 3)
    want = seg_sort_keys(keys, offsets, kt, desc)
    for in_place in (False, True):
        assert_words(seg_keys(keys, offsets, kt, desc, in_place), want, f"ragged n={n} in_place={in_place}")
        check_pairs(keys, offsets, kt, desc, in_place, f"ragged n={n} in_place={in_place}")


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_one_segment_equals_the_1d_sort(order):
    import torch
    kt, desc = order
    dt = {ko.KEY_I16: torch.int16, ko.KEY_U16: torch.uint16, ko.KEY_F16: torch.float16, ko.KEY_BF16: torch.bfloat16}[kt]
    for n in (5000, 300001, (1 << 21) + 7):
        keys = mixed_keys(n, kt, n)
        got = seg_keys(keys, np.array([0, n]), kt, desc, False)
        x = torch.from_numpy(ko.bits(keys).view(np.int16)).cuda().view(dt)
        want = b200sort.sort16(x, descending=bool(desc))
        assert got.tobytes() == want.view(torch.int16).cpu().numpy().tobytes(), n
        v = torch.arange(n, dtype=torch.int32, device="cuda")
        wk, wv = b200sort.sort16_by_key(x, v, descending=bool(desc))
        gk, gv = seg_pairs(keys, np.arange(n, dtype=np.int32), np.array([0, n]), kt, desc, False)
        assert gk.tobytes() == wk.view(torch.int16).cpu().numpy().tobytes() and gv.tobytes() == wv.cpu().numpy().tobytes()


def test_more_segments_than_keys():
    rng = np.random.default_rng(3)
    n, S = 20000, 200000
    cuts = np.sort(rng.integers(0, n + 1, S - 1))
    offsets = np.concatenate([[0], cuts, [n]]).astype(np.int32)
    for kt, desc in ko.ORDERS:
        keys = mixed_keys(n, kt, 9)
        assert_words(seg_keys(keys, offsets, kt, desc, False), seg_sort_keys(keys, offsets, kt, desc), (kt, desc))
        check_pairs(keys, offsets, kt, desc, False, (kt, desc))


def _low_entropy(kind: str, n: int) -> np.ndarray:
    r = datagen.uniform_u32(n, 4)
    if kind == "all_equal":
        return np.full(n, 0x4049, np.uint16)
    if kind == "int16_pm100":
        return ((r % np.uint32(201)).astype(np.int32) - 100).astype(np.int16).view(np.uint16)
    hot = np.full(n, 0x3F80, np.uint16)                        # one hot value, 1 key in 64 different
    idx = np.flatnonzero(r % np.uint32(64) == 0)
    hot[idx] = r[idx].astype(np.uint16)
    return hot


@pytest.mark.parametrize("kind", ["all_equal", "int16_pm100", "one_hot"])
def test_low_entropy_rows(kind):
    for L_ in (16, 700, 5000, 70001):
        B = max(1, (1 << 21) // L_)
        keys = _low_entropy(kind, B * L_)
        offsets = np.arange(B + 1) * L_
        for kt, desc in ((ko.KEY_BF16, 1), (ko.KEY_U16, 0), (ko.KEY_I16, 0), (ko.KEY_F16, 1)):
            k = keys.view(ko.DTYPES[kt])
            assert_words(seg_keys(k, offsets, kt, desc, False), seg_sort_keys(k, offsets, kt, desc), f"{kind} L={L_} {kt},{desc}")
            check_pairs(k, offsets, kt, desc, False, f"{kind} L={L_} {kt},{desc}")


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_float_specials_and_unaligned_pointers(order):
    kt, desc = order
    spec = ko.float_specials(ko.KEY_BF16 if kt == ko.KEY_BF16 else ko.KEY_F16)
    offsets = ragged_offsets(11, total_segments=400, big=0)
    n = int(offsets[-1])
    keys = np.resize(spec, n).copy()
    keys[::3] = datagen.uniform_u32(keys[::3].size, n).astype(np.uint16)
    keys = keys.view(ko.DTYPES[kt])
    want = seg_sort_keys(keys, offsets, kt, desc)
    for offset in (0, 1, 3, 9):            # words: 2 bytes past a 4-byte boundary (1), past 8 (3), past 16 (9)
        assert_words(seg_keys(keys, offsets, kt, desc, False, offset), want, f"offset={offset}")
        check_pairs(keys, offsets, kt, desc, False, f"offset={offset}", offset)


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_pairs_are_stable_in_every_class(order):
    kt, desc = order
    offsets = ragged_offsets(21 + kt, total_segments=2000, big=1)
    n = int(offsets[-1])
    r = (datagen.uniform_u32(n, 23) % np.uint32(100)).astype(np.uint16)      # many duplicates
    keys = {ko.KEY_I16: (r.astype(np.int16) - 50), ko.KEY_U16: r,
            ko.KEY_F16: r.astype(np.float16), ko.KEY_BF16: ko.bf16_bits(r.astype(np.float32))}[kt]
    for in_place in (False, True):
        check_pairs(keys, offsets, kt, desc, in_place, f"in_place={in_place}")


def test_pairs_keys_in_place_values_copied_is_rejected():
    import torch
    n = 1000
    k = torch.zeros(n, dtype=torch.int16, device="cuda"); t = torch.zeros_like(k)
    v = torch.zeros(n, dtype=torch.int32, device="cuda"); v2 = torch.zeros_like(v); tv = torch.zeros_like(v)
    offs = torch.tensor([0, n], dtype=torch.int32, device="cuda")
    ws, ptr, nbytes = _ws(n, 1)
    L = lib()
    L.b200sort_launch_count_reset()
    st = L.b200sort_segmented_pairs_keys16(ko.KEY_I16, 0, k.data_ptr(), v.data_ptr(), k.data_ptr(), v2.data_ptr(),
                                           t.data_ptr(), tv.data_ptr(), n, offs.data_ptr(), 1, ptr, nbytes, stream_ptr())
    assert st == 1 and L.b200sort_launch_count() == 0


def test_independent_of_the_1d_variant_and_skip_switches():
    L = lib()
    offsets = ragged_offsets(31, total_segments=1000, big=1)
    keys = mixed_keys(int(offsets[-1]), ko.KEY_BF16, 2)
    base = seg_keys(keys, offsets, ko.KEY_BF16, 1, False)
    vals = np.arange(keys.size, dtype=np.int32)
    bk, bv = seg_pairs(keys, vals, offsets, ko.KEY_BF16, 1, False)
    try:
        assert L.b200sort_radix_set_variant(2) == 0
        L.b200sort_radix_set_skip(0)
        assert seg_keys(keys, offsets, ko.KEY_BF16, 1, False).tobytes() == base.tobytes()
        gk, gv = seg_pairs(keys, vals, offsets, ko.KEY_BF16, 1, False)
        assert gk.tobytes() == bk.tobytes() and gv.tobytes() == bv.tobytes()
    finally:
        L.b200sort_radix_set_variant(0)
        L.b200sort_radix_set_skip(1)
    assert_words(base, seg_sort_keys(keys, offsets, ko.KEY_BF16, 1), "reference")


def test_rank_safe_fallback_gives_the_same_bytes():
    """With B200SORT_RANK_SAFE=1 the ballot-ranked forms run, in every class, for keys and for pairs."""
    code = (
        "import sys; sys.path.insert(0, '.'); sys.path.insert(0, 'tests')\n"
        "import numpy as np\n"
        "from b200sort._lib import lib\n"
        "import key_orders16 as ko\n"
        "import test_segmented16_gpu as t\n"
        "assert lib().b200sort_radix_atomic_order_ok() == 0\n"
        "offsets = t.ragged_offsets(41, total_segments=2000, big=1)\n"
        "n = int(offsets[-1])\n"
        "for kt, desc in ko.ORDERS:\n"
        "    k = t.mixed_keys(n, kt, kt + desc)\n"
        "    t.assert_words(t.seg_keys(k, offsets, kt, desc, False), t.seg_sort_keys(k, offsets, kt, desc), (kt, desc))\n"
        "    k = (k.view(np.uint16) % np.uint16(100)).view(ko.DTYPES[kt])\n"
        "    t.check_pairs(k, offsets, kt, desc, False, ('pairs', kt, desc))\n"
        "print('ok')\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", code], cwd=root, env={**os.environ, "B200SORT_RANK_SAFE": "1"},
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


def test_launch_count_does_not_depend_on_the_number_of_segments():
    L = lib()
    n = 1 << 20
    keys = mixed_keys(n, ko.KEY_U16, 1)
    counts = []
    for S in (1, 1000, 10 ** 6):
        offsets = (np.arange(S + 1, dtype=np.int64) * n // S).astype(np.int32)
        for pairs in (False, True):
            L.b200sort_launch_count_reset()
            if pairs:
                check_pairs(keys, offsets, ko.KEY_U16, 0, False, f"S={S}")
            else:
                assert_words(seg_keys(keys, offsets, ko.KEY_U16, 0, False), seg_sort_keys(keys, offsets, ko.KEY_U16, 0),
                             f"S={S}")
            counts.append((pairs, L.b200sort_launch_count()))
    assert len(set(counts)) == 2, counts


def test_cuda_graph_capture_and_replay():
    import torch
    L = lib()
    check(L.b200sort_device_check())
    B, Lr = 64, 3000
    x = torch.empty((B, Lr), dtype=torch.bfloat16, device="cuda")
    v = torch.arange(Lr, dtype=torch.int32, device="cuda").repeat(B).view(B, Lr)
    ko_, vo = torch.empty_like(x), torch.empty_like(v)
    kt_, vt = torch.empty_like(x), torch.empty_like(v)
    offs = (torch.arange(B + 1, dtype=torch.int32, device="cuda") * Lr)
    ws, ptr, nbytes = _ws(B * Lr, B)
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        check(L.b200sort_segmented_pairs_keys16(ko.KEY_BF16, 1, x.data_ptr(), v.data_ptr(), ko_.data_ptr(),
                                                vo.data_ptr(), kt_.data_ptr(), vt.data_ptr(), B * Lr, offs.data_ptr(), B,
                                                ptr, nbytes, s.cuda_stream))
    for seed in (1, 2):
        a = (datagen.uniform_u32(B * Lr, seed) % np.uint32(500)).astype(np.float32) - np.float32(250.5)
        x.copy_(torch.from_numpy(a).view(B, Lr))
        g.replay()
        torch.cuda.synchronize()
        tv, ti = torch.sort(x, dim=-1, stable=True, descending=True)
        assert torch.equal(ko_, tv) and torch.equal(vo, ti.to(torch.int32)), seed


def _normal_rows(torch, B, L_, dtype, seed):
    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    x = torch.randn((B, L_), device="cuda", generator=g).to(dtype)
    return torch.where(x == 0, torch.ones_like(x), x)                 # no +-0.0: torch.sort treats them as equal


@pytest.mark.parametrize("L_", [8, 64, 256, 1024, 32000, 128256])
def test_python_calls_match_torch_sort(L_):
    import torch
    B = max(1, (1 << 22) // L_)
    idx = torch.arange(L_, dtype=torch.int32, device="cuda").repeat(B).view(B, L_)
    for dtype in (torch.bfloat16, torch.float16):
        x = _normal_rows(torch, B, L_, dtype, L_)
        pristine = x.clone()
        for desc in (True, False):
            tv, ti = torch.sort(x, dim=-1, stable=True, descending=desc)
            k = b200sort.segmented_sort16(x, descending=desc)
            assert k.shape == x.shape and k.dtype == dtype and torch.equal(k, tv), (dtype, desc)
            k, v = b200sort.segmented_sort16_by_key(x, idx, descending=desc)
            assert torch.equal(k, tv) and torch.equal(v, ti.to(torch.int32)), (dtype, desc)
            offs = torch.arange(B + 1, device="cuda") * L_                   # the same rows as 1-D keys and offsets
            for o in (offs, offs.to(torch.int32)):
                k1, v1 = b200sort.segmented_sort16_by_key(x.view(-1), idx.view(-1), o, descending=desc)
                assert torch.equal(k1.view(B, L_), tv) and torch.equal(v1.view(B, L_), ti.to(torch.int32)), (dtype, o.dtype)
        assert torch.equal(x.view(torch.int16), pristine.view(torch.int16))
    for dtype in (torch.int16, torch.uint16):
        x = torch.from_numpy((datagen.uniform_u32(B * L_, 3) % np.uint32(3000)).astype(np.int16)).cuda().view(B, L_)
        x = x.view(dtype)
        tv, ti = torch.sort(x.to(torch.int32), dim=-1, stable=True, descending=True)
        k, v = b200sort.segmented_sort16_by_key(x, idx, descending=True)
        assert torch.equal(k.to(torch.int32), tv) and torch.equal(v, ti.to(torch.int32)), dtype


def test_python_call_rejects_invalid_offsets_before_any_launch():
    import torch
    L = lib()
    x = torch.zeros(100, dtype=torch.bfloat16, device="cuda")
    bad = [[1, 100], [0, 99], [0, 101], [0, 60, 40, 100], [-1, 50, 100]]
    for b in bad:
        for dt in (torch.int32, torch.int64):
            L.b200sort_launch_count_reset()
            with pytest.raises(ValueError):
                b200sort.segmented_sort16(x, torch.tensor(b, dtype=dt, device="cuda"))
            with pytest.raises(ValueError):
                b200sort.segmented_sort16_by_key(x, torch.zeros(100, dtype=torch.int32, device="cuda"),
                                                 torch.tensor(b, dtype=dt, device="cuda"))
            assert L.b200sort_launch_count() == 0, b
    with pytest.raises(ValueError):
        b200sort.segmented_sort16(x, torch.tensor([0, 100], dtype=torch.int32))            # offsets on the CPU


def test_malformed_offsets_stay_in_bounds():
    """Through the C-ABI malformed offsets give an undefined order, but every key and value written lies in the
    output: the guard words around out and tmp are untouched."""
    import torch
    n, g = 50000, 64
    keys = mixed_keys(n, ko.KEY_U16, 77)
    cases = ([0, 30000, 10000, 50000], [0, 60000, -5, 20000, 99999], [5, 4, 3, 2, 1, 0], [0, 40000, 9000, 45000, 50000],
             [0, 9000, 3, 20000, 19000, 50000])
    for offs in cases:
        src, p_in = _dev(keys)
        out, p_out = _dev(np.zeros(n, np.uint16), 0, g)
        tmp, p_tmp = _dev(np.zeros(n, np.uint16), 0, g)
        vin = torch.arange(n, dtype=torch.int32, device="cuda")
        vout = torch.full((n + 2 * g,), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
        vtmp = torch.full((n + 2 * g,), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
        d_off = torch.tensor(offs, dtype=torch.int32, device="cuda")
        ws, ptr, nbytes = _ws(n, len(offs) - 1)
        check(lib().b200sort_segmented_sort_keys16(ko.KEY_U16, 0, p_in, p_out, p_tmp, n, d_off.data_ptr(), len(offs) - 1,
                                                   ptr, nbytes, stream_ptr()))
        check(lib().b200sort_segmented_pairs_keys16(ko.KEY_U16, 1, p_in, vin.data_ptr(), p_out, vout.data_ptr() + 4 * g,
                                                    p_tmp, vtmp.data_ptr() + 4 * g, n, d_off.data_ptr(), len(offs) - 1,
                                                    ptr, nbytes, stream_ptr()))
        torch.cuda.synchronize()
        for b in (out, tmp):
            assert bool((b[:g] == GUARD).all()) and bool((b[g + n:] == GUARD).all()), offs
        for b in (vout, vtmp):
            assert bool((b[:g] == 0x5A5A5A5A).all()) and bool((b[-g:] == 0x5A5A5A5A).all()), offs


def test_python_call_on_a_non_default_device():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible")
    dev = torch.device("cuda", torch.cuda.device_count() - 1)
    B, L_ = 300, 3001
    w = datagen.uniform_u32(B * L_, 5).astype(np.uint16)
    x = torch.from_numpy(w.view(np.int16)).to(dev).view(B, L_).view(torch.bfloat16)
    assert torch.cuda.current_device() != dev.index
    offsets = np.arange(B + 1) * L_
    got = b200sort.segmented_sort16(x, descending=True)
    assert got.device == dev
    assert_words(got.view(torch.int16).cpu().numpy().reshape(-1).view(np.uint16),
                 seg_sort_keys(w, offsets, ko.KEY_BF16, 1), "keys")
    v = torch.arange(L_, dtype=torch.int32, device=dev).repeat(B).view(B, L_)
    k, vv = b200sort.segmented_sort16_by_key(x, v)
    wk, wv = seg_sort_pairs(w, np.tile(np.arange(L_, dtype=np.int32), B), offsets, ko.KEY_BF16, 0)
    assert_words(k.view(torch.int16).cpu().numpy().reshape(-1).view(np.uint16), wk, "pairs keys")
    assert vv.cpu().numpy().reshape(-1).tobytes() == wv.tobytes()


@pytest.mark.parametrize("layout", ["rows_2_17", "rows_128256"])
def test_full_size_2_28(layout):
    """2^28 bfloat16 keys in rows, descending pairs: every row sorted, a permutation of its row, stable."""
    import torch
    n = 1 << 28
    L_ = 1 << 17 if layout == "rows_2_17" else 128256
    B = n // L_
    n = B * L_
    g = torch.Generator(device="cuda"); g.manual_seed(12)
    x = torch.randint(-2**15, 2**15, (n,), dtype=torch.int32, device="cuda", generator=g).to(torch.int16)
    v = torch.arange(L_, dtype=torch.int32, device="cuda").repeat(B)
    k, vo = b200sort.segmented_sort16_by_key(x.view(torch.bfloat16), v, torch.arange(B + 1, device="cuda") * L_,
                                             descending=True)
    torch.cuda.synchronize()
    k = k.view(torch.int16).view(B, L_).to(torch.int32) & 0xFFFF
    neg, pos = ko.MASKS[(ko.KEY_BF16, 1)]
    img = k ^ torch.where(k >= 0x8000, torch.tensor(neg, device="cuda"), torch.tensor(pos, device="cuda"))
    vo = vo.view(B, L_)
    assert not bool((img[:, 1:] < img[:, :-1]).any()), "a row is not sorted"
    ties = img[:, 1:] == img[:, :-1]
    assert not bool((ties & (vo[:, 1:] <= vo[:, :-1])).any()), "equal keys out of input order"
    del img, ties
    assert torch.equal(torch.sort(vo, dim=-1)[0], v.view(B, L_)), "values are not a permutation of each row"
    assert torch.equal(torch.gather(x.view(B, L_).to(torch.int32) & 0xFFFF, 1, vo.to(torch.int64)), k)
