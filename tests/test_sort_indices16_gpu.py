"""Sort with indices of 16-bit keys on the GPU (b200sort_radix_sort_indices_keys16,
b200sort_segmented_sort_indices_keys16 and the torch-facing b200sort.sort16_with_indices /
segmented_sort16_with_indices): keys byte for byte and int64 indices exactly against the numpy reference of
tests/test_sort_indices16_cpu.py, and against torch.sort.

Every C-ABI call here writes into canary-guarded buffers (digit_patterns.DevBuf) whose arrays start out holding
canaries too, so the index output must be fully overwritten, nothing may be written around any output or scratch
buffer, and garbage in the scratch buffers must change nothing.  The 1-D and segmented calls share one workspace
that is filled with 0xFF once and never cleared."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import b200sort
from b200sort import datagen
from b200sort._lib import check, lib
from helpers import stream_ptr

import digit_patterns as dp
import key_orders16 as ko
from test_segmented_gpu import ragged_offsets
from test_segmented16_gpu import mixed_keys
from test_sort_indices16_cpu import sort16_indices_ref

pytestmark = pytest.mark.gpu

ORDER_IDS = [f"{ko.NAMES[k]}_{'desc' if d else 'asc'}" for k, d in ko.ORDERS]
TILE = 8192                        # keys per tile of the 1-D and segmented passes (csrc/radix16.cu, segmented16.cuh)
MAX_1D = (1 << 20) + 7
MAX_SEG_N, MAX_SEG_S = 1 << 22, 1 << 22
CLAMP_SITE = 15                    # the check site that counts clamped destinations of malformed offsets

_WS = None
_STATE = {"start": 0, "clamps": 0}


def shared_ws():
    """The module's never-cleared workspace, sized for every call below but the 2^28-key ones."""
    global _WS
    if _WS is None:
        L = lib()
        _WS = dp.Workspace(max(L.b200sort_keys16_workspace_bytes(MAX_1D),
                               L.b200sort_segmented16_workspace_bytes(MAX_SEG_N, MAX_SEG_S)))
    return _WS


def _sites():
    sites = (ctypes.c_ulonglong * 16)()
    lib().b200sort_debug_check_failures_by_site(ctypes.cast(sites, ctypes.c_void_p))
    return list(sites)


@pytest.fixture(scope="module", autouse=True)
def _module_checks():
    L = lib()
    if L.b200sort_debug_checked_build():
        _STATE["start"] = L.b200sort_debug_check_failures()
    yield
    if _WS is not None:
        _WS.check_tail()
    if L.b200sort_debug_checked_build():
        assert L.b200sort_debug_check_failures() - _STATE["start"] == _STATE["clamps"]


def _call(seg, keys, kt, desc, in_place, offsets=None, word_offset=0):
    """One guarded call; returns (sorted key words, int64 indices).  word_offset: the keys' 2-byte words past a
    16-byte boundary."""
    import torch
    L = lib()
    n = keys.size
    kin = dp.DevBuf(n, word_offset, 2, 1).load(ko.bits(keys))
    kout = kin if in_place else dp.DevBuf(n, (word_offset + 2) % 8, 2, 2).load()
    idx = dp.DevBuf(n, 2 * (word_offset & 1), 8, 3).load()
    tk = dp.DevBuf(n, (word_offset + 5) % 8, 2, 4).load()
    ti = dp.DevBuf(n, word_offset % 4, 4, 5).load()
    ws = shared_ws()
    if seg:
        d_off = torch.from_numpy(np.asarray(offsets, np.int32)).cuda()
        S = d_off.numel() - 1
        nbytes = L.b200sort_segmented16_workspace_bytes(n, S)
        assert nbytes <= ws.cap - ws.GUARD
        before = ws.guard(nbytes).clone()
        check(L.b200sort_segmented_sort_indices_keys16(kt, desc, kin.ptr, kout.ptr, idx.ptr, tk.ptr, ti.ptr, n,
                                                       d_off.data_ptr(), S, ws.ptr, nbytes, stream_ptr()))
    else:
        nbytes = L.b200sort_keys16_workspace_bytes(n)
        assert nbytes <= ws.cap - ws.GUARD
        before = ws.guard(nbytes).clone()
        check(L.b200sort_radix_sort_indices_keys16(kt, desc, kin.ptr, kout.ptr, idx.ptr, tk.ptr, ti.ptr, n,
                                                   ws.ptr, nbytes, stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(ws.guard(nbytes), before), "workspace written past ws_bytes"
    tk.read("tmp keys"); ti.read("tmp indices")
    if not in_place:
        assert kin.read("keys in").tobytes() == ko.bits(keys).tobytes(), "the copy form modified its input"
    return kout.read("keys out"), idx.read("indices").view(np.int64)


def check_1d(keys, kt, desc, in_place, what="", word_offset=0):
    gk, gi = _call(False, keys, kt, desc, in_place, word_offset=word_offset)
    wk, wi = sort16_indices_ref(keys, [0, keys.size], kt, desc)
    assert gk.tobytes() == ko.bits(wk).tobytes(), f"{what}: keys differ"
    assert gi.tobytes() == wi.tobytes(), f"{what}: indices differ at {np.flatnonzero(gi != wi)[:5]}"
    return gk, gi


def check_seg(keys, offsets, kt, desc, in_place, what="", word_offset=0):
    gk, gi = _call(True, keys, kt, desc, in_place, offsets=offsets, word_offset=word_offset)
    wk, wi = sort16_indices_ref(keys, offsets, kt, desc)
    assert gk.tobytes() == ko.bits(wk).tobytes(), f"{what}: keys differ"
    assert gi.tobytes() == wi.tobytes(), f"{what}: indices differ at {np.flatnonzero(gi != wi)[:5]}"
    return gk, gi


def dup_keys(n, kt, seed, distinct=300):
    """Keys with many ties, so that stability shows in the indices."""
    w = (datagen.uniform_u32(n, seed) % np.uint32(distinct)).astype(np.uint16) * np.uint16(0x0101)
    return w.view(ko.DTYPES[kt])


def plan_keys(n, S, order, seed):
    """Keys of `order` whose image byte p (pass p: 0 low, 1 high) takes one value over all keys exactly for p in S,
    so the 1-D sort skips exactly those passes (n >= 2)."""
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 1 << 16, n, dtype=np.uint32).astype(np.uint16)
    for p in (0, 1):
        sh = np.uint16(8 * p)
        if p in S:
            c = np.uint16(int(rng.integers(0, 256)) << (8 * p))
            img = (img & ~np.uint16(0xFF << (8 * p))) | c
        elif bool((((img >> sh) & np.uint16(0xFF)) == ((img[0] >> sh) & np.uint16(0xFF))).all()):
            img[1] ^= np.uint16(1 << (8 * p))
    return ko.inverse(img, *order)


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_1d_orders_and_sizes_in_place_and_copied(order):
    kt, desc = order
    for n in (0, 1, 2, TILE - 1, TILE, TILE + 1, (1 << 16) + 3, MAX_1D):
        for in_place in (False, True):
            for i, keys in enumerate((mixed_keys(n, kt, n + kt), dup_keys(n, kt, n + desc))):
                check_1d(keys, kt, desc, in_place, f"n={n} in_place={in_place} set {i}",
                         word_offset=(1, 3, 5, 7)[(n + i) % 4])


@pytest.mark.parametrize("n", [TILE + 1, (1 << 16) + 3])
def test_every_pass_plan(n):
    """Keys whose image bytes are constant in exactly the passes of S, for every S, in place and copied: both passes
    (the int32 indices go through tmp_idx), one (made and stored as int64 by the same pass, also in place where the
    keys land in tmp), and none (the final kernel writes 0..n-1)."""
    for m, S in enumerate((set(), {0}, {1}, {0, 1})):
        for kt, desc in ko.ORDERS:
            keys = plan_keys(n, S, (kt, desc), seed=m * 8 + kt + desc)
            for in_place in (False, True):
                check_1d(keys, kt, desc, in_place, f"constant passes {sorted(S)} in_place={in_place}",
                         word_offset=m)
    for in_place in (False, True):
        keys = np.full(n, 0x3F80, np.uint16).view(ko.DTYPES[ko.KEY_BF16])       # all keys equal: the identity
        gk, gi = check_1d(keys, ko.KEY_BF16, 1, in_place, "all equal")
        assert gi.tobytes() == np.arange(n, dtype=np.int64).tobytes()


def test_skipping_off():
    L = lib()
    try:
        L.b200sort_radix_set_skip(0)
        for m, S in enumerate((set(), {0}, {1}, {0, 1})):
            keys = plan_keys((1 << 16) + 3, S, (ko.KEY_F16, 1), seed=m)
            for in_place in (False, True):
                check_1d(keys, ko.KEY_F16, 1, in_place, f"skip off, constant {sorted(S)}")
    finally:
        L.b200sort_radix_set_skip(1)


def test_rank_safe_fallback():
    """With B200SORT_RANK_SAFE=1 the ballot-ranked passes and classes give the same bytes."""
    code = (
        "import sys; sys.path.insert(0, '.'); sys.path.insert(0, 'tests')\n"
        "from b200sort._lib import lib\n"
        "import key_orders16 as ko\n"
        "import test_sort_indices16_gpu as t\n"
        "assert lib().b200sort_radix_atomic_order_ok() == 0\n"
        "offsets = t.ragged_offsets(43, total_segments=2000, big=1)\n"
        "for kt, desc in ko.ORDERS:\n"
        "    for in_place in (False, True):\n"
        "        t.check_1d(t.dup_keys((1 << 18) + 5, kt, kt + desc), kt, desc, in_place, 'safe 1-D')\n"
        "        t.check_1d(t.plan_keys(70001, {1}, (kt, desc), 3), kt, desc, in_place, 'safe plan')\n"
        "        t.check_seg(t.dup_keys(int(offsets[-1]), kt, desc), offsets, kt, desc, in_place, 'safe segmented')\n"
        "t.shared_ws().check_tail()\n"
        "print('ok')\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", code], cwd=root, env={**os.environ, "B200SORT_RANK_SAFE": "1"},
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_segmented_every_class_boundary(order):
    kt, desc = order
    check_seg(dup_keys(0, kt, 1), np.zeros(9, np.int32), kt, desc, False, "empty segments")
    for length in (1, 2, 127, 128, 129, 1023, 1024, 1025, TILE - 1, TILE, TILE + 1, 2 * TILE + 1, (1 << 17) + 5):
        rows = max(1, min(64, (1 << 21) // length))
        offsets = (np.arange(rows + 1, dtype=np.int64) * length).astype(np.int32)
        n = rows * length
        for in_place in (False, True):
            check_seg(dup_keys(n, kt, length + kt, distinct=50 + length % 7), offsets, kt, desc, in_place,
                      f"rows of {length} in_place={in_place}", word_offset=length % 8)


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_segmented_ragged(order):
    kt, desc = order
    offsets = ragged_offsets(11 + kt + desc)
    n = int(offsets[-1])
    assert n <= MAX_SEG_N
    for in_place in (False, True):
        check_seg(mixed_keys(n, kt, kt * 2 + desc), offsets, kt, desc, in_place, "ragged", word_offset=3)
        check_seg(dup_keys(n, kt, 9 + desc), offsets, kt, desc, in_place, "ragged, ties")


def test_segmented_more_segments_than_keys():
    rng = np.random.default_rng(3)
    n = 5000
    S = 3 * n
    offsets = np.concatenate([[0], np.sort(rng.integers(0, n + 1, S - 1)), [n]]).astype(np.int32)
    for kt, desc in ko.ORDERS:
        check_seg(dup_keys(n, kt, kt, distinct=20), offsets, kt, desc, desc == 1, "more segments than keys")


def test_length_one_segments_beside_onesweep_segments():
    """The classify kernel writes index 0 for a one-key segment while the onesweep passes move the long segments
    around it: nothing may overwrite it."""
    lens = [1, 20000, 1, 1, TILE + 1, 1, 0, 3 * TILE, 1, 1, 70001, 1]
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    n = int(offsets[-1])
    for kt, desc in ko.ORDERS:
        for in_place in (False, True):
            gk, gi = check_seg(mixed_keys(n, kt, kt + desc), offsets, kt, desc, in_place, "length 1 beside onesweep")
            assert not gi[offsets[:-1][np.asarray(lens) == 1]].any()


def test_one_segment_equals_the_1d_call():
    for n in (2, TILE + 1, 70001, MAX_1D):
        for kt, desc in ko.ORDERS:
            keys = dup_keys(n, kt, n + kt + desc)
            a = _call(True, keys, kt, desc, False, offsets=[0, n])
            b = _call(False, keys, kt, desc, False)
            assert a[0].tobytes() == b[0].tobytes() and a[1].tobytes() == b[1].tobytes(), (n, kt, desc)


def test_malformed_offsets_stay_in_bounds():
    """Malformed offsets give an undefined order, but every key and index written lies in its output: the guard
    words around every output and scratch buffer are untouched.  The checked build counts the clamped destinations at
    their check site and nowhere else."""
    import torch
    L = lib()
    n = 50000
    keys = mixed_keys(n, ko.KEY_U16, 77)
    cases = ([0, 30000, 10000, 50000], [0, 60000, -5, 20000, 99999], [5, 4, 3, 2, 1, 0], [0, 40000, 9000, 45000, 50000],
             [0, 9000, 3, 20000, 19000, 50000], [0, 20000, 20001, 19000, 50000])
    checked = L.b200sort_debug_checked_build() == 1
    for offs in cases:
        for in_place in (False, True):
            before = _sites() if checked else None
            kin = dp.DevBuf(n, 1, 2, 1).load(ko.bits(keys))
            kout = kin if in_place else dp.DevBuf(n, 3, 2, 2).load()
            idx, tk, ti = dp.DevBuf(n, 0, 8, 3).load(), dp.DevBuf(n, 5, 2, 4).load(), dp.DevBuf(n, 1, 4, 5).load()
            d_off = torch.tensor(offs, dtype=torch.int32, device="cuda")
            ws = shared_ws()
            nbytes = L.b200sort_segmented16_workspace_bytes(n, len(offs) - 1)
            check(L.b200sort_segmented_sort_indices_keys16(ko.KEY_U16, 1, kin.ptr, kout.ptr, idx.ptr, tk.ptr, ti.ptr,
                                                           n, d_off.data_ptr(), len(offs) - 1, ws.ptr, nbytes,
                                                           stream_ptr()))
            torch.cuda.synchronize()
            for b, what in ((kout, "keys out"), (idx, "indices"), (tk, "tmp keys"), (ti, "tmp indices")):
                b.read(f"{what}, offsets {offs}")
            if checked:
                grew = [s for s, (a, b) in enumerate(zip(before, _sites())) if b != a]
                assert set(grew) <= {CLAMP_SITE}, (offs, grew)
                _STATE["clamps"] += _sites()[CLAMP_SITE] - before[CLAMP_SITE]


def _normal(torch, shape, dtype, seed):
    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    x = torch.randn(shape, device="cuda", generator=g).to(dtype)
    return torch.where(x == 0, torch.ones_like(x), x)                 # no +-0.0: torch.sort treats them as equal


def _against_torch(torch, x, v, i, desc):
    tv, ti = torch.sort(x, dim=-1, stable=True, descending=desc)
    assert i.dtype == torch.int64 and i.shape == x.shape and v.dtype == x.dtype and v.shape == x.shape
    assert torch.equal(v.view(torch.int16), tv.view(torch.int16))
    assert torch.equal(i, ti)


@pytest.mark.parametrize("dtype", ["int16", "float16", "bfloat16"])
def test_python_1d_matches_torch_sort(dtype):
    import torch
    n = (1 << 20) + 3
    if dtype == "int16":
        x = torch.from_numpy(datagen.uniform_u32(n, 7).astype(np.uint16).view(np.int16) % 3000).cuda()
    else:
        x = _normal(torch, n, getattr(torch, dtype), 8)
    for desc in (False, True):
        x0 = x.clone()
        v, i = b200sort.sort16_with_indices(x, descending=desc)
        _against_torch(torch, x, v, i, desc)
        assert torch.equal(x.view(torch.int16), x0.view(torch.int16)), "the input changed"


@pytest.mark.parametrize("L_", [8, 64, 256, 1024, 32000, 128256])
def test_python_rows_match_torch_sort(L_):
    import torch
    B = max(1, (1 << 21) // L_)
    for dtype in (torch.bfloat16, torch.float16):
        x = _normal(torch, (B, L_), dtype, L_)
        v, i = b200sort.segmented_sort16_with_indices(x, descending=True)
        _against_torch(torch, x, v, i, True)


def test_python_offsets_and_uint16():
    import torch
    offsets = ragged_offsets(21, total_segments=500, big=0)
    n = int(offsets[-1])
    keys = mixed_keys(n, ko.KEY_U16, 4)
    for off_dtype in (torch.int32, torch.int64):
        for desc in (0, 1):
            x = torch.from_numpy(keys.view(np.int16)).cuda().view(torch.uint16)
            v, i = b200sort.segmented_sort16_with_indices(x, torch.from_numpy(offsets).to(off_dtype).cuda(),
                                                          descending=bool(desc))
            wk, wi = sort16_indices_ref(keys, offsets, ko.KEY_U16, desc)
            assert v.dtype == torch.uint16 and i.dtype == torch.int64
            assert ko.bits(v.view(torch.int16).cpu().numpy()).tobytes() == ko.bits(wk).tobytes()
            assert i.cpu().numpy().tobytes() == wi.tobytes()
            v, i = b200sort.sort16_with_indices(x, descending=bool(desc))
            wk, wi = sort16_indices_ref(keys, [0, n], ko.KEY_U16, desc)
            assert ko.bits(v.view(torch.int16).cpu().numpy()).tobytes() == ko.bits(wk).tobytes()
            assert i.cpu().numpy().tobytes() == wi.tobytes()
    v, i = b200sort.sort16_with_indices(torch.empty(0, dtype=torch.bfloat16, device="cuda"))
    assert v.numel() == 0 and i.dtype == torch.int64
    v, i = b200sort.segmented_sort16_with_indices(torch.empty((3, 0), dtype=torch.float16, device="cuda"))
    assert v.shape == (3, 0) and i.shape == (3, 0) and i.dtype == torch.int64


def test_python_call_on_a_non_default_device():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible")
    dev = torch.device("cuda", torch.cuda.device_count() - 1)
    assert torch.cuda.current_device() != dev.index
    x = _normal(torch, (300, 3001), torch.bfloat16, 5).to(dev)
    v, i = b200sort.segmented_sort16_with_indices(x, descending=True)
    assert v.device == dev and i.device == dev
    _against_torch(torch, x, v, i, True)
    v, i = b200sort.sort16_with_indices(x.view(-1))
    assert v.device == dev and i.device == dev
    _against_torch(torch, x.view(-1), v, i, False)


def test_launch_count_does_not_depend_on_data_or_segments():
    L = lib()
    counts = []
    for n in (2, TILE + 1, (1 << 18) + 3):
        for S in (set(), {0}, {1}, {0, 1}):
            for in_place in (False, True):
                L.b200sort_launch_count_reset()
                check_1d(plan_keys(n, S, (ko.KEY_BF16, 1), 5), ko.KEY_BF16, 1, in_place)
                counts.append(L.b200sort_launch_count())
    assert len(set(counts)) == 1, counts
    seg = []
    n = (1 << 18) + 3
    for S in (1, 1000, 10 ** 5, 2 * n):
        offsets = (np.arange(S + 1, dtype=np.int64) * n // S).astype(np.int32)
        L.b200sort_launch_count_reset()
        check_seg(mixed_keys(n, ko.KEY_F16, S), offsets, ko.KEY_F16, 1, False)
        seg.append(L.b200sort_launch_count())
    assert len(set(seg)) == 1, seg


def test_cuda_graph_capture_and_replay():
    import torch
    L = lib()
    check(L.b200sort_device_check())
    n, B = 300001, 100
    Lr = n // B
    x = torch.empty(n, dtype=torch.int16, device="cuda")
    ko_, io, kt_ = torch.empty_like(x), torch.empty(n, dtype=torch.int64, device="cuda"), torch.empty_like(x)
    ti = torch.empty(n, dtype=torch.int32, device="cuda")
    so, sio = torch.empty_like(x), torch.empty(n, dtype=torch.int64, device="cuda")
    offs = torch.arange(B + 1, dtype=torch.int32, device="cuda") * Lr
    offs[-1] = n
    ws1 = torch.empty(L.b200sort_keys16_workspace_bytes(n) + 256, dtype=torch.uint8, device="cuda")
    ws2 = torch.empty(L.b200sort_segmented16_workspace_bytes(n, B) + 256, dtype=torch.uint8, device="cuda")
    p1, p2 = ws1.data_ptr() + (-ws1.data_ptr()) % 256, ws2.data_ptr() + (-ws2.data_ptr()) % 256
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        check(L.b200sort_radix_sort_indices_keys16(ko.KEY_I16, 1, x.data_ptr(), ko_.data_ptr(), io.data_ptr(),
                                                   kt_.data_ptr(), ti.data_ptr(), n, p1, ws1.numel() - 256,
                                                   s.cuda_stream))
        check(L.b200sort_segmented_sort_indices_keys16(ko.KEY_I16, 0, x.data_ptr(), so.data_ptr(), sio.data_ptr(),
                                                       kt_.data_ptr(), ti.data_ptr(), n, offs.data_ptr(), B, p2,
                                                       ws2.numel() - 256, s.cuda_stream))
    o = offs.cpu().numpy()
    for keys in (np.full(n, 3, np.int16), plan_keys(n, {0}, (ko.KEY_I16, 1), 1), mixed_keys(n, ko.KEY_I16, 2)):
        x.copy_(torch.from_numpy(keys))
        g.replay()
        torch.cuda.synchronize()
        wk, wi = sort16_indices_ref(keys, [0, n], ko.KEY_I16, 1)
        assert ko_.cpu().numpy().tobytes() == wk.tobytes() and io.cpu().numpy().tobytes() == wi.tobytes()
        wk, wi = sort16_indices_ref(keys, o, ko.KEY_I16, 0)
        assert so.cpu().numpy().tobytes() == wk.tobytes() and sio.cpu().numpy().tobytes() == wi.tobytes()


@pytest.mark.parametrize("layout", ["1d", "rows128256"])
def test_full_size_2_28(layout):
    import torch
    n = 1 << 28
    if layout == "1d":
        x = _normal(torch, n, torch.bfloat16, 28)
        v, i = b200sort.sort16_with_indices(x)
        tv, ti = torch.sort(x, stable=True)
    else:
        L_ = 128256
        x = _normal(torch, (n // L_, L_), torch.bfloat16, 29)
        v, i = b200sort.segmented_sort16_with_indices(x, descending=True)
        tv, ti = torch.sort(x, dim=-1, stable=True, descending=True)
    assert torch.equal(v.view(torch.int16), tv.view(torch.int16))
    del v, tv
    assert torch.equal(i, ti)
