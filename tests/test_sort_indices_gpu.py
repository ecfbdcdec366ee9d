"""Sort with indices on the GPU (b200sort_radix_sort_indices_keys, b200sort_segmented_sort_indices_keys and the
torch-facing b200sort.sort_with_indices / segmented_sort_with_indices): keys byte for byte and int64 indices exactly
against the numpy reference of tests/test_sort_indices_cpu.py, and against torch.sort.

Every C-ABI call here writes into canary-guarded buffers (digit_patterns.DevBuf) whose arrays start out holding
canaries too, so the index output must be fully overwritten, nothing may be written around any output or scratch
buffer, and garbage in the scratch buffers must change nothing.  The 1-D and segmented calls share one workspace
that is filled with 0xFF once and never cleared."""
import os
import subprocess
import sys

import numpy as np
import pytest

import b200sort
from b200sort import datagen
from b200sort._lib import ALGO_RADIX, check, lib
from helpers import stream_ptr

import digit_patterns as dp
import key_orders as ko
from test_segmented_gpu import mixed_keys, ragged_offsets, row_lengths
from test_sort_indices_cpu import sort_indices_ref

pytestmark = pytest.mark.gpu

ORDER_IDS = [f"{ko.NAMES[k]}_{'desc' if d else 'asc'}" for k, d in ko.ORDERS]
PAIRS_TILE = 5120                  # keys per tile of the generic pairs pass (512 threads x 10)
MAX_1D = (1 << 20) + 7
MAX_SEG_N, MAX_SEG_S = 1 << 22, 1 << 22

_WS = None


def shared_ws():
    """The module's never-cleared workspace, sized for every call below but the 2^28-key ones."""
    global _WS
    if _WS is None:
        L = lib()
        _WS = dp.Workspace(max(L.b200sort_workspace_bytes(MAX_1D, ALGO_RADIX),
                               L.b200sort_segmented_workspace_bytes(MAX_SEG_N, MAX_SEG_S)))
    return _WS


@pytest.fixture(scope="module", autouse=True)
def _module_checks():
    yield
    if _WS is not None:
        _WS.check_tail()
    L = lib()
    if L.b200sort_debug_checked_build():
        assert L.b200sort_debug_check_failures() == 0


def _call(seg, keys, kt, desc, in_place, offsets=None, word_offset=0):
    """One guarded call; returns (sorted key words, int64 indices)."""
    import torch
    L = lib()
    n = keys.size
    kin = dp.DevBuf(n, word_offset, 4, 1).load(ko.bits(keys))
    kout = kin if in_place else dp.DevBuf(n, word_offset, 4, 2).load()
    idx = dp.DevBuf(n, 2 * (word_offset & 1), 8, 3).load()
    tk = dp.DevBuf(n, 0, 4, 4).load()
    ti = dp.DevBuf(n, 0, 4, 5).load()
    ws = shared_ws()
    if seg:
        d_off = torch.from_numpy(np.asarray(offsets, np.int32)).cuda()
        S = d_off.numel() - 1
        nbytes = L.b200sort_segmented_workspace_bytes(n, S)
        assert nbytes <= ws.cap - ws.GUARD
        before = ws.guard(nbytes).clone()
        check(L.b200sort_segmented_sort_indices_keys(kt, desc, kin.ptr, kout.ptr, idx.ptr, tk.ptr, ti.ptr, n,
                                                     d_off.data_ptr(), S, ws.ptr, nbytes, stream_ptr()))
    else:
        nbytes = L.b200sort_workspace_bytes(n, ALGO_RADIX)
        assert nbytes <= ws.cap - ws.GUARD
        before = ws.guard(nbytes).clone()
        check(L.b200sort_radix_sort_indices_keys(kt, desc, kin.ptr, kout.ptr, idx.ptr, tk.ptr, ti.ptr, n,
                                                 ws.ptr, nbytes, stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(ws.guard(nbytes), before), "workspace written past ws_bytes"
    tk.read("tmp keys"); ti.read("tmp indices")
    if not in_place:
        assert kin.read("keys in").tobytes() == ko.bits(keys).tobytes(), "the copy form modified its input"
    return kout.read("keys out"), idx.read("indices").view(np.int64)


def check_1d(keys, kt, desc, in_place, what="", word_offset=0):
    gk, gi = _call(False, keys, kt, desc, in_place, word_offset=word_offset)
    wk, wi = sort_indices_ref(keys, [0, keys.size], kt, desc)
    assert gk.tobytes() == ko.bits(wk).tobytes(), f"{what}: keys differ"
    assert gi.tobytes() == wi.tobytes(), f"{what}: indices differ at {np.flatnonzero(gi != wi)[:5]}"


def check_seg(keys, offsets, kt, desc, in_place, what=""):
    gk, gi = _call(True, keys, kt, desc, in_place, offsets=offsets)
    wk, wi = sort_indices_ref(keys, offsets, kt, desc)
    assert gk.tobytes() == ko.bits(wk).tobytes(), f"{what}: keys differ"
    assert gi.tobytes() == wi.tobytes(), f"{what}: indices differ at {np.flatnonzero(gi != wi)[:5]}"
    return gk, gi


def dup_keys(n, kt, seed, distinct=300):
    """Keys with many ties, so that stability shows in the indices."""
    w = (datagen.uniform_u32(n, seed) % np.uint32(distinct)) * np.uint32(0x01010101)
    return w.view(ko.DTYPES[kt])


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_1d_sizes_in_place_and_copied(order):
    kt, desc = order
    for n in (0, 1, 2, 31, PAIRS_TILE - 1, PAIRS_TILE, PAIRS_TILE + 1, (1 << 16) + 3, MAX_1D):
        for in_place in (False, True):
            for i, keys in enumerate((mixed_keys(n, kt, n + kt), dup_keys(n, kt, n + desc))):
                check_1d(keys, kt, desc, in_place, f"n={n} in_place={in_place} set {i}", word_offset=(n + i) % 4)


@pytest.mark.parametrize("n", [PAIRS_TILE + 1, (1 << 16) + 3])
def test_every_pass_plan(n):
    """Keys whose image digits are constant in exactly the passes of S, for every S: no pass (indices 0..n-1) up to
    all four executed, in place and copied, so the in-place odd counts end in the tmp -> out widening."""
    for m in range(16):
        S = {p for p in range(4) if m >> p & 1}
        kt, desc = ko.ORDERS[m % len(ko.ORDERS)]
        keys = dp.with_constant_digits(n, S, (kt, desc), seed=m)
        for in_place in (False, True):
            check_1d(keys, kt, desc, in_place, f"constant passes {sorted(S)} in_place={in_place}")
    keys = np.full(n, 7, np.int32)                                      # all keys equal: the identity
    gk, gi = _call(False, keys, ko.KEY_I32, 1, False)
    assert gi.tobytes() == np.arange(n, dtype=np.int64).tobytes()


def test_skipping_off():
    L = lib()
    try:
        L.b200sort_radix_set_skip(0)
        for S in ({0, 1, 2, 3}, {1, 3}, set()):
            keys = dp.with_constant_digits((1 << 16) + 3, S, (ko.KEY_F32, 1), seed=len(S))
            for in_place in (False, True):
                check_1d(keys, ko.KEY_F32, 1, in_place, f"skip off, constant {sorted(S)}")
    finally:
        L.b200sort_radix_set_skip(1)


def test_rank_safe_fallback():
    """With B200SORT_RANK_SAFE=1 the ballot-ranked passes and classes give the same results."""
    code = (
        "import sys; sys.path.insert(0, '.'); sys.path.insert(0, 'tests')\n"
        "from b200sort._lib import lib\n"
        "import digit_patterns as dp, key_orders as ko\n"
        "import test_sort_indices_gpu as t\n"
        "assert lib().b200sort_radix_atomic_order_ok() == 0\n"
        "offsets = t.ragged_offsets(43, total_segments=2000, big=1)\n"
        "for kt, desc in ko.ORDERS:\n"
        "    for in_place in (False, True):\n"
        "        t.check_1d(t.dup_keys((1 << 18) + 5, kt, kt + desc), kt, desc, in_place, 'safe 1-D')\n"
        "        t.check_1d(dp.with_constant_digits(70001, {1, 2}, (kt, desc), 3), kt, desc, in_place, 'safe plan')\n"
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
    for length in row_lengths():
        rows = max(1, min(64, (1 << 21) // length))
        offsets = (np.arange(rows + 1, dtype=np.int64) * length).astype(np.int32)
        n = rows * length
        check_seg(dup_keys(n, kt, length + kt, distinct=50 + length % 7), offsets, kt, desc, length % 2 == 1,
                  f"rows of {length}")


@pytest.mark.parametrize("order", ko.ORDERS, ids=ORDER_IDS)
def test_segmented_ragged(order):
    kt, desc = order
    offsets = ragged_offsets(11 + kt + desc)
    n = int(offsets[-1])
    assert n <= MAX_SEG_N
    for in_place in (False, True):
        check_seg(mixed_keys(n, kt, kt * 2 + desc), offsets, kt, desc, in_place, "ragged")
        check_seg(dup_keys(n, kt, 9 + desc), offsets, kt, desc, in_place, "ragged, ties")


def test_segmented_more_segments_than_keys():
    rng = np.random.default_rng(3)
    n = 5000
    S = 3 * n
    offsets = np.concatenate([[0], np.sort(rng.integers(0, n + 1, S - 1)), [n]]).astype(np.int32)
    for kt, desc in ko.ORDERS:
        check_seg(dup_keys(n, kt, kt, distinct=20), offsets, kt, desc, desc == 1, "more segments than keys")


def test_one_segment_equals_the_1d_call():
    for n in (2, 5121, 8193, (1 << 20) + 7):
        for kt, desc in ko.ORDERS:
            keys = dup_keys(n, kt, n + kt + desc)
            a = _call(True, keys, kt, desc, False, offsets=[0, n])
            b = _call(False, keys, kt, desc, False)
            assert a[0].tobytes() == b[0].tobytes() and a[1].tobytes() == b[1].tobytes(), (n, kt, desc)


def _torch_cases(n, seed):
    import torch
    r = datagen.uniform_u32(n, seed)
    g = torch.Generator().manual_seed(seed)
    return {"float32": torch.randn(n, generator=g).numpy(), "int32": r.view(np.int32) % 5000,
            "uint32": r % np.uint32(5000) + np.uint32(0x7FFFF000)}


@pytest.mark.parametrize("layout", ["1d", "rows16", "rows1000", "rows70001"])
def test_python_calls_match_torch_sort(layout):
    """Values and int64 indices equal torch.sort(stable=True); uint32 is compared through int64, which torch sorts."""
    import torch
    n = 1 << 20
    for dtype, a in _torch_cases(n, 5).items():
        if layout != "1d":
            L_ = int(layout[4:])
            a = a[: n // L_ * L_].reshape(-1, L_)
        for desc in (False, True):
            x = torch.from_numpy(np.ascontiguousarray(a)).cuda()
            if layout == "1d":
                v, i = b200sort.sort_with_indices(x, descending=desc)
            else:
                v, i = b200sort.segmented_sort_with_indices(x, descending=desc)
            cmp = torch.from_numpy(a.astype(np.int64) if dtype == "uint32" else np.ascontiguousarray(a)).cuda()
            tv, ti = torch.sort(cmp, dim=-1, stable=True, descending=desc)
            assert i.dtype == torch.int64 and tuple(i.shape) == a.shape and v.dtype == x.dtype
            assert v.cpu().numpy().tobytes() == tv.cpu().numpy().astype(a.dtype).tobytes(), (layout, dtype, desc)
            assert torch.equal(i, ti), (layout, dtype, desc)
            assert x.cpu().numpy().tobytes() == np.ascontiguousarray(a).tobytes(), "the input changed"


def test_python_offsets_call():
    import torch
    offsets = ragged_offsets(21, total_segments=500, big=0)
    n = int(offsets[-1])
    keys = dup_keys(n, ko.KEY_F32, 4)
    for off_dtype in (torch.int32, torch.int64):
        v, i = b200sort.segmented_sort_with_indices(torch.from_numpy(keys).cuda(),
                                                    torch.from_numpy(offsets).to(off_dtype).cuda(), descending=True)
        wk, wi = sort_indices_ref(keys, offsets, ko.KEY_F32, 1)
        assert ko.bits(v.cpu().numpy()).tobytes() == ko.bits(wk).tobytes() and i.cpu().numpy().tobytes() == wi.tobytes()
    v, i = b200sort.sort_with_indices(torch.empty(0, dtype=torch.int32, device="cuda"))
    assert v.numel() == 0 and i.dtype == torch.int64


def test_launch_count_does_not_depend_on_data_or_segments():
    L = lib()
    n = (1 << 18) + 3
    counts = []
    for keys in (np.full(n, 5, np.int32), dp.with_constant_digits(n, {2}, (ko.KEY_I32, 0), 1), mixed_keys(n, 0, 2)):
        for in_place in (False, True):
            L.b200sort_launch_count_reset()
            check_1d(keys, ko.KEY_I32, 0, in_place)
            counts.append(L.b200sort_launch_count())
    assert len(set(counts)) == 1, counts
    seg = []
    for S in (1, 1000, 10 ** 5):
        offsets = (np.arange(S + 1, dtype=np.int64) * n // S).astype(np.int32)
        L.b200sort_launch_count_reset()
        check_seg(mixed_keys(n, ko.KEY_U32, S), offsets, ko.KEY_U32, 1, False)
        seg.append(L.b200sort_launch_count())
    assert len(set(seg)) == 1, seg


def test_cuda_graph_capture_and_replay():
    import torch
    L = lib()
    check(L.b200sort_device_check())
    n, B = 300001, 100
    Lr = n // B
    x = torch.empty(n, dtype=torch.int32, device="cuda")
    ko_, io, kt_ = torch.empty_like(x), torch.empty(n, dtype=torch.int64, device="cuda"), torch.empty_like(x)
    ti = torch.empty_like(x)
    so, sio = torch.empty_like(x), torch.empty(n, dtype=torch.int64, device="cuda")
    offs = torch.arange(B + 1, dtype=torch.int32, device="cuda") * Lr
    offs[-1] = n
    ws1 = torch.empty(L.b200sort_workspace_bytes(n, ALGO_RADIX) + 256, dtype=torch.uint8, device="cuda")
    ws2 = torch.empty(L.b200sort_segmented_workspace_bytes(n, B) + 256, dtype=torch.uint8, device="cuda")
    p1, p2 = ws1.data_ptr() + (-ws1.data_ptr()) % 256, ws2.data_ptr() + (-ws2.data_ptr()) % 256
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        check(L.b200sort_radix_sort_indices_keys(ko.KEY_I32, 1, x.data_ptr(), ko_.data_ptr(), io.data_ptr(),
                                                 kt_.data_ptr(), ti.data_ptr(), n, p1, ws1.numel() - 256,
                                                 s.cuda_stream))
        check(L.b200sort_segmented_sort_indices_keys(ko.KEY_I32, 0, x.data_ptr(), so.data_ptr(), sio.data_ptr(),
                                                     kt_.data_ptr(), ti.data_ptr(), n, offs.data_ptr(), B, p2,
                                                     ws2.numel() - 256, s.cuda_stream))
    o = offs.cpu().numpy()
    for keys in (np.full(n, 3, np.int32), mixed_keys(n, 0, 1) & np.int32(0x00FF00FF), mixed_keys(n, 0, 2)):
        x.copy_(torch.from_numpy(keys))
        g.replay()
        torch.cuda.synchronize()
        wk, wi = sort_indices_ref(keys, [0, n], ko.KEY_I32, 1)
        assert ko_.cpu().numpy().tobytes() == wk.tobytes() and io.cpu().numpy().tobytes() == wi.tobytes()
        wk, wi = sort_indices_ref(keys, o, ko.KEY_I32, 0)
        assert so.cpu().numpy().tobytes() == wk.tobytes() and sio.cpu().numpy().tobytes() == wi.tobytes()


@pytest.mark.parametrize("layout", ["1d", "rows1024", "rows131072"])
def test_full_size_2_28(layout):
    import torch
    n = 1 << 28
    g = torch.Generator(device="cuda").manual_seed(28)
    x = torch.randn(n, generator=g, device="cuda")
    if layout == "1d":
        v, i = b200sort.sort_with_indices(x)
        tv, ti = torch.sort(x, stable=True)
    else:
        x = x.view(-1, int(layout[4:]))
        v, i = b200sort.segmented_sort_with_indices(x, descending=True)
        tv, ti = torch.sort(x, dim=-1, stable=True, descending=True)
    assert torch.equal(v, tv)
    del v, tv
    assert torch.equal(i, ti)
