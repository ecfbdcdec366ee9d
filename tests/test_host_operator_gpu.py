"""The host-array operator (b200sort_order_array_host, b200sort_order_with_trust_host: the C++ order_array and
order_with_trust) on a GPU, above all its streamed path for device-accessible arrays of kStreamMinKeys keys or more
(order_host_streamed in csrc/api.cu; tests/host_stream_model.py models its schedule).

Every result is compared byte for byte with np.sort of the input (at 2^28, with torch.sort on the device).  Host
arrays sit between 4 KiB canaries, checked after every call.  The module's pinned and registered buffers are sized
for the largest streamed case, 2^26 keys, so the pinned memory held at once stays bounded: 256 MiB each, plus 1 GiB
for the 2^28 case, the operator's staging chunks and one 128 MiB array of the memory-kind cases."""
import ctypes
import glob
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

import host_stream_model as hsm
import oracle
from b200sort import datagen
from b200sort._lib import ALGO_LAB, ALGO_MERGE, ALGO_RADIX, MAX_N, check, lib
from helpers import stream_ptr

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
C, T, MIN = hsm.STREAM_CHUNKS, hsm.SORT_TILE, hsm.STREAM_MIN_KEYS
CANARY = 1024                      # keys (4 KiB) of guard on each side of every host array
CAP = 1 << 26                      # the largest array the module's pinned and registered buffers take
ALGOS = {"radix": ALGO_RADIX, "merge": ALGO_MERGE, "lab": ALGO_LAB}
ENTRIES = [("radix", ALGO_RADIX), ("merge", ALGO_MERGE), ("lab", ALGO_LAB), ("trust", None)]
PATTERN = (np.arange(CANARY, dtype=np.uint32) * np.uint32(0x9E3779B1) ^ np.uint32(0x5EED1234)).view(np.int32)


class Guarded:
    """An int32 host region that holds one array at a time, CANARY keys of PATTERN on each side."""

    def __init__(self, raw: np.ndarray):
        self.raw, self.lo, self.hi = raw, CANARY, CANARY

    def place(self, keys: np.ndarray, offset: int = 0) -> np.ndarray:
        lo, hi = CANARY + offset, CANARY + offset + keys.size
        assert hi + CANARY <= self.raw.size
        self.raw[lo - CANARY:lo] = PATTERN
        self.raw[hi:hi + CANARY] = PATTERN
        a = self.raw[lo:hi]
        a[:] = keys
        self.lo, self.hi = lo, hi
        return a

    def check(self, what: str) -> None:
        assert np.array_equal(self.raw[self.lo - CANARY:self.lo], PATTERN), f"{what}: wrote before the array"
        assert np.array_equal(self.raw[self.hi:self.hi + CANARY], PATTERN), f"{what}: wrote past the array"


def raw_of(ptr: int, keys: int) -> np.ndarray:
    return np.ctypeslib.as_array((ctypes.c_int32 * keys).from_address(ptr))


def same(got: np.ndarray, want: np.ndarray, what: str) -> None:
    if not np.array_equal(got, want):
        bad = np.flatnonzero(got != want)
        raise AssertionError(f"{what}: {bad.size} of {got.size} keys differ, first at {bad[0]}: "
                             f"got {got[bad[0]]}, want {want[bad[0]]}")


def host_sort(a: np.ndarray, algo) -> None:
    """algo None: order_with_trust_host."""
    L = lib()
    check(L.b200sort_order_with_trust_host(a.ctypes.data, a.size) if algo is None
          else L.b200sort_order_array_host(a.ctypes.data, a.size, algo))


def sort_guarded(buf: Guarded, keys: np.ndarray, want: np.ndarray, algo, what: str, offset: int = 0) -> None:
    a = buf.place(keys, offset)
    host_sort(a, algo)
    same(a, want, what)
    buf.check(what)


def uniform_with_ties(n: int, seed: int) -> np.ndarray:
    keys = datagen.uniform(n, seed)
    keys[::13] = np.iinfo(np.int32).max
    keys[5::17] = -7
    return keys


@pytest.fixture(scope="module")
def pinned():
    import torch
    t = torch.empty(CAP + 2 * CANARY + 8, dtype=torch.int32, pin_memory=True)
    yield Guarded(t.numpy())
    del t


@pytest.fixture(scope="module")
def registered():
    import torch
    keys = CAP + 2 * CANARY + 8
    raw = np.empty(keys + 1024, np.int32)
    view = raw[(-raw.ctypes.data % 4096) // 4:][:keys]
    cudart = torch.cuda.cudart()
    assert int(cudart.cudaHostRegister(view.ctypes.data, view.nbytes, 0)) == 0
    yield Guarded(view)
    assert int(cudart.cudaHostUnregister(view.ctypes.data)) == 0


# ---- every entry point on the streamed path -------------------------------------------------------------------------
STREAM_SIZES = [MIN, MIN + 1, MIN + 12345, 3 * (1 << 24) + 77, (1 << 26) - 1, hsm.shortest_last_chunk(5 << 20)]


@pytest.mark.parametrize("n", STREAM_SIZES)
def test_every_algorithm_on_the_streamed_path(pinned, n):
    """Radix, merge and lab through order_array_host, and order_with_trust_host, on pinned memory.  The last size
    has the shortest last chunk the chunk rounding allows (2 C T - 1 keys short of the others)."""
    keys = uniform_with_ties(n, n % 1000)
    want = np.sort(keys)
    for name, algo in ENTRIES:
        sort_guarded(pinned, keys, want, algo, f"{name} n={n}")


def test_streamed_path_with_every_merge_variant(pinned):
    """The last level's tile ranges run the compiled merge-pass kernel the variant selects."""
    L = lib()
    n = MIN + 4 * T + 3
    keys = uniform_with_ties(n, 8)
    want = np.sort(keys)
    try:
        for v in range(L.b200sort_merge_num_variants()):
            assert L.b200sort_merge_set_variant(v) == 0
            for name in ("radix", "merge"):
                sort_guarded(pinned, keys, want, ALGOS[name], f"variant {v} {name}")
    finally:
        L.b200sort_merge_set_variant(0)


def _launches(a: np.ndarray, keys: np.ndarray, algo: int) -> int:
    L = lib()
    a[:] = keys
    before = L.b200sort_launch_count()
    host_sort(a, algo)
    return L.b200sort_launch_count() - before


def test_one_key_below_the_switch(pinned):
    """At kStreamMinKeys - 1 pinned memory takes the one-shot path (the launches of a call with streaming off) and
    gives the same bytes; at kStreamMinKeys it streams (other launches)."""
    L = lib()
    for n in (MIN - 1, MIN):
        keys = uniform_with_ties(n, 3)
        want = np.sort(keys)
        for name, algo in ALGOS.items():
            a = pinned.place(keys)
            streamed = _launches(a, keys, algo)
            same(a, want, f"{name} n={n}")
            try:
                L.b200sort_host_set_streaming(0)
                one_shot = _launches(a, keys, algo)
            finally:
                L.b200sort_host_set_streaming(1)
            same(a, want, f"{name} n={n} streaming off")
            pinned.check(f"{name} n={n}")
            assert (streamed == one_shot) == (n < MIN), (name, n, streamed, one_shot)


# ---- inputs that stress the chunk merges ----------------------------------------------------------------------------
@pytest.mark.parametrize("kind", hsm.STRESS)
def test_streamed_chunk_merges_on_stress_inputs(pinned, kind):
    n = MIN + 12345
    s = hsm.schedule(n)
    keys = hsm.stress_keys(kind, n, s.chunk, [e0 for e0, _ in s.copies[1:]], T, seed=11)
    want = np.sort(keys)
    for name, algo in ALGOS.items():
        sort_guarded(pinned, keys, want, algo, f"{kind} {name}")


# ---- memory kinds ---------------------------------------------------------------------------------------------------
def _cudart():
    """The CUDA runtime through ctypes (for managed memory), or None."""
    import torch
    cands = ["libcudart.so.12", "libcudart.so"]
    cands += glob.glob(os.path.join(os.path.dirname(torch.__file__), "..", "nvidia", "cuda_runtime", "lib",
                                    "libcudart.so*"))
    cands += glob.glob("/usr/local/cuda/lib64/libcudart.so*")
    for c in cands:
        try:
            rt = ctypes.CDLL(c)
            rt.cudaMallocManaged.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_size_t, ctypes.c_uint]
            rt.cudaFree.argtypes = [ctypes.c_void_p]
            return rt
        except (OSError, AttributeError):
            continue
    return None


@pytest.mark.parametrize("offset", [0, 1])
@pytest.mark.parametrize("kind", ["torch_pinned", "alloc_pinned", "registered", "managed", "pageable"])
def test_memory_kinds(pinned, registered, kind, offset):
    """Pinned (torch and b200sort_host_alloc_pinned), registered and managed memory stream; pageable memory goes
    through the staged copy.  Arrays start at the allocation's 4 KiB boundary, or 4 bytes past it."""
    L = lib()
    n = MIN + 777
    keys = uniform_with_ties(n, 21 + offset)
    want = np.sort(keys)
    total = n + 2 * CANARY + 8
    free = None
    if kind == "torch_pinned":
        buf = pinned
    elif kind == "registered":
        buf = registered
    elif kind == "alloc_pinned":
        p = ctypes.c_void_p()
        check(L.b200sort_host_alloc_pinned(ctypes.byref(p), total * 4))
        buf, free = Guarded(raw_of(p.value, total)), lambda: check(L.b200sort_host_free_pinned(p))
    elif kind == "managed":
        rt = _cudart()
        if rt is None:
            pytest.skip("the CUDA runtime library is not reachable through ctypes")
        p = ctypes.c_void_p()
        assert rt.cudaMallocManaged(ctypes.byref(p), total * 4, 1) == 0          # cudaMemAttachGlobal
        buf, free = Guarded(raw_of(p.value, total)), lambda: rt.cudaFree(p)
    else:
        buf = Guarded(np.empty(total, np.int32))
    try:
        for name, algo in ALGOS.items():
            sort_guarded(buf, keys, want, algo, f"{kind}+{offset} {name}", offset)
    finally:
        if free is not None:
            free()


_STAGED_SCRIPT = r"""
import sys
import numpy as np
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
import host_stream_model as hsm
from b200sort import datagen
from b200sort._lib import ALGO_MERGE, ALGO_RADIX, check, lib
canary = (np.arange(1024, dtype=np.uint32) * np.uint32(0x9E3779B1) ^ np.uint32(0x5EED1234)).view(np.int32)
for i, n in enumerate(hsm.STAGED_SIZES):
    raw = np.empty(n + 2048 + 1, np.int32)
    off = 1024 + i % 2                      # every other array starts 4 bytes further on
    raw[off - 1024:off] = canary
    raw[off + n:off + n + 1024] = canary
    keys = datagen.uniform(n, n)
    keys[::9] = -1
    a = raw[off:off + n]
    a[:] = keys
    algo = ALGO_MERGE if i % 2 else ALGO_RADIX
    check(lib().b200sort_order_array_host(a.ctypes.data, n, algo))
    assert np.array_equal(a, np.sort(keys)), (n, algo)
    assert np.array_equal(raw[off - 1024:off], canary) and np.array_equal(raw[off + n:off + n + 1024], canary), n
print("staged ok")
"""


@pytest.mark.parametrize("threads", hsm.COPY_THREADS)
def test_staged_pageable_copy(threads, tmp_path):
    """Pageable arrays around the direct-copy limit (kDirectBytes) and around whole 8 MiB staging chunks +- 1 key,
    with 1, 3 and 16 copy threads.  B200SORT_COPY_THREADS is read once per process, hence the subprocesses."""
    env = dict(os.environ, B200SORT_COPY_THREADS=str(threads))
    r = subprocess.run([sys.executable, "-c", _STAGED_SCRIPT, ROOT], env=env, cwd=tmp_path, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0 and "staged ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


# ---- the arena across calls -----------------------------------------------------------------------------------------
def test_arena_reuse_sequence(pinned):
    """One arena through growth, smaller requests, a change of algorithm, streaming off and on, and a release."""
    L = lib()
    L.b200sort_host_release()
    cache = {}

    def step(n, algo, what, pageable=False):
        if n not in cache:
            keys = uniform_with_ties(n, n % 977)
            cache[n] = (keys, np.sort(keys))
        keys, want = cache[n]
        buf = Guarded(np.empty(n + 2 * CANARY, np.int32)) if pageable else pinned
        sort_guarded(buf, keys, want, ALGOS[algo], what)

    try:
        step(MIN + 5, "radix", "streamed radix")
        step(1000, "radix", "1000 keys")
        step(1 << 26, "merge", "2^26 streamed merge, the arena grows")
        step(MIN, "lab", "streamed lab")
        L.b200sort_host_set_streaming(0)
        step(MIN + 5, "radix", "streaming off")
        L.b200sort_host_set_streaming(1)
        step(MIN + 5, "radix", "streaming on again")
        L.b200sort_host_release()
        step(MIN, "radix", "after release")
        step(1 << 22, "radix", "pageable", pageable=True)
        step(1 << 22, "merge", "pageable merge", pageable=True)
    finally:
        L.b200sort_host_set_streaming(1)


def test_two_host_threads(pinned, registered):
    """Two Python threads sort their own pinned arrays at once (ctypes releases the GIL); the arena's mutex must
    serialise the calls."""
    jobs = [(pinned, MIN + 3, ALGO_RADIX), (registered, MIN + 7, ALGO_MERGE)]
    data = [(uniform_with_ties(n, 100 + i), None) for i, (_, n, _) in enumerate(jobs)]
    data = [(k, np.sort(k)) for k, _ in data]
    errors = []
    barrier = threading.Barrier(len(jobs))

    def worker(i):
        buf, n, algo = jobs[i]
        keys, want = data[i]
        try:
            for rep in range(3):
                a = buf.place(keys)
                barrier.wait()
                host_sort(a, algo)
                same(a, want, f"thread {i} rep {rep}")
                buf.check(f"thread {i} rep {rep}")
        except Exception as e:          # noqa: BLE001  (reported below)
            errors.append(e)
            barrier.abort()

    threads = [threading.Thread(target=worker, args=(i,)) for i in range(len(jobs))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors


# ---- full size ------------------------------------------------------------------------------------------------------
def test_full_size_pinned():
    """n = 2^28 from pinned memory, as bench.py runs it, against torch.sort of a device copy taken before the call."""
    import torch
    L = lib()
    n = 1 << 28
    total = n + 2 * CANARY
    p = ctypes.c_void_p()
    check(L.b200sort_host_alloc_pinned(ctypes.byref(p), total * 4))
    try:
        buf = Guarded(raw_of(p.value, total))
        g = torch.Generator(device="cuda")
        g.manual_seed(28)
        d = torch.randint(-2**31, 2**31, (n,), dtype=torch.int64, device="cuda", generator=g).to(torch.int32)
        d[::11] = 2**31 - 1
        d[3::29] = -2**31
        want = torch.sort(d).values
        buf.lo, buf.hi = CANARY, CANARY + n
        buf.raw[:CANARY] = PATTERN
        buf.raw[CANARY + n:] = PATTERN
        a = buf.raw[CANARY:CANARY + n]
        host = torch.from_numpy(a)
        for name, algo in ALGOS.items():
            host.copy_(d)
            host_sort(a, algo)
            assert torch.equal(host.cuda(), want), name
            buf.check(f"2^28 {name}")
        del want, d
    finally:
        check(L.b200sort_host_free_pinned(p))


# ---- errors before any work -----------------------------------------------------------------------------------------
def test_errors_before_any_work(pinned):
    L = lib()
    keys = uniform_with_ties(MIN, 4)
    a = pinned.place(keys)
    count = L.b200sort_launch_count()
    for algo in ALGOS.values():
        assert L.b200sort_order_array_host(a.ctypes.data, MAX_N + 1, algo) == 1
        assert L.b200sort_order_array_host(None, MIN, algo) == 1
        assert L.b200sort_order_array_host(a.ctypes.data, 0, algo) == 0
        assert L.b200sort_order_array_host(a.ctypes.data, 1, algo) == 0
    for bad in (-1, 3):
        assert L.b200sort_order_array_host(a.ctypes.data, MIN, bad) == 1
    assert L.b200sort_order_with_trust_host(a.ctypes.data, MAX_N + 1) == 1
    assert L.b200sort_order_with_trust_host(None, 2) == 1
    assert L.b200sort_order_with_trust_host(a.ctypes.data, 1) == 0
    assert L.b200sort_launch_count() == count
    same(a, keys, "untouched")
    pinned.check("errors")


# ---- the merge stage kernels at the runs the streamed path uses -----------------------------------------------------
MERGE_CHUNKS = [3 * 2 * T, 5 * 2 * T, 1025 * 2 * T]


def _sorted_windows(keys: np.ndarray, run: int, kind=None) -> np.ndarray:
    """keys with every window of `run` sorted; kind="stable" on windows that are two sorted runs merges them."""
    out = keys.copy()
    for base in range(0, keys.size, run):
        out[base:base + run] = np.sort(out[base:base + run], kind=kind)
    return out


@pytest.mark.parametrize("chunk", MERGE_CHUNKS)
def test_merge_stages_at_streamed_runs(chunk):
    """b200sort_merge_partition_i32 + b200sort_merge_pass_i32 at runs of chunk, 2 chunk and 4 chunk, chunk an odd
    multiple of 2T (the runs are not powers of two), n = 8 chunk - r: a full last pair (r = 0), a short one
    (r = 1, T - 1) and a last pair with no second run (r = 3 chunk / 2).  Split points against oracle.merge_path,
    output against oracle.rank_merge (numpy's merge of the pair, checked against it at the small chunks, at the
    largest one), every compiled merge-pass kernel, guard words around the output.  The largest chunk (2^26 keys)
    takes the two inputs that stress ties most, to keep the test's time down."""
    import torch
    L = lib()
    kinds = hsm.STRESS if chunk < 1024 * T else ("straddle", "extremes")
    variants = range(L.b200sort_merge_num_variants())
    try:
        for r in (0, 1, T - 1, 3 * chunk // 2):
            n = 8 * chunk - r
            tiles = hsm.div_up(n, T)
            edges = [k * hsm.div_up(tiles, C) * T for k in range(1, C)]
            for kind in kinds:
                keys = hsm.stress_keys(kind, n, chunk, edges, T, seed=r + 1)
                merged = _sorted_windows(keys, chunk)
                for run in (chunk, 2 * chunk, 4 * chunk):
                    runs, merged = merged, _sorted_windows(merged, 2 * run, "stable")
                    what = f"chunk={chunk} r={r} run={run} {kind}"
                    if chunk < 1024 * T:
                        want = runs.copy()
                        for base in range(0, n, 2 * run):
                            want[base:base + 2 * run] = oracle.rank_merge(runs[base:base + run],
                                                                          runs[base + run:base + 2 * run])
                        same(merged, want, what + " numpy merge vs rank_merge")
                    d_in = torch.from_numpy(runs).cuda()
                    splits = torch.zeros(tiles + 1, dtype=torch.int32, device="cuda")
                    check(L.b200sort_merge_partition_i32(d_in.data_ptr(), n, run, splits.data_ptr(), stream_ptr()))
                    torch.cuda.synchronize()
                    sp = splits.cpu().numpy().view(np.uint32)
                    for t in range(tiles):
                        g = t * T
                        base = g // (2 * run) * (2 * run)
                        assert sp[t] == oracle.merge_path(runs[base:base + run], runs[base + run:base + 2 * run],
                                                          g - base), (what, t)
                    out = torch.full((n + 2 * CANARY,), -123456789, dtype=torch.int32, device="cuda")
                    for v in variants:
                        assert L.b200sort_merge_set_variant(v) == 0
                        out.fill_(-123456789)
                        check(L.b200sort_merge_pass_i32(d_in.data_ptr(), out[CANARY:].data_ptr(), n, run,
                                                        splits.data_ptr(), stream_ptr()))
                        got = out.cpu().numpy()
                        same(got[CANARY:CANARY + n], merged, f"{what} variant {v}")
                        assert np.all(got[:CANARY] == -123456789) and np.all(got[CANARY + n:] == -123456789), what
                    L.b200sort_merge_set_variant(0)
    finally:
        L.b200sort_merge_set_variant(0)
