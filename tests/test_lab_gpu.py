"""The drop-in boundary on a GPU: host-array operator, the exported C++ symbols, the reference's
unmodified drivers linked against this library, and the reference's own GPU sort run beside ours."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import b200sort
import oracle
from b200sort import datagen
from helpers import assert_bit_exact

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("n", [0, 1, 32, 256, 65536, (1 << 20) + 3, 1 << 23])
def test_host_operator_both_entry_points(n):
    keys = datagen.uniform(n, 17)
    want = oracle.radix_sort(keys)
    a = keys.copy(); b200sort.order_array(a)
    assert_bit_exact(a, want, "order_array")
    b = keys.copy(); b200sort.order_with_trust(b)
    assert_bit_exact(b, want, "order_with_trust")


def test_host_operator_with_pinned_memory():
    import torch
    keys = datagen.uniform(1 << 22, 18)
    t = torch.from_numpy(keys.copy()).pin_memory()
    a = t.numpy()
    b200sort.order_array(a)
    assert_bit_exact(a, oracle.radix_sort(keys), "pinned")


@pytest.mark.parametrize("n", [1 << 25, (1 << 25) + 12345, 3 * (1 << 24) + 77])
def test_streamed_host_operator_large_arrays(n):
    """From 2^25 keys on the host-array operator streams (chunked H2D, chunk sorts, progressive
    merge-path merges, output ranges copied back as they are merged).  Pageable and pinned arrays,
    radix and merge, and the one-shot path on the same input: all the same bytes as the oracle."""
    import torch
    from b200sort._lib import ALGO_MERGE, ALGO_RADIX, check
    L = b200sort.lib()
    keys = datagen.uniform(n, 41)
    keys[: n // 16] = np.iinfo(np.int32).max               # sentinel-valued keys in quantity
    keys[n // 3: n // 3 + 100000] = -7                     # a long run of equal keys across a chunk boundary
    want = oracle.radix_sort(keys)
    try:
        for algo in (ALGO_RADIX, ALGO_MERGE):
            a = keys.copy()
            check(L.b200sort_order_array_host(a.ctypes.data, n, algo))
            assert_bit_exact(a, want, f"pageable algo={algo}")
        pinned = torch.from_numpy(keys.copy()).pin_memory().numpy()
        check(L.b200sort_order_array_host(pinned.ctypes.data, n, ALGO_RADIX))
        assert_bit_exact(pinned, want, "pinned")
        L.b200sort_host_set_streaming(0)
        a = keys.copy()
        check(L.b200sort_order_array_host(a.ctypes.data, n, ALGO_RADIX))
        assert_bit_exact(a, want, "one-shot")
    finally:
        L.b200sort_host_set_streaming(1)


def test_host_operator_matches_the_stored_reference_outputs(golden_small, golden_mixed):
    """Both drop-in entry points against what the reference's own code returned (its CPU path, stored by
    tests/golden/make_golden.py): the same bytes on its sign domain; on mixed signs its unsigned order rotated
    to signed order."""
    for fn in (b200sort.order_array, b200sort.order_with_trust):
        for name, (keys, ref_out) in golden_small.items():
            a = keys.copy(); fn(a)
            assert_bit_exact(a, ref_out, f"{fn.__name__} {name}")
        for name, (keys, ref_out) in golden_mixed.items():
            a = keys.copy(); fn(a)
            assert_bit_exact(a, np.roll(ref_out, int((keys < 0).sum())), f"{fn.__name__} {name}")


def test_cxx_symbols_sort_in_place_like_the_reference_header_says():
    L = b200sort.lib()
    for sym in ("_Z11order_arrayPii", "_Z16order_with_trustPii"):
        keys = datagen.lab_rand(65536, 100, seed=3)            # SRM/main.cpp:10
        a = keys.copy()
        getattr(L, sym)(a.ctypes.data, a.size)
        assert_bit_exact(a, oracle.order_array(keys), sym)


def test_reference_drivers_link_and_run_unmodified(tmp_path):
    """build/sort and build/performaceTest are the reference's main.cpp / performanceTest.cpp,
    compiled from the reference checkout by `make drivers`, linked against libb200sort.so."""
    for exe in ("sort", "performaceTest"):
        path = os.path.join(ROOT, "build", exe)
        if not os.path.exists(path):
            pytest.skip("build/%s not prebuilt (make drivers needs /root/reference)" % exe)
        r = subprocess.run([path], cwd=tmp_path, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
    rows = open(tmp_path / "output.txt").read().strip().splitlines()
    assert rows[0] == "Size,Time,Algorithm" and len(rows) == 1 + 2 * 9      # SRM/main.cpp:21,35-44
    assert rows[1].startswith("256,") and rows[1].endswith(",Our")


def test_checked_driver(tmp_path):
    path = os.path.join(ROOT, "build", "b200sort_driver")
    if not os.path.exists(path):
        pytest.skip("build/b200sort_driver not built")
    r = subprocess.run([path, "--min", "256", "--max", "1048576", "--dist", "uniform", "--check"],
                       cwd=tmp_path, capture_output=True, text=True, timeout=300)   # it writes output.txt
    assert r.returncode == 0, r.stdout + r.stderr
    assert "MISMATCH" not in r.stdout


@pytest.mark.skipif(not oracle.ref.available, reason="oracle/_ref not prebuilt")
def test_reference_gpu_sort_side_by_side():
    """The reference's own order_array (SRM/lab.cu:303-402) run on this GPU where it is launchable
    and well defined: n <= 512 (stages 1-2 only), non-negative keys.  Same bytes as ours."""
    for n in (32, 64, 256, 512):
        for dist in ("lab_rand100", "uniform_nonneg"):
            keys = datagen.make(dist, n, 4)
            ours = keys.copy(); b200sort.order_array(ours)
            assert_bit_exact(ours, oracle.ref.order_array(keys), f"{dist} n={n}")
