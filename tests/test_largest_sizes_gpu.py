"""Every sort family at the top of its range, checked exactly: n = 2^29 + 1 (the first n at which an 8-byte array
passes 4 GiB), 2^30 - 3 (a ragged last tile) and 2^30 = B200SORT_MAX_N, and segment lists filled to their worst-case
capacity.  Inputs are the constructions of tests/large_refs.py, whose sorted output is known in closed form; outputs
are compared with that form, with the exact characterization of the stable sort, or byte for byte with torch.sort.
Nothing is sorted on the host.  Every case frees what it allocated before the next, and skips (naming the bytes it
needs and the bytes free) on a card with less memory.  The checked library runs the 64-bit, indices and capacity
cases first, in a subprocess, and must count no violated kernel invariant."""
import gc
import os
import subprocess
import sys

import pytest

import b200sort
from b200sort._lib import ALGO_LAB, ALGO_MERGE, ALGO_RADIX, check, lib
from helpers import stream_ptr

import key_orders as ko32
import key_orders16 as ko16
import key_orders64 as ko64
import large_refs as R

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N30, N30M3, N29P1 = 1 << 30, (1 << 30) - 3, (1 << 29) + 1
GiB = 1 << 30
INVALID = 1
ITEM = {16: 2, 32: 4, 64: 8}
DEV = "cuda"


def _release():
    import torch
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def _need(nbytes: int) -> None:
    """Skip unless the card has ``nbytes`` (plus room for the checker's chunks) free."""
    import torch
    _release()
    want = nbytes + 4 * GiB
    free, _ = torch.cuda.mem_get_info()
    if free < want:
        pytest.skip(f"needs {want} bytes of device memory, {free} free")


@pytest.fixture(autouse=True)
def _peak_memory():
    """Frees the previous case's memory; prints this case's peak (pytest -rP shows it)."""
    import torch
    _release()
    torch.cuda.reset_peak_memory_stats()
    yield
    print(f"peak allocated: {torch.cuda.max_memory_allocated()} bytes")
    _release()


def _ws(nbytes: int):
    import torch
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=DEV)
    return ws, ws.data_ptr() + (-ws.data_ptr()) % 256, nbytes


# ---- C-ABI calls ----------------------------------------------------------------------------------------------------
def _ws_1d(b: int, n: int, algo: int = ALGO_RADIX):
    L = lib()
    return {32: lambda: L.b200sort_workspace_bytes(n, algo), 64: lambda: L.b200sort_keys64_workspace_bytes(n),
            16: lambda: L.b200sort_keys16_workspace_bytes(n)}[b]()


def sort_keys(keys, kt: int, desc: int, algo: int = ALGO_RADIX):
    """b200sort_sort_keys (32-bit, radix or merge), b200sort_sort_keys64 or b200sort_sort_keys16, out of place."""
    import torch
    L, n, b = lib(), keys.numel(), R.BITS[kt]
    out = torch.empty_like(keys)
    tmp = torch.empty_like(keys) if b != 16 else None
    ws, ptr, nb = _ws(_ws_1d(b, n, algo))
    if b == 32:
        check(L.b200sort_sort_keys(algo, kt, desc, keys.data_ptr(), out.data_ptr(), tmp.data_ptr(), n, ptr, nb,
                                   stream_ptr()))
    elif b == 64:
        check(L.b200sort_sort_keys64(kt, desc, keys.data_ptr(), out.data_ptr(), tmp.data_ptr(), n, ptr, nb,
                                     stream_ptr()))
    else:
        check(L.b200sort_sort_keys16(kt, desc, keys.data_ptr(), out.data_ptr(), n, ptr, nb, stream_ptr()))
    torch.cuda.synchronize()
    return out


def _pairs_fn(b: int):
    L = lib()
    return {32: L.b200sort_radix_pairs_keys, 64: L.b200sort_radix_pairs_keys64, 16: L.b200sort_radix_pairs_keys16}[b]


def sort_pairs(keys, vals, kt: int, desc: int, n: int | None = None):
    """(status, keys out, values out) of the 1-D radix pairs sort of the first n keys (all by default)."""
    import torch
    b = R.BITS[kt]
    n = keys.numel() if n is None else n
    kout, vout = torch.empty_like(keys), torch.empty_like(vals)
    ktmp, vtmp = torch.empty_like(keys), torch.empty_like(vals)
    ws, ptr, nb = _ws(_ws_1d(b, keys.numel()))
    st = _pairs_fn(b)(kt, desc, keys.data_ptr(), vals.data_ptr(), kout.data_ptr(), vout.data_ptr(), ktmp.data_ptr(),
                      vtmp.data_ptr(), n, ptr, nb, stream_ptr())
    torch.cuda.synchronize()
    return st, kout, vout


def sort_indices(keys, kt: int, desc: int):
    """(keys out, int64 indices) of b200sort_radix_sort_indices_keys or its 16-bit twin."""
    import torch
    L, n, b = lib(), keys.numel(), R.BITS[kt]
    kout, ktmp = torch.empty_like(keys), torch.empty_like(keys)
    idx = torch.empty(n, dtype=torch.int64, device=DEV)
    itmp = torch.empty(n, dtype=torch.int32, device=DEV)
    ws, ptr, nb = _ws(_ws_1d(b, n))
    fn = L.b200sort_radix_sort_indices_keys if b == 32 else L.b200sort_radix_sort_indices_keys16
    check(fn(kt, desc, keys.data_ptr(), kout.data_ptr(), idx.data_ptr(), ktmp.data_ptr(), itmp.data_ptr(), n, ptr, nb,
             stream_ptr()))
    torch.cuda.synchronize()
    return kout, idx


def _check_arange(v, n: int, what: str) -> None:
    import torch
    for s in range(0, n, R.CHUNK):
        e = min(n, s + R.CHUNK)
        assert torch.equal(v[s:e].to(torch.int64), torch.arange(s, e, dtype=torch.int64, device=v.device)), \
            f"{what}: not 0..n-1 in [{s}, {e})"


def _bytes_1d(n: int, b: int, copies: int, vals: int = 0) -> int:
    return n * (ITEM[b] * copies + vals)


# ---- the checked library --------------------------------------------------------------------------------------------
# what runs under it: the 64-bit and indices cases and every capacity case
CHECKED = ["test_keys_distinct[keys64_i64_asc_2^30]", "test_pairs[u64_asc_T_2^30]", "test_pairs[i64_desc_D_2^30-3]",
           "test_indices[u32_asc_D_2^29+1]", "test_indices[i32_desc_D_2^30]", "test_indices[f16_asc_T_2^30]",
           "test_indices_all_equal_2_30[f32]", "test_indices_all_equal_2_30[i16]"] + [
    f"test_segmented[{f}-{s}]" for f in ("keys32", "pairs32", "indices32", "keys16", "pairs16", "indices16", "keys64",
                                         "pairs64")
    for s in ("one_segment", "cap0", "cap1", "cap2", "cap3", "ones")
    if s.startswith("cap") or f.startswith("indices") or f.endswith("64")]


def test_checked_library_counts_no_violations():
    """The self-asserting build (make checked) runs the 64-bit, indices and capacity cases of this module: its bounds
    checks count a bad position instead of writing through it, and check site 15 counts segments a full list drops.
    Defined first, so it runs before the product library meets these cases."""
    lib_path = os.path.join(ROOT, os.path.basename(os.path.dirname(b200sort.__file__)), "libb200sort_checked.so")
    if not os.path.exists(lib_path):
        pytest.skip("checked library not built (make checked)")
    here = os.path.abspath(__file__)
    code = f"""
import ctypes, sys
import pytest
rc = pytest.main(["-q", "-p", "no:cacheprovider", *[{here!r} + "::" + c for c in {CHECKED!r}]])
from b200sort._lib import lib
assert lib().b200sort_debug_checked_build() == 1
sites = (ctypes.c_ulonglong * 16)()
fails = int(lib().b200sort_debug_check_failures_by_site(ctypes.cast(sites, ctypes.c_void_p)))
print('per check site:', list(sites), flush=True)
print(f'CHECKED BUILD: {{fails}} violated', flush=True)
sys.exit(int(rc))
"""
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT,
                       env={**os.environ, "B200SORT_LIB": "libb200sort_checked.so"},
                       capture_output=True, text=True, timeout=3000)
    assert r.returncode == 0 and "CHECKED BUILD: 0 violated" in r.stdout and " passed" in r.stdout, \
        r.stdout[-6000:] + r.stderr[-3000:]
    assert "skipped" not in r.stdout, r.stdout[-6000:]
    print(r.stdout[-1500:])


# ---- 1-D: keys only -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kt,desc,n,algo", [
    (ko32.KEY_U32, 1, N30M3, ALGO_RADIX),
    (ko32.KEY_I32, 0, N30, ALGO_MERGE), (ko32.KEY_I32, 0, N30M3, ALGO_MERGE),
    (ko32.KEY_F32, 1, N30, ALGO_MERGE), (ko32.KEY_F32, 1, N30M3, ALGO_MERGE),
    (ko64.KEY_I64, 0, N30, ALGO_RADIX),
], ids=["radix_u32_desc_2^30-3", "merge_i32_asc_2^30", "merge_i32_asc_2^30-3", "merge_f32_desc_2^30",
        "merge_f32_desc_2^30-3", "keys64_i64_asc_2^30"])
def test_keys_distinct(kt, desc, n, algo):
    """Construction D: every digit varies (the 64-bit sort runs all 8 passes); keys byte for byte."""
    _need(_bytes_1d(n, R.BITS[kt], 3) + (n * 8 if algo == ALGO_MERGE else 0))
    keys, case = R.build(n, kt, desc, None, DEV)
    out = sort_keys(keys, kt, desc, algo)
    del keys
    R.check_keys(out, case, f"{R.NAMES[kt]} desc={desc} n={n} algo={algo}")


def test_lab_i32_distinct_2_30():
    """The lab's staged pipeline (b200sort_sort_i32 with ALGO_LAB) at n = 2^30, in place."""
    import torch
    n = N30
    _need(_bytes_1d(n, 32, 2) + lib().b200sort_workspace_bytes(n, ALGO_LAB))
    keys, case = R.build(n, ko32.KEY_I32, 0, None, DEV)
    tmp = torch.empty_like(keys)
    ws, ptr, nb = _ws(lib().b200sort_workspace_bytes(n, ALGO_LAB))
    check(lib().b200sort_sort_i32(ALGO_LAB, keys.data_ptr(), tmp.data_ptr(), n, ptr, nb, stream_ptr()))
    torch.cuda.synchronize()
    del tmp, ws
    R.check_keys(keys, case, "lab n=2^30")


def _random_bits(n: int, kt: int, seed: int):
    """Random bit patterns of kt's width, with -0.0, +0.0 and NaNs of both signs planted at spread positions."""
    import torch
    b = R.BITS[kt]
    g = torch.Generator(device=DEV); g.manual_seed(seed)
    out = torch.empty(n, dtype=R.int_dtype(torch, kt), device=DEV)
    for s in range(0, n, R.CHUNK):
        e = min(n, s + R.CHUNK)
        w = torch.randint(-(1 << 63), (1 << 63) - 1, (e - s,), dtype=torch.int64, device=DEV, generator=g)
        if b < 64:                                                # the low b bits, sign-extended: no narrowing cast
            w = ((w & ((1 << b) - 1)) ^ (1 << (b - 1))) - (1 << (b - 1))
        out[s:e] = w
    top = -(1 << (b - 1))
    specials = torch.tensor([top, 0, -1, (1 << (b - 1)) - 1, top + 1, 1], dtype=out.dtype, device=DEV)
    at = torch.arange(specials.numel(), device=DEV) * (n // specials.numel()) + 17
    out[at] = specials
    out[n - 1] = top
    return out.view(R.torch_dtype(torch, kt))


@pytest.mark.parametrize("kt,desc,n", [(ko32.KEY_F32, 0, N30), (ko64.KEY_F64, 1, N29P1), (ko16.KEY_U16, 1, N30M3)],
                         ids=["radix_f32_asc_2^30", "keys64_f64_desc_2^29+1", "keys16_u16_desc_2^30-3"])
def test_keys_random_equal_torch_sort_of_images(kt, desc, n):
    """Random bit patterns, float NaNs and -0.0 included, byte for byte against torch.sort of the images."""
    _need(_bytes_1d(n, R.BITS[kt], 2) + n * 8 * 4)
    keys = _random_bits(n, kt, 30 + kt)
    out = sort_keys(keys, kt, desc)
    _release()
    R.check_sorted_like_torch(out, keys, kt, desc, f"{R.NAMES[kt]} desc={desc} n={n}")


# ---- 1-D: pairs -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kt,desc,n,t", [
    (ko32.KEY_I32, 0, N30, 8), (ko32.KEY_F32, 1, N30M3, None),
    (ko64.KEY_U64, 0, N30, 8), (ko64.KEY_I64, 1, N30M3, None),
    (ko16.KEY_BF16, 1, N30, 14), (ko16.KEY_I16, 0, N30M3, 14),
], ids=["i32_asc_T_2^30", "f32_desc_D_2^30-3", "u64_asc_T_2^30", "i64_desc_D_2^30-3", "bf16_desc_T_2^30",
        "i16_asc_T_2^30-3"])
def test_pairs(kt, desc, n, t):
    """Stable sort-by-key with values 0..n-1: D checked against pi^-1, T by the characterization."""
    import torch
    _need(_bytes_1d(n, R.BITS[kt], 3, 12))
    keys, case = R.build(n, kt, desc, t, DEV)
    vals = torch.arange(n, dtype=torch.int32, device=DEV)
    st, kout, vout = sort_pairs(keys, vals, kt, desc)
    check(st)
    del vals
    _release()
    what = f"pairs {R.NAMES[kt]} desc={desc} n={n} t={t}"
    R.check_keys(kout, case, what)
    if t is None:
        R.check_values_d(vout, case, what)
    else:
        R.check_pairs(keys, kout, vout, kt, desc, what)


def test_pairs_all_equal_2_30_skips_every_pass():
    import torch
    n = N30
    _need(_bytes_1d(n, 32, 3, 12))
    keys = torch.full((n,), -0x2468ACE, dtype=torch.int32, device=DEV)
    vals = torch.arange(n, dtype=torch.int32, device=DEV)
    st, kout, vout = sort_pairs(keys, vals, ko32.KEY_I32, 1)
    check(st)
    del keys, vals
    assert bool((kout == -0x2468ACE).all())
    _check_arange(vout, n, "all-equal pairs")


@pytest.mark.parametrize("b", [32, 64])
def test_pairs_with_skipping_off(b):
    """With b200sort_radix_set_skip(0) a digit count of 2^30 cannot be held: n = 2^30 is refused before any device
    work; for 32-bit keys n = 2^30 - 1 (construction D) still sorts, every pass executed."""
    import torch
    n = N30
    kt = ko32.KEY_U32 if b == 32 else ko64.KEY_I64
    _need(_bytes_1d(n, b, 3, 12))
    L = lib()
    keys = torch.zeros(n, dtype=R.torch_dtype(torch, kt), device=DEV)
    vals = torch.arange(n, dtype=torch.int32, device=DEV)
    try:
        L.b200sort_radix_set_skip(0)
        st, kout, vout = sort_pairs(keys, vals, kt, 0)
        assert st == INVALID, f"n = 2^30 with skipping off: status {st}"
        if b == 32:
            d, case = R.build(n - 1, kt, 1, None, DEV)
            keys[:n - 1] = d
            del d, kout, vout
            st, kout, vout = sort_pairs(keys, vals, kt, 1, n - 1)
            check(st)
            del keys, vals
            _release()
            R.check_keys(kout[:n - 1], case, "skip off, n = 2^30 - 1")
            R.check_values_d(vout[:n - 1], case, "skip off, n = 2^30 - 1")
    finally:
        L.b200sort_radix_set_skip(1)


# ---- 1-D: indices ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kt,desc,n,t", [
    (ko32.KEY_U32, 0, N29P1, None), (ko32.KEY_I32, 1, N30, None), (ko16.KEY_F16, 0, N30, 14),
], ids=["u32_asc_D_2^29+1", "i32_desc_D_2^30", "f16_asc_T_2^30"])
def test_indices(kt, desc, n, t):
    _need(_bytes_1d(n, R.BITS[kt], 3, 12))
    keys, case = R.build(n, kt, desc, t, DEV)
    kout, idx = sort_indices(keys, kt, desc)
    _release()
    what = f"indices {R.NAMES[kt]} desc={desc} n={n} t={t}"
    R.check_keys(kout, case, what)
    if t is None:
        R.check_values_d(idx, case, what)
    else:
        R.check_pairs(keys, kout, idx, kt, desc, what)


@pytest.mark.parametrize("kt", [ko32.KEY_F32, ko16.KEY_I16], ids=["f32", "i16"])
def test_indices_all_equal_2_30(kt):
    """Every pass skipped: the final kernel writes 0..2^30 - 1 as int64, 8 GiB."""
    import torch
    n = N30
    _need(_bytes_1d(n, R.BITS[kt], 3, 12))
    keys = torch.full((n,), 0x1357, dtype=R.int_dtype(torch, kt), device=DEV).view(R.torch_dtype(torch, kt))
    kout, idx = sort_indices(keys, kt, 1)
    assert torch.equal(R.ints(kout, kt), R.ints(keys, kt))
    del keys, kout
    _check_arange(idx, n, "all-equal indices")


def test_sort_with_indices_randn_equals_torch_sort():
    """b200sort.sort_with_indices on float32 randn at 2^30 against torch.sort(stable=True), values and indices."""
    import torch
    n = N30
    _need(n * (4 * 4 + 8 * 3))
    g = torch.Generator(device=DEV); g.manual_seed(2030)
    x = torch.randn(n, device=DEV, generator=g)
    vals, idx = b200sort.sort_with_indices(x)
    _release()
    torch.cuda.reset_peak_memory_stats()
    before = torch.cuda.memory_allocated()
    ref = torch.sort(x, stable=True)
    torch.cuda.synchronize()
    print(f"torch.sort(stable=True) of 2^30 float32: peak {torch.cuda.max_memory_allocated() - before} bytes above "
          f"what was allocated before it")
    assert torch.equal(vals.view(torch.int32), ref.values.view(torch.int32)), "values differ from torch.sort"
    assert torch.equal(idx, ref.indices), "indices differ from torch.sort"


# ---- segmented ------------------------------------------------------------------------------------------------------
FAMILIES = [("keys", 32), ("pairs", 32), ("indices", 32), ("keys", 16), ("pairs", 16), ("indices", 16),
            ("keys", 64), ("pairs", 64)]
FAMILY_IDS = [f"{f}{b}" for f, b in FAMILIES]
WIDTH_ORDERS = {32: ko32.ORDERS, 16: ko16.ORDERS, 64: ko64.ORDERS}
SHAPES = ["one_segment", "cap0", "cap1", "cap2", "cap3", "rows_2^17_desc", "rows_1024_asc", "ones", "mixed"]


def _class_max(b: int, c: int) -> int:
    L = lib()
    return {32: L.b200sort_segmented_class_max, 16: L.b200sort_segmented16_class_max,
            64: L.b200sort_segmented64_class_max}[b](c)


def _seg_ws_bytes(b: int, n: int, S: int) -> int:
    L = lib()
    return {32: L.b200sort_segmented_workspace_bytes, 16: L.b200sort_segmented16_workspace_bytes,
            64: L.b200sort_segmented64_workspace_bytes}[b](n, S)


def offsets_for(shape: str, b: int, n: int = N30):
    """int32 device offsets of a shape."""
    import torch
    if shape == "one_segment":
        return torch.tensor([0, n], dtype=torch.int32, device=DEV)
    if shape.startswith("cap"):
        # every segment one longer than class c's longest, so the list of the class after c receives exactly
        # n // (class_max(c) + 1) segments: its worst-case capacity.  The remainder is a shorter trailing segment.
        ln = _class_max(b, int(shape[3:])) + 1
        count = n // ln
        offs = torch.arange(count + 1, dtype=torch.int64, device=DEV) * ln
        if offs[-1] != n:
            offs = torch.cat([offs, torch.tensor([n], dtype=torch.int64, device=DEV)])
        return offs.to(torch.int32)
    if shape.startswith("rows"):
        ln = 1 << 17 if "17" in shape else 1024
        return (torch.arange(n // ln + 1, dtype=torch.int64, device=DEV) * ln).to(torch.int32)
    if shape == "ones":
        return torch.arange(n + 1, dtype=torch.int32, device=DEV)
    assert shape == "mixed"
    # 2^30 segments again, periods of 512: 506 empty ones between lengths 300, 129 (CTA classes), 60, 20, 2 (warp
    # class) and 1 (copied)
    period = torch.zeros(512, dtype=torch.int32, device=DEV)
    period[torch.tensor([1, 7, 100, 200, 301, 511], device=DEV)] = torch.tensor(
        [300, 129, 60, 20, 2, 1], dtype=torch.int32, device=DEV)
    assert int(period.sum()) == 512 and n % 512 == 0
    offs = torch.zeros(n + 1, dtype=torch.int32, device=DEV)
    offs[1:] = period.repeat(n // 512).cumsum(0, dtype=torch.int32)
    return offs


def _order(family_index: int, shape: str, b: int):
    """(key type, descending): rotated over the width's orders so every (family, shape) meets another one; the rows
    shapes fix the direction."""
    orders = WIDTH_ORDERS[b]
    kt, desc = orders[(family_index + SHAPES.index(shape)) % len(orders)]
    if shape.startswith("rows"):
        desc = 1 if "17" in shape else 0
    return kt, desc


def _python_rows(form: str, b: int, keys, rows: int, desc: int):
    """The torch-facing rows path of each family."""
    import torch
    x = keys.view(rows, -1)
    fn = {("keys", 32): b200sort.segmented_sort, ("keys", 16): b200sort.segmented_sort16,
          ("keys", 64): b200sort.segmented_sort64, ("pairs", 32): b200sort.segmented_sort_by_key,
          ("pairs", 16): b200sort.segmented_sort16_by_key, ("pairs", 64): b200sort.segmented_sort64_by_key,
          ("indices", 32): b200sort.segmented_sort_with_indices,
          ("indices", 16): b200sort.segmented_sort16_with_indices}[(form, b)]
    if form == "pairs":
        v = torch.arange(x.shape[1], dtype=torch.int32, device=DEV).repeat(rows).view(rows, -1)
        k, vo = fn(x, v, descending=bool(desc))
        return k.view(-1), vo.view(-1)
    if form == "indices":
        k, vo = fn(x, descending=bool(desc))
        return k.view(-1), vo.view(-1)
    return fn(x, descending=bool(desc)).view(-1), None


def seg_sort(form: str, keys, offs, kt: int, desc: int):
    """(keys out, local positions or None) of a segmented C-ABI call, out of place."""
    import torch
    L, n, b, S = lib(), keys.numel(), R.BITS[kt], offs.numel() - 1
    kout, ktmp = torch.empty_like(keys), torch.empty_like(keys)
    ws, ptr, nb = _ws(_seg_ws_bytes(b, n, S))
    st = stream_ptr()
    v = None
    if form == "keys":
        fn = {32: L.b200sort_segmented_sort_keys, 16: L.b200sort_segmented_sort_keys16,
              64: L.b200sort_segmented_sort_keys64}[b]
        check(fn(kt, desc, keys.data_ptr(), kout.data_ptr(), ktmp.data_ptr(), n, offs.data_ptr(), S, ptr, nb, st))
    elif form == "pairs":
        fn = {32: L.b200sort_segmented_pairs_keys, 16: L.b200sort_segmented_pairs_keys16,
              64: L.b200sort_segmented_pairs_keys64}[b]
        vin = R.local_positions(offs)
        v, vtmp = torch.empty_like(vin), torch.empty_like(vin)
        check(fn(kt, desc, keys.data_ptr(), vin.data_ptr(), kout.data_ptr(), v.data_ptr(), ktmp.data_ptr(),
                 vtmp.data_ptr(), n, offs.data_ptr(), S, ptr, nb, st))
    else:
        fn = {32: L.b200sort_segmented_sort_indices_keys, 16: L.b200sort_segmented_sort_indices_keys16}[b]
        v = torch.empty(n, dtype=torch.int64, device=DEV)
        itmp = torch.empty(n, dtype=torch.int32, device=DEV)
        check(fn(kt, desc, keys.data_ptr(), kout.data_ptr(), v.data_ptr(), ktmp.data_ptr(), itmp.data_ptr(), n,
                 offs.data_ptr(), S, ptr, nb, st))
    torch.cuda.synchronize()
    return kout, v


def run_segmented(family_index: int, shape: str) -> None:
    form, b = FAMILIES[family_index]
    kt, desc = _order(family_index, shape, b)
    n = N30
    S = n if shape in ("ones", "mixed") else 0
    _need(n * (3 * ITEM[b] + (12 if form == "pairs" else 12 if form == "indices" else 0)) + S * 4 + (
        _seg_ws_bytes(b, n, max(S, 1))))
    offs = offsets_for(shape, b, n)
    S = offs.numel() - 1
    if shape.startswith("cap"):
        c = int(shape[3:])
        ln = _class_max(b, c) + 1
        assert n // ln == min(S, n // ln), "the class after c receives exactly its worst-case capacity"
    keys, case = R.build_segmented(offs, kt, desc)
    if shape.startswith("rows"):
        kout, v = _python_rows(form, b, keys, S, desc)
    else:
        kout, v = seg_sort(form, keys, offs, kt, desc)
    _release()
    what = f"segmented {form} {R.NAMES[kt]} desc={desc} shape={shape} S={S} t={case.t}"
    R.check_seg_keys(kout, offs, case, what)
    if v is not None:
        R.check_seg_pairs(keys, kout, v, offs, kt, desc, what)


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("family_index", range(len(FAMILIES)), ids=FAMILY_IDS)
def test_segmented(family_index, shape):
    """(a) one segment of 2^30 keys, no pass skipped; (b) every list of the classifier filled to exactly its
    worst-case capacity; (c) rows of 2^17 descending and of 1024 ascending through the Python rows path; (d) 2^30
    segments: all of length 1, and empty ones mixed with longer ones (4 GiB of offsets)."""
    run_segmented(family_index, shape)
