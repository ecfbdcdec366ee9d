#!/usr/bin/env python
"""What compute-sanitizer runs (tools/sanitize.sh): every kernel family once at smoke sizes, each result checked
against the oracle.  `python tools/sanitize_target.py [big | keys16 | segmented16]` -- `big` adds one 2^20-key radix sort; `keys16` runs
only the 16-bit sorts, `segmented16` only the segmented sort of 16-bit keys,
`segmented64` only the segmented sort of 64-bit keys."""
import ctypes
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

import oracle
from b200sort import datagen
from b200sort import dist as b200dist
from b200sort._lib import ALGO_LAB, ALGO_MERGE, ALGO_RADIX, check, lib
from helpers import gpu_sort, stream_ptr, to_device, workspace

L = lib()
check(L.b200sort_device_check())
big = len(sys.argv) > 1 and sys.argv[1] == "big"
n = 1 << 16


def same(a, b, what):
    assert a.tobytes() == b.tobytes(), what
    print("  ok", what, flush=True)


def keys16_runs(full_size):
    """16-bit keys: the counting sort and the pairs passes, keys off a 16-byte boundary, a skipped pass."""
    import key_orders16 as ko16
    from test_keys16_gpu import check_both, low_entropy, random_keys
    sizes = (n + 123, (1 << 22) + 77) if full_size else (n + 123,)
    for m in sizes:
        check_both(random_keys(m, ko16.KEY_BF16, 14), ko16.KEY_BF16, 1, f"16-bit keys and pairs n={m} bfloat16 desc",
                   offs_k=(6, 2), offs_p=(6, 2, 14))
        check_both(low_entropy("constant_high_byte", m).view(np.int16), ko16.KEY_I16, 0,
                   f"16-bit n={m} int16, pass 1 skipped")
        print("  ok 16-bit keys and pairs n =", m, flush=True)


def segmented16_runs():
    """Segmented 16-bit keys: a ragged mix covering every size class, bfloat16 descending, keys and pairs."""
    import key_orders16 as ko16
    from test_segmented16_gpu import check_pairs, mixed_keys, ragged_offsets, seg_keys, seg_sort_keys
    offs = ragged_offsets(5, total_segments=2000, big=1)
    m = int(offs[-1])
    k = mixed_keys(m, ko16.KEY_BF16, 11)
    same(seg_keys(k, offs, ko16.KEY_BF16, 1, False), ko16.bits(seg_sort_keys(k, offs, ko16.KEY_BF16, 1)),
         f"segmented 16-bit keys n={m}, {offs.size - 1} segments, bfloat16 desc")
    check_pairs(k, offs, ko16.KEY_BF16, 1, False, "segmented 16-bit pairs")
    check_pairs((k.view(np.uint16) % np.uint16(50)).view(np.int16), offs, ko16.KEY_I16, 0, True,
                "segmented 16-bit pairs in place, many ties")
    print("  ok segmented 16-bit pairs (stable)", flush=True)


def segmented64_runs():
    """Segmented 64-bit keys: a ragged mix covering every size class, every order, keys and pairs, copied and in place,
    with executed and skipped passes."""
    import key_orders64 as ko64
    from test_segmented64_gpu import check_all, every_class_layout, random_keys, varying_bytes
    offs = ragged_offsets(5, total_segments=2000, big=1)
    m = int(offs[-1])
    for kt, desc in ko64.ORDERS:
        check_all(random_keys(m, kt, 11 + kt + desc), offs, kt, desc, f"segmented 64-bit n={m} {kt},{desc}")
        print(f"  ok segmented 64-bit keys and pairs n={m}, {offs.size - 1} segments, order {kt},{desc}", flush=True)
    offs = every_class_layout(6)
    for mask in (0x00, 0x0F, 0xF0, 0x5A, 0x81, 0xFF):
        check_all(varying_bytes(int(offs[-1]), mask, mask).view(np.int64), offs, ko64.KEY_I64, 0, f"mask {mask:#x}")
    print("  ok segmented 64-bit skipped-pass patterns", flush=True)


def report_checked():
    sites = (ctypes.c_ulonglong * 16)()
    fails = int(L.b200sort_debug_check_failures_by_site(ctypes.cast(sites, ctypes.c_void_p)))
    print('per check site:', list(sites), flush=True)
    print(f"CHECKED BUILD: {fails} violated kernel invariants (staged positions, destination indices, bulk-copy alignment)", flush=True)
    assert fails == 0


if len(sys.argv) > 1 and sys.argv[1] == "keys16":      # only the 16-bit sorts, at smoke and full size
    keys16_runs(True)
    if L.b200sort_debug_checked_build():
        report_checked()
    print("SANITIZE TARGET PASSED", flush=True)
    sys.exit(0)


if len(sys.argv) > 1 and sys.argv[1] == "segmented64":  # only the segmented sort of 64-bit keys
    from test_segmented_gpu import ragged_offsets  # noqa: E402
    segmented64_runs()
    if L.b200sort_debug_checked_build():
        report_checked()
    print("SANITIZE TARGET PASSED", flush=True)
    sys.exit(0)
if len(sys.argv) > 1 and sys.argv[1] == "segmented16":  # only the segmented sort of 16-bit keys
    segmented16_runs()
    if L.b200sort_debug_checked_build():
        report_checked()
    print("SANITIZE TARGET PASSED", flush=True)
    sys.exit(0)


keys = datagen.uniform(n, 3)
want = oracle.radix_sort(keys)
skew = datagen.skewed(n + 123, 4)
for v in range(L.b200sort_radix_num_variants()):
    name = L.b200sort_radix_variant_name(v).decode()
    if name.startswith("TIMING_"):
        continue
    check(L.b200sort_radix_set_variant(v))
    same(gpu_sort(keys, ALGO_RADIX), want, f"radix shape {v} {name} n=2^16 uniform")
    same(gpu_sort(skew, ALGO_RADIX), oracle.radix_sort(skew), f"radix shape {v} n=2^16+123 skewed90 (hot-digit path, ragged tile)")
check(L.b200sort_radix_set_variant(0))
if big:
    k20 = datagen.uniform(1 << 20, 5)
    same(gpu_sort(k20, ALGO_RADIX), oracle.radix_sort(k20), "radix default n=2^20 uniform")
small = datagen.uniform(5000, 6)
same(gpu_sort(small, ALGO_RADIX), oracle.radix_sort(small), "one-CTA kernel n=5000")
same(gpu_sort(keys, ALGO_MERGE), want, "merge sort n=2^16")
same(gpu_sort(skew, ALGO_MERGE), oracle.radix_sort(skew), "merge sort n=2^16+123")
same(gpu_sort(keys, ALGO_LAB), want, "lab pipeline n=2^16")
# sort-by-key
vals = np.arange(n, dtype=np.int32)
ties = datagen.lab_rand(n, 100, seed=2)
wk, wv = oracle.sort_pairs(ties, vals)
dk, dv = to_device(ties), to_device(vals)
tk, tv = torch.empty_like(dk), torch.empty_like(dv)
ws, ptr, nb = workspace(n, ALGO_RADIX)
check(L.b200sort_radix_pairs_i32(dk.data_ptr(), dv.data_ptr(), tk.data_ptr(), tv.data_ptr(), n, ptr, nb, stream_ptr()))
torch.cuda.synchronize()
same(dk.cpu().numpy(), wk, "pairs: keys"); same(dv.cpu().numpy(), wv, "pairs: values (stable)")
# multi-GPU kernels with simulated ranks on one device
world, bits = 4, 12
srcs = [datagen.make("uniform", 40000 + 100 * r, seed=20 + r) for r in range(world)]
all_hist = np.stack([b200dist.host_histogram(k, bits) for k in srcs])
plans = [b200dist.plan(all_hist, r, bits) for r in range(world)]
owner, recv = plans[0][0], plans[0][1]
bufs = [torch.full((max(int(recv[r]), 1),), -7, dtype=torch.int32, device="cuda") for r in range(world)]
base = (ctypes.c_void_p * world)(*[b.data_ptr() for b in bufs])
owner_dev = to_device(owner)
pws = torch.zeros(512, dtype=torch.uint8, device="cuda")
pws_ptr = pws.data_ptr() + (-pws.data_ptr()) % 256
for s in range(world):
    d = to_device(srcs[s])
    hist = torch.zeros(1 << bits, dtype=torch.int64, device="cuda")
    check(L.b200sort_dist_histogram_i32(d.data_ptr(), d.numel(), bits, hist.data_ptr(), stream_ptr()))
    assert (hist.cpu().numpy().astype(np.uint64) == all_hist[s]).all()
    check(L.b200sort_dist_partition_i32(d.data_ptr(), d.numel(), bits, world, base, owner_dev.data_ptr(),
                                        plans[s][3].ctypes.data, pws_ptr, 256, stream_ptr()))
    torch.cuda.synchronize()
everything = np.concatenate(srcs)
top = (everything.view(np.uint32) ^ np.uint32(0x80000000)) >> np.uint32(32 - bits)
dest = owner[top.astype(np.int64)]
for r in range(world):
    same(np.sort(bufs[r].cpu().numpy()[:int(recv[r])]), np.sort(everything[dest == r]), f"dist partition: destination {r}")
# segmented sort: every size class at once (empty, one-key, warp, both CTA capacities, onesweep), keys and pairs
import key_orders as ko  # noqa: E402
from test_segmented_gpu import ragged_offsets, seg_keys, seg_pairs, seg_sort_keys, seg_sort_pairs  # noqa: E402
seg_offs = ragged_offsets(5, total_segments=2000, big=1)
seg_n = int(seg_offs[-1])
seg_k = (datagen.uniform_u32(seg_n, 11) % np.uint32(1000)).astype(np.float32)
same(seg_keys(seg_k, seg_offs, ko.KEY_F32, 1, False), ko.bits(seg_sort_keys(seg_k, seg_offs, ko.KEY_F32, 1)),
     f"segmented keys n={seg_n}, {seg_offs.size - 1} segments")
seg_gk, seg_gv = seg_pairs(seg_k, np.arange(seg_n, dtype=np.int32), seg_offs, ko.KEY_F32, 0, True)
seg_wk, seg_wv = seg_sort_pairs(seg_k, np.arange(seg_n, dtype=np.int32), seg_offs, ko.KEY_F32, 0)
same(seg_gk, ko.bits(seg_wk), "segmented pairs: keys"); same(seg_gv, seg_wv, "segmented pairs: values (stable)")
# 64-bit keys: keys only and pairs, a ragged last tile, every pass executed and a skipped half
import key_orders64 as ko64  # noqa: E402
from test_keys64_gpu import low_entropy, random_keys, sort64_keys, sort64_pairs  # noqa: E402
k64 = random_keys(n + 123, ko64.KEY_F64, 12)
same(sort64_keys(k64, ko64.KEY_F64, 1, False), ko64.bits(ko64.sort_keys(k64, ko64.KEY_F64, 1)), "64-bit keys n=2^16+123 float64 desc")
k64 = low_entropy("below_2_32", n + 45).view(np.int64)
k64_gk, k64_gv = sort64_pairs(k64, np.arange(k64.size, dtype=np.int32), ko64.KEY_I64, 0, True)
k64_wk, k64_wv = ko64.sort_pairs(k64, np.arange(k64.size, dtype=np.int32), ko64.KEY_I64, 0)
same(k64_gk, ko64.bits(k64_wk), "64-bit pairs: keys (4 passes skipped)"); same(k64_gv, k64_wv, "64-bit pairs: values (stable)")
keys16_runs(False)
segmented16_runs()
# host operator
h = datagen.lab_rand(4096, 100, seed=1)
wh = oracle.order_array(h)
a = h.copy(); check(L.b200sort_order_array_host(a.ctypes.data, a.size, ALGO_RADIX)); same(a, wh, "order_array host operator")
L.b200sort_host_release()
if L.b200sort_debug_checked_build():
    # full-size runs too: the checks cost little
    for dist_name in ("uniform", "skewed90", "ascending"):
        k = datagen.make(dist_name, (1 << 24) + 4321, 8)
        same(gpu_sort(k, ALGO_RADIX), oracle.radix_sort(k), f"radix default n=2^24+4321 {dist_name}")
    check(L.b200sort_radix_set_variant(1))
    k = datagen.uniform((1 << 24) + 4321, 9)
    same(gpu_sort(k, ALGO_RADIX), oracle.radix_sort(k), "radix small-tile shape n=2^24+4321 uniform")
    check(L.b200sort_radix_set_variant(0))
    for dist_name in ("zipf16", "and3", "edge_mix"):
        k = datagen.make(dist_name, (1 << 23) + 77, 10)
        same(gpu_sort(k, ALGO_RADIX), oracle.radix_sort(k), f"radix default n=2^23+77 {dist_name}")
    k64 = random_keys((1 << 22) + 77, ko64.KEY_I64, 13)
    same(sort64_keys(k64, ko64.KEY_I64, 0, True), ko64.bits(ko64.sort_keys(k64, ko64.KEY_I64, 0)), "64-bit keys n=2^22+77 int64")
    k64_gk, k64_gv = sort64_pairs(k64, np.arange(k64.size, dtype=np.int32), ko64.KEY_I64, 1, False)
    k64_wk, k64_wv = ko64.sort_pairs(k64, np.arange(k64.size, dtype=np.int32), ko64.KEY_I64, 1)
    same(k64_gk, ko64.bits(k64_wk), "64-bit pairs n=2^22+77: keys"); same(k64_gv, k64_wv, "64-bit pairs: values")
    keys16_runs(True)
    report_checked()
print("SANITIZE TARGET PASSED", flush=True)
