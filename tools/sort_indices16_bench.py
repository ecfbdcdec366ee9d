#!/usr/bin/env python
"""Sort with indices of 16-bit keys against the routes a caller has without it, at 2^28 keys (DESIGN section 4.2j).

    python tools/sort_indices16_bench.py [--log2n 28] [--reps 10] [--out profiles/r09_sort_indices16.json]

Routes, each timed with CUDA events around the whole route (buffers allocated once, outside the timed window):
  new     b200sort_radix_sort_indices_keys16 / b200sort_segmented_sort_indices_keys16: keys and int64 indices in one
          call;
  route3  torch.arange (1-D) or arange(L).repeat(B) (rows) as int32, b200sort_radix_pairs_keys16 /
          b200sort_segmented_pairs_keys16, then .long() of the sorted values: the three calls the docstrings printed;
  torch   torch.sort(stable=True), values and int64 indices;
  widen   the keys widened to float32 (int16: int32), b200sort_radix_sort_indices_keys /
          b200sort_segmented_sort_indices_keys, the values narrowed back.
Inputs: bfloat16 normals 1-D ascending; bfloat16 normals in rows of L = 256, 1024, 32000 and 128256, descending
(B = 2^28 // L rows); int16 in [-100, 100] 1-D ascending (narrow digits: the high byte takes two values); all-equal
bfloat16 keys 1-D (both passes skipped).  Every route's outputs are checked against torch.sort in the same run.  The
card's name, power limit and SM clock limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

from b200sort._lib import ALGO_RADIX, check, lib

KEY_I32, KEY_F32, KEY_I16, KEY_BF16 = 0, 2, 6, 9
# bytes per key of each route's algorithmic traffic (DESIGN 4.2j): 1-D and onesweep class / CTA classes
BYTE_MODEL = {"new": (26, 12), "route3": (42, 28)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else ""
    return {"name": torch.cuda.get_device_name(), "nvidia_smi": line}


def aligned_ws(nbytes):
    t = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
    return t, t.data_ptr() + (-t.data_ptr()) % 256, nbytes


def timed(fn, reps):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    ms.sort()
    return {"ms_median": ms[len(ms) // 2], "ms_min": ms[0], "ms_max": ms[-1], "reps": reps}


def workload(name, x, kt, desc, L_row, reps):
    Ls = lib()
    s = torch.cuda.current_stream().cuda_stream
    n = x.numel()
    flat = x.view(-1)
    rows = n // L_row if L_row else 1
    k_out, k_tmp = torch.empty_like(flat), torch.empty_like(flat)
    i_out = torch.empty(n, dtype=torch.int64, device="cuda")
    i_tmp = torch.empty(n, dtype=torch.int32, device="cuda")
    v_out = torch.empty(n, dtype=torch.int32, device="cuda")
    wide_dtype = torch.int32 if kt == KEY_I16 else torch.float32
    wide_kt = KEY_I32 if kt == KEY_I16 else KEY_F32
    w_in, w_out, w_tmp = (torch.empty(n, dtype=wide_dtype, device="cuda") for _ in range(3))
    if L_row:
        offs = torch.arange(rows + 1, dtype=torch.int32, device="cuda") * L_row
        ws = aligned_ws(Ls.b200sort_segmented16_workspace_bytes(n, rows))
        ws32 = aligned_ws(Ls.b200sort_segmented_workspace_bytes(n, rows))
    else:
        ws = aligned_ws(Ls.b200sort_keys16_workspace_bytes(n))
        ws32 = aligned_ws(Ls.b200sort_workspace_bytes(n, ALGO_RADIX))
    out = {}

    def new():
        if L_row:
            check(Ls.b200sort_segmented_sort_indices_keys16(kt, desc, flat.data_ptr(), k_out.data_ptr(),
                                                            i_out.data_ptr(), k_tmp.data_ptr(), i_tmp.data_ptr(), n,
                                                            offs.data_ptr(), rows, ws[1], ws[2], s))
        else:
            check(Ls.b200sort_radix_sort_indices_keys16(kt, desc, flat.data_ptr(), k_out.data_ptr(), i_out.data_ptr(),
                                                        k_tmp.data_ptr(), i_tmp.data_ptr(), n, ws[1], ws[2], s))
        out["r"] = (k_out, i_out)

    def route3():
        if L_row:
            vals = torch.arange(L_row, dtype=torch.int32, device="cuda").repeat(rows)
            check(Ls.b200sort_segmented_pairs_keys16(kt, desc, flat.data_ptr(), vals.data_ptr(), k_out.data_ptr(),
                                                     v_out.data_ptr(), k_tmp.data_ptr(), i_tmp.data_ptr(), n,
                                                     offs.data_ptr(), rows, ws[1], ws[2], s))
        else:
            vals = torch.arange(n, dtype=torch.int32, device="cuda")
            check(Ls.b200sort_radix_pairs_keys16(kt, desc, flat.data_ptr(), vals.data_ptr(), k_out.data_ptr(),
                                                 v_out.data_ptr(), k_tmp.data_ptr(), i_tmp.data_ptr(), n, ws[1], ws[2],
                                                 s))
        out["r"] = (k_out, v_out.long())

    def tsort():
        v, i = torch.sort(x, dim=-1, stable=True, descending=bool(desc))
        out["r"] = (v.view(-1), i.view(-1))

    def widen():
        w_in.copy_(flat)
        if L_row:
            check(Ls.b200sort_segmented_sort_indices_keys(wide_kt, desc, w_in.data_ptr(), w_out.data_ptr(),
                                                          i_out.data_ptr(), w_tmp.data_ptr(), i_tmp.data_ptr(), n,
                                                          offs.data_ptr(), rows, ws32[1], ws32[2], s))
        else:
            check(Ls.b200sort_radix_sort_indices_keys(wide_kt, desc, w_in.data_ptr(), w_out.data_ptr(),
                                                      i_out.data_ptr(), w_tmp.data_ptr(), i_tmp.data_ptr(), n,
                                                      ws32[1], ws32[2], s))
        out["r"] = (w_out.to(x.dtype), i_out)

    tv, ti = torch.sort(x, dim=-1, stable=True, descending=bool(desc))
    tv, ti = tv.view(-1).view(torch.int16), ti.view(-1)
    res = {"workload": name, "dtype": str(x.dtype), "n": n, "row_length": L_row or None, "descending": desc,
           "matches_torch": {}, "routes": {}}
    routes = (("new", new), ("route3", route3), ("torch", tsort), ("widen", widen))
    for rname, fn in routes:                                  # every route's output against torch.sort, first
        fn()
        torch.cuda.synchronize()
        v, i = out.pop("r")
        res["matches_torch"][rname] = bool(torch.equal(v.view(torch.int16), tv) and torch.equal(i, ti))
    del tv, ti
    for rname, fn in routes:
        r = timed(fn, reps)
        out.clear()
        r["gkeys_per_s"] = n / (r["ms_median"] * 1e-3) / 1e9
        res["routes"][rname] = r
        print(f"{name:>26s} {rname:>7s} {r['ms_median']:8.3f} ms  ({r['gkeys_per_s']:.2f} Gkeys/s)", flush=True)
    res["new_over_route3_time"] = res["routes"]["new"]["ms_median"] / res["routes"]["route3"]["ms_median"]
    print(f"{name:>26s} outputs equal torch.sort: {res['matches_torch']}; new / route3 time "
          f"{res['new_over_route3_time']:.3f}", flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2n", type=int, default=28)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    check(lib().b200sort_device_check())
    n = 1 << a.log2n
    info = card()
    print(info, flush=True)
    g = torch.Generator(device="cuda").manual_seed(9)
    results = []
    x = torch.randn(n, generator=g, device="cuda").to(torch.bfloat16)
    x = torch.where(x == 0, torch.ones_like(x), x)           # no +-0.0: torch.sort treats them as equal
    results.append(workload("bf16_normal_1d_asc", x, KEY_BF16, 0, 0, a.reps))
    for L_row in (256, 1024, 32000, 128256):
        rows = n // L_row
        results.append(workload(f"bf16_normal_rows{L_row}_desc", x[:rows * L_row].view(rows, L_row), KEY_BF16, 1,
                                L_row, a.reps))
    del x
    xi = torch.randint(-100, 101, (n,), generator=g, device="cuda", dtype=torch.int16)
    results.append(workload("i16_pm100_1d_asc", xi, KEY_I16, 0, 0, a.reps))
    del xi
    xe = torch.full((n,), 1.5, dtype=torch.bfloat16, device="cuda")
    results.append(workload("bf16_all_equal_1d_asc", xe, KEY_BF16, 0, 0, a.reps))
    doc = {"tool": "tools/sort_indices16_bench.py", "card": info, "log2n": a.log2n,
           "byte_model_bytes_per_key": {"note": "(1-D and onesweep class, CTA classes)", **BYTE_MODEL},
           "results": results}
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(doc, f, indent=1)
    assert all(all(r["matches_torch"].values()) for r in results), "an output differs from torch.sort"


if __name__ == "__main__":
    main()
