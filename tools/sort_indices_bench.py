#!/usr/bin/env python
"""Sort with indices against the routes a caller has without it, at 2^28 keys (DESIGN section 4.2i).

    python tools/sort_indices_bench.py [--log2n 28] [--reps 10] [--out profiles/r08_sort_indices.json]

Routes, each timed with CUDA events around the whole route (buffers allocated once, outside the timed window):
  new     b200sort_radix_sort_indices_keys / b200sort_segmented_sort_indices_keys: keys and int64 indices in one call;
  route3  torch.arange (1-D) or arange(L).repeat(B) (rows) as int32, b200sort_radix_pairs_keys /
          b200sort_segmented_pairs_keys, then .long() of the sorted values: the three calls the docstrings printed;
  torch   torch.sort(stable=True), values and int64 indices.
Inputs: float32 normals 1-D ascending; float32 normals in rows of L = 256, 1024, 8192 and 2^17, descending; int32 in
[0, 2^16) 1-D, whose two upper digit passes the 1-D sorts skip.  Every route's outputs are checked against torch.sort
(or, for route3, against the new call) before timing.  The card's name and power limit are read in the same run.
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

KEY_I32, KEY_F32 = 0, 2


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
    if L_row:
        offs = torch.arange(rows + 1, dtype=torch.int32, device="cuda") * L_row
        ws = aligned_ws(Ls.b200sort_segmented_workspace_bytes(n, rows))
    else:
        ws = aligned_ws(Ls.b200sort_workspace_bytes(n, ALGO_RADIX))

    def new():
        if L_row:
            check(Ls.b200sort_segmented_sort_indices_keys(kt, desc, flat.data_ptr(), k_out.data_ptr(), i_out.data_ptr(),
                                                          k_tmp.data_ptr(), i_tmp.data_ptr(), n, offs.data_ptr(), rows,
                                                          ws[1], ws[2], s))
        else:
            check(Ls.b200sort_radix_sort_indices_keys(kt, desc, flat.data_ptr(), k_out.data_ptr(), i_out.data_ptr(),
                                                      k_tmp.data_ptr(), i_tmp.data_ptr(), n, ws[1], ws[2], s))

    out3 = {}

    def route3():
        if L_row:
            vals = torch.arange(L_row, dtype=torch.int32, device="cuda").repeat(rows)
            check(Ls.b200sort_segmented_pairs_keys(kt, desc, flat.data_ptr(), vals.data_ptr(), k_out.data_ptr(),
                                                   v_out.data_ptr(), k_tmp.data_ptr(), i_tmp.data_ptr(), n,
                                                   offs.data_ptr(), rows, ws[1], ws[2], s))
        else:
            vals = torch.arange(n, dtype=torch.int32, device="cuda")
            check(Ls.b200sort_radix_pairs_keys(kt, desc, flat.data_ptr(), vals.data_ptr(), k_out.data_ptr(),
                                               v_out.data_ptr(), k_tmp.data_ptr(), i_tmp.data_ptr(), n, ws[1], ws[2], s))
        out3["idx"] = v_out.long()

    def tsort():
        out3["t"] = torch.sort(x, dim=-1, stable=True, descending=bool(desc))

    # outputs first: new against torch.sort, route3 against new
    tsort()
    tv, ti = out3.pop("t")
    new()
    torch.cuda.synchronize()
    ok_new = torch.equal(k_out.view_as(x), tv) and torch.equal(i_out.view_as(x), ti)
    del tv, ti
    keys_new, idx_new = k_out.clone(), i_out.clone()
    route3()
    torch.cuda.synchronize()
    ok_r3 = torch.equal(k_out, keys_new) and torch.equal(out3.pop("idx"), idx_new)
    del keys_new, idx_new
    res = {"workload": name, "n": n, "row_length": L_row or None, "descending": desc, "new_matches_torch": ok_new,
           "route3_matches_new": ok_r3, "routes": {}}
    for rname, fn in (("new", new), ("route3", route3), ("torch", tsort)):
        r = timed(fn, reps)
        out3.clear()
        r["gkeys_per_s"] = n / (r["ms_median"] * 1e-3) / 1e9
        res["routes"][rname] = r
        print(f"{name:>22s} {rname:>7s} {r['ms_median']:8.3f} ms  ({r['gkeys_per_s']:.2f} Gkeys/s)", flush=True)
    print(f"{name:>22s} outputs: new == torch.sort {ok_new}, route3 == new {ok_r3}", flush=True)
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
    g = torch.Generator(device="cuda").manual_seed(8)
    results = []
    x = torch.randn(n, generator=g, device="cuda")
    results.append(workload("f32_normal_1d_asc", x, KEY_F32, 0, 0, a.reps))
    for L_row in (256, 1024, 8192, 1 << 17):
        results.append(workload(f"f32_normal_rows{L_row}_desc", x.view(-1, L_row), KEY_F32, 1, L_row, a.reps))
    del x
    xi = torch.randint(0, 1 << 16, (n,), generator=g, device="cuda", dtype=torch.int32)
    results.append(workload("i32_below_2^16_1d_asc", xi, KEY_I32, 0, 0, a.reps))
    doc = {"tool": "tools/sort_indices_bench.py", "card": info, "log2n": a.log2n, "results": results}
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(doc, f, indent=1)
    assert all(r["new_matches_torch"] and r["route3_matches_new"] for r in results), "an output differs"


if __name__ == "__main__":
    main()
