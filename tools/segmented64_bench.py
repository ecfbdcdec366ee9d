"""Time the segmented sort of 64-bit keys (b200sort_segmented_*_keys64) against torch.sort over rows, against the flat
1-D 64-bit sort of the same n, and, for ids below 2^32, against sort64 of packed (segment << 32) | key keys, on one
GPU; writes profiles/r08_segmented64.json.

Workloads at 2^28 keys in rows of L = 16, 256, 1024, 8192, 2^15, 2^17 and 2^20: uniform 64-bit int64 keys; int64 ids
below 2^32, keys only and with int32 arange values per row; float64 normal rows, descending pairs.  Then a ragged
Pareto layout of int64 ids below 2^32 (the neighbour lists of a CSR graph), keys and pairs.
Arms: "segmented64" (this library), "torch" (torch.sort(x.view(B, L), dim=-1, stable=True), with indices for pairs),
"flat" (sort64 / sort64_by_key of all n keys as one array: no segments at all), "packed" (ids only: the route a
caller has without this feature, (segment << 32) | key built and sort64 run on it, the low words taken back; for
pairs sort64_by_key on the packed keys).

Every step sorts the same pristine input out of place, larger than L2.  After a warm-up the arms take turns inside
each round and the rounds repeat, so drift of the shared machine hits every arm alike; reported per arm: the median
over rounds of the mean step time and its min / max.  After the timed steps every arm's output is checked: the
segmented one against torch.sort (rows) or for order inside every segment and an unchanged per-segment sum (ragged),
the packed one against the segmented one, the flat one for order.  The card's name and power limit are read through
NVML in the same run and stored beside the numbers.

    python tools/segmented64_bench.py [--steps 3] [--rounds 3] [--out profiles/r08_segmented64.json] [--quick]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

KEY_I64, KEY_F64 = 3, 5


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--quick", action="store_true", help="2^24 keys, for a rehearsal")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_segmented64.json"))
    args = ap.parse_args()

    import torch
    from b200sort._lib import check, lib
    from key_types_bench import card_info
    from segmented_bench import power_law_offsets

    if not torch.cuda.is_available():
        print("segmented64_bench: no GPU", file=sys.stderr)
        return 2
    torch.cuda.set_device(0)
    L = lib()
    check(L.b200sort_device_check())
    stream = torch.cuda.current_stream().cuda_stream

    def aligned(nbytes):
        ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
        return ws, ws.data_ptr() + (-ws.data_ptr()) % 256

    def sorted_in_segments(w, offs, desc):
        starts = torch.zeros(w.numel(), dtype=torch.bool, device="cuda")
        starts[offs[1:-1].to(torch.int64)] = True
        bad = (w[1:] > w[:-1]) if desc else (w[1:] < w[:-1])
        return not bool((bad & ~starts[1:]).any())

    def workload(name, src, offs, pairs, kt, desc, rows=None, ids=False):
        n = src.numel()
        S = offs.numel() - 1
        out, tmp = torch.empty_like(src), torch.empty_like(src)
        vals = (torch.arange(rows[1], dtype=torch.int32, device="cuda").repeat(rows[0]) if rows
                else torch.arange(n, dtype=torch.int32, device="cuda"))
        vout, vtmp = torch.empty_like(vals), torch.empty_like(vals)
        pvout = torch.empty_like(vals)
        seg_bytes = L.b200sort_segmented64_workspace_bytes(n, S)
        seg_ws, seg_ptr = aligned(seg_bytes)
        flat_bytes = L.b200sort_keys64_workspace_bytes(n)
        flat_ws, flat_ptr = aligned(flat_bytes)
        f_out = torch.empty_like(src)
        pristine = src.clone()
        seg_id = torch.repeat_interleave(torch.arange(S, device="cuda"), (offs[1:] - offs[:-1]).to(torch.int64))
        p_out, p_low = torch.empty_like(src), torch.empty_like(src)

        def seg():
            if pairs:
                check(L.b200sort_segmented_pairs_keys64(kt, desc, src.data_ptr(), vals.data_ptr(), out.data_ptr(),
                                                        vout.data_ptr(), tmp.data_ptr(), vtmp.data_ptr(), n,
                                                        offs.data_ptr(), S, seg_ptr, seg_bytes, stream))
            else:
                check(L.b200sort_segmented_sort_keys64(kt, desc, src.data_ptr(), out.data_ptr(), tmp.data_ptr(), n,
                                                       offs.data_ptr(), S, seg_ptr, seg_bytes, stream))

        def flat():
            if pairs:
                check(L.b200sort_radix_pairs_keys64(kt, desc, src.data_ptr(), vals.data_ptr(), f_out.data_ptr(),
                                                    vtmp.data_ptr(), tmp.data_ptr(), pvout.data_ptr(), n, flat_ptr,
                                                    flat_bytes, stream))
            else:
                check(L.b200sort_sort_keys64(kt, desc, src.data_ptr(), f_out.data_ptr(), tmp.data_ptr(), n, flat_ptr,
                                             flat_bytes, stream))

        def packed():
            p = (seg_id << 32) | src                       # ids below 2^32: the key in the low word
            if pairs:
                check(L.b200sort_radix_pairs_keys64(KEY_I64, 0, p.data_ptr(), vals.data_ptr(), p_out.data_ptr(),
                                                    pvout.data_ptr(), tmp.data_ptr(), vtmp.data_ptr(), n, flat_ptr,
                                                    flat_bytes, stream))
            else:
                check(L.b200sort_sort_keys64(KEY_I64, 0, p.data_ptr(), p_out.data_ptr(), tmp.data_ptr(), n, flat_ptr,
                                             flat_bytes, stream))
            torch.bitwise_and(p_out, 0xFFFFFFFF, out=p_low)

        arms = {"segmented64": seg, "flat": flat}
        if ids:
            arms["packed"] = packed
        if rows:
            tview = src.view(*rows)

            def tsort():
                torch.sort(tview, dim=-1, stable=True, descending=bool(desc))
            arms["torch"] = tsort
        for fn in arms.values():
            for _ in range(args.warmup):
                fn()
        torch.cuda.synchronize()
        per_round = {a: [] for a in arms}
        for _ in range(args.rounds):
            for a, fn in arms.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.steps):
                    fn()
                e1.record()
                e1.synchronize()
                per_round[a].append(e0.elapsed_time(e1) / args.steps)
        seg()
        flat()
        torch.cuda.synchronize()
        ok = bool(torch.equal(src, pristine))
        ok = ok and not bool(((f_out[1:] > f_out[:-1]) if desc else (f_out[1:] < f_out[:-1])).any())   # no NaN here
        if rows:
            tv, ti = torch.sort(src.view(*rows), dim=-1, stable=True, descending=bool(desc))
            ok = ok and bool(torch.equal(out.view(*rows), tv))
            ok = ok and (not pairs or bool(torch.equal(vout.view(*rows).to(torch.int64), ti)))
            del tv, ti
        else:
            ok = ok and sorted_in_segments(out, offs, desc)
            a = torch.zeros(S, dtype=torch.int64, device="cuda").index_add_(0, seg_id, src)
            b = torch.zeros(S, dtype=torch.int64, device="cuda").index_add_(0, seg_id, out)
            ok = ok and bool(torch.equal(a, b))
            del a, b
        if ids:
            packed()
            torch.cuda.synchronize()
            ok = ok and bool(torch.equal(p_low, out)) and (not pairs or bool(torch.equal(pvout, vout)))
        res = {"n": n, "segments": S, "rows": list(rows) if rows else None, "pairs": pairs,
               "key_type": "f64" if kt == KEY_F64 else "i64", "descending": bool(desc), "verified": ok, "arms": {}}
        for a, ms in per_round.items():
            med = statistics.median(ms)
            res["arms"][a] = {"ms_median": med, "ms_min": min(ms), "ms_max": max(ms), "gkeys_per_s": n / med / 1e6}
        seg_ms = res["arms"]["segmented64"]["ms_median"]
        for a in ("torch", "flat", "packed"):
            res[f"segmented64_vs_{a}"] = res["arms"][a]["ms_median"] / seg_ms if a in res["arms"] else None
        line = "  ".join(f"{a} {r['ms_median']:.3f} [{r['ms_min']:.3f},{r['ms_max']:.3f}]" for a, r in res["arms"].items())
        print(f"{name:34s} {line}  verified={ok}", flush=True)
        del seg_ws, flat_ws, f_out, seg_id, p_out, p_low, out, tmp
        torch.cuda.synchronize()
        return res

    result = {"card": card_info(0), "library": L.b200sort_version().decode(), "steps_per_round": args.steps,
              "rounds": args.rounds, "warmup": args.warmup, "workloads": {}}
    g = torch.Generator(device="cuda"); g.manual_seed(1)
    log2n = 24 if args.quick else 28
    for Lr in (16, 256, 1024, 8192, 1 << 15, 1 << 17, 1 << 20):
        B = max(1, (1 << log2n) // Lr)
        n = B * Lr
        offs = torch.arange(0, n + 1, Lr, dtype=torch.int32, device="cuda")
        key = f"rows_2^{log2n}_L{Lr}"
        u = torch.randint(-2**63, 2**63 - 1, (n,), dtype=torch.int64, device="cuda", generator=g)
        result["workloads"][key + "_i64_keys"] = workload(key + " i64 keys", u, offs, False, KEY_I64, 0, (B, Lr))
        del u
        ids = torch.randint(0, 2**32, (n,), dtype=torch.int64, device="cuda", generator=g)
        result["workloads"][key + "_ids_keys"] = workload(key + " ids<2^32 keys", ids, offs, False, KEY_I64, 0, (B, Lr),
                                                          ids=True)
        result["workloads"][key + "_ids_pairs"] = workload(key + " ids<2^32 pairs", ids, offs, True, KEY_I64, 0, (B, Lr),
                                                           ids=True)
        del ids
        f = torch.randn(n, device="cuda", generator=g, dtype=torch.float64)
        result["workloads"][key + "_f64_desc_pairs"] = workload(key + " f64 desc pairs", f, offs, True, KEY_F64, 1,
                                                                (B, Lr))
        del f
        torch.cuda.synchronize()
        w = result["workloads"]
        w[key + "_ids_keys"]["time_vs_uniform_keys"] = (w[key + "_ids_keys"]["arms"]["segmented64"]["ms_median"] /
                                                        w[key + "_i64_keys"]["arms"]["segmented64"]["ms_median"])
    n = 1 << log2n
    ids = torch.randint(0, 2**32, (n,), dtype=torch.int64, device="cuda", generator=g)
    offs = power_law_offsets(torch, n, 3)
    result["workloads"][f"ragged_pareto_2^{log2n}_ids_keys"] = workload("ragged Pareto ids keys", ids, offs, False,
                                                                        KEY_I64, 0, ids=True)
    result["workloads"][f"ragged_pareto_2^{log2n}_ids_pairs"] = workload("ragged Pareto ids pairs", ids, offs, True,
                                                                         KEY_I64, 0, ids=True)
    del ids
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    return 0 if all(w["verified"] for w in result["workloads"].values()) else 1


if __name__ == "__main__":
    sys.exit(main())
