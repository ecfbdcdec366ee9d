"""Time the segmented sort of 16-bit keys (b200sort_segmented_*_keys16) against torch.sort over rows, against the
widened route (float32 + b200sort_segmented_pairs_keys + narrowing) and against the flat 1-D 16-bit sort of the same
total n, on one GPU; writes profiles/r07_segmented16.json.

Workloads: rows of L keys with B x L about 2^26 and 2^28 (bfloat16 descending pairs with arange values per row: the
top-p sampling shape; uint16 keys only), small batches at a vocabulary size (B = 1, 8, 64 at L = 128256, where launch
latency counts), all-equal rows (the contended-atomic case) and a ragged Pareto mix of segment lengths.
Arms: "segmented16" (this library), "torch" (torch.sort(x.view(B, L), dim=-1, stable=True) in the same process, with
indices for pairs; uint16 rows are sorted as int32, widened before the timed steps), "widened" (the route a caller
has without this feature: x.float(), the 32-bit segmented sort, then narrowing back; keys only for uint16 rows),
"flat" (the 1-D sort16 / sort16_by_key of all n keys: the bound the onesweep class should approach).

Every step sorts the same pristine input out of place.  After a warm-up the arms take turns inside each round and the
rounds repeat, so drift of the shared machine hits every arm alike; reported per arm: the median over rounds of the
mean step time and its min / max.  After the timed steps the segmented output is checked against torch.sort (rows) or
for sortedness inside every segment and an unchanged per-segment sum (ragged), and the widened route's output against
it.  The card's name and power limit are read through NVML and stored beside the numbers.

    python tools/segmented16_bench.py [--steps 5] [--rounds 3] [--out profiles/r07_segmented16.json] [--quick]
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

KEY_U32, KEY_F32, KEY_U16, KEY_BF16 = 1, 2, 7, 9


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--quick", action="store_true", help="2^26 rows only, for a rehearsal")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_segmented16.json"))
    args = ap.parse_args()

    import torch
    from b200sort._lib import check, lib
    from key_types_bench import card_info
    from segmented_bench import power_law_offsets

    if not torch.cuda.is_available():
        print("segmented16_bench: no GPU", file=sys.stderr)
        return 2
    torch.cuda.set_device(0)
    L = lib()
    check(L.b200sort_device_check())
    stream = torch.cuda.current_stream().cuda_stream

    def aligned(nbytes):
        ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
        return ws, ws.data_ptr() + (-ws.data_ptr()) % 256

    def workload(name, src, offs, pairs, kt, desc, rows=None):
        n = src.numel()
        S = offs.numel() - 1
        out, tmp = torch.empty_like(src), torch.empty_like(src)
        vals = (torch.arange(rows[1], dtype=torch.int32, device="cuda").repeat(rows[0]) if rows
                else torch.arange(n, dtype=torch.int32, device="cuda"))
        vout, vtmp = torch.empty_like(vals), torch.empty_like(vals)
        seg_bytes = L.b200sort_segmented16_workspace_bytes(n, S)
        seg_ws, seg_ptr = aligned(seg_bytes)
        flat_bytes = L.b200sort_keys16_workspace_bytes(n)
        flat_ws, flat_ptr = aligned(flat_bytes)
        wide_bytes = L.b200sort_segmented_workspace_bytes(n, S)
        wide_ws, wide_ptr = aligned(wide_bytes)
        f_out, f_tmp = torch.empty(n, dtype=torch.float32, device="cuda"), torch.empty(n, dtype=torch.float32, device="cuda")
        w_out = torch.empty_like(src)
        pristine = src.clone()
        # uint16 widens to int32 exactly (a value below 2^16 as a float32 would too; int32 keeps the bytes obvious)
        wide_kt = KEY_F32 if kt == KEY_BF16 else KEY_U32

        def seg():
            if pairs:
                check(L.b200sort_segmented_pairs_keys16(kt, desc, src.data_ptr(), vals.data_ptr(), out.data_ptr(),
                                                        vout.data_ptr(), tmp.data_ptr(), vtmp.data_ptr(), n,
                                                        offs.data_ptr(), S, seg_ptr, seg_bytes, stream))
            else:
                check(L.b200sort_segmented_sort_keys16(kt, desc, src.data_ptr(), out.data_ptr(), tmp.data_ptr(), n,
                                                       offs.data_ptr(), S, seg_ptr, seg_bytes, stream))

        def widened():
            w = src.float() if kt == KEY_BF16 else src.view(torch.int16).to(torch.int32) & 0xFFFF
            if pairs:
                check(L.b200sort_segmented_pairs_keys(wide_kt, desc, w.data_ptr(), vals.data_ptr(), f_out.data_ptr(),
                                                      vout.data_ptr(), f_tmp.data_ptr(), vtmp.data_ptr(), n,
                                                      offs.data_ptr(), S, wide_ptr, wide_bytes, stream))
            else:
                check(L.b200sort_segmented_sort_keys(wide_kt, desc, w.data_ptr(), f_out.data_ptr(), f_tmp.data_ptr(), n,
                                                     offs.data_ptr(), S, wide_ptr, wide_bytes, stream))
            if kt == KEY_BF16:
                w_out.copy_(f_out)
            else:
                w_out.view(torch.int16).copy_(f_out.view(torch.int32))       # int32 -> int16 keeps the low half

        def flat():
            if pairs:
                check(L.b200sort_radix_pairs_keys16(kt, desc, src.data_ptr(), vals.data_ptr(), out.data_ptr(),
                                                    vout.data_ptr(), tmp.data_ptr(), vtmp.data_ptr(), n, flat_ptr,
                                                    flat_bytes, stream))
            else:
                check(L.b200sort_sort_keys16(kt, desc, src.data_ptr(), out.data_ptr(), n, flat_ptr, flat_bytes, stream))

        arms = {"segmented16": seg, "widened": widened, "flat": flat}
        if rows:
            # widened once, outside the timed steps: the torch arm times the sort alone
            tview = src.view(*rows) if kt == KEY_BF16 else (src.view(torch.int16).to(torch.int32) & 0xFFFF).view(*rows)

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
        widened()
        seg()
        torch.cuda.synchronize()
        assert torch.equal(src.view(torch.int16), pristine.view(torch.int16)), "the input was modified"
        ok = bool(torch.equal(w_out.view(torch.int16), out.view(torch.int16)))       # the widened route agrees
        if rows:
            tv, ti = torch.sort(tview, dim=-1, stable=True, descending=bool(desc))
            got = out.view(*rows) if kt == KEY_BF16 else out.view(torch.int16).view(*rows).to(torch.int32) & 0xFFFF
            ok = ok and bool(torch.equal(got, tv)) and (not pairs or bool(torch.equal(vout.view(*rows).to(torch.int64), ti)))
            del tv, ti, got
        else:                                   # ragged, uint16 ascending keys
            w = out.view(torch.int16).to(torch.int64) & 0xFFFF
            starts = torch.zeros(n, dtype=torch.bool, device="cuda")
            starts[offs[1:-1].to(torch.int64)] = True
            ok = ok and not bool(((w[1:] < w[:-1]) & ~starts[1:]).any().item())
            seg_id = torch.repeat_interleave(torch.arange(S, device="cuda"), (offs[1:] - offs[:-1]).to(torch.int64))
            a = torch.zeros(S, dtype=torch.int64, device="cuda").index_add_(0, seg_id, src.view(torch.int16).to(torch.int64) & 0xFFFF)
            b = torch.zeros(S, dtype=torch.int64, device="cuda").index_add_(0, seg_id, w)
            ok = ok and bool(torch.equal(a, b))
            del w, starts, seg_id, a, b
        res = {"n": n, "segments": S, "rows": list(rows) if rows else None, "pairs": pairs,
               "key_type": "bf16" if kt == KEY_BF16 else "u16", "descending": bool(desc), "verified": ok, "arms": {}}
        for a, ms in per_round.items():
            med = statistics.median(ms)
            res["arms"][a] = {"ms_median": med, "ms_min": min(ms), "ms_max": max(ms), "gkeys_per_s": n / med / 1e6}
        seg_ms = res["arms"]["segmented16"]["ms_median"]
        for a in ("torch", "widened", "flat"):
            res[f"segmented16_vs_{a}"] = res["arms"][a]["ms_median"] / seg_ms if a in res["arms"] else None
        line = "  ".join(f"{a} {r['ms_median']:.3f} [{r['ms_min']:.3f},{r['ms_max']:.3f}]" for a, r in res["arms"].items())
        print(f"{name:36s} {line}  verified={ok}", flush=True)
        del seg_ws, flat_ws, wide_ws, f_out, f_tmp
        torch.cuda.synchronize()
        return res

    result = {"card": card_info(0), "library": L.b200sort_version().decode(), "steps_per_round": args.steps,
              "rounds": args.rounds, "warmup": args.warmup, "workloads": {}}
    g = torch.Generator(device="cuda"); g.manual_seed(1)
    for log2n in ((26,) if args.quick else (26, 28)):
        for Lr in (16, 256, 1024, 8192, 32000, 128256, 1 << 20):
            B = max(1, (1 << log2n) // Lr)
            n = B * Lr
            u = torch.randint(-2**15, 2**15, (n,), dtype=torch.int32, device="cuda", generator=g).to(torch.int16)
            u = u.view(torch.uint16)
            f = torch.randn(n, device="cuda", generator=g).to(torch.bfloat16)
            offs = torch.arange(0, n + 1, Lr, dtype=torch.int32, device="cuda")
            key = f"rows_2^{log2n}_L{Lr}"
            result["workloads"][key + "_bf16_desc_pairs"] = workload(key + " bf16 desc pairs", f, offs, True, KEY_BF16, 1,
                                                                     (B, Lr))
            result["workloads"][key + "_u16_keys"] = workload(key + " u16 keys", u, offs, False, KEY_U16, 0, (B, Lr))
            del u, f
            torch.cuda.synchronize()
    Lr = 128256
    for B in (1, 8, 64):
        f = torch.randn(B * Lr, device="cuda", generator=g).to(torch.bfloat16)
        offs = torch.arange(0, B * Lr + 1, Lr, dtype=torch.int32, device="cuda")
        result["workloads"][f"batch_B{B}_L{Lr}_bf16_desc_pairs"] = workload(f"batch B{B} L{Lr} bf16 desc pairs", f, offs,
                                                                             True, KEY_BF16, 1, (B, Lr))
    Lr, n2 = 32000, (1 << 26) // 32000 * 32000
    eq = torch.full((n2,), 0x3FC0, dtype=torch.int16, device="cuda").view(torch.bfloat16)
    offs = torch.arange(0, n2 + 1, Lr, dtype=torch.int32, device="cuda")
    result["workloads"]["all_equal_rows_2^26_L32000_bf16_desc_pairs"] = workload(
        "all-equal rows L32000 bf16 desc pairs", eq, offs, True, KEY_BF16, 1, (n2 // Lr, Lr))
    n = 1 << (26 if args.quick else 28)
    u = torch.randint(-2**15, 2**15, (n,), dtype=torch.int32, device="cuda", generator=g).to(torch.int16).view(torch.uint16)
    offs = power_law_offsets(torch, n, 3)
    result["workloads"][f"ragged_powerlaw_2^{n.bit_length() - 1}_u16_keys"] = workload(
        "ragged power law u16 keys", u, offs, False, KEY_U16, 0)
    del u
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    return 0 if all(w["verified"] for w in result["workloads"].values()) else 1


if __name__ == "__main__":
    sys.exit(main())
