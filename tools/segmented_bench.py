"""Time the segmented sort (b200sort_segmented_*) against torch.sort over rows and against the 1-D sort of the same
total n, on one GPU; writes profiles/r04_segmented.json.

Workloads: rows of L keys with B x L = 2^26 and 2^28 (float32 descending pairs: the top-k / top-p sampling shape;
uint32 keys only), a ragged power-law mix at 2^28 and all-equal rows at L = 2^17 (the contended-atomic case).
Arms: "segmented" (this library), "torch" (torch.sort(x.view(B, L), dim=-1) in the same process: stable, with
indices for pairs; the uint32 rows are sorted as int32, the same bytes, since torch.sort takes no uint32), "flat"
(the 1-D b200sort sort of all n keys: the bound the onesweep class should approach) and, for 1024 rows of 2^16 keys,
"loop" (one 1-D sort per row, what a caller does without this feature).

Every step sorts the same pristine input out of place (256 MiB and up: larger than the 126 MB L2).  After a warm-up
the arms take turns inside each round and the rounds repeat, so drift of the shared machine hits every arm alike;
reported per arm: the median over rounds of the mean step time and its min / max.  After the timed steps the
segmented output is checked against torch.sort (rows) or for sortedness inside every segment and an unchanged
per-segment sum (ragged).  The card's name and power limit are read through NVML and stored beside the numbers.

    python tools/segmented_bench.py [--steps 5] [--rounds 3] [--out profiles/r04_segmented.json] [--quick]
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

KEY_U32, KEY_F32 = 1, 2


def power_law_offsets(torch, n: int, seed: int):
    """Segment lengths drawn from a Pareto law (alpha 1.1, scale 64) and capped at 2^22, until n is covered."""
    import numpy as np
    rng = np.random.default_rng(seed)
    lens = np.minimum((rng.pareto(1.1, 4 * n // 64 + 16) + 1) * 64, 1 << 22).astype(np.int64)
    cum = np.cumsum(lens)
    k = int(np.searchsorted(cum, n))
    offs = np.concatenate([[0], cum[:k], [n]])
    return torch.from_numpy(offs.astype(np.int32)).cuda()


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--quick", action="store_true", help="2^26 rows only, for a rehearsal")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_segmented.json"))
    args = ap.parse_args()

    import torch
    from b200sort._lib import ALGO_RADIX, check, lib
    from key_types_bench import card_info

    if not torch.cuda.is_available():
        print("segmented_bench: no GPU", file=sys.stderr)
        return 2
    torch.cuda.set_device(0)
    L = lib()
    check(L.b200sort_device_check())
    stream = torch.cuda.current_stream().cuda_stream

    def aligned(nbytes):
        ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
        return ws, ws.data_ptr() + (-ws.data_ptr()) % 256

    def workload(name, src, offs, pairs, kt, desc, rows=None, loop=False):
        n = src.numel()
        S = offs.numel() - 1
        out, tmp = torch.empty_like(src), torch.empty_like(src)
        vals = (torch.arange(rows[1], dtype=torch.int32, device="cuda").repeat(rows[0]) if rows
                else torch.arange(n, dtype=torch.int32, device="cuda"))
        vout, vtmp = torch.empty_like(vals), torch.empty_like(vals)
        seg_bytes = L.b200sort_segmented_workspace_bytes(n, S)
        seg_ws, seg_ptr = aligned(seg_bytes)
        flat_bytes = L.b200sort_workspace_bytes(n, ALGO_RADIX)
        flat_ws, flat_ptr = aligned(flat_bytes)
        pristine = src.clone()

        def seg():
            if pairs:
                check(L.b200sort_segmented_pairs_keys(kt, desc, src.data_ptr(), vals.data_ptr(), out.data_ptr(),
                                                      vout.data_ptr(), tmp.data_ptr(), vtmp.data_ptr(), n,
                                                      offs.data_ptr(), S, seg_ptr, seg_bytes, stream))
            else:
                check(L.b200sort_segmented_sort_keys(kt, desc, src.data_ptr(), out.data_ptr(), tmp.data_ptr(), n,
                                                     offs.data_ptr(), S, seg_ptr, seg_bytes, stream))

        def flat():
            if pairs:
                check(L.b200sort_radix_pairs_keys(kt, desc, src.data_ptr(), vals.data_ptr(), out.data_ptr(),
                                                  vout.data_ptr(), tmp.data_ptr(), vtmp.data_ptr(), n, flat_ptr,
                                                  flat_bytes, stream))
            else:
                check(L.b200sort_sort_keys(ALGO_RADIX, kt, desc, src.data_ptr(), out.data_ptr(), tmp.data_ptr(), n,
                                           flat_ptr, flat_bytes, stream))

        arms = {"segmented": seg, "flat": flat}
        if rows:
            tview = (src if kt == KEY_F32 else src.view(torch.int32)).view(*rows)

            def tsort():
                torch.sort(tview, dim=-1, stable=True, descending=bool(desc))
            arms["torch"] = tsort
        if loop:
            B, Lr = rows
            row_bytes = L.b200sort_workspace_bytes(Lr, ALGO_RADIX)
            row_ws, row_ptr = aligned(row_bytes)

            def loop_arm():
                for b in range(B):
                    o = 4 * b * Lr
                    check(L.b200sort_sort_keys(ALGO_RADIX, kt, desc, src.data_ptr() + o, out.data_ptr() + o,
                                               tmp.data_ptr() + o, Lr, row_ptr, row_bytes, stream))
            arms["loop"] = loop_arm
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
        torch.cuda.synchronize()
        assert torch.equal(src, pristine), "the input was modified"
        if rows:
            tv, ti = torch.sort(tview if kt == KEY_F32 else (src.to(torch.int64) & 0xFFFFFFFF).view(*rows), dim=-1,
                                stable=True, descending=bool(desc))
            got = out.view(*rows) if kt == KEY_F32 else (out.to(torch.int64) & 0xFFFFFFFF).view(*rows)
            ok = bool(torch.equal(got, tv)) and (not pairs or bool(torch.equal(vout.view(*rows).to(torch.int64), ti)))
            del tv, ti, got
        else:                                   # ragged, uint32 ascending keys
            w = out.to(torch.int64) & 0xFFFFFFFF
            starts = torch.zeros(n, dtype=torch.bool, device="cuda")
            starts[offs[1:-1].to(torch.int64)] = True
            ok = not bool(((w[1:] < w[:-1]) & ~starts[1:]).any().item())
            seg_id = torch.repeat_interleave(torch.arange(S, device="cuda"), (offs[1:] - offs[:-1]).to(torch.int64))
            a = torch.zeros(S, dtype=torch.int64, device="cuda").index_add_(0, seg_id, src.to(torch.int64) & 0xFFFFFFFF)
            b = torch.zeros(S, dtype=torch.int64, device="cuda").index_add_(0, seg_id, w)
            ok = ok and bool(torch.equal(a, b))
            del w, starts, seg_id, a, b
        res = {"n": n, "segments": S, "pairs": pairs, "key_type": "f32" if kt == KEY_F32 else "u32",
               "descending": bool(desc), "verified": ok, "arms": {}}
        for a, ms in per_round.items():
            med = statistics.median(ms)
            res["arms"][a] = {"ms_median": med, "ms_min": min(ms), "ms_max": max(ms), "gkeys_per_s": n / med / 1e6}
        res["segmented_vs_torch"] = (res["arms"]["torch"]["ms_median"] / res["arms"]["segmented"]["ms_median"]
                                     if "torch" in res["arms"] else None)
        res["segmented_vs_flat"] = res["arms"]["flat"]["ms_median"] / res["arms"]["segmented"]["ms_median"]
        line = "  ".join(f"{a} {r['ms_median']:.3f} [{r['ms_min']:.3f},{r['ms_max']:.3f}]" for a, r in res["arms"].items())
        print(f"{name:34s} {line}  verified={ok}", flush=True)
        del seg_ws, flat_ws
        torch.cuda.synchronize()
        return res

    result = {"card": card_info(0), "library": L.b200sort_version().decode(), "steps_per_round": args.steps,
              "rounds": args.rounds, "warmup": args.warmup, "workloads": {}}
    g = torch.Generator(device="cuda"); g.manual_seed(1)
    for log2n in ((26,) if args.quick else (26, 28)):
        n = 1 << log2n
        u = torch.randint(-2**31, 2**31, (n,), dtype=torch.int64, device="cuda", generator=g).to(torch.int32)
        f = torch.randn(n, device="cuda", generator=g)
        for Lr in (16, 256, 1024, 8192, 1 << 15, 1 << 17, 1 << 20):
            B = n // Lr
            offs = torch.arange(0, n + 1, Lr, dtype=torch.int32, device="cuda")
            key = f"rows_2^{log2n}_L{Lr}"
            result["workloads"][key + "_f32_desc_pairs"] = workload(key + " f32 desc pairs", f, offs, True, KEY_F32, 1, (B, Lr))
            result["workloads"][key + "_u32_keys"] = workload(key + " u32 keys", u, offs, False, KEY_U32, 0, (B, Lr))
        if log2n == 26:
            Lr = 1 << 16
            offs = torch.arange(0, n + 1, Lr, dtype=torch.int32, device="cuda")
            result["workloads"]["rows_2^26_L65536_u32_keys"] = workload("rows 2^26 L65536 u32 keys (+loop)", u, offs,
                                                                        False, KEY_U32, 0, (n // Lr, Lr), loop=True)
        del u, f
        torch.cuda.synchronize()
    if not args.quick:
        n = 1 << 28
        u = torch.randint(-2**31, 2**31, (n,), dtype=torch.int64, device="cuda", generator=g).to(torch.int32)
        offs = power_law_offsets(torch, n, 3)
        result["workloads"]["ragged_powerlaw_2^28_u32_keys"] = workload("ragged power law 2^28 u32 keys", u, offs,
                                                                        False, KEY_U32, 0)
        del u
        Lr, n2 = 1 << 17, 1 << 26
        eq = torch.full((n2,), 0x3FC00000, dtype=torch.int32, device="cuda").view(torch.float32)
        offs = torch.arange(0, n2 + 1, Lr, dtype=torch.int32, device="cuda")
        result["workloads"]["all_equal_rows_2^26_L131072_f32_desc_pairs"] = workload(
            "all-equal rows L2^17 f32 desc pairs", eq, offs, True, KEY_F32, 1, (n2 // Lr, Lr))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    return 0 if all(w["verified"] for w in result["workloads"].values()) else 1


if __name__ == "__main__":
    sys.exit(main())
