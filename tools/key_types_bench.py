"""Time every key order of b200sort_sort_keys against int32 ascending, at n = 2^28 on one GPU.

Each step sorts the same pristine input out of place (1 GiB, larger than the 126 MB L2).  The orders take turns:
one round times K steps of every order in sequence, int32 ascending among them, and the rounds repeat, so drift
of the shared machine hits all orders alike.  Reported per order: the median over rounds of the mean step time,
the spread (min / max over rounds) and the ratio to int32 ascending of the same algorithm.  After the timed
steps every output is checked: its images are the sorted images of the input (sorted + same multiset).

    python tools/key_types_bench.py [--log2n 28] [--steps 20] [--rounds 5] [--out profiles/r03_key_types.json]

The card's name and power limit are read through NVML (read only) and stored beside the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ORDERS = [("i32", 0, 0), ("i32", 0, 1), ("u32", 1, 0), ("u32", 1, 1), ("f32", 2, 0), ("f32", 2, 1)]
MASKS = {(0, 0): (0x80000000, 0x80000000), (0, 1): (0x7FFFFFFF, 0x7FFFFFFF), (1, 0): (0, 0),
         (1, 1): (0xFFFFFFFF, 0xFFFFFFFF), (2, 0): (0xFFFFFFFF, 0x80000000), (2, 1): (0, 0x7FFFFFFF)}


def card_info(index: int) -> dict:
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        name = pynvml.nvmlDeviceGetName(h)
        return {"name": name.decode() if isinstance(name, bytes) else name,
                "power_limit_w": pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0,
                "sm_max_mhz": int(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))}
    except Exception as e:          # the numbers are still recorded, without the card's limits
        import torch
        return {"name": torch.cuda.get_device_name(index), "power_limit_w": None, "nvml_error": str(e)}


def key_of(name: str, desc: int) -> str:
    return f"{name}_{'desc' if desc else 'asc'}"


def images(torch, words, kt: int, desc: int):
    """image(k) as int64 in [0, 2^32)."""
    neg, pos = MASKS[(kt, desc)]
    w = words.to(torch.int64) & 0xFFFFFFFF
    return w ^ torch.where(w >= 2**31, torch.full_like(w, neg), torch.full_like(w, pos))


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2n", type=int, default=28)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_key_types.json"))
    args = ap.parse_args()

    import torch
    from b200sort._lib import ALGO_MERGE, ALGO_RADIX, check, lib

    if not torch.cuda.is_available():
        print("key_types_bench: no GPU", file=sys.stderr)
        return 2
    torch.cuda.set_device(0)
    L = lib()
    check(L.b200sort_device_check())
    n = 1 << args.log2n
    g = torch.Generator(device="cuda"); g.manual_seed(args.seed)
    src = torch.randint(-2**31, 2**31, (n,), dtype=torch.int64, device="cuda", generator=g).to(torch.int32)
    pristine = src.clone()
    out = torch.empty_like(src); tmp = torch.empty_like(src)
    stream = torch.cuda.current_stream().cuda_stream
    result = {"n": n, "input": "uniform random 32-bit patterns (torch.randint, seed %d)" % args.seed,
              "steps_per_round": args.steps, "rounds": args.rounds, "card": card_info(0),
              "library": L.b200sort_version().decode(), "algos": {}}
    for algo_name, algo in (("radix", ALGO_RADIX), ("merge", ALGO_MERGE)):
        ws_bytes = L.b200sort_workspace_bytes(n, algo)
        ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device="cuda")
        ws_ptr = ws.data_ptr() + (-ws.data_ptr()) % 256

        def step(kt, desc):
            check(L.b200sort_sort_keys(algo, kt, desc, src.data_ptr(), out.data_ptr(), tmp.data_ptr(), n, ws_ptr,
                                       ws_bytes, stream))

        for _, kt, desc in ORDERS:
            for _ in range(args.warmup):
                step(kt, desc)
        torch.cuda.synchronize()
        per_round = {key_of(name, desc): [] for name, _, desc in ORDERS}
        for _ in range(args.rounds):
            for name, kt, desc in ORDERS:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.steps):
                    step(kt, desc)
                e1.record()
                e1.synchronize()
                per_round[key_of(name, desc)].append(e0.elapsed_time(e1) / args.steps)
        verified = {}
        for name, kt, desc in ORDERS:
            step(kt, desc)
            torch.cuda.synchronize()
            got = images(torch, out, kt, desc)
            want = torch.sort(images(torch, src, kt, desc)).values
            verified[key_of(name, desc)] = bool(torch.equal(got, want))
            del got, want
        assert torch.equal(src, pristine), "the input was modified"
        base = statistics.median(per_round["i32_asc"])
        rows = {}
        for key, ms in per_round.items():
            med = statistics.median(ms)
            rows[key] = {"ms_median": med, "ms_min": min(ms), "ms_max": max(ms), "keys_per_s": n / (med / 1e3),
                         "vs_i32_asc": med / base, "verified": verified[key], "per_round_ms": ms}
        spread = (max(per_round["i32_asc"]) - min(per_round["i32_asc"])) / base
        result["algos"][algo_name] = {"orders": rows, "i32_asc_spread": spread}
        del ws
        torch.cuda.synchronize()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    for algo_name, a in result["algos"].items():
        for key, r in a["orders"].items():
            print(f"{algo_name:5s} {key:8s} {r['ms_median']:8.3f} ms  [{r['ms_min']:.3f}, {r['ms_max']:.3f}]  "
                  f"x{r['vs_i32_asc']:.3f} of i32_asc  verified={r['verified']}")
    return 0 if all(r["verified"] for a in result["algos"].values() for r in a["orders"].values()) else 1


if __name__ == "__main__":
    sys.exit(main())
