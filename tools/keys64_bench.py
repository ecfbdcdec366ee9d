"""Time the 64-bit key sorts (b200sort_sort_keys64, b200sort_radix_pairs_keys64) at n = 2^28 on one GPU, against
torch.sort on the same tensors and against the 32-bit uint32 sort of 2^28 keys.

Each step sorts the same pristine input out of place (2 GiB of keys, far above the 126 MB L2).  The arms take turns:
one round times K steps of every arm in sequence, and the rounds repeat, so drift of the shared machine hits all arms
alike.  Reported per arm and input distribution: the median, min and max over rounds of the mean step time, Gkeys/s,
the algorithmic bytes per key (8 for the histogram read plus 16 per executed pass for keys, 24 for pairs; the 32-bit
sort: 4 plus 8 per pass) and the resulting bytes/s.  The executed passes are counted from the images of the input,
as the sort's own plan skips a pass in which one digit value holds every key.  After the timed steps every output is
checked: its images are the sorted images of the input, pairs' values follow their keys and are stable.

    python tools/keys64_bench.py [--log2n 28] [--steps 5] [--rounds 5] [--out profiles/r05_keys64.json]

The card's name and power limit are read through NVML (read only) and stored beside the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(ROOT))
sys.path.insert(0, ROOT)

from key_types_bench import card_info  # noqa: E402

ORDERS = [("i64", 3, 0), ("i64", 3, 1), ("u64", 4, 0), ("u64", 4, 1), ("f64", 5, 0), ("f64", 5, 1)]
TOP, ALL = 1 << 63, (1 << 64) - 1
MASKS = {(3, 0): (TOP, TOP), (3, 1): (ALL ^ TOP, ALL ^ TOP), (4, 0): (0, 0), (4, 1): (ALL, ALL),
         (5, 0): (ALL, TOP), (5, 1): (0, ALL ^ TOP)}
DISTS = ["uniform64", "nonneg_below_2_32", "small_signed", "float64_normal"]


def as_i64(m: int) -> int:
    return m - (1 << 64) if m >= TOP else m


def images(torch, words, kt: int, desc: int):
    """image(k) ^ (1 << 63) as int64: the signed order of these is the unsigned order of the images."""
    neg, pos = MASKS[(kt, desc)]
    w = words.view(torch.int64)
    img = w ^ torch.where(w < 0, torch.full_like(w, as_i64(neg)), torch.full_like(w, as_i64(pos)))
    return img ^ as_i64(TOP)


def executed_passes(torch, img) -> int:
    """Passes in which the digits of the images are not all equal (the others are skipped by the sort's plan)."""
    count = 0
    for p in range(8):
        d = (img >> (8 * p)) & 0xFF
        count += int(bool((d != d[0]).any()))
    return count


def make_input(torch, dist: str, n: int, seed: int):
    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    if dist == "uniform64":
        x = torch.randint(-2**31, 2**31, (n, 2), dtype=torch.int64, device="cuda", generator=g).to(torch.int32)
        return x.view(torch.int64).view(-1).clone()
    if dist == "nonneg_below_2_32":
        return torch.randint(0, 2**32, (n,), dtype=torch.int64, device="cuda", generator=g)
    if dist == "small_signed":
        return torch.randint(-1000, 1001, (n,), dtype=torch.int64, device="cuda", generator=g)
    if dist == "float64_normal":
        return torch.randn(n, dtype=torch.float64, device="cuda", generator=g).view(torch.int64)
    raise ValueError(dist)


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2n", type=int, default=28)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--dists", default=",".join(DISTS))
    ap.add_argument("--out", default=os.path.join(os.path.dirname(ROOT), "profiles", "r05_keys64.json"))
    args = ap.parse_args()

    import torch
    from b200sort._lib import ALGO_RADIX, check, lib

    if not torch.cuda.is_available():
        print("keys64_bench: no GPU", file=sys.stderr)
        return 2
    torch.cuda.set_device(0)
    L = lib()
    check(L.b200sort_device_check())
    n = 1 << args.log2n
    stream = torch.cuda.current_stream().cuda_stream
    out = torch.empty(n, dtype=torch.int64, device="cuda"); tmp = torch.empty_like(out)
    vals = torch.arange(n, dtype=torch.int32, device="cuda")
    vout = torch.empty_like(vals); vtmp = torch.empty_like(vals)
    ws_bytes = L.b200sort_keys64_workspace_bytes(n)
    ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device="cuda")
    ws_ptr = ws.data_ptr() + (-ws.data_ptr()) % 256
    ws32_bytes = L.b200sort_workspace_bytes(n, ALGO_RADIX)
    ws32 = torch.empty(ws32_bytes + 256, dtype=torch.uint8, device="cuda")
    ws32_ptr = ws32.data_ptr() + (-ws32.data_ptr()) % 256
    result = {"n": n, "steps_per_round": args.steps, "rounds": args.rounds, "card": card_info(0),
              "library": L.b200sort_version().decode(), "out_of_place": True,
              "bytes_per_key_model": "keys: 8 (histogram) + 16 per executed pass; pairs: 8 + 24 per executed pass; "
                                     "u32 reference: 4 + 8 per pass", "dists": {}}

    for dist in args.dists.split(","):
        src = make_input(torch, dist, n, args.seed)
        pristine = src.clone()
        fsrc = src.view(torch.float64)
        tsrc = fsrc if dist == "float64_normal" else src          # what torch.sort is given
        src32 = src.to(torch.int32)                                # the low words: uniform for the uniform inputs
        out32 = torch.empty_like(src32); tmp32 = torch.empty_like(src32)

        def keys_arm(kt, desc):
            return lambda: check(L.b200sort_sort_keys64(kt, desc, src.data_ptr(), out.data_ptr(), tmp.data_ptr(), n,
                                                        ws_ptr, ws_bytes, stream))

        def pairs_arm(kt):
            return lambda: check(L.b200sort_radix_pairs_keys64(kt, 0, src.data_ptr(), vals.data_ptr(), out.data_ptr(),
                                                               vout.data_ptr(), tmp.data_ptr(), vtmp.data_ptr(), n,
                                                               ws_ptr, ws_bytes, stream))
        arms = {f"{name}_{'desc' if d else 'asc'}_keys": keys_arm(kt, d) for name, kt, d in ORDERS}
        arms["i64_asc_pairs"] = pairs_arm(3)
        arms["f64_asc_pairs"] = pairs_arm(5)
        arms["torch_sort"] = lambda: torch.sort(tsrc)
        arms["torch_sort_stable"] = lambda: torch.sort(tsrc, stable=True)
        arms["u32_asc_keys_32bit_sort"] = lambda: check(L.b200sort_sort_keys(ALGO_RADIX, 1, 0, src32.data_ptr(),
                                                                             out32.data_ptr(), tmp32.data_ptr(), n,
                                                                             ws32_ptr, ws32_bytes, stream))
        for fn in arms.values():
            for _ in range(args.warmup):
                fn()
        torch.cuda.synchronize()
        per_round = {k: [] for k in arms}
        for _ in range(args.rounds):
            for name, fn in arms.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.steps):
                    fn()
                e1.record()
                e1.synchronize()
                per_round[name].append(e0.elapsed_time(e1) / args.steps)

        # verification and the byte model, arm by arm
        verified, bpk = {}, {}
        for name, kt, d in ORDERS:
            arm = f"{name}_{'desc' if d else 'asc'}_keys"
            arms[arm]()
            torch.cuda.synchronize()
            want = images(torch, src, kt, d)
            bpk[arm] = 8 + 16 * executed_passes(torch, want)
            want = torch.sort(want).values
            verified[arm] = bool(torch.equal(images(torch, out, kt, d), want))
            del want
        for kt, arm in ((3, "i64_asc_pairs"), (5, "f64_asc_pairs")):
            arms[arm]()
            torch.cuda.synchronize()
            img = images(torch, out, kt, 0)
            ok = bool(torch.equal(img, torch.sort(images(torch, src, kt, 0)).values))
            ok = ok and bool(torch.equal(src[vout.to(torch.int64)], out))            # values follow their keys
            ok = ok and not bool(((img[1:] == img[:-1]) & (vout[1:] <= vout[:-1])).any())   # stable
            verified[arm] = ok
            bpk[arm] = 8 + 24 * executed_passes(torch, images(torch, src, kt, 0))
            del img
        # torch.sort agrees with the library where totalOrder and torch's order coincide (no NaN, no -0.0 here)
        ref = "f64_asc_keys" if dist == "float64_normal" else "i64_asc_keys"
        arms[ref]()
        torch.cuda.synchronize()
        mine = out.view(torch.float64) if dist == "float64_normal" else out
        for arm in ("torch_sort", "torch_sort_stable"):
            verified[arm] = bool(torch.equal(arms[arm]().values, mine))
            bpk[arm] = None
        arms["u32_asc_keys_32bit_sort"]()
        torch.cuda.synchronize()
        verified["u32_asc_keys_32bit_sort"] = bool(torch.equal(
            out32.to(torch.int64) & 0xFFFFFFFF, torch.sort(src32.to(torch.int64) & 0xFFFFFFFF).values))
        bpk["u32_asc_keys_32bit_sort"] = 4 + 8 * 4
        assert torch.equal(src, pristine), "the input was modified"

        rows = {}
        for arm, ms in per_round.items():
            med = statistics.median(ms)
            rows[arm] = {"ms_median": med, "ms_min": min(ms), "ms_max": max(ms), "gkeys_per_s": n / (med / 1e3) / 1e9,
                         "bytes_per_key": bpk[arm],
                         "gbytes_per_s": None if bpk[arm] is None else bpk[arm] * n / (med / 1e3) / 1e9,
                         "verified": verified[arm], "per_round_ms": ms}
        result["dists"][dist] = rows
        del src, pristine, fsrc, tsrc, src32, out32, tmp32
        torch.cuda.synchronize()
        torch.cuda.empty_cache()

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(f"card: {result['card']}")
    for dist, rows in result["dists"].items():
        for arm, r in rows.items():
            gbs = "" if r["gbytes_per_s"] is None else f"{r['bytes_per_key']:3d} B/key {r['gbytes_per_s']:7.1f} GB/s"
            print(f"{dist:18s} {arm:24s} {r['ms_median']:8.3f} ms [{r['ms_min']:.3f}, {r['ms_max']:.3f}] "
                  f"{r['gkeys_per_s']:6.2f} Gkeys/s {gbs}  verified={r['verified']}")
    return 0 if all(r["verified"] for rows in result["dists"].values() for r in rows.values()) else 1


if __name__ == "__main__":
    sys.exit(main())
