"""Time the 16-bit key sorts (b200sort_sort_keys16, b200sort_radix_pairs_keys16) on one GPU, against torch.sort on
the same tensor and against the widened route (x.to(int32 or float32) -> b200sort.sort / sort_by_key -> back).

Each step sorts the same pristine input out of place.  At n = 2^28 the keys are 512 MiB per array, above the 126 MB
L2; at n = 2^24 (32 MiB per array) input and output stay in L2 between steps.  The arms take turns: one round times
K steps of every arm in sequence, and the rounds repeat, so drift of the shared machine hits all arms alike.  Reported
per size, input distribution and arm: the median, min and max over rounds of the mean step time, Gkeys/s, the
algorithmic bytes per key and the resulting bytes/s.  Bytes per key: the counting sort 4 (read 2, write 2); pairs 2
(histogram read) + 12 per executed pass (the plan skips a pass in which one digit value holds every key); the widened
routes 48 (keys: 6 to widen, 36 for the 32-bit sort, 6 to narrow) and 80 (pairs: 6 + 68 + 6).  After the timed steps
every output is checked: its images are the sorted images of the input, pairs' values follow their keys and are
stable, and torch.sort and the widened routes give the same values (the float inputs hold no +-0.0 or NaN).

    python tools/keys16_bench.py [--log2n 28,24] [--steps 5] [--rounds 5] [--out profiles/r06_keys16.json]

--variants (with B200SORT_LIB=libb200sort_exp.so, built by make experiments) adds the shapes the shipped ones were
measured against: the histogram without run aggregation, and pairs tiles of 4096 and 16384 keys.  The card's name and
power limit are read through NVML (read only) and stored beside the numbers.
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

KEY = {"int16": 6, "uint16": 7, "float16": 8, "bfloat16": 9}
MASKS = {6: (0x8000, 0x8000), 7: (0, 0), 8: (0xFFFF, 0x8000), 9: (0xFFFF, 0x8000)}   # ascending (neg, pos)
DISTS = {"uniform16": "int16", "bf16_normal": "bfloat16", "f16_normal": "float16", "int16_small": "int16",
         "all_equal": "int16", "ascending": "int16"}
VARIANTS = {"keys_hist_plain_atomics": ("keys", {"B200SORT_R16_HIST_RUNS": "0"}),
            "pairs_tile_4096": ("pairs", {"B200SORT_R16_IPT": "8"}),
            "pairs_tile_16384": ("pairs", {"B200SORT_R16_IPT": "32"})}
ENV_KEYS = ("B200SORT_R16_HIST_RUNS", "B200SORT_R16_IPT")


def images(torch, x, kt: int):
    """Ascending image of each key as int32 in [0, 65536)."""
    neg, pos = MASKS[kt]
    w = x.view(torch.int16).to(torch.int32) & 0xFFFF
    return w ^ torch.where(w >= 0x8000, torch.full_like(w, neg), torch.full_like(w, pos))


def executed_passes(img) -> int:
    return sum(int(bool((((img >> (8 * p)) & 0xFF) != ((img[0] >> (8 * p)) & 0xFF)).any())) for p in range(2))


def make_input(torch, dist: str, n: int, seed: int):
    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    if dist == "uniform16":
        return torch.randint(-2**15, 2**15, (n,), dtype=torch.int32, device="cuda", generator=g).to(torch.int16)
    if dist in ("bf16_normal", "f16_normal"):
        # zeros (either sign) become 0.5: torch.sort(stable=True) ties -0.0 with +0.0, totalOrder does not
        x = torch.randn(n, device="cuda", generator=g).to(torch.bfloat16 if dist == "bf16_normal" else torch.float16)
        x[x == 0] = 0.5
        return x
    if dist == "int16_small":
        return torch.randint(-100, 101, (n,), dtype=torch.int32, device="cuda", generator=g).to(torch.int16)
    if dist == "all_equal":
        return torch.full((n,), 1234, dtype=torch.int16, device="cuda")
    if dist == "ascending":
        return torch.sort(torch.randint(-2**15, 2**15, (n,), dtype=torch.int32, device="cuda", generator=g)
                          .to(torch.int16)).values
    raise ValueError(dist)


def run_size(torch, L, b200sort, n: int, args) -> dict:
    from b200sort._lib import check
    stream = torch.cuda.current_stream().cuda_stream
    vals = torch.arange(n, dtype=torch.int32, device="cuda")
    vout = torch.empty_like(vals); vtmp = torch.empty_like(vals)
    ws_bytes = L.b200sort_keys16_workspace_bytes(n)
    ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device="cuda")
    ws_ptr = ws.data_ptr() + (-ws.data_ptr()) % 256
    rows_by_dist = {}
    for dist, dtype_name in DISTS.items():
        dtype = getattr(torch, dtype_name)
        kt = KEY[dtype_name]
        wide = torch.int32 if dtype_name in ("int16", "uint16") else torch.float32
        src = make_input(torch, dist, n, args.seed)
        pristine = src.clone()
        out = torch.empty_like(src); tmp = torch.empty_like(src)

        def keys16():
            check(L.b200sort_sort_keys16(kt, 0, src.data_ptr(), out.data_ptr(), n, ws_ptr, ws_bytes, stream))

        def pairs16():
            check(L.b200sort_radix_pairs_keys16(kt, 0, src.data_ptr(), vals.data_ptr(), out.data_ptr(), vout.data_ptr(),
                                                tmp.data_ptr(), vtmp.data_ptr(), n, ws_ptr, ws_bytes, stream))
        arms = {"sort16_keys": keys16,
                "torch_sort": lambda: torch.sort(src),
                "widened_keys": lambda: b200sort.sort(src.to(wide)).to(dtype),
                "sort16_by_key_pairs": pairs16,
                "torch_sort_stable": lambda: torch.sort(src, stable=True),
                "widened_pairs": lambda: b200sort.sort_by_key(src.to(wide), vals)}
        env = {name: {} for name in arms}
        if args.variants:
            for name, (kind, e) in VARIANTS.items():
                arms[name] = keys16 if kind == "keys" else pairs16
                env[name] = e

        def set_env(e):
            for k in ENV_KEYS:
                os.environ.pop(k, None)
            os.environ.update(e)
        for name, fn in arms.items():
            set_env(env[name])
            for _ in range(args.warmup):
                fn()
        torch.cuda.synchronize()
        per_round = {k: [] for k in arms}
        for _ in range(args.rounds):
            for name, fn in arms.items():
                set_env(env[name])
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.steps):
                    fn()
                e1.record()
                e1.synchronize()
                per_round[name].append(e0.elapsed_time(e1) / args.steps)
        set_env({})

        # verification and the byte model, arm by arm
        img_in = images(torch, src, kt)
        hist_in = torch.bincount(img_in, minlength=1 << 16)
        passes = executed_passes(img_in)

        def keys_ok():
            img = images(torch, out, kt)
            return bool((img[1:] >= img[:-1]).all()) and bool(torch.equal(torch.bincount(img, minlength=1 << 16), hist_in))

        def pairs_ok():
            img = images(torch, out, kt)
            return (keys_ok() and bool(torch.equal(src.view(torch.int16)[vout.to(torch.int64)], out.view(torch.int16)))
                    and not bool(((img[1:] == img[:-1]) & (vout[1:] <= vout[:-1])).any()))
        verified, bpk = {}, {}
        for name in arms:
            kind = "keys" if name in ("sort16_keys", "torch_sort", "widened_keys") else "pairs"
            if name in VARIANTS:
                kind = VARIANTS[name][0]
            if name in ("sort16_keys", "sort16_by_key_pairs") or name in VARIANTS:
                set_env(env[name])
                arms[name]()
                torch.cuda.synchronize()
                verified[name] = keys_ok() if kind == "keys" else pairs_ok()
                bpk[name] = 4 if kind == "keys" else 2 + 12 * passes
        set_env({})
        keys16(); torch.cuda.synchronize()
        mine = out.clone()
        verified["torch_sort"] = bool(torch.equal(arms["torch_sort"]().values, mine))
        verified["widened_keys"] = bool(torch.equal(arms["widened_keys"](), mine))
        pairs16(); torch.cuda.synchronize()
        tv, ti = arms["torch_sort_stable"]()
        verified["torch_sort_stable"] = bool(torch.equal(tv, out)) and bool(torch.equal(ti.to(torch.int32), vout))
        wk, wv = arms["widened_pairs"]()
        verified["widened_pairs"] = bool(torch.equal(wk.to(dtype), out)) and bool(torch.equal(wv, vout))
        bpk.update({"torch_sort": None, "torch_sort_stable": None, "widened_keys": 48, "widened_pairs": 80})
        assert torch.equal(src.view(torch.int16), pristine.view(torch.int16)), "the input was modified"

        rows = {}
        for arm, ms in per_round.items():
            med = statistics.median(ms)
            rows[arm] = {"ms_median": med, "ms_min": min(ms), "ms_max": max(ms), "gkeys_per_s": n / (med / 1e3) / 1e9,
                         "bytes_per_key": bpk[arm],
                         "gbytes_per_s": None if bpk[arm] is None else bpk[arm] * n / (med / 1e3) / 1e9,
                         "verified": verified[arm], "per_round_ms": ms}
        rows_by_dist[dist] = {"dtype": dtype_name, "executed_pairs_passes": passes, "arms": rows}
        del src, pristine, out, tmp, img_in, hist_in, mine
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
    return rows_by_dist


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2n", default="28,24")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--variants", action="store_true")
    ap.add_argument("--out", default=os.path.join(os.path.dirname(ROOT), "profiles", "r06_keys16.json"))
    args = ap.parse_args()

    import torch
    import b200sort
    from b200sort._lib import check, lib

    if not torch.cuda.is_available():
        print("keys16_bench: no GPU", file=sys.stderr)
        return 2
    torch.cuda.set_device(0)
    L = lib()
    check(L.b200sort_device_check())
    result = {"card": card_info(0), "library": L.b200sort_version().decode(), "out_of_place": True,
              "steps_per_round": args.steps, "rounds": args.rounds,
              "bytes_per_key_model": "sort16 keys 4; sort16 pairs 2 + 12 per executed pass; widened keys 48 "
                                     "(6 + 36 + 6), widened pairs 80 (6 + 68 + 6)",
              "l2_note": "n = 2^28: 512 MiB per key array, above the 126 MB L2; n = 2^24: 32 MiB, held in L2",
              "sizes": {}}
    for lg in (int(x) for x in args.log2n.split(",")):
        result["sizes"][f"2^{lg}"] = run_size(torch, L, b200sort, 1 << lg, args)

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(f"card: {result['card']}")
    ok = True
    for size, dists in result["sizes"].items():
        for dist, d in dists.items():
            for arm, r in d["arms"].items():
                ok = ok and r["verified"]
                gbs = "" if r["gbytes_per_s"] is None else f"{r['bytes_per_key']:3d} B/key {r['gbytes_per_s']:7.1f} GB/s"
                print(f"{size:5s} {dist:12s} {arm:24s} {r['ms_median']:8.3f} ms [{r['ms_min']:.3f}, {r['ms_max']:.3f}] "
                      f"{r['gkeys_per_s']:7.2f} Gkeys/s {gbs}  verified={r['verified']}")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
