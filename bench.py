#!/usr/bin/env python
"""bench.py -- the sort hot path on B200, measured the way BASELINE.json's metric is quoted.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--algo radix|merge] [--dist uniform|...] [--log2n L] [--dump-outputs DIR]

A step is ONE full sort of one batch of keys.

--dump-outputs DIR writes DIR/sorted_keys.npy: the sorted keys of the last timed step as float64 (exact for int32), all
of them up to 2^22 keys, else the keys at the positions dump_positions(n) picks (a fixed, seeded sample).  The input
depends only on the arguments, so two builds can be compared output for output.  Our arm on one GPU and the reference
arm (its host sample, see below) write it; the multi-GPU sort does not.

N = 1   workload = BASELINE configs[1..3]' single-GPU case at the size the metric is quoted on:
        n = 2^28 uniform int32 keys, onesweep radix sort (``--algo merge`` gives configs[2]).
        `value`  keys/s with the input resident in HBM (out-of-place form: every step sorts the same
                 pristine 1 GiB input, which is larger than L2, into the output buffer);
        `e2e`    keys/s through the reference-facing operator b200sort_order_array_host (what the
                 exported C++ order_array calls) on a pinned HOST buffer: H2D + sort + D2H per step;
        `roofline` the dominant kernel (one onesweep pass, 8 B/key) timed live with CUDA events;
        `cpu_baseline` the reference's own CPU path (order_with_trust, oracle/_ref) on a bounded sample.
N > 1   torchrun launches one process per GPU; the distributed sort (MSD partition + exchange over
        NVLink + local sort) runs on n = 2^28 keys PER GPU (weak scaling); see dist.py.

--impl reference times the reference's CPU implementation of the path (oracle/_ref when present,
else the oracle port) on the host cores, rank 0 only.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "32-bit keys sorted/sec at n=2^28"
UNIT = "keys/s"


def _ncu_traffic(kernel_substr: str, variant: str | None = None):
    """DRAM bytes per launch of the dominant kernel from the newest committed ncu --set full summary
    (profiles/rNN_ncu_*.json, written by tools/ncu_summary.py --json), or None.  A summary that names the
    shape it was captured on (`variant`) is only used while that shape is still the one being launched, so the
    figure cannot go stale when the kernel changes."""
    import glob
    best = None
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_*.json"))):
        try:
            for item in json.load(open(path)):
                if kernel_substr in item.get("kernel", "") and "dram_bytes_total" in item:
                    if variant is not None and item.get("variant") not in (None, variant):
                        continue
                    if variant is not None and item.get("variant") is None and os.path.basename(path).startswith("r01_"):
                        continue                          # round 1's capture: a different kernel
                    best = {"bytes": item["dram_bytes_total"], "source": os.path.relpath(path, ROOT),
                            "variant": item.get("variant")}
                    try:     # the pipe that actually bounds these kernels (DESIGN.md section 7)
                        best["lsu_pct"] = float(item["LSU wavefronts % of peak"].split()[0])
                    except Exception:
                        pass
        except Exception:
            pass
    return best


def _peaks() -> dict:
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm_gbs": float(p["hbm_gbs"]), "source": "measured (MEASURED_PEAKS.json)"}
    except Exception:
        return {"hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


# ---- clocks during the timed region ---------------------------------------------------------------
_REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown",
            0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting"}


class ClockSampler(threading.Thread):
    def __init__(self, cuda_index: int):
        super().__init__(daemon=True)
        self.samples = []
        self.stop_flag = False
        self.h = None
        self.sm_max = None
        try:
            import pynvml
            import torch
            self.nv = pynvml
            pynvml.nvmlInit()
            try:
                uuid = "GPU-" + str(torch.cuda.get_device_properties(cuda_index).uuid)
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(cuda_index)
            self.sm_max = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None

    def run(self):
        if self.h is None:
            return
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.samples.append((time.perf_counter(), sm, rs))
            except Exception:
                pass
            time.sleep(0.004)

    def summary(self, t0: float, t1: float) -> dict:
        inside = [s for s in self.samples if t0 <= s[0] <= t1]
        how = "sampled inside the timed region"
        if not inside and self.samples:
            mid = 0.5 * (t0 + t1)
            inside = [min(self.samples, key=lambda s: abs(s[0] - mid))]
            how = "nearest sample (timed region shorter than the sampling period)"
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": [], "samples": 0, "how": "nvml unavailable"}
        clocks = sorted(s[1] for s in inside)
        bits = 0
        for s in inside:
            bits |= s[2]
        return {"sm_mhz": clocks[len(clocks) // 2], "sm_max_mhz": self.sm_max,
                "reasons": sorted(name for bit, name in _REASONS.items() if bits & bit),
                "samples": len(inside), "how": how}


# ---- --dump-outputs ----------------------------------------------------------------------------------
DUMP_KEYS = 1 << 22          # 32 MiB of float64


def dump_positions(n: int):
    """Output positions --dump-outputs writes: all n up to DUMP_KEYS, else one position in each of DUMP_KEYS
    equal strata, drawn from a fixed seed, so the sample covers the whole output and depends on n alone."""
    import numpy as np
    if n <= DUMP_KEYS:
        return np.arange(n, dtype=np.int64)
    stride = n // DUMP_KEYS
    return np.arange(DUMP_KEYS, dtype=np.int64) * stride + np.random.default_rng(0).integers(0, stride, DUMP_KEYS)


def _save_dump(dump_dir: str, sorted_keys_sample) -> None:
    import numpy as np
    os.makedirs(dump_dir, exist_ok=True)
    np.save(os.path.join(dump_dir, "sorted_keys.npy"), sorted_keys_sample.astype(np.float64))


# ---- reference arm -----------------------------------------------------------------------------------
def _cpu_sorter():
    """(callable sorting a numpy int32 array in place, kind, description)."""
    import oracle
    if oracle.ref.available:
        return (oracle.ref.order_with_trust_inplace, "reference",
                "oracle/_ref/libreflab.so order_with_trust = reference SRM/lab.cu:404-406 "
                "(Thrust sequential host sort), unmodified")
    return oracle.radix_sort_inplace, "port", "oracle/oracle_sort.c oracle_radix_sort_i32 (LSD byte radix, 1 thread)"


def reference_arm(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np
    from b200sort import datagen
    sort_inplace, kind, what = _cpu_sorter()
    total_steps = args.steps + args.warmup
    log2m = 24 if total_steps <= 110 else 22
    m = 1 << log2m
    pristine = datagen.make(args.dist, m, 1)
    work = np.empty_like(pristine)
    for _ in range(args.warmup):
        work[:] = pristine
        sort_inplace(work)
    elapsed = 0.0
    for _ in range(args.steps):
        work[:] = pristine
        t = time.perf_counter()
        sort_inplace(work)
        elapsed += time.perf_counter() - t
    if args.dump_outputs:
        _save_dump(args.dump_outputs, work[dump_positions(m)])
    value = m * args.steps / elapsed
    sample = (f"each step sorts a bounded sample of 2^{log2m} {args.dist} keys (seed 1) of the 2^{args.log2n} "
              f"workload on the host; {what}")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * elapsed / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
        "data": "synthetic",
        "config": {"workload": f"radix sort of 2^{args.log2n} {args.dist} int32 keys (CPU arm: 2^{log2m}-key sample per step)",
                   "dist": args.dist, "seed": 1},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": kind, "sample": sample,
                         "host_cores_available": os.cpu_count()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---- our arm -------------------------------------------------------------------------------------------
def _make_device_keys(torch, n: int, dist: str, seed: int, device):
    """Synthetic keys generated on the device (the host generators in b200sort.datagen are the
    recipes of record; these are their torch twins for sizes where a host round trip is slow)."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)

    def u32():
        return torch.randint(-2**31, 2**31, (n,), dtype=torch.int64, device=device, generator=g).to(torch.int32)

    if dist == "uniform":
        return u32()
    if dist == "uniform_nonneg":
        return u32() & 0x7FFFFFFF
    if dist in ("and2", "and3", "and4"):
        d = u32()
        for _ in range(int(dist[3]) - 1):
            d &= u32()
        return d
    if dist == "mask_0000ffff":
        return u32() & 0x0000FFFF
    if dist == "mask_00ff00ff":
        return u32() & 0x00FF00FF
    if dist == "skewed90":
        d = u32()
        hot = torch.rand(n, device=device, generator=g) < 0.9
        return torch.where(hot, (d & 0x00FFFFFF) | 0x40000000, d)
    if dist == "ascending":
        return (torch.arange(n, dtype=torch.int64, device=device) - n // 2).to(torch.int32)
    if dist == "descending":
        return (n // 2 - 1 - torch.arange(n, dtype=torch.int64, device=device)).to(torch.int32)
    if dist == "all_equal":
        return torch.full((n,), 7, dtype=torch.int32, device=device)
    raise SystemExit(f"unknown --dist {dist}")


def _check_sorted(torch, out, src) -> None:
    assert bool((out[1:] >= out[:-1]).all().item()), "bench: output is not sorted"
    assert int(out.sum(dtype=torch.int64).item()) == int(src.sum(dtype=torch.int64).item()), \
        "bench: output is not a permutation of the input (sum differs)"



def _measure_config(L, torch, dev, algo_name: str, dist: str, log2n: int, steps: int, peaks: dict, bufs: dict) -> dict:
    """One row of the `configs` block: `steps` timed sorts (after 3 warm-up sorts) of 2^log2n `dist` keys
    with `algo_name`, the per-kernel CUDA-event times of one more sort, and the checks the bench can afford
    at this size (sortedness + multiset sum)."""
    import ctypes

    from b200sort._lib import ALGO_MERGE, ALGO_RADIX, check
    algo = {"radix": ALGO_RADIX, "merge": ALGO_MERGE}[algo_name]
    n = 1 << log2n
    key = (dist, log2n)
    if bufs.get("key") != key:                      # the same keys serve radix and merge
        bufs["src"] = None
        bufs["src"] = _make_device_keys(torch, n, dist, 1, dev)
        bufs["key"] = key
    if bufs.get("n") != n:
        bufs["out"] = bufs["tmp"] = None
        bufs["out"] = torch.empty(n, dtype=torch.int32, device=dev)
        bufs["tmp"] = torch.empty(n, dtype=torch.int32, device=dev)
        bufs["n"] = n
    src, out, tmp = bufs["src"], bufs["out"], bufs["tmp"]
    ws_bytes = L.b200sort_workspace_bytes(n, algo)
    ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=dev)
    ws_ptr = ws.data_ptr() + (-ws.data_ptr()) % 256
    stream = torch.cuda.current_stream().cuda_stream

    def step():
        check(L.b200sort_sort_copy_i32(algo, src.data_ptr(), out.data_ptr(), tmp.data_ptr(), n, ws_ptr, ws_bytes, stream))
    for _ in range(3):
        step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    _check_sorted(torch, out, src)
    kms = (ctypes.c_float * 8)()
    check(L.b200sort_sort_timed_i32(algo, src.data_ptr(), out.data_ptr(), tmp.data_ptr(), n, ws_ptr, ws_bytes, stream,
                                    ctypes.cast(kms, ctypes.c_void_p)))
    row = {"algo": algo_name, "dist": dist, "log2n": log2n, "steps": steps, "ms_per_step": ms,
           "keys_per_s": n / (ms / 1e3), "checked": "sorted + multiset sum",
           "l2": "input larger than L2" if 4 * n > 126e6 else "input fits L2 (64 MiB of 126 MB): flushed by the "
                 "sort's own 2x64 MiB ping-pong traffic only; HBM fractions are quoted all the same"}
    if algo == ALGO_RADIX:
        pass_ms = [kms[i] for i in range(1, 5)]
        ran = [p for p in pass_ms if p > 0.25 * max(pass_ms)] or pass_ms
        executed = len(ran) if n >= (1 << 22) else 4
        k_ms = sum(ran) / len(ran)
        row.update({"histogram_ms": kms[0], "pass_ms": pass_ms, "passes_executed": executed,
                    "pass_frac": 8.0 * n / (k_ms / 1e3) / 1e9 / peaks["hbm_gbs"],
                    "whole_sort_frac": (4.0 + 8.0 * executed) * n / (ms / 1e3) / 1e9 / peaks["hbm_gbs"]})
    else:
        passes = int(round(kms[2]))
        row.update({"block_sort_ms": kms[0], "merge_passes_ms": kms[1], "merge_passes": passes,
                    "pass_frac": 8.0 * n / (kms[1] / max(passes, 1) / 1e3) / 1e9 / peaks["hbm_gbs"],
                    "block_sort_frac": 8.0 * n / (kms[0] / 1e3) / 1e9 / peaks["hbm_gbs"] if kms[0] > 0 else None,
                    "whole_sort_frac": 8.0 * (1 + passes) * n / (ms / 1e3) / 1e9 / peaks["hbm_gbs"]})
    return row


# BASELINE.json configs 2-5 on one GPU: every row is measured in the default run (config 1 is the parity
# suite's size; the headline line itself is config 2/3's radix sort at the metric's n)
CONFIG_ROWS = (
    ("config3: merge sort, 2^28 uniform", "merge", "uniform", 28),
    ("config4: radix, 2^28 skewed90", "radix", "skewed90", 28),
    ("config4: merge, 2^28 skewed90", "merge", "skewed90", 28),
    ("config4: radix, 2^28 ascending (already sorted)", "radix", "ascending", 28),
    ("config4: merge, 2^28 ascending (already sorted)", "merge", "ascending", 28),
    ("config4: radix, 2^28 descending (reverse sorted)", "radix", "descending", 28),
    ("config4: merge, 2^28 descending (reverse sorted)", "merge", "descending", 28),
    ("config2: radix, 2^24 uniform", "radix", "uniform", 24),
    ("config2: radix, 2^24 and3 (AND of 3 uniform words)", "radix", "and3", 24),
    ("config2: radix, 2^24 mask_0000ffff", "radix", "mask_0000ffff", 24),
    ("config2: radix, 2^24 mask_00ff00ff", "radix", "mask_00ff00ff", 24),
    ("config5 denominator: radix, 2^30 uniform on ONE GPU", "radix", "uniform", 30),
)


def _configs_block(L, torch, dev, peaks: dict, steps: int) -> list:
    rows, bufs = [], {}
    for name, algo_name, dist, log2n in CONFIG_ROWS:
        try:
            row = _measure_config(L, torch, dev, algo_name, dist, log2n, steps, peaks, bufs)
        except Exception as e:                      # a row that cannot run says so instead of vanishing
            row = {"algo": algo_name, "dist": dist, "log2n": log2n, "error": repr(e)[:200]}
        row["config"] = name
        rows.append(row)
    bufs.clear()
    torch.cuda.empty_cache()
    return rows


def ours_single(args) -> None:
    import ctypes

    import numpy as np
    import torch

    import b200sort
    from b200sort._lib import ALGO_MERGE, ALGO_RADIX, check, lib

    L = lib()
    torch.cuda.set_device(0)
    dev = torch.device("cuda:0")
    check(L.b200sort_device_check())
    algo = {"radix": ALGO_RADIX, "merge": ALGO_MERGE, "lab": 2}[args.algo]
    n = 1 << args.log2n
    if args.variant is not None:
        check(L.b200sort_radix_set_variant(args.variant))
    if args.merge_variant is not None:
        check(L.b200sort_merge_set_variant(args.merge_variant))

    src = _make_device_keys(torch, n, args.dist, 1, dev)
    out = torch.empty_like(src)
    tmp = torch.empty_like(src)
    ws_bytes = L.b200sort_workspace_bytes(n, algo)
    ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=dev)
    ws_ptr = ws.data_ptr() + (-ws.data_ptr()) % 256
    stream = torch.cuda.current_stream().cuda_stream

    def step():
        check(L.b200sort_sort_copy_i32(algo, src.data_ptr(), out.data_ptr(), tmp.data_ptr(), n, ws_ptr,
                                       ws_bytes, stream))

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    _check_sorted(torch, out, src)

    sampler = ClockSampler(0)
    sampler.start()
    time.sleep(0.02)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    L.b200sort_launch_count_reset()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    launches = int(L.b200sort_launch_count())
    sampler.stop_flag = True
    sampler.join(timeout=2)
    ms_total = e0.elapsed_time(e1)
    ms_per_step = ms_total / args.steps
    value = n / (ms_per_step / 1000.0)
    _check_sorted(torch, out, src)
    if args.dump_outputs:                 # before the per-kernel timing below sorts into `out` again
        _save_dump(args.dump_outputs, out[torch.from_numpy(dump_positions(n)).to(dev)].cpu().numpy())

    # ---- per-kernel timing (CUDA events between the kernels, on the launching stream) ----------
    peaks = _peaks()
    kms = (ctypes.c_float * 8)()
    acc = [0.0] * 8
    reps = 5
    for _ in range(reps):
        check(L.b200sort_sort_timed_i32(algo, src.data_ptr(), out.data_ptr(), tmp.data_ptr(), n, ws_ptr,
                                        ws_bytes, stream, ctypes.cast(kms, ctypes.c_void_p)))
        for i in range(8):
            acc[i] += kms[i] / reps
    if algo == ALGO_RADIX:
        pass_ms = [acc[i] for i in range(1, 5)]
        ran = [p for p in pass_ms if p > 0.25 * max(pass_ms)] if n >= (1 << 22) else pass_ms   # skipped passes exit at once
        kernel_ms = sum(ran) / max(len(ran), 1)
        bytes_per_launch = 8.0 * n
        kernels = {"histogram_ms": acc[0], "pass_ms": pass_ms, "final_copy_ms": acc[5],
                   "histogram_gbs": 4.0 * n / (acc[0] / 1e3) / 1e9 if acc[0] > 0 else None}
        dominant = "radix_onesweep_kernel (one 8-bit-digit pass: 4 B/key read + 4 B/key written)"
        algo_bytes_total = 36.0 * n
    else:
        passes = int(round(acc[2]))
        kernel_ms = acc[1] / max(passes, 1)
        bytes_per_launch = 8.0 * n
        kernels = {"block_sort_ms": acc[0], "merge_passes_ms": acc[1], "merge_passes": passes,
                   "block_sort_gbs": 8.0 * n / (acc[0] / 1e3) / 1e9 if acc[0] > 0 else None,
                   "tile": int(L.b200sort_block_sort_tile()),
                   "merge_variant": L.b200sort_merge_variant_name(args.merge_variant or 0).decode()}
        dominant = "merge_pass_kernel (+ its partition kernel; one merge pass: 8 B/key)"
        algo_bytes_total = 8.0 * n * (1 + passes)
    achieved = bytes_per_launch / (kernel_ms / 1e3) / 1e9
    traffic = None
    if args.log2n == 28:
        traffic = (_ncu_traffic("radix_onesweep", L.b200sort_radix_effective_variant_name().decode()) if algo == ALGO_RADIX
                   else _ncu_traffic("merge_pass"))
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"], "traffic": traffic["bytes"] if traffic else None,
                "traffic_source": traffic["source"] if traffic else None,
                "algorithmic_bytes": bytes_per_launch, "kernel": dominant,
                "kernel_ms": kernel_ms, "peak_source": peaks["source"],
                "whole_sort_gbs": algo_bytes_total / (ms_per_step / 1e3) / 1e9,
                "whole_sort_frac": algo_bytes_total / (ms_per_step / 1e3) / 1e9 / peaks["hbm_gbs"],
                "frac_of_nominal_8tbs": achieved / 8000.0, "kernels": kernels}
    if traffic and "lsu_pct" in traffic:
        roofline["shared_memory_pipe"] = {
            "busy_pct": traffic["lsu_pct"], "source": traffic["source"],
            "note": "l1tex data-pipe wavefronts, % of peak, from the same ncu capture: the kernel's real bound "
                    "(about 17.5 wavefronts per 32 keys and pass for the onesweep pass, 11 for the merge pass)"}

    # ---- end to end through the reference-facing operator, host buffers -------------------------
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    pristine = torch.empty(n, dtype=torch.int32, pin_memory=True)
    pristine.copy_(src)
    torch.cuda.synchronize()
    work = torch.empty(n, dtype=torch.int32, pin_memory=True)
    work_np = work.numpy()
    def host_runs(steps):
        elapsed = 0.0
        for i in range(steps + 1):                         # first call warms the arena, untimed
            work.copy_(pristine)
            t = time.perf_counter()
            check(L.b200sort_order_array_host(work.data_ptr(), n, algo))
            dt = time.perf_counter() - t
            if i > 0:
                elapsed += dt
        assert bool(np.all(work_np[1:] >= work_np[:-1])), "bench: e2e output not sorted"
        return elapsed
    e2e_elapsed = host_runs(e2e_steps)
    # the same call with the streaming switched off (one H2D, one sort, one D2H), for comparison
    L.b200sort_host_set_streaming(0)
    one_shot_ms = 1000.0 * host_runs(min(e2e_steps, 2)) / min(e2e_steps, 2)
    L.b200sort_host_set_streaming(1)
    e2e = {"value": n * e2e_steps / e2e_elapsed, "unit": UNIT, "h2d_bytes_per_step": 4 * n,
           "d2h_bytes_per_step": 4 * n, "steps": e2e_steps, "ms_per_step": 1000.0 * e2e_elapsed / e2e_steps,
           "one_shot_ms_per_step": one_shot_ms,
           "api": "b200sort_order_array_host (what the exported C++ order_array(int*,int) calls), pinned host buffer; "
                  "from 2^25 keys on it streams: chunked H2D, chunk sorts and merges behind the transfers, "
                  "merged output ranges copied back as they finish (one_shot_ms_per_step = the same call with "
                  "b200sort_host_set_streaming(0))"}
    L.b200sort_host_release()
    del pristine, work

    # ---- CPU baseline: the reference's own CPU path on a bounded sample -----------------------------
    cpu = None
    if not args.no_cpu_baseline:
        from b200sort import datagen
        sort_inplace, kind, what = _cpu_sorter()
        log2m = min(args.log2n, args.cpu_log2n)
        m = 1 << log2m
        sample_keys = datagen.make(args.dist if args.dist in datagen.DISTRIBUTIONS else "uniform", m, 1)
        t = time.perf_counter()
        sort_inplace(sample_keys)
        dt = time.perf_counter() - t
        cpu = {"value": m / dt, "unit": UNIT, "cores": 1, "kind": kind,
               "sample": f"one sort of 2^{log2m} {args.dist} keys (seed 1), {dt:.2f} s; {what}",
               "host_cores_available": os.cpu_count()}

    del src, out, tmp, ws
    torch.cuda.empty_cache()
    configs = None if args.no_configs else _configs_block(L, torch, dev, peaks, args.config_steps)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": f"{args.algo} sort of n=2^{args.log2n} {args.dist} int32 keys on 1 B200 "
                               f"(BASELINE configs[{1 if args.algo == 'radix' else 2}] at the metric's n)",
                   "algo": args.algo, "dist": args.dist, "seed": 1, "n": n,
                   "form": "out-of-place (b200sort_sort_copy_i32): each step sorts the same pristine input",
                   "l2": "inputs larger than L2 (1 GiB input vs 126 MB L2), no explicit flush",
                   "radix_variant": L.b200sort_radix_effective_variant_name().decode(),
                   "atomic_order_selftest": bool(L.b200sort_radix_atomic_order_ok()),
                   "radix_tile": int(L.b200sort_radix_tile())},
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches,
        "clocks": sampler.summary(t0, t1), "configs": configs,
    }
    print(json.dumps(line), flush=True)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--algo", default="radix", choices=["radix", "merge", "lab"])
    ap.add_argument("--dist", default="uniform")
    ap.add_argument("--log2n", type=int, default=28)
    ap.add_argument("--variant", type=int, default=None, help="onesweep tile shape (sweeps only)")
    ap.add_argument("--merge-variant", type=int, default=None, help="merge-pass kernel (sweeps only)")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-log2n", type=int, default=27, help="size of the CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE configs 2-5 rows")
    ap.add_argument("--config-steps", type=int, default=4, help="timed sorts per row of the configs block")
    ap.add_argument("--total-log2n", type=int, default=None,
                    help="multi-GPU: 2^T keys IN TOTAL split over the ranks (strong scaling; BASELINE config 5: 30)")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                    help="multi-GPU exchange: fused peer-write scatter (default) or NCCL all-to-all")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's sorted keys to DIR/sorted_keys.npy (one GPU)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and args.impl == "ours" and (world > 1 or args.gpus > 1):
        ap.error("--dump-outputs is not implemented for the multi-GPU sort")
    if args.impl == "reference":
        reference_arm(args)
        return
    if world > 1 or args.gpus > 1:
        from b200sort import dist as b200dist
        b200dist.bench_main(args, METRIC, UNIT, ClockSampler, _peaks)
        return
    ours_single(args)


if __name__ == "__main__":
    main()
