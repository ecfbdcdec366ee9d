// radix_misc.cuh -- the plan's final copy and the lane-order self-test (included by radix.cu).
#pragma once
#include "radix_tile.cuh"

namespace b200sort {

// The plan's final copy (only ever needed with pass skipping): tmp -> out when an in-place sort
// executed an odd number of passes, in -> out when an out-of-place sort executed none.
__global__ void __launch_bounds__(256)
radix_final_copy_kernel(const int32_t *in_buf, int32_t *out_buf, const int32_t *tmp_buf, size_t n,
                        const RadixControl *ctl, uint32_t n_from_ctl = 0)
{
    if (n_from_ctl) n = ctl->n_dev;
    const uint32_t sel = ctl->final_copy;
    if (sel == 0) return;
    const int32_t *src = (sel == kSelIn) ? in_buf : tmp_buf;
    if (src == out_buf) return;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t nvec = n / 4;
    const int4 *s4 = reinterpret_cast<const int4 *>(src);
    int4 *d4 = reinterpret_cast<int4 *>(out_buf);
    const bool aligned = ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(out_buf)) & 15) == 0;
    const size_t start = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (aligned) {
        for (size_t i = start; i < nvec; i += stride) d4[i] = s4[i];
        for (size_t i = nvec * 4 + start; i < n; i += stride) out_buf[i] = src[i];
    } else {
        for (size_t i = start; i < n; i += stride) out_buf[i] = src[i];
    }
}

// The final step of the sort with indices (radix_sort_indices), in place of the final copy.  Keys: the final copy's
// plan.  Indices, which only the executed passes wrote:
//   no pass executed (one bin held every key in every pass): the sort is the identity, the indices are 0..n-1;
//   the last executed pass landed in tmp (in place, an odd number of passes): widen tmp_idx -> out_idx;
//   else the last executed pass stored them as int64 already.
__global__ void __launch_bounds__(256)
radix_final_indices_kernel(const int32_t *in_buf, int32_t *out_buf, const int32_t *tmp_buf, int64_t *out_idx,
                           const int32_t *tmp_idx, size_t n, const RadixControl *ctl)
{
    const uint32_t sel = ctl->final_copy;
    uint32_t executed = 0;
    for (int p = 0; p < kRadixPasses; ++p) executed += ctl->skip[p] ? 0u : 1u;
    if (sel == 0 && executed != 0) return;
    const int32_t *src = (sel == kSelIn) ? in_buf : tmp_buf;
    const bool copy_keys = sel != 0 && src != out_buf;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    B200_CHECK((reinterpret_cast<uintptr_t>(out_idx) & 7) == 0);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        if (copy_keys) out_buf[i] = src[i];
        out_idx[i] = executed == 0 ? (int64_t)i : (int64_t)tmp_idx[i];
    }
}

// Self-test behind kRankAdd: that mode is stable only if same-address shared-memory atomics issued by one
// warp instruction are resolved in lane order.  PTX does not promise that; every B200 tried does it
// (tools/atomic_order_probe.cu: 245 M same-address pairs, 0 violations).  The library checks it once per
// DEVICE (radix.cu: atomic_order_ok) and falls back to the ballot-ranked shape if it ever fails.  The test
// reproduces what the pass kernels actually do:
//   * packed rows: the two warps of a pair add 1 << 16 / 1 to the SAME words at the same time, unsynchronised;
//   * counters that start anywhere in the 16-bit range (a warp adds at most 640 per tile, so a half never
//     carries into its neighbour -- the test stays below 65535 as the kernels do);
//   * conflict patterns from none to 32-way, and sets of digits that share a bank;
//   * the hot-digit path: one lane adds the whole group's count, the other lanes add 1, in ONE instruction;
//   * ordinary shared-memory loads and stores from every warp in between (the staging traffic).
__global__ void __launch_bounds__(512)
radix_atomic_order_selftest_kernel(uint32_t *violations)
{
    __shared__ uint32_t table[8][kRadixBins];
    __shared__ uint32_t traffic[1024];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t *row = table[warp >> 1];
    const uint32_t sh = (warp & 1) * 16;
    const uint32_t lt = lanemask_lt();
    uint32_t x = (blockIdx.x * 512u + tid) * 2654435761u + 12345u;
    uint32_t bad = 0;
    for (int round = 0; round < 96; ++round) {
        // both halves of every counter start at the same pseudo-random level
        const uint32_t level = ((uint32_t)round * 7919u + blockIdx.x * 131u) % 65000u;
        asm volatile("bar.sync %0, 64;" :: "r"(3 + (warp >> 1)) : "memory");
        for (int j = lane + 32 * (warp & 1); j < kRadixBins; j += 64) row[j] = level | (level << 16);
        asm volatile("bar.sync %0, 64;" :: "r"(3 + (warp >> 1)) : "memory");
        x ^= x << 13; x ^= x >> 17; x ^= x << 5;
        const uint32_t bins = 1u << (round & 7);                 // 1, 2, 4 ... 128 distinct digits
        const uint32_t d = ((x >> 8) % bins) * ((round & 8) ? 32u : 1u) % kRadixBins;   // also same-bank sets
        traffic[(tid * 5 + round) & 1023] = x;                   // staging-like traffic around the atomic
        uint32_t got, want;
        const uint32_t peers = __match_any_sync(0xffffffffu, d);
        if ((round & 3) != 3) {
            got = ((atomicAdd(row + d, 1u << sh) >> sh) & 0xffffu) - level;
            want = __popc(peers & lt);
        } else {
            // hot-digit path of the pass kernels: lane 0's digit is ranked by ballot and ONE atomic
            const uint32_t hd = __shfl_sync(0xffffffffu, d, 0);
            const bool same = (d == hd);
            const uint32_t sm = __ballot_sync(0xffffffffu, same);
            const uint32_t leader = (uint32_t)(__ffs(sm) - 1) & 31u;
            uint32_t r = 0;
            if (!same || lane == leader)
                r = ((atomicAdd(row + d, (same ? (uint32_t)__popc(sm) : 1u) << sh) >> sh) & 0xffffu) - level;
            const uint32_t r0 = __shfl_sync(0xffffffffu, r, leader);
            if (same) r = r0 + __popc(sm & lt);
            got = r;
            want = __popc(peers & lt);
        }
        x += traffic[(tid * 11 + round * 3) & 1023];
        bad += (got != want);
        // the halves must not have leaked into each other: every counter holds level + its digit's count
        __syncwarp();
        const uint32_t after = (row[d] >> sh) & 0xffffu;
        bad += (after != level + __popc(peers));
    }
    if (bad) atomicAdd(violations, bad);
    if (x == 0x12345678u) violations[0] += 1;                    // keeps the traffic loads alive
}


}  // namespace b200sort
