// radix_hist.cuh -- k1: the digit-histogram kernel of the onesweep radix sort (included by radix.cu).
#pragma once
#include "radix.cuh"
#include "radix_async.cuh"

#include <cooperative_groups.h>

namespace cg = cooperative_groups;

namespace b200sort {

// ================================================================================================
// k1: digit histograms
// ================================================================================================
constexpr int kHistThreads = 512;
constexpr int kHistUnroll  = 4;                  // 128-bit loads in flight per thread
constexpr int kHistBlocksPerSM = 3;
// Shared-memory counters are 16-bit and LANE-PRIVATE: counter (place p, digit d, lane l) lives in half (p & 1) of
// word ((p >> 1) * 256 + d) * 32 + l.  The bank is l: no two lanes of an atomic instruction ever meet, whatever the
// key distribution -- one wavefront per instruction (32 random words on 32 banks cost ~3.5; round 1's layout, two
// lanes per word, cost 2.2 and held the kernel at 91 % of the load/store pipe) -- and the half is a compile-time
// constant of the place, so the address costs the same two instructions as before.  16-bit counters overflow after
// 65535 hits, so the block flushes to the global histogram every kHistFlushIters iterations (<= 32768 hits each).
constexpr int kHistSmemWords  = (kRadixPasses / 2) * kRadixBins * 32;            // 64 KiB
constexpr size_t kHistSmemBytes = (size_t)kHistSmemWords * 4;
constexpr int kHistFlushIters = 128;   // 128 iters * (4 keys * 4 loads) * 16 warps = 32768 per lane column

// col_s = shared-memory address of the lane's column (sh + lane).  Three instructions per counter: the digit by a
// byte permute, the address by one shift-add, the add itself without a return value.
__device__ __forceinline__ void hist_add(uint32_t col_s, int32_t key) {
    const uint32_t k = (uint32_t)key;                   // raw bytes: the top byte's sign flip (key_bits) is applied by hist_flush
    const uint32_t d0 = __byte_perm(k, 0u, 0x4440u), d1 = __byte_perm(k, 0u, 0x4441u), d2 = __byte_perm(k, 0u, 0x4442u),
                   d3 = __byte_perm(k, 0u, 0x4443u);
    asm volatile("red.shared.add.u32 [%0], 1;"           :: "r"(col_s + (d0 << 7)) : "memory");
    asm volatile("red.shared.add.u32 [%0], 65536;"       :: "r"(col_s + (d1 << 7)) : "memory");
    asm volatile("red.shared.add.u32 [%0+32768], 1;"     :: "r"(col_s + (d2 << 7)) : "memory");
    asm volatile("red.shared.add.u32 [%0+32768], 65536;" :: "r"(col_s + (d3 << 7)) : "memory");
}

// Sum the 32 lane columns of every (place, digit), add into the global histogram, clear.  Thread = one word row
// = one digit of two places.
__device__ __forceinline__ void hist_flush(uint32_t *sh, RadixControl *ctl, uint32_t tid) {
    static_assert(kHistThreads == (kRadixPasses / 2) * kRadixBins, "one thread per word row");
    __syncthreads();
    uint32_t lo = 0, hi = 0;
#pragma unroll
    for (uint32_t l = 0; l < 32; ++l) {
        const uint32_t idx = tid * 32 + ((l + tid) & 31);        // rotate: conflict-free across threads
        const uint32_t v = sh[idx];
        sh[idx] = 0;
        lo += v & 0xffffu;
        hi += v >> 16;
    }
    const uint32_t pp = tid >> kRadixBits, d = tid & (kRadixBins - 1);
    if (lo) atomicAdd(&ctl->hist[2 * pp][d], lo);
    if (hi) atomicAdd(&ctl->hist[2 * pp + 1][pp == 1 ? (d ^ 0x80u) : d], hi);       // place 3 was counted by its raw top byte
    __syncthreads();
}

// What the last block of the histogram kernel does once the four digit histograms are complete: exclusive bases,
// skippable passes, hot digits, the buffer plan.  Also run on its own (radix_plan_kernel) when the histograms were
// counted elsewhere -- the multi-GPU exchange counts them at the source, under the NVLink transfer.
__device__ __forceinline__ void radix_finish_plan(RadixControl *ctl, size_t n, uint32_t skip_enabled, uint32_t in_place,
                                                  uint32_t tid, uint32_t *s_warp_sums, uint32_t *s_skip, uint32_t *s_hot)
{
    const uint32_t lane = tid & 31, warp = tid >> 5;
    for (int p = 0; p < kRadixPasses; ++p) {
        const uint32_t c = (tid < kRadixBins) ? __ldcg(&ctl->hist[p][tid]) : 0u;
        uint32_t x = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= (uint32_t)o) x += y;
        }
        if (tid < kRadixBins && lane == 31) s_warp_sums[warp] = x;
        __syncthreads();
        if (tid < kRadixBins) {
            uint32_t add = 0;
            for (uint32_t w = 0; w < warp; ++w) add += s_warp_sums[w];
            ctl->base[p][tid] = x - c + add;
            if (skip_enabled && n > 0 && c == (uint32_t)n) s_skip[p] = 1;
            if ((size_t)c * 8 > n) atomicMax(&s_hot[p], ((c >> 6) << 8) | tid);   // the most frequent such digit wins
        }
        __syncthreads();
    }
    // The buffer plan: executed pass j reads what pass j-1 wrote (the input for j = 0).
    //   in place     : writes alternate tmp, out, tmp, ...; an odd count leaves the result in tmp
    //                  and the final-copy kernel brings it home;
    //   out of place : writes alternate so that the LAST executed pass lands in out; the input
    //                  is never written.  No executed pass at all (all keys equal): copy in -> out.
    if (tid == 0) {
        ctl->n_dev = (uint32_t)n;
        uint32_t executed = 0;
        for (int p = 0; p < kRadixPasses; ++p) executed += s_skip[p] ? 0u : 1u;
        uint32_t j = 0, cur = kSelIn;
        for (int p = 0; p < kRadixPasses; ++p) {
            ctl->skip[p] = s_skip[p];
            ctl->hot[p] = s_hot[p] ? 1u + (s_hot[p] & 255u) : 0u;
            ctl->src_sel[p] = cur;
            uint32_t dst = cur;
            if (!s_skip[p]) {
                if (in_place) dst = (j % 2 == 0) ? kSelTmp : kSelOut;
                else          dst = ((executed - 1 - j) % 2 == 0) ? kSelOut : kSelTmp;
                ++j;
                cur = dst;
            }
            ctl->dst_sel[p] = dst;
        }
        uint32_t final_copy = 0;
        if (in_place) { if (cur == kSelTmp) final_copy = kSelTmp; }
        else          { if (executed == 0) final_copy = kSelIn; }
        ctl->final_copy = final_copy;
    }
}

// The plan from histograms that already exist: d_hist[p][d] (uint32) = keys whose digit p is d; *d_n keys in all.
__global__ void __launch_bounds__(kHistThreads)
radix_plan_kernel(const uint32_t *__restrict__ d_hist, const uint32_t *d_n, RadixControl *ctl, uint32_t skip_enabled,
                  uint32_t in_place)
{
    __shared__ uint32_t s_warp_sums[kRadixBins / 32];
    __shared__ uint32_t s_skip[kRadixPasses];
    __shared__ uint32_t s_hot[kRadixPasses];
    const uint32_t tid = threadIdx.x;
    for (uint32_t i = tid; i < kRadixPasses * kRadixBins; i += kHistThreads) ctl->hist[i >> kRadixBits][i & (kRadixBins - 1)] = d_hist[i];
    if (tid < kRadixPasses) { s_skip[tid] = 0; s_hot[tid] = 0; }
    __threadfence();
    __syncthreads();
    radix_finish_plan(ctl, (size_t)*d_n, skip_enabled, in_place, tid, s_warp_sums, s_skip, s_hot);
}

// KEYS = 1: any key order; the bytes of every key's image k ^ (k < 0 ? order.neg : order.pos) are counted, and the
// order is left in the control block for the generic pass kernels.  0: int32 ascending.
template <int KEYS>
__device__ __forceinline__ void
radix_histogram_body(const int32_t *__restrict__ keys, size_t n, RadixControl *ctl, uint32_t *status_to_zero,
                     size_t status_words, uint32_t skip_enabled, uint32_t in_place, const uint32_t *d_n, SignXor order)
{
    if (d_n != nullptr) n = *d_n;                       // key count produced on the device (<= the n the grid was sized for)
    extern __shared__ __align__(16) uint32_t sh[];
    __shared__ uint32_t s_warp_sums[kRadixBins / 32];
    __shared__ uint32_t s_skip[kRadixPasses];
    __shared__ uint32_t s_hot[kRadixPasses];
    __shared__ uint32_t s_is_last;

    const uint32_t tid = threadIdx.x;
    if (KEYS && blockIdx.x == 0 && tid == 0) {
        ctl->key_neg = order.neg;
        ctl->key_pos = order.pos;
        ctl->key_pad = key_of_last_image(order);
    }
    // hist_flush flips the top byte of what it was given back: hand it image ^ 0x80000000
    const uint32_t xneg = order.neg ^ 0x80000000u, xpos = order.pos ^ 0x80000000u;
    {
        uint4 *z = reinterpret_cast<uint4 *>(sh);
        for (uint32_t i = tid; i < kHistSmemWords / 4; i += kHistThreads) z[i] = make_uint4(0, 0, 0, 0);
    }

    // Zero the tile-status buffer the first pass will use.
    if (status_to_zero != nullptr) {
        uint4 *z = reinterpret_cast<uint4 *>(status_to_zero);
        const size_t nz = status_words / 4;
        for (size_t i = (size_t)blockIdx.x * kHistThreads + tid; i < nz;
             i += (size_t)gridDim.x * kHistThreads)
            z[i] = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();

    const uint32_t col = smem_u32(sh + (tid & 31));
    auto add = [&](int32_t k) { hist_add(col, KEYS ? (int32_t)sign_xor((uint32_t)k, xneg, xpos) : k); };

    // Scalar head up to 16-byte alignment, 128-bit body, scalar tail.
    size_t head = ((16 - (reinterpret_cast<uintptr_t>(keys) & 15)) & 15) / 4;
    if (head > n) head = n;
    const size_t nvec = (n - head) / 4;
    const size_t tail_start = head + nvec * 4;
    const int4 *v = reinterpret_cast<const int4 *>(keys + head);

    constexpr size_t kChunk = (size_t)kHistThreads * kHistUnroll;
    int iters = 0;
    for (size_t base = (size_t)blockIdx.x * kChunk; base < nvec; base += (size_t)gridDim.x * kChunk) {
        // the chunk this CTA reads next is sent for (TMA prefetch into L2): three CTAs of this size leave an SM 60 KB of
        // L1, which bounds the loads in flight, so L2 hits instead of HBM reads are what lifts the load rate
        if (tid == 0) {
            const size_t far = base + (size_t)gridDim.x * kChunk;
            if (far < nvec)
                bulk_prefetch_l2(v + far, (uint32_t)((nvec - far < kChunk ? nvec - far : kChunk) * sizeof(int4)));
        }
        int4 r[kHistUnroll];
        bool ok[kHistUnroll];
#pragma unroll
        for (int u = 0; u < kHistUnroll; ++u) {
            const size_t idx = base + (size_t)u * kHistThreads + tid;
            ok[u] = idx < nvec;
            if (ok[u]) r[u] = ld_stream_v4(v + idx);
        }
#pragma unroll
        for (int u = 0; u < kHistUnroll; ++u) {
            if (ok[u]) {
                add(r[u].x); add(r[u].y);
                add(r[u].z); add(r[u].w);
            }
        }
        if (++iters == kHistFlushIters) { hist_flush(sh, ctl, tid); iters = 0; }
    }
    if (blockIdx.x == 0) {   // < 8 keys in total: cannot overflow anything
        for (size_t i = tid; i < head; i += kHistThreads) add(keys[i]);
        for (size_t i = tail_start + tid; i < n; i += kHistThreads) add(keys[i]);
    }
    hist_flush(sh, ctl, tid);

    // The last block to finish turns counts into exclusive bases.
    __threadfence();
    __syncthreads();
    if (tid == 0) s_is_last = (atomicAdd(&ctl->hist_blocks_done, 1u) == gridDim.x - 1) ? 1u : 0u;
    if (tid < kRadixPasses) { s_skip[tid] = 0; s_hot[tid] = 0; }
    __syncthreads();
    if (!s_is_last) return;
    __threadfence();

    radix_finish_plan(ctl, n, skip_enabled, in_place, tid, s_warp_sums, s_skip, s_hot);
}

__global__ void __launch_bounds__(kHistThreads)
radix_histogram_kernel(const int32_t *__restrict__ keys, size_t n, RadixControl *ctl,
                       uint32_t *status_to_zero, size_t status_words, uint32_t skip_enabled,
                       uint32_t in_place, const uint32_t *d_n = nullptr)
{
    radix_histogram_body<0>(keys, n, ctl, status_to_zero, status_words, skip_enabled, in_place, d_n,
                            SignXor{0x80000000u, 0x80000000u});
}
__global__ void __launch_bounds__(kHistThreads)
radix_histogram_keys_kernel(const int32_t *__restrict__ keys, size_t n, RadixControl *ctl, uint32_t *status_to_zero,
                            size_t status_words, uint32_t skip_enabled, uint32_t in_place, SignXor order)
{
    radix_histogram_body<1>(keys, n, ctl, status_to_zero, status_words, skip_enabled, in_place, nullptr, order);
}

}  // namespace b200sort
