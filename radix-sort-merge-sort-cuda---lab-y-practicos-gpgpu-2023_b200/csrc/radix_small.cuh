// radix_small.cuh -- k0: the whole sort in ONE CTA for arrays of up to kSmallTile keys (included by radix.cu).
//
// The lab's own sizes (SRM/main.cpp:17: 2^8 .. 2^16) and the sizes its report publishes are small: there the
// onesweep pipeline is seven launches of mostly launch latency.  Up to 8192 keys fit one CTA's shared
// memory, so the four 8-bit passes run back to back in one kernel: rank with one shared-memory atomicAdd per
// key on the warp's counters (the same lane-ordered rank as the pass kernel, same self-test gate), scan,
// scatter into the other shared-memory buffer, next digit.  Slots past n hold INT_MAX (any other order: the key whose
// image is 0xFFFFFFFF): they are last in tile order and carry the largest digit in every pass, so they stay behind the
// n real keys.
#pragma once
#include "radix_pipelined.cuh"

namespace b200sort {

constexpr int kSmallThreads = 512;
constexpr int kSmallWarps = kSmallThreads / 32;
constexpr int kSmallIpt = 16;
constexpr int kSmallTile = kSmallThreads * kSmallIpt;          // 8192
constexpr size_t kSmallSmemBytes = (size_t)2 * kSmallTile * 4 + (size_t)kSmallWarps * kRadixBins * 4 + 64;

// KEYS = 1: any key order, `order` = its masks; 0: int32 ascending.
template <int KEYS>
__device__ __forceinline__ void radix_small_body(const int32_t *in, int32_t *out, uint32_t n, SignXor order)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    int32_t  *s_buf   = reinterpret_cast<int32_t *>(smem_raw);                       // [2][kSmallTile]
    uint32_t *s_table = reinterpret_cast<uint32_t *>(s_buf + 2 * kSmallTile);        // [16][256]
    uint32_t *s_sums  = s_table + kSmallWarps * kRadixBins;                          // [8] warp sums of the scan

    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t *wt = s_table + warp * kRadixBins;
    const uint32_t wofs = warp * (32 * kSmallIpt) + lane;

    const int32_t pad_key = KEYS ? (int32_t)key_of_last_image(order) : 0x7FFFFFFF;
    for (uint32_t i = tid; i < (uint32_t)kSmallTile; i += kSmallThreads) s_buf[i] = (i < n) ? in[i] : pad_key;
    __syncthreads();

    int cur = 0;
#pragma unroll 1
    for (int pass = 0; pass < kRadixPasses; ++pass) {
        const int shift = pass * kRadixBits;
        const uint32_t flip = (pass == kRadixPasses - 1) ? 0x80u : 0u;
        const uint32_t flips = flips_of(order.neg, order.pos, shift);
        auto dig = [&](int32_t k) -> uint32_t { return KEYS ? digit_of_image(k, shift, flips) : digit_of(k, shift, flip); };
        const int32_t *src = s_buf + cur * kSmallTile;
        int32_t *dst = s_buf + (cur ^ 1) * kSmallTile;
        for (int j = lane; j < kRadixBins; j += 32) wt[j] = 0;
        __syncwarp();
        int32_t key[kSmallIpt];
        uint32_t rank[kSmallIpt];
#pragma unroll
        for (int i = 0; i < kSmallIpt; ++i) {
            key[i] = src[wofs + i * 32];                      // warp-striped: tile order = memory order
            rank[i] = atomicAdd(wt + dig(key[i]), 1u);
        }
        __syncthreads();                                      // counts final, src fully read
        if (tid < kRadixBins) {
            uint32_t total = 0;
#pragma unroll
            for (int w = 0; w < kSmallWarps; ++w) total += s_table[w * kRadixBins + tid];
            uint32_t x = total;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
                if (lane >= (uint32_t)o) x += y;
            }
            if (lane == 31) s_sums[warp] = x;
            bar_sync(1, kRadixBins);
            uint32_t add = 0;
#pragma unroll
            for (int w = 0; w < kRadixBins / 32; ++w) add += (w < (int)warp) ? s_sums[w] : 0u;
            uint32_t run = x - total + add;                   // first position of this digit
#pragma unroll
            for (int w = 0; w < kSmallWarps; ++w) {
                const uint32_t c = s_table[w * kRadixBins + tid];
                s_table[w * kRadixBins + tid] = run;
                run += c;
            }
        }
        __syncthreads();                                      // positions final
#pragma unroll
        for (int i = 0; i < kSmallIpt; ++i) {
            B200_CHECK_AT(8, wt[dig(key[i])] + rank[i] < (uint32_t)kSmallTile);
            dst[wt[dig(key[i])] + rank[i]] = key[i];
        }
        __syncthreads();                                      // dst complete; the counters may be cleared
        cur ^= 1;
    }
    const int32_t *res = s_buf + cur * kSmallTile;
    for (uint32_t i = tid; i < n; i += kSmallThreads) out[i] = res[i];
}

__global__ void __launch_bounds__(kSmallThreads, 1)
radix_small_kernel(const int32_t *in, int32_t *out, uint32_t n)
{
    radix_small_body<0>(in, out, n, SignXor{0x80000000u, 0x80000000u});
}
__global__ void __launch_bounds__(kSmallThreads, 1)
radix_small_keys_kernel(const int32_t *in, int32_t *out, uint32_t n, SignXor order)
{
    radix_small_body<1>(in, out, n, order);
}

}  // namespace b200sort
