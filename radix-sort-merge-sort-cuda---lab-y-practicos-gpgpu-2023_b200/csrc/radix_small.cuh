// radix_small.cuh -- k0: the whole sort in ONE CTA for arrays of up to kSmallTile keys (included by radix.cu).
//
// The lab's own sizes (SRM/main.cpp:17: 2^8 .. 2^16) and the sizes its report publishes are small: there the
// onesweep pipeline is seven launches of mostly launch latency.  Up to 8192 keys fit one CTA's shared
// memory, so the four 8-bit passes run back to back in one kernel: rank with one shared-memory atomicAdd per
// key on the warp's counters (the same lane-ordered rank as the pass kernel, same self-test gate), scan,
// scatter into the other shared-memory buffer, next digit.  Slots past n hold INT_MAX (any other order: the key whose
// image is 0xFFFFFFFF): they are last in tile order and carry the largest digit in every pass, so they stay behind the
// n real keys.
// The segmented sort (segmented.cu) runs the same body on one segment per CTA, with smaller tiles, values riding
// beside the keys, or ballot ranks (SAFE: one atomicAdd per distinct digit of a warp instruction, by its leader).
#pragma once
#include "radix_digit.cuh"

namespace b200sort {

constexpr int kSmallThreads = 512;
constexpr int kSmallWarps = kSmallThreads / 32;
constexpr int kSmallIpt = 16;
constexpr int kSmallTile = kSmallThreads * kSmallIpt;          // 8192
constexpr size_t kSmallSmemBytes = (size_t)2 * kSmallTile * 4 + (size_t)kSmallWarps * kRadixBins * 4 + 64;
// Shared memory of radix_small_body<KEYS, THREADS, IPT, VALS>: key (and value) buffers, warp counters, scan sums.
constexpr size_t small_smem_bytes(int threads, int ipt, int vals) {
    return (size_t)2 * threads * ipt * 4 * (vals ? 2 : 1) + (size_t)(threads / 32) * kRadixBins * 4 + 64;
}

// KEYS = 1: any key order, `order` = its masks; 0: int32 ascending.  THREADS >= 256 (the digit scan).
// VALS = 1: vin[i] moves with in[i] (stable); 2: the values are the positions 0..n-1, made here (vin is not read), and
// vout is an int64 output viewed as int32.  SAFE = 1: ranks from ballots instead of lane-ordered atomics.
// SKIP_PAD = 1: the slots past n are neither ranked nor moved.  They would stay last anyway, but ranking them sends
// every padded lane of a warp to the same counter (digit 255) in every pass: with a short segment in a large tile
// that contended atomicAdd is most of the work.
template <int KEYS, int THREADS = kSmallThreads, int IPT = kSmallIpt, int VALS = 0, int SAFE = 0, int SKIP_PAD = 0>
__device__ __forceinline__ void radix_small_body(const int32_t *in, int32_t *out, uint32_t n, SignXor order,
                                                 const int32_t *vin = nullptr, int32_t *vout = nullptr)
{
    static_assert(THREADS >= kRadixBins && THREADS % 32 == 0, "the digit scan needs 256 threads");
    constexpr int kWarps = THREADS / 32;
    constexpr int kTile = THREADS * IPT;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    int32_t  *s_buf   = reinterpret_cast<int32_t *>(smem_raw);                       // [2][kTile]
    int32_t  *s_vbuf  = s_buf + 2 * kTile;                                           // [2][kTile] if VALS
    uint32_t *s_table = reinterpret_cast<uint32_t *>(s_buf + (VALS ? 4 : 2) * kTile); // [kWarps][256]
    uint32_t *s_sums  = s_table + kWarps * kRadixBins;                               // [8] warp sums of the scan

    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t *wt = s_table + warp * kRadixBins;
    const uint32_t wofs = warp * (32 * IPT) + lane;

    const int32_t pad_key = KEYS ? (int32_t)key_of_last_image(order) : 0x7FFFFFFF;
    for (uint32_t i = tid; i < (uint32_t)kTile; i += THREADS) s_buf[i] = (i < n) ? in[i] : pad_key;
    if constexpr (VALS == 2)
        for (uint32_t i = tid; i < n; i += THREADS) s_vbuf[i] = (int32_t)i;
    else if constexpr (VALS != 0)
        for (uint32_t i = tid; i < n; i += THREADS) s_vbuf[i] = vin[i];
    __syncthreads();

    int cur = 0;
#pragma unroll 1
    for (int pass = 0; pass < kRadixPasses; ++pass) {
        const int shift = pass * kRadixBits;
        const uint32_t flip = (pass == kRadixPasses - 1) ? 0x80u : 0u;
        const uint32_t flips = flips_of(order.neg, order.pos, shift);
        auto dig = [&](int32_t k) -> uint32_t { return KEYS ? digit_of_image(k, shift, flips) : digit_of(k, shift, flip); };
        const int32_t *src = s_buf + cur * kTile;
        int32_t *dst = s_buf + (cur ^ 1) * kTile;
        for (int j = lane; j < kRadixBins; j += 32) wt[j] = 0;
        __syncwarp();
        int32_t key[IPT];
        uint32_t rank[IPT];
#pragma unroll
        for (int i = 0; i < IPT; ++i) {
            key[i] = src[wofs + i * 32];                      // warp-striped: tile order = memory order
            const bool ranked = SKIP_PAD == 0 || wofs + i * 32 < n;
            if constexpr (SAFE != 0) {
                const uint32_t d = ranked ? dig(key[i]) : (uint32_t)kRadixBins;
                const uint32_t peers = __match_any_sync(0xffffffffu, d);
                const uint32_t leader = __ffs(peers) - 1;
                uint32_t base = 0;
                if (ranked && lane == leader) base = atomicAdd(wt + d, (uint32_t)__popc(peers));
                rank[i] = __shfl_sync(0xffffffffu, base, leader) + __popc(peers & lanemask_lt());
            } else if constexpr (SKIP_PAD != 0) {
                rank[i] = ranked ? atomicAdd(wt + dig(key[i]), 1u) : 0u;
            } else {
                rank[i] = atomicAdd(wt + dig(key[i]), 1u);
            }
        }
        __syncthreads();                                      // counts final, src fully read
        if (tid < kRadixBins) {
            uint32_t total = 0;
#pragma unroll
            for (int w = 0; w < kWarps; ++w) total += s_table[w * kRadixBins + tid];
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
            for (int w = 0; w < kWarps; ++w) {
                const uint32_t c = s_table[w * kRadixBins + tid];
                s_table[w * kRadixBins + tid] = run;
                run += c;
            }
        }
        __syncthreads();                                      // positions final
#pragma unroll
        for (int i = 0; i < IPT; ++i) {
            if (SKIP_PAD != 0 && wofs + i * 32 >= n) continue;
            B200_CHECK_AT(8, wt[dig(key[i])] + rank[i] < (uint32_t)kTile);
            dst[wt[dig(key[i])] + rank[i]] = key[i];
        }
        if constexpr (VALS != 0) {                            // values follow their keys' moves
            const int32_t *vsrc = s_vbuf + cur * kTile;
            int32_t *vdst = s_vbuf + (cur ^ 1) * kTile;
#pragma unroll
            for (int i = 0; i < IPT; ++i) {
                const uint32_t at = wofs + i * 32;
                if (at < n) vdst[wt[dig(key[i])] + rank[i]] = vsrc[at];
            }
        }
        __syncthreads();                                      // dst complete; the counters may be cleared
        cur ^= 1;
    }
    const int32_t *res = s_buf + cur * kTile;
    for (uint32_t i = tid; i < n; i += THREADS) out[i] = res[i];
    if constexpr (VALS == 2) {
        const int32_t *vres = s_vbuf + cur * kTile;
        int64_t *wide = reinterpret_cast<int64_t *>(vout);
        B200_CHECK((reinterpret_cast<uintptr_t>(wide) & 7) == 0);
        for (uint32_t i = tid; i < n; i += THREADS) wide[i] = vres[i];
    } else if constexpr (VALS != 0) {
        const int32_t *vres = s_vbuf + cur * kTile;
        for (uint32_t i = tid; i < n; i += THREADS) vout[i] = vres[i];
    }
}

}  // namespace b200sort
