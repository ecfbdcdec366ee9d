// radix_digit.cuh -- what every radix kernel shares about digits and tile-status words: the digit of a key in a
// pass, the {flag:2, count:30} status words of the decoupled look-back, a named barrier and the 256-digit scan
// (radix.cu, segmented.cu, radix64.cu).
#pragma once
#include "radix.cuh"

namespace b200sort {

constexpr uint32_t kFlagLocal = 1u << 30;   // this tile's own digit count
constexpr uint32_t kFlagIncl  = 2u << 30;   // inclusive count over tiles 0..this
constexpr uint32_t kValueMask = (1u << 30) - 1;

// digit of `key` for the pass with this shift; `flip` is 0x80 for the top digit (signed order)
__device__ __forceinline__ uint32_t digit_of(int32_t key, int shift, uint32_t flip) {
    return ((static_cast<uint32_t>(key) >> shift) & (kRadixBins - 1)) ^ flip;
}
// The generic pass kernels (KEYS = 1): the digit of the key's image key ^ (key < 0 ? key_neg : key_pos).  `flips`
// (flips_of) holds this pass's byte of key_pos in byte 0 and of key_neg in byte 1, so the order costs one register,
// as `flip` does, and two instructions more per digit: the sign as a byte selector, and the byte permute.
__device__ __forceinline__ uint32_t flips_of(uint32_t key_neg, uint32_t key_pos, int shift) {
    return ((key_pos >> shift) & (kRadixBins - 1)) | (((key_neg >> shift) & (kRadixBins - 1)) << 8);
}
__device__ __forceinline__ uint32_t digit_of_image(int32_t key, int shift, uint32_t flips) {
    return ((static_cast<uint32_t>(key) >> shift) ^ __byte_perm(flips, 0u, static_cast<uint32_t>(key) >> 31)) & (kRadixBins - 1);
}

__device__ __forceinline__ void bar_sync(int id, int count) {
    asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(count) : "memory");
}

// Exclusive scan of one value per thread over threads 0..255 (named barrier 1); `sums` holds 8 words.
__device__ __forceinline__ uint32_t scan256(uint32_t v, uint32_t *sums) {
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= (uint32_t)o) x += y;
    }
    if (lane == 31) sums[warp] = x;
    bar_sync(1, kRadixBins);
    uint32_t add = 0;
#pragma unroll
    for (int w = 0; w < kRadixBins / 32; ++w) add += (w < (int)warp) ? sums[w] : 0u;
    return x - v + add;
}

}  // namespace b200sort
