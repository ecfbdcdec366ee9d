// common.cuh -- shared helpers of libb200sort (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

#include "../../include/b200sort.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libb200sort is written for sm_100a only"
#endif

namespace b200sort {

// ---- host-side error plumbing -----------------------------------------------------------------
extern thread_local cudaError_t g_last_cuda_error;
extern thread_local unsigned long long g_launch_count;

inline int record_cuda(cudaError_t e) {
    if (e == cudaSuccess) return B200SORT_OK;
    g_last_cuda_error = e;
    return B200SORT_ERR_CUDA;
}

#define B200_CUDA_TRY(expr)                                              \
    do {                                                                 \
        cudaError_t e__ = (expr);                                        \
        if (e__ != cudaSuccess) return ::b200sort::record_cuda(e__);     \
    } while (0)

// After every kernel launch: count it and surface launch-configuration errors.
#define B200_LAUNCH_CHECK()                                              \
    do {                                                                 \
        ++::b200sort::g_launch_count;                                    \
        cudaError_t e__ = cudaGetLastError();                            \
        if (e__ != cudaSuccess) return ::b200sort::record_cuda(e__);     \
    } while (0)

#define B200_TRY(expr)                                                   \
    do {                                                                 \
        int s__ = (expr);                                                \
        if (s__ != B200SORT_OK) return s__;                              \
    } while (0)

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs

// ---- checked build (make CHECKED=1) ------------------------------------------------------------------
// compute-sanitizer is closed on the pool this library is developed on (profiles/r02_sanitizer_closed_on_this_pool.txt),
// so the bounds and alignment invariants of the kernels are asserted by the kernels themselves in a checked build:
// a violated B200_CHECK counts into a per-translation-unit device counter instead of touching the address (the access
// that follows is skipped by the caller where that is possible), and b200sort_debug_check_failures() adds them up.
// tools/sanitize_target.py runs every kernel family under it; the product build compiles the checks away.
#ifdef B200SORT_CHECKED
static __device__ unsigned long long g_check_failures[16];      // one counter per check site (B200_CHECK_AT)
#define B200_CHECK_AT(site, cond) do { if (!(cond)) atomicAdd(&::b200sort::g_check_failures[site], 1ull); } while (0)
#define B200_CHECK(cond) B200_CHECK_AT(0, cond)
static inline unsigned long long tu_check_failures(unsigned long long *per_site = nullptr) {
    unsigned long long v[16] = {0}, sum = 0;
    cudaMemcpyFromSymbol(v, g_check_failures, sizeof v);
    for (int i = 0; i < 16; ++i) { sum += v[i]; if (per_site) per_site[i] += v[i]; }
    return sum;
}
#else
#define B200_CHECK_AT(site, cond) do {} while (0)
#define B200_CHECK(cond) do {} while (0)
static inline unsigned long long tu_check_failures(unsigned long long * = nullptr) { return 0; }
#endif

inline size_t div_up(size_t a, size_t b) { return (a + b - 1) / b; }
inline size_t align_up(size_t a, size_t b) { return div_up(a, b) * b; }

// ---- device helpers ---------------------------------------------------------------------------
// Order-preserving map int32 -> uint32 (signed ascending == unsigned ascending of the image).
__host__ __device__ __forceinline__ uint32_t key_bits(int32_t k) {
    return static_cast<uint32_t>(k) ^ 0x80000000u;
}

// ---- key orders (b200sort_sort_keys) ------------------------------------------------------------
// Every supported order of 32-bit keys is a bijection onto uint32 of the form
//   image(k) = k ^ (k has its top bit set ? neg : pos)
// and the keys are sorted by their images, unsigned ascending.  The same form with other masks maps an
// image back to its key, or a key to a signed-comparable int32 (image ^ 0x80000000: the merge sort).
struct SignXor {
    uint32_t neg, pos;
};
__host__ __device__ __forceinline__ uint32_t sign_xor(uint32_t k, uint32_t neg, uint32_t pos) {
    return k ^ ((k & 0x80000000u) ? neg : pos);
}
// The (neg, pos) masks of an order; false for an unknown key type.
inline bool key_order(int key_type, int descending, SignXor *m) {
    static const SignXor kOrders[3][2] = {
        {{0x80000000u, 0x80000000u}, {0x7fffffffu, 0x7fffffffu}},   // int32   ascending / descending
        {{0x00000000u, 0x00000000u}, {0xffffffffu, 0xffffffffu}},   // uint32
        {{0xffffffffu, 0x80000000u}, {0x00000000u, 0x7fffffffu}},   // float32: IEEE-754 totalOrder on the bits
    };
    if (key_type < B200SORT_KEY_I32 || key_type > B200SORT_KEY_F32 || (descending != 0 && descending != 1)) return false;
    *m = kOrders[key_type][descending];
    return true;
}
// The masks that map an image back to its key.  Each order sends the keys with the top bit set to one half
// of the images (top bit of the image = 1 ^ top bit of `neg`), so the inverse is keyed on the image's top bit.
__host__ __device__ __forceinline__ SignXor image_inverse(SignXor m) {
    return (m.neg & 0x80000000u) ? SignXor{m.pos, m.neg} : SignXor{m.neg, m.pos};
}
// The key whose image is 0xFFFFFFFF: last in every order, digit 255 in every pass (the radix tiles' padding).
__host__ __device__ __forceinline__ uint32_t key_of_last_image(SignXor m) {
    const SignXor inv = image_inverse(m);
    return sign_xor(0xFFFFFFFFu, inv.neg, inv.pos);
}

__device__ __forceinline__ uint32_t lane_id() {
    uint32_t l;
    asm volatile("mov.u32 %0, %%laneid;" : "=r"(l));
    return l;
}
__device__ __forceinline__ uint32_t lanemask_lt() {
    uint32_t m;
    asm volatile("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

// Streaming loads/stores: keys are touched once per pass, keep them out of L1.
__device__ __forceinline__ int4 ld_stream_v4(const int4 *p) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ int32_t ld_stream(const int32_t *p) {
    int32_t r;
    asm volatile("ld.global.L1::no_allocate.s32 %0, [%1];" : "=r"(r) : "l"(p) : "memory");
    return r;
}
__device__ __forceinline__ void st_stream(int32_t *p, int32_t v) {
    asm volatile("st.global.L1::no_allocate.s32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_stream_s64(int64_t *p, int64_t v) {
    asm volatile("st.global.L1::no_allocate.s64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}

// Tile-status words of the decoupled look-back are single 32-bit words read and written at GPU
// scope with relaxed ordering: flag and value travel together, so no fence is needed.
__device__ __forceinline__ uint32_t ld_relaxed_gpu(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_gpu(uint32_t *p, uint32_t v) {
    asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}

}  // namespace b200sort
