// radix64.cuh -- internal interface of the LSD radix sort of 64-bit keys (radix64.cu): int64, uint64 and float64,
// ascending or descending, keys only or with a 32-bit value (stable).  DESIGN section 4.2e.
#pragma once
#include "common.cuh"

namespace b200sort {

// Every order of 64-bit keys is the 32-bit form of section 4.2c widened:
//   image(k) = k ^ (bit 63 of k set ? neg : pos), sorted as uint64 ascending.
struct SignXor64 {
    uint64_t neg, pos;
};
// The (neg, pos) masks of an order; false for a key type outside B200SORT_KEY_I64..F64 or descending not 0/1.
inline bool key_order64(int key_type, int descending, SignXor64 *m) {
    constexpr uint64_t kTop = 1ull << 63, kAll = ~0ull;
    static const SignXor64 kOrders[3][2] = {
        {{kTop, kTop}, {kAll ^ kTop, kAll ^ kTop}},   // int64   ascending / descending
        {{0, 0}, {kAll, kAll}},                       // uint64
        {{kAll, kTop}, {0, kAll ^ kTop}},             // float64: IEEE-754 totalOrder on the bits
    };
    if (key_type < B200SORT_KEY_I64 || key_type > B200SORT_KEY_F64 || (descending != 0 && descending != 1)) return false;
    *m = kOrders[key_type - B200SORT_KEY_I64][descending];
    return true;
}

size_t radix64_workspace_bytes(size_t n);
// d_in may equal d_out (then v_in must equal v_out); v_in == nullptr sorts keys only.  The caller has checked the
// pointers; the workspace and the 30-bit count limit are checked here, before any device work.
int radix64_sort(const uint64_t *d_in, uint64_t *d_out, uint64_t *d_tmp, const int32_t *v_in, int32_t *v_out,
                 int32_t *v_tmp, size_t n, void *d_ws, size_t ws_bytes, cudaStream_t s, SignXor64 order);
unsigned long long radix64_check_failures(unsigned long long *per_site);

}  // namespace b200sort
