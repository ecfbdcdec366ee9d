// radix16.cuh -- internal interface of the sorts of 16-bit keys (radix16.cu): int16, uint16, float16 and bfloat16,
// ascending or descending; keys only by counting, or with a 32-bit value (stable) by two radix passes.  DESIGN
// section 4.2f.
#pragma once
#include "common.cuh"

namespace b200sort {

// Every order of 16-bit keys is the 32-bit form of section 4.2c on 16-bit words:
//   image(k) = k ^ (bit 15 of k set ? neg : pos), sorted as uint16 ascending.
struct SignXor16 {
    uint32_t neg, pos;   // 16-bit masks in the low half
};
// The (neg, pos) masks of an order; false for a key type outside B200SORT_KEY_I16..BF16 or descending not 0/1.
inline bool key_order16(int key_type, int descending, SignXor16 *m) {
    static const SignXor16 kOrders[3][2] = {
        {{0x8000u, 0x8000u}, {0x7fffu, 0x7fffu}},   // int16   ascending / descending
        {{0x0000u, 0x0000u}, {0xffffu, 0xffffu}},   // uint16
        {{0xffffu, 0x8000u}, {0x0000u, 0x7fffu}},   // float16 and bfloat16: IEEE-754 totalOrder on the bits
    };
    if (key_type < B200SORT_KEY_I16 || key_type > B200SORT_KEY_BF16 || (descending != 0 && descending != 1)) return false;
    *m = kOrders[key_type == B200SORT_KEY_BF16 ? 2 : key_type - B200SORT_KEY_I16][descending];
    return true;
}

__host__ __device__ __forceinline__ uint32_t image16(uint32_t k, SignXor16 o) {
    return k ^ ((k & 0x8000u) ? o.neg : o.pos);
}
// The masks that map an image back to its key (common.cuh's image_inverse on 16-bit words).
__host__ __device__ __forceinline__ SignXor16 inverse16(SignXor16 o) {
    return (o.neg & 0x8000u) ? SignXor16{o.pos, o.neg} : SignXor16{o.neg, o.pos};
}

size_t radix16_workspace_bytes(size_t n);
// d_in may equal d_out.  v_in == nullptr sorts keys only, by counting (d_tmp unused); otherwise the pairs are sorted
// stably by two radix passes, in place iff d_in == d_out (then v_in must equal v_out).  The caller has checked the
// pointers; the workspace and the 30-bit count limit of the pairs are checked here, before any device work.
int radix16_sort(const uint16_t *d_in, uint16_t *d_out, uint16_t *d_tmp, const int32_t *v_in, int32_t *v_out,
                 int32_t *v_tmp, size_t n, void *d_ws, size_t ws_bytes, cudaStream_t s, SignXor16 order);
// Sort with indices: the keys sorted stably as by the pairs sort, and idx_out[i] = the input position of d_out[i], as
// int64 (no index input; tmp_idx holds n int32 of scratch).  d_in may equal d_out.  Same workspace and checks as the
// pairs sort; n == 1 writes idx_out[0] = 0 without a workspace.
int radix16_sort_indices(const uint16_t *d_in, uint16_t *d_out, uint16_t *d_tmp, int64_t *idx_out, int32_t *tmp_idx,
                         size_t n, void *d_ws, size_t ws_bytes, cudaStream_t s, SignXor16 order);
unsigned long long radix16_check_failures(unsigned long long *per_site);

}  // namespace b200sort
