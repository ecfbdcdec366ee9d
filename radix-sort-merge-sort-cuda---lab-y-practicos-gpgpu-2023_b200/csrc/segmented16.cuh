// segmented16.cuh -- internal interface of the segmented sort of 16-bit keys (segmented16.cu): int16, uint16, float16
// and bfloat16 in the orders of radix16.cuh, keys only or with a 32-bit value (stable), every segment on its own, in
// a number of launches that does not depend on the number of segments.  DESIGN section 4.2g.
#pragma once
#include "radix16.cuh"

namespace b200sort {

// Size classes by segment length (b200sort_segmented16_class_max), those of segmented.cuh on 2-byte keys:
//   0  length 0-1         nothing to sort; the classify kernel copies a single key (and value) when out of place
//   1  2 .. 128           one warp per segment, rank = number of keys before it in (image, position) order
//   2  129 .. 1024        one 256-thread CTA per segment, two 8-bit passes in shared memory, 4 keys per thread
//   3  1025 .. 8192       one 512-thread CTA per segment, two 8-bit passes in shared memory, 16 keys per thread
//   4  above 8192         the segmented onesweep: 2 passes over a global list of tiles that never straddle a segment
constexpr uint32_t kSeg16Max0 = 1, kSeg16Max1 = 128, kSeg16Max2 = 1024, kSeg16Max3 = 8192;
constexpr int kSeg16Threads = 512;
constexpr int kSeg16Ipt = 16;
constexpr uint32_t kSeg16Tile = kSeg16Threads * kSeg16Ipt;   // 8192 keys per onesweep tile

size_t segmented16_class_max(int c);
size_t segmented16_workspace_bytes(size_t n, size_t num_segments);
// d_in may equal d_out (then v_in must equal v_out); v_in == nullptr sorts keys only.  All arguments checked by the
// caller, workspace included; n > 0.
int segmented16_sort(const uint16_t *d_in, uint16_t *d_out, uint16_t *d_tmp, const int32_t *v_in, int32_t *v_out,
                     int32_t *v_tmp, size_t n, const int32_t *d_offsets, size_t num_segments, void *d_ws,
                     cudaStream_t s, SignXor16 order);
// Sort with indices: idx_out[i] = position of d_out[i] inside its segment, as int64 (no index input).  tmp_idx holds
// n int32.  Checked by the caller like segmented16_sort.
int segmented16_sort_indices(const uint16_t *d_in, uint16_t *d_out, uint16_t *d_tmp, int64_t *idx_out, int32_t *tmp_idx,
                             size_t n, const int32_t *d_offsets, size_t num_segments, void *d_ws, cudaStream_t s,
                             SignXor16 order);
unsigned long long segmented16_check_failures(unsigned long long *per_site);

}  // namespace b200sort
