// segmented.cuh -- internal interface of the segmented radix sort (segmented.cu): many independent segments of one
// array, each sorted in its own key order, in a number of launches that does not depend on the number of segments.
#pragma once
#include "common.cuh"

namespace b200sort {

// Size classes by segment length (b200sort_segmented_class_max):
//   0  length 0-1         nothing to sort; the classify kernel copies a single key when out of place
//   1  2 .. 128           one warp per segment, rank = number of keys before it in (image, position) order
//   2  129 .. 1024        one 256-thread CTA per segment, radix_small_body with 4 keys per thread
//   3  1025 .. 8192       one 512-thread CTA per segment, radix_small_body with 16 keys per thread
//   4  above 8192         the segmented onesweep: 4 passes over a global list of tiles that never straddle a segment
constexpr uint32_t kSegMax0 = 1, kSegMax1 = 128, kSegMax2 = 1024, kSegMax3 = 8192;   // longest segment of class c
constexpr int kSegThreads = 512;
constexpr int kSegIpt = 12;
constexpr uint32_t kSegTile = kSegThreads * kSegIpt;     // 6144 keys per onesweep tile

size_t segmented_class_max(int c);
size_t segmented_workspace_bytes(size_t n, size_t num_segments);
// d_in may equal d_out (then v_in must equal v_out); v_in == nullptr sorts keys only.  All arguments checked by the
// caller, workspace included; n > 0.
int segmented_sort(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, const int32_t *v_in, int32_t *v_out,
                   int32_t *v_tmp, size_t n, const int32_t *d_offsets, size_t num_segments, void *d_ws,
                   cudaStream_t s, SignXor order);
unsigned long long segmented_check_failures(unsigned long long *per_site);

}  // namespace b200sort
