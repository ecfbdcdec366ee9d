// segmented64.cuh -- internal interface of the segmented sort of 64-bit keys (segmented64.cu): int64, uint64 and
// float64 in the orders of radix64.cuh, keys only or with a 32-bit value (stable), every segment on its own, in a
// number of launches that depends neither on the number of segments nor on the data.  DESIGN section 4.2h.
#pragma once
#include "radix64.cuh"

namespace b200sort {

// Size classes by segment length (b200sort_segmented64_class_max), those of segmented16.cuh on 8-byte keys:
//   0  length 0-1         nothing to sort; the classify kernel copies a single key (and value) when out of place
//   1  2 .. 128           one warp per segment, rank = number of keys before it in (image, position) order
//   2  129 .. 1024        one 256-thread CTA per segment, 8-bit passes in shared memory, 4 keys per thread
//   3  1025 .. 8192       one 512-thread CTA per segment, 8-bit passes in shared memory, 16 keys per thread
//   4  above 8192         the segmented onesweep: 8 passes over a global list of tiles that never straddle a segment
// Classes 2-4 skip every pass whose digit is the same for all keys of the segment (class 4: of every large segment).
constexpr uint32_t kSeg64Max0 = 1, kSeg64Max1 = 128, kSeg64Max2 = 1024, kSeg64Max3 = 8192;
constexpr int kSeg64Threads = 512;
constexpr int kSeg64Ipt = 8;
constexpr uint32_t kSeg64Tile = kSeg64Threads * kSeg64Ipt;   // 4096 keys per onesweep tile, as radix64.cu's

size_t segmented64_class_max(int c);
size_t segmented64_workspace_bytes(size_t n, size_t num_segments);
// d_in may equal d_out (then v_in must equal v_out); v_in == nullptr sorts keys only.  All arguments checked by the
// caller, workspace included; 0 < n <= 2^30.
int segmented64_sort(const uint64_t *d_in, uint64_t *d_out, uint64_t *d_tmp, const int32_t *v_in, int32_t *v_out,
                     int32_t *v_tmp, size_t n, const int32_t *d_offsets, size_t num_segments, void *d_ws,
                     cudaStream_t s, SignXor64 order);
unsigned long long segmented64_check_failures(unsigned long long *per_site);

}  // namespace b200sort
