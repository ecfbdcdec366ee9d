// merge.cuh -- internal interface of the merge sort (merge.cu).
#pragma once
#include "common.cuh"

namespace b200sort {

size_t merge_block_tile();
size_t merge_tile();
size_t merge_workspace_bytes(size_t n);
// A/B switch between the compiled merge-pass kernels (0 = default); process-wide, for sweeps.
int merge_set_variant(int v);
int merge_num_variants();
const char *merge_variant_name(int v);

// lab_stages: produce the sorted tiles with the assignment's staged pipeline (1-bit warp split +
// in-block rank merges) instead of the register bitonic network + merge-path rounds.
int merge_block_sort(const int32_t *d_in, int32_t *d_out, size_t n, cudaStream_t s, bool lab_stages = false);
int merge_partition(const int32_t *d_in, size_t n, size_t run, uint32_t *d_splits, cudaStream_t s);
int merge_pass(const int32_t *d_in, int32_t *d_out, size_t n, size_t run, const uint32_t *d_splits,
               cudaStream_t s);
// Output tiles [tile_begin, tile_end) of the same pass (the host-array path copies each finished range
// back while the next one is merged).  st: every key is stored as sign_xor(k, *st) (the last pass of merge_sort_keys).
int merge_pass_range(const int32_t *d_in, int32_t *d_out, size_t n, size_t run, const uint32_t *d_splits,
                     size_t tile_begin, size_t tile_end, cudaStream_t s, const SignXor *st = nullptr);
// d_in may equal d_out.  ms (optional): [0] block sort ms, [1] merge passes ms, [2] pass count.
int merge_sort(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, size_t n, void *d_ws,
               size_t ws_bytes, cudaStream_t s, float *ms, bool lab_stages = false);
// Any key order (key_order's masks): the block sort maps every key to the signed-comparable image ^ 0x80000000, the
// int32 passes sort those, and the last kernel maps them back on store.  Not with the lab's stages.
int merge_sort_keys(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, size_t n, void *d_ws,
                    size_t ws_bytes, cudaStream_t s, SignXor order);

}  // namespace b200sort
