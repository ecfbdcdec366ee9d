// radix.cuh -- internal interface of the onesweep LSD radix sort (radix.cu).
#pragma once
#include "common.cuh"

namespace b200sort {

constexpr int kRadixBits   = 8;
constexpr int kRadixBins   = 1 << kRadixBits;   // 256
constexpr int kRadixPasses = 4;                 // 32-bit keys

// Control block at the head of the radix workspace.  Zeroed (first kZeroBytes) by one
// cudaMemsetAsync per sort; everything else is written before it is read.
struct RadixControl {
    uint32_t hist[kRadixPasses][kRadixBins];   // raw digit counts (global atomics)
    uint32_t ticket[kRadixPasses];             // tile tickets of each pass
    uint32_t hist_blocks_done;                 // last-block detection in the histogram kernel
    uint32_t pad0[3];
    // ---- not zeroed: written by the histogram kernel's last block ----
    uint32_t base[kRadixPasses][kRadixBins];   // exclusive scan of hist[p]
    uint32_t skip[kRadixPasses];               // 1 = one bin holds every key: pass is the identity
    uint32_t src_sel[kRadixPasses];            // buffer pass p reads : kSelIn / kSelTmp / kSelOut
    uint32_t dst_sel[kRadixPasses];            // buffer pass p writes: kSelTmp / kSelOut
    uint32_t final_copy;                       // 0 none, else copy from that kSel* buffer to out
    uint32_t hot[kRadixPasses];                // 0, or 1 + the most frequent digit value of the pass if it
                                               // holds > 1/8 of the keys
    uint32_t n_dev;                            // number of keys, as the kernels use it (see radix_sort_devn)
    uint32_t key_neg, key_pos;                 // the key order's masks (SignXor), written by the generic histogram
                                               // kernel and read by the generic pass kernels; unused for int32 ascending
    uint32_t key_pad;                          // the key whose image is 0xFFFFFFFF: pads the ragged last tile
    uint32_t pad1[3];
};
constexpr uint32_t kSelIn = 1, kSelTmp = 2, kSelOut = 3;
constexpr size_t kRadixZeroBytes    = offsetof(RadixControl, base);
constexpr size_t kRadixControlBytes = (sizeof(RadixControl) + 255) / 256 * 256;

// Smallest tile of any compiled variant: the workspace is sized for it so that variants can be
// switched without reallocating.
constexpr size_t kRadixMinTile = 2048;

size_t radix_workspace_bytes(size_t n);
size_t radix_current_tile();

int radix_histogram(const int32_t *d_keys, size_t n, uint32_t *d_hist, cudaStream_t s);
int radix_single_pass(const int32_t *d_in, int32_t *d_out, size_t n, int pass,
                      void *d_ws, size_t ws_bytes, cudaStream_t s);
// d_in may equal d_out (in-place sort); otherwise d_in is left untouched.
// order: nullptr = int32 ascending (the kernels specialised for it); else the key order's masks (key_order), served by
// the generic instantiations.  B200SORT_ERR_INVALID if the selected shape has no generic instantiation.
int radix_sort(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, size_t n, void *d_ws,
               size_t ws_bytes, cudaStream_t s, const SignXor *order = nullptr);
// Sort-by-key: (key, value) pairs ordered by key, stable.  Same workspace as radix_sort.  Either both of
// d_in == d_out and v_in == v_out (in place) or neither.
int radix_sort_pairs(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, const int32_t *v_in, int32_t *v_out,
                     int32_t *v_tmp, size_t n, void *d_ws, size_t ws_bytes, cudaStream_t s,
                     const SignXor *order = nullptr);
// The same sort with the key count taken from DEVICE memory (*d_n <= n_max, read by the kernels when they run):
// lets a caller whose n is produced by an earlier kernel (the multi-GPU exchange) enqueue the sort without a
// host synchronisation.  Grids, workspace and status rows are sized for n_max.
// d_hist (may be null): uint32[4][256] digit histograms of exactly those *d_n keys, counted elsewhere -- then the
// histogram kernel is skipped (the multi-GPU exchange counts them at the source, under the NVLink transfer).
int radix_sort_devn(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, size_t n_max, const uint32_t *d_n,
                    const uint32_t *d_hist, void *d_ws, size_t ws_bytes, cudaStream_t s);
// Same, with CUDA events around every kernel: ms[0] histogram, ms[1..4] passes, ms[5] final copy.
int radix_sort_timed(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, size_t n, void *d_ws,
                     size_t ws_bytes, cudaStream_t s, float *ms);

}  // namespace b200sort
