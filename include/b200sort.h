/*
 * b200sort.h -- C-ABI of libb200sort.so, the B200 (sm_100a) sort library that sits behind the
 * lab's operator boundary.
 *
 * Plain C: pointers, sizes and ints only.  Every function returns a B200SORT_* status (0 = ok)
 * unless stated otherwise, never exits the process, and is stream-ordered: it enqueues work on
 * `stream` (a cudaStream_t passed as void*, NULL = the legacy default stream) and returns without
 * synchronising unless its comment says it blocks.
 *
 * Reference interface each entry point replaces ("SRM/" = "/root/reference/Sord Radix y Merge/"):
 *
 *   b200sort_order_array_host   SRM/include/lab.h:9  + SRM/lab.cu:303-402  order_array(int*,int)
 *   b200sort_order_with_trust_host  SRM/include/lab.h:10 + SRM/lab.cu:404-406 order_with_trust(int*,int)
 *   b200sort_radix_i32          SRM/lab.cu:47-87   radix_sort_kernel (the radix stage), rebuilt as a
 *                               full onesweep LSD sort
 *   b200sort_radix_histogram_i32 / b200sort_radix_pass_i32
 *                               SRM/lab.cu:11-41 exlusiveScan + :63-76 split, i.e. the count/scan/
 *                               scatter the lab does per bit, here per 8-bit digit
 *   b200sort_merge_i32          SRM/lab.cu:192-197 orderedJoin + :209-300 separators_kernel /
 *                               merge_segments_kernel (the merge stages), rebuilt as block sort +
 *                               merge-path merges
 *   b200sort_block_sort_i32     SRM/lab.cu:328-344 (stage 1 + stage 2: sorted runs inside a block)
 *   b200sort_merge_partition_i32 SRM/lab.cu:209-270 separators_kernel
 *   b200sort_merge_pass_i32     SRM/lab.cu:272-300 merge_segments_kernel
 *   b200sort_lab_i32            SRM/lab.cu:303-402 the assignment's staged pipeline kept as a third
 *                               algorithm (warp-tile split -> rank merge -> merge path)
 *   b200sort_dist_*             no reference counterpart (north_star (c)): one-box multi-GPU sort
 *   b200sort_sort_keys64 / b200sort_radix_pairs_keys64
 *                               no reference counterpart: int64, uint64 and float64 keys (8 radix passes),
 *                               keys only or with an int32 value
 *   b200sort_sort_keys16 / b200sort_radix_pairs_keys16
 *                               no reference counterpart: int16, uint16, float16 and bfloat16 keys (a counting
 *                               sort for keys only, 2 radix passes with an int32 value)
 *   b200sort_segmented_sort_keys16 / b200sort_segmented_pairs_keys16
 *                               no reference counterpart: every segment (row) of 16-bit keys sorted on its own
 *                               in one call, keys only or with an int32 value
 *   b200sort_segmented_sort_keys64 / b200sort_segmented_pairs_keys64
 *                               no reference counterpart: every segment (row) of 64-bit keys sorted on its own
 *                               in one call, keys only or with an int32 value, skipping the digit passes that no
 *                               segment needs
 *   b200sort_radix_sort_indices_keys / b200sort_segmented_sort_indices_keys
 *                               no reference counterpart: 32-bit keys sorted with their int64 positions (the
 *                               values and indices of torch.sort), 1-D or segmented, with no index input
 *   b200sort_radix_sort_indices_keys16 / b200sort_segmented_sort_indices_keys16
 *                               no reference counterpart: the same for 16-bit keys
 *
 * The C++ symbols order_array(int*,int) / order_with_trust(int*,int) that SRM/main.cpp and
 * SRM/performanceTest.cpp link against are exported by the same library (csrc/lab_shim.cu) with
 * the reference's abort-on-error convention (SRM/include/utils.h:18-26); see include/lab.h.
 */
#ifndef B200SORT_H
#define B200SORT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status ------------------------------------------------------------------------------------ */
#define B200SORT_OK                 0
#define B200SORT_ERR_INVALID        1   /* bad argument (NULL pointer, unknown algorithm, n too large) */
#define B200SORT_ERR_WORKSPACE      2   /* workspace NULL / too small / misaligned */
#define B200SORT_ERR_CUDA           3   /* a CUDA runtime call failed; see b200sort_last_cuda_error */
#define B200SORT_ERR_NO_DEVICE      4   /* no usable sm_100 device: there is NO CPU fallback */
#define B200SORT_ERR_ALLOC          5   /* host-path allocation failed */

/* ---- algorithms -------------------------------------------------------------------------------- */
#define B200SORT_ALGO_RADIX         0   /* onesweep LSD radix, 8-bit digits, 4 passes */
#define B200SORT_ALGO_MERGE         1   /* register bitonic block sort + merge-path merges */
#define B200SORT_ALGO_LAB           2   /* the assignment's staged pipeline (radix tiles -> merges) */

/* Largest n any entry point accepts (tile-status words carry 30-bit counts; a digit count can reach 2^30 only
 * when one bin holds every key, which pass skipping removes -- with b200sort_radix_set_skip(0) the radix
 * sorts therefore refuse n = 2^30 with B200SORT_ERR_INVALID). */
#define B200SORT_MAX_N              ((size_t)1 << 30)

const char *b200sort_version(void);
const char *b200sort_status_string(int status);
/* cudaError_t (as int) of the most recent failing CUDA call on this host thread, 0 if none. */
int         b200sort_last_cuda_error(void);
const char *b200sort_last_cuda_error_string(void);
/* B200SORT_OK iff the current device exists and is compute capability 10.x.  Also the explicit per-device
 * initialisation: runs the lane-order self-test of the radix sort for the current device if it has not run
 * yet (launches on a private stream and BLOCKS; allocates nothing).  Call it once per device before timing: the
 * first sort on a device otherwise does it lazily.  That lazy test may run inside a CUDA graph capture, on this
 * thread or another: it switches the thread to relaxed capture mode for its few calls, which stay outside the graph,
 * and caches only a verdict its kernel returned. */
int         b200sort_device_check(void);

/* ---- device-array sorts (the layer measured against the HBM roofline) --------------------------
 * d_keys  n keys, sorted in place (ascending, signed).
 * d_tmp   n keys of scratch (ping-pong buffer); contents undefined on return.
 * d_ws    workspace of at least b200sort_workspace_bytes(n, algo) bytes, 256-byte aligned;
 *         need not be initialised; may be reused by the next call on the same stream.
 * Any n in [0, B200SORT_MAX_N]; the lab's n (power of two, multiple of 32) is the tested case,
 * ragged n is handled. */
size_t b200sort_workspace_bytes(size_t n, int algo);
/* b200sort_radix_i32: the pass kernels rank keys with shared-memory atomicAdds (one per key, or a counting one and a
 * positioning one), whose return value is a stable rank only if the GPU resolves same-address lanes of one warp
 * instruction in lane order.  B200 does
 * (tools/atomic_order_probe.cu), PTX does not promise it.  GUARD: a self-test that reproduces the kernels'
 * exact access pattern runs once per DEVICE -- in b200sort_device_check(), or lazily (blocking) in the first
 * sort on that device -- and on failure, or with B200SORT_RANK_SAFE=1 in the environment, every radix entry
 * point (keys, pairs, small arrays) runs the ballot-ranked shape of the same kernel instead, which relies on
 * documented behaviour only.  b200sort_radix_atomic_order_ok() reports the verdict. */
int    b200sort_radix_i32(int32_t *d_keys, int32_t *d_tmp, size_t n,
                          void *d_ws, size_t ws_bytes, void *stream);
int    b200sort_merge_i32(int32_t *d_keys, int32_t *d_tmp, size_t n,
                          void *d_ws, size_t ws_bytes, void *stream);
/* Sort-by-key (SURVEY section 8(f)-4): (key, 32-bit value) pairs ordered by key, ascending signed, STABLE --
 * equal keys keep their input order, the A-before-B tie rule of SRM/lab.cu:163-170 carried through the
 * whole sort; with values 0..n-1 the result is the index permutation the doc comment at
 * SRM/lab.cu:44-45 ("positions") had in mind.  The onesweep passes with the value riding beside the key
 * (16 B/key per pass).  Workspace: b200sort_workspace_bytes(n, B200SORT_ALGO_RADIX).  The _copy form
 * leaves the inputs untouched.  Falls back to the ballot-ranked shape like b200sort_radix_i32. */
int    b200sort_radix_pairs_i32(int32_t *d_keys, int32_t *d_vals, int32_t *d_tmp_keys, int32_t *d_tmp_vals,
                                size_t n, void *d_ws, size_t ws_bytes, void *stream);
int    b200sort_radix_pairs_copy_i32(const int32_t *d_keys_in, const int32_t *d_vals_in, int32_t *d_keys_out,
                                     int32_t *d_vals_out, int32_t *d_tmp_keys, int32_t *d_tmp_vals, size_t n,
                                     void *d_ws, size_t ws_bytes, void *stream);
/* The assignment's staged pipeline (SRM/letra.pdf p.3 parts a-d, SRM/lab.cu:303-402) as a third
 * algorithm: 1-bit warp split on 32-key groups -> in-block rank merges -> merge-path merges. */
int    b200sort_lab_i32(int32_t *d_keys, int32_t *d_tmp, size_t n,
                        void *d_ws, size_t ws_bytes, void *stream);
int    b200sort_sort_i32(int algo, int32_t *d_keys, int32_t *d_tmp, size_t n,
                         void *d_ws, size_t ws_bytes, void *stream);
/* Out-of-place form: d_out = sorted d_in; d_in is only read (it may also equal d_out).  No extra
 * traffic compared with the in-place form: the first pass simply reads d_in. */
int    b200sort_sort_copy_i32(int algo, const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, size_t n,
                              void *d_ws, size_t ws_bytes, void *stream);
/* Same as b200sort_sort_copy_i32 with CUDA events around the kernels; BLOCKS until done.
 * radix: ms[0] histogram, ms[1..4] the four passes, ms[5] final copy (6 floats).
 * merge: ms[0] block sort, ms[1] all merge passes together, ms[2] number of merge passes. */
int    b200sort_sort_timed_i32(int algo, const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, size_t n,
                               void *d_ws, size_t ws_bytes, void *stream, float *ms);

/* ---- other key types and descending order ------------------------------------------------------
 * Keys are 32-bit words; key_type says how they compare:
 *   B200SORT_KEY_I32  signed integers, numeric order (the _i32 entry points' order);
 *   B200SORT_KEY_U32  unsigned integers, numeric order;
 *   B200SORT_KEY_F32  IEEE-754 binary32 in totalOrder on the bit pattern:
 *                     -NaN (sign bit set, any payload) < -inf < negatives < -0.0 < +0.0 < positives < +inf < +NaN,
 *                     NaNs of one sign ordered by payload.  Bits are never changed: the output is the input's bit
 *                     patterns permuted.  This is NOT the order of torch.sort / np.sort, which treat -0.0 == +0.0
 *                     and put every NaN last.
 * descending = 1 is the reverse order of the same key type.  Distinct bit patterns never compare equal, so a keys-only
 * result is unique.  Sort-by-key stays STABLE in both directions (equal keys keep their input order), so a descending
 * pairs result is not the reverse of the ascending one; without NaN or -0.0 it equals
 * torch.sort(stable=True, descending=True).
 * Internally every order is image(k) = k ^ (top bit of k set ? M_neg : M_pos) sorted as uint32 (DESIGN section 4.2c).
 * (B200SORT_KEY_I32, ascending) runs exactly the code of the _i32 entry points. */
#define B200SORT_KEY_I32            0
#define B200SORT_KEY_U32            1
#define B200SORT_KEY_F32            2
/* d_out = d_in sorted (d_in may equal d_out; otherwise it is only read).  algo: RADIX or MERGE; LAB only with
 * (B200SORT_KEY_I32, 0) -- its 1-bit split is signed by construction.  Workspace: b200sort_workspace_bytes(n, algo),
 * unchanged.  Unknown key_type, descending not 0/1, NULL pointers, n > B200SORT_MAX_N, a radix shape selected with
 * b200sort_radix_set_variant that has no generic instantiation (make EXPERIMENTS=1 shapes) -> B200SORT_ERR_INVALID;
 * missing or small workspace -> B200SORT_ERR_WORKSPACE; all checked before any device work. */
int    b200sort_sort_keys(int algo, int key_type, int descending, const void *d_in, void *d_out, void *d_tmp,
                          size_t n, void *d_ws, size_t ws_bytes, void *stream);
/* Stable sort-by-key on the radix path; same in-place / copy rules as b200sort_radix_pairs_copy_i32 (in place iff
 * d_keys_in == d_keys_out and d_vals_in == d_vals_out). */
int    b200sort_radix_pairs_keys(int key_type, int descending, const void *d_keys_in, const int32_t *d_vals_in,
                                 void *d_keys_out, int32_t *d_vals_out, void *d_tmp_keys, int32_t *d_tmp_vals,
                                 size_t n, void *d_ws, size_t ws_bytes, void *stream);

/* ---- 64-bit keys: int64, uint64 and float64 on the radix path -------------------------------------------
 * Keys are 8-byte words; key_type says how they compare:
 *   B200SORT_KEY_I64  signed integers, numeric order;
 *   B200SORT_KEY_U64  unsigned integers, numeric order;
 *   B200SORT_KEY_F64  IEEE-754 binary64 in totalOrder on the bit pattern, as B200SORT_KEY_F32:
 *                     -NaN (any payload) < -inf < negatives < -0.0 < +0.0 < positives < +inf < +NaN, NaNs of one
 *                     sign ordered by payload.  Bits are never changed.  This is NOT the order of torch.sort /
 *                     np.sort, which treat -0.0 == +0.0 and put every NaN last.
 * The 32-bit entry points (b200sort_sort_keys, b200sort_radix_pairs_keys, the segmented sort) reject these key types,
 * and these entry points reject B200SORT_KEY_I32..F32.  descending = 1 is the reverse order; sort-by-key is STABLE in
 * both directions (without NaN or -0.0 it equals torch.sort(stable=True, descending=...)).  Internally every order is
 * image(k) = k ^ (bit 63 of k set ? M_neg : M_pos) sorted as uint64: 8 stable passes of 8-bit digits, of which
 * those where one digit value holds every key are skipped on the device (b200sort_radix_set_skip applies; the
 * variant switch b200sort_radix_set_variant does not).  DESIGN section 4.2e.
 * Like the other radix sorts the passes rank with lane-ordered shared-memory atomics only after the self-test of
 * b200sort_radix_i32 has passed on the device; otherwise, or with B200SORT_RANK_SAFE=1, their ballot-ranked form runs.
 * A call enqueues one memset and the same ten kernels for every n >= 2 and every distribution, never synchronises and
 * never reads device results on the host, so it can be captured in a CUDA graph.
 * Arrays of up to 8192 keys pay that whole sequence too: there is no one-CTA path for 64-bit keys.
 * d_in may equal d_out (in place); otherwise d_in is only read.  d_tmp: n keys of scratch.  Workspace:
 * b200sort_keys64_workspace_bytes(n) bytes, 256-byte aligned, sized from n alone.
 * Key type outside B200SORT_KEY_I64..F64, descending not 0/1, n > B200SORT_MAX_N, NULL data pointers with n > 0, key
 * pointers not 8-byte aligned -> B200SORT_ERR_INVALID; missing, small or misaligned workspace ->
 * B200SORT_ERR_WORKSPACE; all checked before any device work.  n == 0, and n == 1 in place, return B200SORT_OK
 * without touching the device.  With b200sort_radix_set_skip(0), n = 2^30 -> B200SORT_ERR_INVALID. */
#define B200SORT_KEY_I64            3
#define B200SORT_KEY_U64            4
#define B200SORT_KEY_F64            5
size_t b200sort_keys64_workspace_bytes(size_t n);
int    b200sort_sort_keys64(int key_type, int descending, const void *d_in, void *d_out, void *d_tmp, size_t n,
                            void *d_ws, size_t ws_bytes, void *stream);
/* Stable sort of (64-bit key, int32 value) pairs by key.  In place iff d_keys_in == d_keys_out and
 * d_vals_in == d_vals_out; a mix of the two -> B200SORT_ERR_INVALID.  Same workspace as b200sort_sort_keys64. */
int    b200sort_radix_pairs_keys64(int key_type, int descending, const void *d_keys_in, const int32_t *d_vals_in,
                                   void *d_keys_out, int32_t *d_vals_out, void *d_tmp_keys, int32_t *d_tmp_vals,
                                   size_t n, void *d_ws, size_t ws_bytes, void *stream);

/* ---- 16-bit keys: int16, uint16, float16 and bfloat16 ------------------------------------------------------
 * Keys are 2-byte words; key_type says how they compare:
 *   B200SORT_KEY_I16   signed integers, numeric order;
 *   B200SORT_KEY_U16   unsigned integers, numeric order;
 *   B200SORT_KEY_F16   IEEE-754 binary16, and
 *   B200SORT_KEY_BF16  bfloat16 (the top half of a binary32), both in totalOrder on the bit pattern, as
 *                      B200SORT_KEY_F32: -NaN (any payload) < -inf < negatives < -0.0 < +0.0 < positives < +inf <
 *                      +NaN, NaNs of one sign ordered by payload.  Bits are never changed.  This is NOT the order of
 *                      torch.sort / np.sort, which treat -0.0 == +0.0 and put every NaN last.
 * F16 and BF16 share one order; both names exist so that callers can name their dtype.  The 32-bit, segmented and
 * 64-bit entry points reject these key types, and these entry points reject B200SORT_KEY_I32..F64.  descending = 1
 * is the reverse order.  Every order is image(k) = k ^ (bit 15 of k set ? M_neg : M_pos) sorted as uint16.
 * The output holds the input's bit patterns, permuted.  DESIGN section 4.2f.
 *
 * b200sort_sort_keys16 sorts by counting: one read of the keys counts each of the 65536 bit patterns, the counts are
 * scanned in image order, and every pattern is written `count` times.  It ranks nothing, so it needs neither the
 * lane-order self-test of b200sort_radix_i32 nor its ballot-ranked fallback, has no scratch buffer and no 2^30 limit.
 * b200sort_radix_pairs_keys16 is a STABLE sort in both directions (without NaN or -0.0 it equals
 * torch.sort(stable=True, descending=...)): after the same count, two radix passes of 8-bit digits of the image, of
 * which one where a single digit value holds every key is skipped on the device (b200sort_radix_set_skip applies).
 * Its passes rank like the other radix sorts: lane-ordered shared-memory atomics after the self-test has passed on
 * the device, otherwise, or with B200SORT_RANK_SAFE=1, the ballot-ranked form.  b200sort_radix_set_variant applies to
 * neither.  A call enqueues one memset and the same kernels for every n >= 2 and every distribution (3 for keys, 5
 * for pairs), never synchronises and never reads device results on the host, so it can be captured in a CUDA graph.
 * Key pointers need only 2-byte alignment.  d_in may equal d_out (in place); otherwise d_in is only read.
 * Workspace: b200sort_keys16_workspace_bytes(n) bytes, 256-byte aligned, sized from n alone, for keys and pairs.
 * Key type outside B200SORT_KEY_I16..BF16, descending not 0/1, n > B200SORT_MAX_N, NULL data pointers with n > 0, key
 * pointers not 2-byte aligned -> B200SORT_ERR_INVALID; missing, small or misaligned workspace ->
 * B200SORT_ERR_WORKSPACE; all checked before any device work.  n == 0, and n == 1 in place, return B200SORT_OK
 * without touching the device.  Pairs with b200sort_radix_set_skip(0) and n = 2^30 -> B200SORT_ERR_INVALID. */
#define B200SORT_KEY_I16            6
#define B200SORT_KEY_U16            7
#define B200SORT_KEY_F16            8
#define B200SORT_KEY_BF16           9
size_t b200sort_keys16_workspace_bytes(size_t n);
int    b200sort_sort_keys16(int key_type, int descending, const void *d_in, void *d_out, size_t n, void *d_ws,
                            size_t ws_bytes, void *stream);
/* Stable sort of (16-bit key, int32 value) pairs by key.  d_tmp_keys, d_tmp_vals: n keys and n values of scratch.
 * In place iff d_keys_in == d_keys_out and d_vals_in == d_vals_out; a mix of the two -> B200SORT_ERR_INVALID. */
int    b200sort_radix_pairs_keys16(int key_type, int descending, const void *d_keys_in, const int32_t *d_vals_in,
                                   void *d_keys_out, int32_t *d_vals_out, void *d_tmp_keys, int32_t *d_tmp_vals,
                                   size_t n, void *d_ws, size_t ws_bytes, void *stream);

/* ---- segmented sort: many independent segments of one array in one call ---------------------------
 * Segment i is keys[d_offsets[i] .. d_offsets[i+1]), for i < num_segments.  d_offsets is a DEVICE array of
 * num_segments + 1 int32 with d_offsets[0] = 0, d_offsets[num_segments] = n, non-decreasing; empty segments allowed.
 * Each segment comes out sorted in the order (key_type, descending) of b200sort_sort_keys; keys never cross segments.
 * The host never reads d_offsets: a call is stream-ordered, enqueues the same kernels whatever the number of segments
 * (no host loop over segments, no host synchronisation), and can be captured in a CUDA graph.  Malformed offsets
 * (decreasing, negative, past n) give an undefined order but never an access out of bounds: every segment is clamped
 * to [0, n] on the device, and the checked build counts what the clamps caught at check site 15.
 * Segments are routed by length to size classes (b200sort_segmented_class_max): copies for length 0-1, a warp per
 * segment, a CTA per segment sorted in shared memory (two capacities), and above that a segmented onesweep whose tiles
 * never straddle a segment.  Like the 1-D radix sort, the ranking kernels rely on lane-ordered shared-memory atomics
 * only after the self-test of b200sort_radix_i32 has passed on the device; otherwise, or with B200SORT_RANK_SAFE=1,
 * their ballot-ranked forms run.  b200sort_radix_set_variant and b200sort_radix_set_skip select shapes and policies
 * of the 1-D sort: the segmented sort ignores both.
 * d_in may equal d_out; otherwise d_in is only read.  d_tmp: n keys of scratch.  Workspace:
 * b200sort_segmented_workspace_bytes(n, num_segments) bytes, 256-byte aligned, sized from (n, num_segments) alone.
 * Unknown key_type, descending not 0/1, NULL data pointers, n or num_segments > B200SORT_MAX_N, NULL d_offsets with
 * num_segments > 0 -> B200SORT_ERR_INVALID; missing, small or misaligned workspace -> B200SORT_ERR_WORKSPACE; all
 * checked before any device work.  n == 0 returns B200SORT_OK without touching the device. */
size_t b200sort_segmented_workspace_bytes(size_t n, size_t num_segments);
int    b200sort_segmented_sort_keys(int key_type, int descending, const void *d_in, void *d_out, void *d_tmp, size_t n,
                                    const int32_t *d_offsets, size_t num_segments,
                                    void *d_ws, size_t ws_bytes, void *stream);
/* Stable within each segment (equal keys keep their input order); in place iff d_keys_in == d_keys_out and
 * d_vals_in == d_vals_out, a mix of the two -> B200SORT_ERR_INVALID. */
int    b200sort_segmented_pairs_keys(int key_type, int descending, const void *d_keys_in, const int32_t *d_vals_in,
                                     void *d_keys_out, int32_t *d_vals_out, void *d_tmp_keys, int32_t *d_tmp_vals,
                                     size_t n, const int32_t *d_offsets, size_t num_segments,
                                     void *d_ws, size_t ws_bytes, void *stream);
/* Largest segment length served by size class c (0, 1, ...); 0 past the last class (the onesweep class, unbounded). */
size_t b200sort_segmented_class_max(int c);

/* ---- sort with indices: 32-bit keys and their int64 positions -------------------------------------------
 * The keys of B200SORT_KEY_I32..F32 sorted in the order (key_type, descending) of b200sort_sort_keys, and beside them
 * d_idx_out[i] = the position that d_keys_out[i] held in its segment of the input, as int64 (the index dtype of
 * torch.sort, torch.gather and friends).  The result is the STABLE sort of (key, position) pairs in both directions:
 * without NaN and -0.0 it equals torch.sort(x, stable=True, descending=...) in values and indices, byte for byte, and
 * for rows torch.sort(x, dim=-1, stable=True, descending=...).  There is no index input: the first pass makes the
 * positions as it loads the keys, they travel as int32 (d_tmp_idx: n int32 of scratch; passes may also use d_idx_out's
 * 8n bytes as int32 scratch) and the pass that stores them for the last time writes them as int64.  Which pass that
 * is depends on the passes skipped, which only the device knows; a final kernel covers a sort in which no pass ran
 * (the indices are then 0..n-1) and an in-place sort whose last pass landed in scratch.  DESIGN section 4.2i.
 * d_keys_in may equal d_keys_out (in place); otherwise d_keys_in is only read.  d_tmp_keys: n keys of scratch.
 * Workspaces are those of the pairs sorts: b200sort_workspace_bytes(n, B200SORT_ALGO_RADIX) for the 1-D form (n >= 2),
 * b200sort_segmented_workspace_bytes(n, num_segments) for the segmented form (n >= 1).
 * Key type outside B200SORT_KEY_I32..F32, descending not 0/1, n or num_segments > B200SORT_MAX_N, NULL pointers with
 * n > 0 (d_offsets: with num_segments > 0), d_idx_out not 8-byte aligned -> B200SORT_ERR_INVALID; missing, small or
 * misaligned workspace -> B200SORT_ERR_WORKSPACE; all checked before any device work.  n == 0 returns B200SORT_OK
 * without touching the device; the 1-D form sorts n == 1 with a memset of d_idx_out (and a copy of the key when out of
 * place).  The 1-D form follows b200sort_radix_pairs_keys: the generic pass kernels, the same self-test gate and
 * ballot-ranked fallback, skipped passes (b200sort_radix_set_skip applies, and with skipping off n = 2^30 ->
 * B200SORT_ERR_INVALID).  The segmented form follows b200sort_segmented_pairs_keys: offsets as there, clamped on the
 * device.  A call enqueues the same kernels for every n >= 2 and every distribution (1-D: one memset and six kernels,
 * five with skipping off; segmented: those of b200sort_segmented_pairs_keys), never synchronises and never reads
 * device results on the host, so it can be captured in a CUDA graph. */
int    b200sort_radix_sort_indices_keys(int key_type, int descending, const void *d_keys_in, void *d_keys_out,
                                        int64_t *d_idx_out, void *d_tmp_keys, int32_t *d_tmp_idx, size_t n,
                                        void *d_ws, size_t ws_bytes, void *stream);
int    b200sort_segmented_sort_indices_keys(int key_type, int descending, const void *d_keys_in, void *d_keys_out,
                                            int64_t *d_idx_out, void *d_tmp_keys, int32_t *d_tmp_idx, size_t n,
                                            const int32_t *d_offsets, size_t num_segments,
                                            void *d_ws, size_t ws_bytes, void *stream);

/* ---- segmented sort of 16-bit keys: int16, uint16, float16 and bfloat16 -----------------------------------
 * The segmented sort above on the 2-byte keys of b200sort_sort_keys16: segment i = keys[d_offsets[i] ..
 * d_offsets[i+1]) comes out sorted in the order (key_type, descending) of b200sort_sort_keys16, image(k) = k ^ (bit 15
 * set ? M_neg : M_pos) sorted as uint16 (float16 and bfloat16: IEEE-754 totalOrder on the bits; bits are never
 * changed).  Only B200SORT_KEY_I16..BF16 are accepted; the 32-bit segmented entry points keep rejecting them.
 * Pairs are STABLE within each segment in both directions: without NaN and -0.0, rows sorted by
 * b200sort_segmented_pairs_keys16 with values 0..L-1 equal torch.sort(x, dim=-1, stable=True, descending=...) in
 * values and indices.
 * d_offsets follows the rules of b200sort_segmented_sort_keys: a DEVICE array of num_segments + 1 int32 the host
 * never reads, segments clamped to [0, n] on the device, malformed offsets giving an undefined order but no access
 * out of bounds (the checked build counts the clamps at check site 15).
 * A call enqueues one memset and the same eight kernels whatever the number of segments and the data, never
 * synchronises, and can be captured in a CUDA graph.  Size classes
 * (b200sort_segmented16_class_max): copies for length 0-1, a warp per segment, a CTA per segment sorted in shared
 * memory by two 8-bit passes (two capacities), and above that a segmented onesweep of two passes whose tiles never
 * straddle a segment.  The ranking kernels use lane-ordered shared-memory atomics only after the self-test of
 * b200sort_radix_i32 has passed on the device; otherwise, or with B200SORT_RANK_SAFE=1, their ballot-ranked forms run.
 * b200sort_radix_set_variant and b200sort_radix_set_skip are ignored.  DESIGN section 4.2g.
 * Key pointers need only 2-byte alignment: segments may begin anywhere.  d_in may equal d_out; otherwise d_in is only
 * read.  d_tmp: n keys of scratch.  Workspace: b200sort_segmented16_workspace_bytes(n, num_segments) bytes, 256-byte
 * aligned, sized from (n, num_segments) alone.
 * Key type outside B200SORT_KEY_I16..BF16, descending not 0/1, NULL data pointers, odd key pointers, n or
 * num_segments > B200SORT_MAX_N, NULL d_offsets with num_segments > 0 -> B200SORT_ERR_INVALID; missing, small or
 * misaligned workspace -> B200SORT_ERR_WORKSPACE; all checked before any device work, in the order of the 32-bit
 * segmented entry points.  n == 0 returns B200SORT_OK without touching the device. */
size_t b200sort_segmented16_workspace_bytes(size_t n, size_t num_segments);
/* Largest segment length served by size class c of the 16-bit segmented sort; 0 past the last bounded class. */
size_t b200sort_segmented16_class_max(int c);
int    b200sort_segmented_sort_keys16(int key_type, int descending, const void *d_in, void *d_out, void *d_tmp,
                                      size_t n, const int32_t *d_offsets, size_t num_segments,
                                      void *d_ws, size_t ws_bytes, void *stream);
/* Stable within each segment; in place iff d_keys_in == d_keys_out and d_vals_in == d_vals_out, a mix of the two ->
 * B200SORT_ERR_INVALID. */
int    b200sort_segmented_pairs_keys16(int key_type, int descending, const void *d_keys_in, const int32_t *d_vals_in,
                                       void *d_keys_out, int32_t *d_vals_out, void *d_tmp_keys, int32_t *d_tmp_vals,
                                       size_t n, const int32_t *d_offsets, size_t num_segments,
                                       void *d_ws, size_t ws_bytes, void *stream);

/* ---- sort with indices: 16-bit keys and their int64 positions -------------------------------------------
 * The keys of B200SORT_KEY_I16..BF16 sorted in the order (key_type, descending) of b200sort_sort_keys16 (float16 and
 * bfloat16: IEEE-754 totalOrder on the bits), and beside them d_idx_out[i] = the position that d_keys_out[i] held in
 * its segment of the input, as int64: the index in the array (1-D), the column (rows), i - d_offsets[s] (offsets).
 * The result is the STABLE sort of (key, position) pairs in both directions: without NaN and -0.0 it equals
 * torch.sort(x, stable=True, descending=...) in values and indices, byte for byte, and for rows
 * torch.sort(x, dim=-1, stable=True, descending=...).  There is no index input: the first executed pass makes the
 * positions as it loads the keys, they travel between the two passes as int32 in d_tmp_idx (n int32 of scratch), and
 * the last executed pass stores them as int64.  DESIGN section 4.2j.
 * d_keys_in may equal d_keys_out (in place); otherwise d_keys_in is only read.  d_tmp_keys: n keys of scratch.  Key
 * pointers need only 2-byte alignment.  Workspaces are those of the 16-bit sorts: b200sort_keys16_workspace_bytes(n)
 * for the 1-D form (n >= 2), b200sort_segmented16_workspace_bytes(n, num_segments) for the segmented form (n >= 1).
 * Key type outside B200SORT_KEY_I16..BF16, descending not 0/1, n or num_segments > B200SORT_MAX_N, NULL pointers with
 * n > 0 (d_offsets: with num_segments > 0), odd key pointers, d_idx_out not 8-byte aligned -> B200SORT_ERR_INVALID;
 * missing, small or misaligned workspace -> B200SORT_ERR_WORKSPACE; all checked before any device work, in the order
 * of b200sort_radix_pairs_keys16.  The 32-bit indices entry points reject the 16-bit key types and these reject every
 * other type.  n == 0 returns B200SORT_OK without touching the device; the 1-D form sorts n == 1 with a memset of
 * d_idx_out (and a copy of the key when out of place).  The 1-D form follows b200sort_radix_pairs_keys16: the same
 * histogram and scan, its two passes with the same self-test gate and ballot-ranked fallback, skipped passes
 * (b200sort_radix_set_skip applies, and with skipping off n = 2^30 -> B200SORT_ERR_INVALID), then one final kernel
 * that copies the keys as the pairs sort's final copy does and writes 0..n-1 when both passes were skipped.  The
 * segmented form follows b200sort_segmented_pairs_keys16: offsets as there, clamped on the device.  A call enqueues the
 * same kernels for every n >= 2 and every distribution (1-D: one memset and five kernels; segmented: those of
 * b200sort_segmented_pairs_keys16), never synchronises and never reads device results on the host, so it can be
 * captured in a CUDA graph. */
int    b200sort_radix_sort_indices_keys16(int key_type, int descending, const void *d_keys_in, void *d_keys_out,
                                          int64_t *d_idx_out, void *d_tmp_keys, int32_t *d_tmp_idx, size_t n,
                                          void *d_ws, size_t ws_bytes, void *stream);
int    b200sort_segmented_sort_indices_keys16(int key_type, int descending, const void *d_keys_in, void *d_keys_out,
                                              int64_t *d_idx_out, void *d_tmp_keys, int32_t *d_tmp_idx, size_t n,
                                              const int32_t *d_offsets, size_t num_segments,
                                              void *d_ws, size_t ws_bytes, void *stream);

/* ---- segmented sort of 64-bit keys: int64, uint64 and float64 -------------------------------------------
 * The segmented sort above on the 8-byte keys of b200sort_sort_keys64: segment i = keys[d_offsets[i] ..
 * d_offsets[i+1]) comes out sorted in the order (key_type, descending) of b200sort_sort_keys64, image(k) = k ^ (bit 63
 * set ? M_neg : M_pos) sorted as uint64 (float64: IEEE-754 totalOrder on the bits; bits are never changed).  Only
 * B200SORT_KEY_I64..F64 are accepted; the 32-bit and 16-bit segmented entry points keep rejecting them.
 * Pairs are STABLE within each segment in both directions: without NaN and -0.0, rows sorted by
 * b200sort_segmented_pairs_keys64 with values 0..L-1 equal torch.sort(x, dim=-1, stable=True, descending=...) in
 * values and indices.
 * d_offsets follows the rules of b200sort_segmented_sort_keys: a DEVICE array of num_segments + 1 int32 the host
 * never reads, segments clamped to [0, n] on the device, malformed offsets giving an undefined order but no access
 * out of bounds (the checked build counts the clamps at check site 15).
 * Size classes (b200sort_segmented64_class_max): copies for length 0-1, a warp per segment, a CTA per segment sorted
 * in shared memory by 8-bit passes (two capacities), and above that a segmented onesweep of 8 passes whose tiles never
 * straddle a segment.  Passes are skipped on the device: a CTA-class segment skips every pass in which all its keys
 * share the digit, and the onesweep class skips pass p when that holds in each of its segments (one large segment
 * whose keys differ in digit p makes pass p run for all of them).  Rows of int64 ids below 2^32 thus run at most 4
 * of the 8 passes.  A call still enqueues one memset and the same fifteen kernels whatever the number of segments
 * and the data, never synchronises, and can be captured in a CUDA graph.  The
 * ranking kernels use lane-ordered shared-memory atomics only after the self-test of b200sort_radix_i32 has passed on
 * the device; otherwise, or with B200SORT_RANK_SAFE=1, their ballot-ranked forms run.  b200sort_radix_set_variant
 * and b200sort_radix_set_skip are ignored: skipping is always on.  DESIGN section 4.2h.
 * Any n up to B200SORT_MAX_N = 2^30 is accepted: a digit count reaches 2^30 only when one segment holds all 2^30 keys
 * and every one of them has that digit, and then that pass is skipped.
 * Key pointers need 8-byte alignment.  d_in may equal d_out; otherwise d_in is only read.  d_tmp: n keys of scratch.
 * Workspace: b200sort_segmented64_workspace_bytes(n, num_segments) bytes, 256-byte aligned, sized from
 * (n, num_segments) alone.
 * Key type outside B200SORT_KEY_I64..F64, descending not 0/1, NULL data pointers, key pointers not 8-byte aligned, n
 * or num_segments > B200SORT_MAX_N, NULL d_offsets with num_segments > 0 -> B200SORT_ERR_INVALID; missing, small or
 * misaligned workspace -> B200SORT_ERR_WORKSPACE; all checked before any device work, in the order of the 32-bit
 * segmented entry points.  n == 0 returns B200SORT_OK without touching the device. */
size_t b200sort_segmented64_workspace_bytes(size_t n, size_t num_segments);
/* Largest segment length served by size class c of the 64-bit segmented sort; 0 past the last bounded class. */
size_t b200sort_segmented64_class_max(int c);
int    b200sort_segmented_sort_keys64(int key_type, int descending, const void *d_in, void *d_out, void *d_tmp,
                                      size_t n, const int32_t *d_offsets, size_t num_segments,
                                      void *d_ws, size_t ws_bytes, void *stream);
/* Stable within each segment; in place iff d_keys_in == d_keys_out and d_vals_in == d_vals_out, a mix of the two ->
 * B200SORT_ERR_INVALID. */
int    b200sort_segmented_pairs_keys64(int key_type, int descending, const void *d_keys_in, const int32_t *d_vals_in,
                                       void *d_keys_out, int32_t *d_vals_out, void *d_tmp_keys, int32_t *d_tmp_vals,
                                       size_t n, const int32_t *d_offsets, size_t num_segments,
                                       void *d_ws, size_t ws_bytes, void *stream);

/* ---- stages, exposed for unit tests and per-kernel timing -------------------------------------- */

/* d_hist[p*256+d] (uint32) = number of keys whose digit p of (key ^ 0x80000000) equals d.
 * One read of the keys with 128-bit loads.  d_hist is overwritten. */
int b200sort_radix_histogram_i32(const int32_t *d_keys, size_t n, uint32_t *d_hist, void *stream);
/* One stable onesweep pass by digit `pass` (0..3): d_out = d_in partitioned by that digit.
 * d_in and d_out must not overlap.  Uses the radix workspace. */
int b200sort_radix_pass_i32(const int32_t *d_in, int32_t *d_out, size_t n, int pass,
                            void *d_ws, size_t ws_bytes, void *stream);
/* Keys per tile of the block sort (every aligned run of this many keys comes out sorted). */
size_t b200sort_block_sort_tile(void);
int b200sort_block_sort_i32(const int32_t *d_in, int32_t *d_out, size_t n, void *stream);
/* The same for tiles of b200sort_merge_tile() keys, produced by the lab's stages 1-2 (warp split +
 * rank merges; SRM/lab.cu:47-197). */
int b200sort_lab_tile_sort_i32(const int32_t *d_in, int32_t *d_out, size_t n, void *stream);
/* Keys per output tile of a merge pass. */
size_t b200sort_merge_tile(void);
/* Merge-path split points for one pass over sorted runs of `run` keys (run a multiple of
 * b200sort_merge_tile()): d_splits[t] = number of keys taken from the pair's first run before
 * output tile t begins.  d_splits holds ceil(n / merge_tile) + 1 uint32. */
int b200sort_merge_partition_i32(const int32_t *d_in, size_t n, size_t run,
                                 uint32_t *d_splits, void *stream);
/* The pass itself: merges run pairs of d_in into d_out using d_splits. */
int b200sort_merge_pass_i32(const int32_t *d_in, int32_t *d_out, size_t n, size_t run,
                            const uint32_t *d_splits, void *stream);

/* ---- tuning / introspection --------------------------------------------------------------------- */
/* Selects one of the compiled onesweep tile shapes (0 = default); returns B200SORT_ERR_INVALID
 * if out of range.  Process-wide; for sweeps only. */
int         b200sort_radix_set_variant(int variant);
int         b200sort_radix_num_variants(void);
const char *b200sort_radix_variant_name(int variant);
size_t      b200sort_radix_tile(void);            /* keys per onesweep tile of the current variant */
/* The same switch for the compiled merge-pass kernels (0 = default). */
int         b200sort_merge_set_variant(int variant);
int         b200sort_merge_num_variants(void);
const char *b200sort_merge_variant_name(int variant);
/* Verdict of the lane-order self-test for the CURRENT device (see b200sort_radix_i32): 1 = ordered, the
 * atomicAdd-ranked shapes are in use; 0 = the ballot-ranked shapes are.  Runs the test if it has not run on
 * this device yet (BLOCKS).  B200SORT_RANK_SAFE=1 in the environment forces 0. */
int         b200sort_radix_atomic_order_ok(void);
/* Profiling aid: TIMING_* shapes stamp clock64() at their phase boundaries into this device buffer
 * (grid x 2 x 10 int64); NULL switches the probe off.  tools/phase_timing.py reads it. */
int         b200sort_debug_set_phase_buffer(void *d_buf);
/* Checked build (make CHECKED=1): the kernels assert their own bounds and alignment invariants (staged positions,
 * destination indices, 16-byte alignment of every bulk copy) and count violations instead of touching the address.
 * b200sort_debug_checked_build() is 1 for such a library; b200sort_debug_check_failures() BLOCKS and returns the
 * violations counted so far on the current device (always 0 for the product build, which compiles the checks away). */
int                b200sort_debug_checked_build(void);
unsigned long long b200sort_debug_check_failures(void);
/* The same per check site (csrc: B200_CHECK_AT(site, ...)); per_site[16] is overwritten. */
unsigned long long b200sort_debug_check_failures_by_site(unsigned long long *per_site);
/* Name of the shape that will actually be launched (after the self-test's verdict). */
const char *b200sort_radix_effective_variant_name(void);
/* Pass skipping: when a digit histogram shows one bin holding every key the pass is the
 * identity and is skipped on the device (no host sync).  1 = on (default), 0 = off. */
int         b200sort_radix_set_skip(int enabled);
/* Kernels this library has launched on this host thread since the last reset (all entry
 * points count their own launches; memsets and copies are not kernels and are not counted). */
unsigned long long b200sort_launch_count(void);
void               b200sort_launch_count_reset(void);

/* ---- host-array operator (the reference's real contract: SRM/include/lab.h:9-10) ---------------
 * Sorts h_keys[0..n) in place and BLOCKS until the result is in h_keys.  The library keeps a
 * per-process device arena (keys, scratch, workspace, pinned staging) that grows on demand and is
 * reused across calls; b200sort_host_release frees it.  h_keys may be pageable or pinned. */
int  b200sort_order_array_host(int32_t *h_keys, size_t n, int algo);
/* From 2^25 keys on, for pinned (device-accessible) arrays, the operator streams: the array moves in 8 chunks, each chunk is sorted while the
 * next one is on the wire, sorted neighbours are merged (merge-path passes) as soon as both exist, and
 * the last merge hands finished output ranges to the copy back.  0 switches that off (one H2D, one
 * sort, one D2H); 1 = default.  Same result either way. */
int  b200sort_host_set_streaming(int enabled);
/* What the exported C++ order_with_trust calls: the same host-array contract served by the
 * merge sort (the drivers' second column).  There is no host/CPU sort in this library. */
int  b200sort_order_with_trust_host(int32_t *h_keys, size_t n);
void b200sort_host_release(void);
/* Pinned host memory helpers for callers that want the fast H2D/D2H path. */
int  b200sort_host_alloc_pinned(void **h_ptr, size_t bytes);
int  b200sort_host_free_pinned(void *h_ptr);

/* ---- one-box multi-GPU sort (one process per GPU; collectives are the caller's plumbing) -------
 * No reference counterpart (north_star (c)).
 * Phase 1  b200sort_dist_histogram_i32   local 2^bits-bin histogram of the top bits of key^0x80000000
 * (caller) all-gather (all-reduce) of the counts over NCCL
 * Phase 2  b200sort_dist_plan            pure host function: contiguous bin ranges -> ranks
 * Phase 3  b200sort_dist_partition_i32   multisplit of the local keys into per-destination blocks;
 *                                        the destination table may hold local pointers (then an
 *                                        NCCL all-to-all moves the blocks) or peer-mapped pointers
 *                                        (then the scatter IS the exchange, over NVLink)
 * Phase 4  b200sort_sort_copy_i32        local sort of what arrived */
#define B200SORT_DIST_BITS_MIN 4
#define B200SORT_DIST_BITS_MAX 14
#define B200SORT_DIST_MAX_WORLD 16
/* d_hist: uint64[2^bits], overwritten. */
int b200sort_dist_histogram_i32(const int32_t *d_keys, size_t n, int bits,
                                unsigned long long *d_hist, void *stream);
/* Host planner (no device work).  all_hist[r*nbins + b] = rank r's count of bin b, nbins = 2^bits.
 * Outputs (each may be NULL except bin_owner):
 *   bin_owner[b]   in [0, world), non-decreasing in b: every rank owns one contiguous value range,
 *                  balanced to about total/world keys;
 *   recv_count[r]  keys rank r will own after the exchange;
 *   send_count[r]  keys THIS rank (`rank`) sends to rank r;
 *   dst_offset[r]  element offset inside rank r's receive buffer at which this rank's block
 *                  starts (receive buffers are laid out source rank by source rank). */
int b200sort_dist_plan(const unsigned long long *all_hist, int world, int rank, int bits,
                       int *bin_owner, unsigned long long *recv_count,
                       unsigned long long *send_count, unsigned long long *dst_offset);
/* h_dst_base[r]  (HOST array of `world` device-visible pointers, each 16-byte aligned) base of rank r's
 *                receive buffer;
 * d_bin_owner    device copy of the planner's bin_owner (int[2^bits]);
 * h_dst_offset   HOST array, the planner's dst_offset;
 * d_ws           b200sort_dist_workspace_bytes(n, bits) bytes, 256-byte aligned. */
size_t b200sort_dist_workspace_bytes(size_t n, int bits);
int b200sort_dist_partition_i32(const int32_t *d_keys, size_t n, int bits, int world,
                                int32_t *const *h_dst_base, const int *d_bin_owner,
                                const unsigned long long *h_dst_offset,
                                void *d_ws, size_t ws_bytes, void *stream);
/* The same without a host synchronisation.  The planner runs on the device over the all-gathered counts
 * (d_all_hist, world x 2^bits uint64 in DEVICE memory) and leaves its result in a device record d_plan
 * (B200SORT_DIST_PLAN_BYTES, 8-byte aligned): recv_count[16], send_count[16], dst_offset[16] (uint64 each), then
 * uint32 m = the number of keys this rank will own, uint32 error = 1 if some rank would receive more than `cap`
 * keys (then the partition kernel writes nothing), 8 bytes of padding, then uint32 top_hist[256] = for bits >= 8 the
 * histogram of the top byte (of key ^ 0x80000000) of the keys this rank will own, which follows from the bin counts;
 * for bits < 8 all zero, because a bin is then coarser than a byte.  Same boundaries as b200sort_dist_plan, bit for
 * bit.
 * b200sort_dist_partition_planned_i32 takes its offsets from that record, and b200sort_radix_copy_devn_i32 sorts
 * what arrived with the key count read from device memory (d_n = the record's m; n_max sizes grids and workspace),
 * so a whole distributed sort is enqueued without the host ever reading a count.
 * d_src_hist (may be NULL; uint32[world][4][256]; needs bits >= 8, else B200SORT_ERR_INVALID before any device work):
 * the partition kernel also counts, per destination, the 8-bit digit histograms 0..2 of the keys it sends there (of
 * key ^ 0x80000000, as b200sort_radix_histogram_i32; row 3, the top byte, stays zero: take it from the plan record's
 * top_hist).  d_src_hist is overwritten by every call, n == 0 included, and holds zeros when the plan's error flag is
 * set.
 * Summed over the source ranks (a reduce-scatter, which doubles as the barrier after the exchange) row r is the
 * histogram of exactly what rank r received; passed as d_hist (may be NULL) to b200sort_radix_copy_devn_i32 it lets
 * the local sort skip its own histogram kernel. */
#define B200SORT_DIST_PLAN_BYTES 1424
int b200sort_dist_plan_device(const unsigned long long *d_all_hist, int world, int rank, int bits,
                              unsigned long long cap, int *d_bin_owner, void *d_plan,
                              void *d_ws, size_t ws_bytes, void *stream);
int b200sort_dist_partition_planned_i32(const int32_t *d_keys, size_t n, int bits, int world,
                                        int32_t *const *h_dst_base, const int *d_bin_owner, const void *d_plan,
                                        unsigned int *d_src_hist, void *d_ws, size_t ws_bytes, void *stream);
int b200sort_radix_copy_devn_i32(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, size_t n_max,
                                 const uint32_t *d_n, const uint32_t *d_hist, void *d_ws, size_t ws_bytes, void *stream);
/* Plain cudaMalloc / cudaFree (receive buffers must be whole allocations to be exported) and the
 * CUDA IPC plumbing that lets ranks (separate processes) map each other's receive buffers. */
#define B200SORT_IPC_HANDLE_BYTES 64
int b200sort_device_malloc(void **d_ptr, size_t bytes);
int b200sort_device_free(void *d_ptr);
int b200sort_ipc_export(void *d_ptr, unsigned char *handle /* [B200SORT_IPC_HANDLE_BYTES] */);
int b200sort_ipc_open(const unsigned char *handle, void **d_ptr);
int b200sort_ipc_close(void *d_ptr);

#ifdef __cplusplus
}
#endif
#endif /* B200SORT_H */
