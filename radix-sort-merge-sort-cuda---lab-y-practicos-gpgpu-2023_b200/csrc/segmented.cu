// segmented.cu -- segmented radix sort: segment i = keys[offsets[i] .. offsets[i+1]) is sorted on its own, in any key
// order of b200sort_sort_keys, keys only or with a 32-bit value (stable).  The host never reads the offsets: every
// call enqueues the same ten kernels whatever the number of segments (DESIGN section 4.2d).
//
//   s0  seg_classify_kernel     clamps every segment to [0, n], routes it by length to a per-class list in the
//                               workspace (class 0 is copied on the spot) and zeroes the histograms of the large ones
//   s1  seg_tile_plan_kernel    one CTA: prefix of the large segments' tile counts = the global tile list
//   s2  seg_hist_kernel         the four digit histograms of every large segment, privatised per CTA in shared memory
//   s3  seg_onesweep_kernel x4  the stable passes over the tile list, look-back bounded by the segment's first tile
//   s4  seg_warp_kernel         class 1: a warp per segment
//   s5  seg_small_kernel x2     classes 2 and 3: a CTA per segment, radix_small_body
//
// VALS: 0 keys only, 1 a 32-bit value beside every key, kValsIdx the key's position in its segment (sort with
// indices): made where the key is first loaded and stored as int64 into vout where it is stored for the last time.
//
// The onesweep passes and the small-segment CTAs rank with lane-ordered shared-memory atomics like the 1-D kernels,
// behind the same self-test (radix_atomic_order_ok); SAFE = 1 is their ballot-ranked form.
#include "segmented.cuh"
#include "radix.cuh"
#include "radix_small.cuh"

namespace b200sort {

int radix_atomic_order_ok();       // radix.cu: the lane-order self-test's verdict for the current device

size_t segmented_class_max(int c) {
    switch (c) {
        case 0: return kSegMax0;
        case 1: return kSegMax1;
        case 2: return kSegMax2;
        case 3: return kSegMax3;
        default: return 0;
    }
}

constexpr int kValsIdx = 2;
constexpr int kSegWarps = kSegThreads / 32;
constexpr int kWarpSegMax = (int)kSegMax1;            // 128
constexpr int kWarpSegIpt = kWarpSegMax / 32;
constexpr int kWarpKernelThreads = 256;
constexpr int kMed1Threads = 256, kMed1Ipt = 4;              // class 2: 1024 slots
constexpr int kMed2Threads = kSmallThreads, kMed2Ipt = kSmallIpt;   // class 3: 8192 slots
static_assert(kMed1Threads * kMed1Ipt == (int)kSegMax2 && kMed2Threads * kMed2Ipt == (int)kSegMax3, "");

// Head of the workspace, zeroed by one memset per call.
struct SegControl {
    uint32_t count[4];       // segments appended to the lists of classes 1, 2, 3 and 4 (large)
    uint32_t ticket[4];      // tile tickets of the four passes
    uint32_t tiles;          // tiles of the global list (s1)
    uint32_t pad[7];
};
constexpr size_t kSegControlBytes = 256;

// Worst-case layout from (n, num_segments) alone.  A class can hold no more segments than n / (its shortest length)
// -- unless the offsets are malformed, and then the lists drop what does not fit.
struct SegLayout {
    size_t cap[4];           // list capacities of classes 1..4
    size_t rows;             // status rows: tiles of the global list, at most n / tile + large segments
    size_t off_list[4], off_prefix, off_hist, off_status, bytes;
};
static SegLayout seg_layout(size_t n, size_t S) {
    SegLayout L;
    for (int c = 0; c < 4; ++c) {
        const size_t most = n / (segmented_class_max(c) + 1);
        L.cap[c] = S < most ? S : most;
    }
    L.rows = n / kSegTile + L.cap[3];
    size_t o = kSegControlBytes;
    for (int c = 0; c < 4; ++c) { L.off_list[c] = o; o = align_up(o + L.cap[c] * sizeof(uint2), 256); }
    L.off_prefix = o; o = align_up(o + (L.cap[3] + 1) * sizeof(uint32_t), 256);
    L.off_hist = o;   o = align_up(o + L.cap[3] * kRadixPasses * kRadixBins * sizeof(uint32_t), 256);
    L.off_status = o; o += 2 * L.rows * kRadixBins * sizeof(uint32_t);
    L.bytes = o;
    return L;
}

struct SegLists {
    uint2 *list[4];          // {begin, end} of the segments of classes 1..4
    uint32_t cap[4];
};

__device__ __forceinline__ uint32_t seg_image(int32_t k, SignXor order) {
    return sign_xor(static_cast<uint32_t>(k), order.neg, order.pos);
}

// ---- s0 -------------------------------------------------------------------------------------------------------------
template <int IDX>
__device__ __forceinline__ void
seg_classify_body(const int32_t *in, int32_t *out, const int32_t *vin, int32_t *vout, uint32_t n,
                  const int32_t *offsets, uint32_t num_segments, SegControl *ctl, SegLists lists, uint32_t *hist)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < num_segments; i += gridDim.x * blockDim.x) {
        const int32_t o0 = offsets[i], o1 = offsets[i + 1];
        const uint32_t b = o0 < 0 ? 0u : ((uint32_t)o0 > n ? n : (uint32_t)o0);
        const uint32_t e = o1 < (int32_t)b ? b : ((uint32_t)o1 > n ? n : (uint32_t)o1);
        const uint32_t len = e - b;
        if (len == 1 && in != out) out[b] = in[b];
        if constexpr (IDX != 0) {
            if (len == 1) {
                B200_CHECK((reinterpret_cast<uintptr_t>(vout) & 7) == 0);
                reinterpret_cast<int64_t *>(vout)[b] = 0;
            }
        } else if (len == 1 && vin != nullptr && vin != vout) {
            vout[b] = vin[b];
        }
        // class c - 1; 4 = nothing to sort.  One atomicAdd per class and warp: with millions of short segments,
        // one per segment serialises on the four counters.
        const int c = len <= kSegMax0 ? 4 : len <= kSegMax1 ? 0 : len <= kSegMax2 ? 1 : len <= kSegMax3 ? 2 : 3;
        const uint32_t active = __activemask();
        const uint32_t peers = __match_any_sync(active, c);
        const uint32_t leader = __ffs(peers) - 1;
        uint32_t first = 0;
        if (c < 4 && lane_id() == leader) first = atomicAdd(&ctl->count[c], (uint32_t)__popc(peers));
        const uint32_t slot = __shfl_sync(active, first, leader) + __popc(peers & lanemask_lt());
        if (c == 4) continue;
        const uint32_t cap = c == 0 ? lists.cap[0] : c == 1 ? lists.cap[1] : c == 2 ? lists.cap[2] : lists.cap[3];
        uint2 *list = c == 0 ? lists.list[0] : c == 1 ? lists.list[1] : c == 2 ? lists.list[2] : lists.list[3];
        B200_CHECK_AT(15, slot < cap);
        if (slot >= cap) continue;                     // only with overlapping (malformed) segments
        list[slot] = make_uint2(b, e);
        if (c == 3) {
            uint4 *h = reinterpret_cast<uint4 *>(hist + (size_t)slot * kRadixPasses * kRadixBins);
            for (int w = 0; w < kRadixPasses * kRadixBins / 4; ++w) h[w] = make_uint4(0, 0, 0, 0);
        }
    }
}
__global__ void __launch_bounds__(256)
seg_classify_kernel(const int32_t *in, int32_t *out, const int32_t *vin, int32_t *vout, uint32_t n,
                    const int32_t *offsets, uint32_t num_segments, SegControl *ctl, SegLists lists, uint32_t *hist)
{
    seg_classify_body<0>(in, out, vin, vout, n, offsets, num_segments, ctl, lists, hist);
}
// Sort with indices: a segment of one key gets index 0 (vout is the int64 index output viewed as int32).
__global__ void __launch_bounds__(256)
seg_classify_indices_kernel(const int32_t *in, int32_t *out, const int32_t *vin, int32_t *vout, uint32_t n,
                            const int32_t *offsets, uint32_t num_segments, SegControl *ctl, SegLists lists, uint32_t *hist)
{
    seg_classify_body<1>(in, out, vin, vout, n, offsets, num_segments, ctl, lists, hist);
}

// ---- s1 -------------------------------------------------------------------------------------------------------------
constexpr int kPlanThreads = 1024;
__global__ void __launch_bounds__(kPlanThreads)
seg_tile_plan_kernel(SegControl *ctl, const uint2 *large, uint32_t cap, uint32_t *prefix, uint32_t max_tiles)
{
    __shared__ uint32_t s_warp[kPlanThreads / 32];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t m = ctl->count[3] < cap ? ctl->count[3] : cap;
    const uint32_t per = (m + kPlanThreads - 1) / kPlanThreads;
    const uint32_t j0 = tid * per, j1 = (j0 + per < m) ? j0 + per : m;
    uint32_t sum = 0;
    for (uint32_t j = j0; j < j1; ++j) sum += (large[j].y - large[j].x + kSegTile - 1) / kSegTile;
    uint32_t x = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= (uint32_t)o) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    uint32_t add = 0;
    for (uint32_t w = 0; w < warp; ++w) add += s_warp[w];
    uint32_t run = x - sum + add;
    for (uint32_t j = j0; j < j1; ++j) {
        prefix[j] = run;
        run += (large[j].y - large[j].x + kSegTile - 1) / kSegTile;
    }
    if (tid == kPlanThreads - 1) {
        prefix[m] = run;
        B200_CHECK_AT(15, run <= max_tiles);
        ctl->tiles = run < max_tiles ? run : max_tiles;
    }
}

// The large segment that holds tile t of the global list: the last j with prefix[j] <= t.
__device__ __forceinline__ uint32_t seg_of_tile(const uint32_t *prefix, uint32_t m, uint32_t t) {
    uint32_t lo = 0, hi = m;                   // prefix[lo] <= t < prefix[hi]
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (prefix[mid] <= t) lo = mid; else hi = mid;
    }
    return lo;
}

// ---- s2 -------------------------------------------------------------------------------------------------------------
// Each CTA counts a contiguous range of tiles into shared counters and flushes them to a segment's 4 x 256 counts when
// the range moves on to the next segment, so global atomics scale with CTAs + segments, not with tiles.  It also zeroes
// the status rows of the first pass.
__global__ void __launch_bounds__(kSegThreads)
seg_hist_kernel(const int32_t *in, const SegControl *ctl, const uint2 *large, uint32_t cap, const uint32_t *prefix,
                uint32_t *hist, uint32_t *status0, SignXor order)
{
    __shared__ uint32_t s_hist[kRadixPasses * kRadixBins];
    const uint32_t tid = threadIdx.x;
    const uint32_t m = ctl->count[3] < cap ? ctl->count[3] : cap;
    const uint32_t tiles = ctl->tiles;
    const uint32_t per = (tiles + gridDim.x - 1) / gridDim.x;
    const uint32_t t0 = blockIdx.x * per, t1 = (t0 + per < tiles) ? t0 + per : tiles;
    if (t0 >= t1) return;
    for (uint32_t i = tid; i < kRadixPasses * kRadixBins; i += kSegThreads) s_hist[i] = 0;
    uint32_t j = seg_of_tile(prefix, m, t0);
    auto flush = [&](uint32_t seg) {
        __syncthreads();
        for (uint32_t i = tid; i < kRadixPasses * kRadixBins; i += kSegThreads) {
            const uint32_t c = s_hist[i];
            if (c) atomicAdd(hist + (size_t)seg * kRadixPasses * kRadixBins + i, c);
            s_hist[i] = 0;
        }
    };
    __syncthreads();
    for (uint32_t t = t0; t < t1; ++t) {
        if (t >= prefix[j + 1]) {
            flush(j);
            while (t >= prefix[j + 1]) ++j;
            __syncthreads();
        }
        const uint2 seg = large[j];
        const uint32_t start = seg.x + (t - prefix[j]) * kSegTile;
        const uint32_t valid = (seg.y - start < kSegTile) ? seg.y - start : kSegTile;
        for (uint32_t i = tid; i < valid; i += kSegThreads) {
            const uint32_t img = seg_image(in[start + i], order);
#pragma unroll
            for (int p = 0; p < kRadixPasses; ++p) atomicAdd(&s_hist[p * kRadixBins + ((img >> (p * kRadixBits)) & 0xFF)], 1u);
        }
        if (tid < kRadixBins) status0[(size_t)t * kRadixBins + tid] = 0;
    }
    flush(j);
}

// ---- s3 -------------------------------------------------------------------------------------------------------------
template <int VALS>
struct SegPassSmem {
    uint32_t cnt[kSegWarps][kRadixBins];   // per-warp digit counts -> the warp's offset inside the digit's run
    int32_t keys[kSegTile];                // the tile in digit order
    int32_t vals[VALS ? kSegTile : 1];
    uint32_t excl[kRadixBins];             // first tile-local position of each digit
    uint32_t dst[kRadixBins];              // segment-relative destination of tile-local position 0 of each digit
    uint32_t sums[2][8];
    uint32_t info[5];                      // ticket, segment begin, length, tile in segment, large-segment index
};

// One stable pass by digit `pass` over the tile list, persistent CTAs drawing tiles by ticket.  A tile publishes its
// digit counts ({flag:2, count:30}: kFlagLocal, or kFlagIncl on the segment's first tile), walks back over the earlier
// tiles OF ITS SEGMENT until an inclusive count, and writes key i of digit d to
//   segment begin + segment base[d] + (keys of digit d in earlier tiles of the segment) + tile-local rank.
// Buffers: pass 0 reads in, passes 0 and 2 write tmp, 1 and 3 write out: four passes land in out.
// VALS = kValsIdx: pass 0 makes the indices, pass 3 stores them as int64 into vout, and pass 1 leaves them as int32 in
// the first half of the segment's own int64 range of vout (vout[2 * begin + pos]).  So no pass writes into another
// segment's part of the index output, which the other kernels of the call fill in any order.
template <int VALS, int SAFE>
__global__ void __launch_bounds__(kSegThreads, 2)
seg_onesweep_kernel(const int32_t *in, int32_t *out, int32_t *tmp, const int32_t *vin, int32_t *vout, int32_t *vtmp,
                    int pass, SegControl *ctl, const uint2 *large, uint32_t cap, const uint32_t *prefix,
                    const uint32_t *hist, uint32_t *status, uint32_t *status_next, SignXor order)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SegPassSmem<VALS> &sm = *reinterpret_cast<SegPassSmem<VALS> *>(smem_raw);
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int shift = pass * kRadixBits;
    const uint32_t flips = flips_of(order.neg, order.pos, shift);
    const int32_t *src = pass == 0 ? in : (pass & 1) ? tmp : out;
    int32_t *dst = (pass & 1) ? out : tmp;
    const int32_t *vsrc = pass == 0 ? vin : (pass & 1) ? vtmp : vout;
    int32_t *vdst = (pass & 1) ? vout : vtmp;
    const int32_t pad_key = (int32_t)key_of_last_image(order);
    const uint32_t m = ctl->count[3] < cap ? ctl->count[3] : cap;
    const uint32_t tiles = ctl->tiles;
    uint32_t *wcnt = sm.cnt[warp];
    const uint32_t wofs = warp * (32 * kSegIpt) + lane;

    for (;;) {
        if (tid == 0) {
            const uint32_t t = atomicAdd(&ctl->ticket[pass], 1u);
            sm.info[0] = t;
            if (t < tiles) {
                const uint32_t j = seg_of_tile(prefix, m, t);
                const uint2 seg = large[j];
                sm.info[1] = seg.x;
                sm.info[2] = seg.y - seg.x;
                sm.info[3] = t - prefix[j];
                sm.info[4] = j;
            }
        }
        for (int d = lane; d < kRadixBins; d += 32) wcnt[d] = 0;
        __syncthreads();
        const uint32_t t = sm.info[0];
        if (t >= tiles) return;
        const uint32_t begin = sm.info[1], len = sm.info[2], k = sm.info[3], j = sm.info[4];
        const uint32_t start = k * kSegTile;                 // segment-relative
        const uint32_t valid = (len - start < kSegTile) ? len - start : kSegTile;

        int32_t key[kSegIpt], val[VALS ? kSegIpt : 1];
        uint32_t rank[kSegIpt];
#pragma unroll
        for (int i = 0; i < kSegIpt; ++i) {
            const uint32_t at = wofs + i * 32;                // warp-striped: tile order = memory order
            key[i] = at < valid ? src[begin + start + at] : pad_key;
            if constexpr (VALS == kValsIdx) {
                if (pass == 0) val[i] = (int32_t)(start + at);
                else if (pass & 1) val[i] = at < valid ? vtmp[begin + start + at] : 0;
                else val[i] = at < valid ? vout[2 * (size_t)begin + start + at] : 0;
            } else if constexpr (VALS != 0) {
                val[i] = at < valid ? vsrc[begin + start + at] : 0;
            }
        }
#pragma unroll
        for (int i = 0; i < kSegIpt; ++i) {
            const bool ok = wofs + i * 32 < valid;           // the padding is not counted
            const uint32_t d = digit_of_image(key[i], shift, flips);
            if constexpr (SAFE != 0) {
                const uint32_t peers = __match_any_sync(0xffffffffu, ok ? d : kRadixBins);
                const uint32_t leader = __ffs(peers) - 1;
                uint32_t base = 0;
                if (ok && lane == leader) base = atomicAdd(wcnt + d, (uint32_t)__popc(peers));
                rank[i] = __shfl_sync(0xffffffffu, base, leader) + __popc(peers & lanemask_lt());
            } else {
                rank[i] = ok ? atomicAdd(wcnt + d, 1u) : 0u;
            }
        }
        __syncthreads();                                       // warp counts final
        if (tid < kRadixBins) {
            uint32_t run = 0;
#pragma unroll
            for (int w = 0; w < kSegWarps; ++w) {
                const uint32_t c = sm.cnt[w][tid];
                sm.cnt[w][tid] = run;
                run += c;
            }
            uint32_t *row = status + (size_t)t * kRadixBins + tid;
            st_relaxed_gpu(row, (k == 0 ? kFlagIncl : kFlagLocal) | run);
            const uint32_t excl = scan256(run, sm.sums[0]);
            const uint32_t seg_base = scan256(hist[(size_t)j * kRadixPasses * kRadixBins + pass * kRadixBins + tid],
                                              sm.sums[1]);
            uint32_t before = 0;                               // keys of this digit in the segment's earlier tiles
            if (k > 0) {
                for (const uint32_t *p = row - kRadixBins;; p -= kRadixBins) {
                    uint32_t w;
                    do { w = ld_relaxed_gpu(p); } while ((w & ~kValueMask) == 0);
                    before += w & kValueMask;
                    if (w & kFlagIncl) break;                  // the segment's first tile is always inclusive
                }
                // a segment's last inclusive count may need 31 bits; no later tile of the segment reads it
                st_relaxed_gpu(row, kFlagIncl | ((before + run) & kValueMask));
            }
            sm.excl[tid] = excl;
            sm.dst[tid] = seg_base + before - excl;
            if (status_next != nullptr) status_next[(size_t)t * kRadixBins + tid] = 0;
        }
        __syncthreads();                                       // offsets final
#pragma unroll
        for (int i = 0; i < kSegIpt; ++i) {
            if (wofs + i * 32 < valid) {
                const uint32_t d = digit_of_image(key[i], shift, flips);
                const uint32_t at = sm.excl[d] + wcnt[d] + rank[i];
                sm.keys[at] = key[i];
                if constexpr (VALS != 0) sm.vals[at] = val[i];
            }
        }
        __syncthreads();                                       // the tile is staged in digit order
        for (uint32_t i = tid; i < valid; i += kSegThreads) {
            const int32_t kk = sm.keys[i];
            const uint32_t pos = sm.dst[digit_of_image(kk, shift, flips)] + i;
            B200_CHECK_AT(15, pos < len);
            if (pos < len) {                                   // only malformed offsets fail this
                dst[begin + pos] = kk;
                if constexpr (VALS == kValsIdx) {
                    if (pass == kRadixPasses - 1) {
                        B200_CHECK((reinterpret_cast<uintptr_t>(vout) & 7) == 0);
                        reinterpret_cast<int64_t *>(vout)[begin + pos] = sm.vals[i];
                    } else if (pass & 1) {
                        vout[2 * (size_t)begin + pos] = sm.vals[i];
                    } else {
                        vtmp[begin + pos] = sm.vals[i];
                    }
                } else if constexpr (VALS != 0) {
                    vdst[begin + pos] = sm.vals[i];
                }
            }
        }
        __syncthreads();                                       // shared memory free for the next tile
    }
}

// ---- s4 -------------------------------------------------------------------------------------------------------------
// Class 1: a warp per segment of 2..128 keys.  The rank of a key is the number of keys before it in (image, position)
// order, counted against the segment's images in shared memory: stable, no atomics, no padding.
template <int VALS>
__global__ void __launch_bounds__(kWarpKernelThreads)
seg_warp_kernel(const int32_t *in, int32_t *out, const int32_t *vin, int32_t *vout, const SegControl *ctl,
                const uint2 *list, uint32_t cap, SignXor order)
{
    __shared__ uint32_t s_img[kWarpKernelThreads / 32][kWarpSegMax];
    const uint32_t lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint32_t count = ctl->count[0] < cap ? ctl->count[0] : cap;
    uint32_t *img_s = s_img[wib];
    for (uint32_t s = blockIdx.x * (kWarpKernelThreads / 32) + wib; s < count; s += gridDim.x * (kWarpKernelThreads / 32)) {
        const uint2 seg = list[s];
        const uint32_t len = seg.y - seg.x;
        int32_t key[kWarpSegIpt], val[kWarpSegIpt];
        uint32_t img[kWarpSegIpt], pos[kWarpSegIpt];
#pragma unroll
        for (int q = 0; q < kWarpSegIpt; ++q) {
            const uint32_t i = lane + 32 * q;
            key[q] = i < len ? in[seg.x + i] : 0;
            if constexpr (VALS == kValsIdx) val[q] = (int32_t)i;
            else if constexpr (VALS != 0) val[q] = i < len ? vin[seg.x + i] : 0;
            img[q] = seg_image(key[q], order);
            pos[q] = 0;
            if (i < len) img_s[i] = img[q];
        }
        __syncwarp();                                          // every key read before any is written
        for (uint32_t i = 0; i < len; ++i) {
            const uint32_t v = img_s[i];
#pragma unroll
            for (int q = 0; q < kWarpSegIpt; ++q) pos[q] += (v < img[q]) | ((v == img[q]) & (i < lane + 32 * q));
        }
#pragma unroll
        for (int q = 0; q < kWarpSegIpt; ++q) {
            if (lane + 32 * q < len) {
                out[seg.x + pos[q]] = key[q];
                if constexpr (VALS == kValsIdx) {
                    B200_CHECK_AT(15, pos[q] < len);
                    B200_CHECK((reinterpret_cast<uintptr_t>(vout) & 7) == 0);
                    reinterpret_cast<int64_t *>(vout)[seg.x + pos[q]] = val[q];
                } else if constexpr (VALS != 0) {
                    vout[seg.x + pos[q]] = val[q];
                }
            }
        }
        __syncwarp();                                          // img_s free for the warp's next segment
    }
}

// ---- s5 -------------------------------------------------------------------------------------------------------------
template <int THREADS, int IPT, int VALS, int SAFE>
__global__ void __launch_bounds__(THREADS)
seg_small_kernel(const int32_t *in, int32_t *out, const int32_t *vin, int32_t *vout, const SegControl *ctl,
                 const uint2 *list, uint32_t cap, int c, SignXor order)
{
    const uint32_t count = ctl->count[c] < cap ? ctl->count[c] : cap;
    for (uint32_t s = blockIdx.x; s < count; s += gridDim.x) {
        const uint2 seg = list[s];
        if constexpr (VALS == kValsIdx)
            radix_small_body<1, THREADS, IPT, VALS, SAFE, 1>(in + seg.x, out + seg.x, seg.y - seg.x, order, nullptr,
                                                          reinterpret_cast<int32_t *>(reinterpret_cast<int64_t *>(vout) + seg.x));
        else
            radix_small_body<1, THREADS, IPT, VALS, SAFE, 1>(in + seg.x, out + seg.x, seg.y - seg.x, order,
                                                          VALS ? vin + seg.x : nullptr, VALS ? vout + seg.x : nullptr);
        __syncthreads();                                       // shared memory free for the next segment
    }
}

static unsigned grid_of(size_t want, size_t most) {
    const size_t g = want < most ? want : most;
    return (unsigned)(g < 1 ? 1 : g);
}

template <int THREADS, int IPT, int VALS, int SAFE>
int launch_small(const int32_t *in, int32_t *out, const int32_t *vin, int32_t *vout, const SegControl *ctl,
                 const uint2 *list, size_t cap, int c, SignXor order, unsigned per_sm, cudaStream_t s) {
    constexpr size_t smem = small_smem_bytes(THREADS, IPT, VALS);
    auto *fn = seg_small_kernel<THREADS, IPT, VALS, SAFE>;
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(fn), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
    fn<<<grid_of(cap, (size_t)kNumSMs * per_sm), THREADS, smem, s>>>(in, out, vin, vout, ctl, list, (uint32_t)cap, c, order);
    B200_LAUNCH_CHECK();
    return B200SORT_OK;
}

template <int VALS, int SAFE>
int seg_sort_impl(const int32_t *in, int32_t *out, int32_t *tmp, const int32_t *vin, int32_t *vout, int32_t *vtmp,
                  size_t n, const int32_t *offsets, size_t S, void *ws, cudaStream_t s, SignXor order) {
    const SegLayout L = seg_layout(n, S);
    auto *base = static_cast<unsigned char *>(ws);
    auto *ctl = reinterpret_cast<SegControl *>(base);
    SegLists lists;
    for (int c = 0; c < 4; ++c) {
        lists.list[c] = reinterpret_cast<uint2 *>(base + L.off_list[c]);
        lists.cap[c] = (uint32_t)L.cap[c];
    }
    auto *prefix = reinterpret_cast<uint32_t *>(base + L.off_prefix);
    auto *hist = reinterpret_cast<uint32_t *>(base + L.off_hist);
    uint32_t *status[2] = {reinterpret_cast<uint32_t *>(base + L.off_status),
                           reinterpret_cast<uint32_t *>(base + L.off_status) + L.rows * kRadixBins};
    const uint32_t cap_large = (uint32_t)L.cap[3];

    B200_CUDA_TRY(cudaMemsetAsync(ctl, 0, sizeof(SegControl), s));
    (VALS == kValsIdx ? seg_classify_indices_kernel : seg_classify_kernel)<<<grid_of(div_up(S, 256), (size_t)kNumSMs * 8), 256, 0, s>>>(
        in, out, vin, vout, (uint32_t)n, offsets, (uint32_t)S, ctl, lists, hist);
    B200_LAUNCH_CHECK();
    seg_tile_plan_kernel<<<1, kPlanThreads, 0, s>>>(ctl, lists.list[3], cap_large, prefix, (uint32_t)L.rows);
    B200_LAUNCH_CHECK();
    seg_hist_kernel<<<grid_of(L.rows, (size_t)kNumSMs * 4), kSegThreads, 0, s>>>(in, ctl, lists.list[3], cap_large,
                                                                               prefix, hist, status[0], order);
    B200_LAUNCH_CHECK();
    constexpr size_t pass_smem = sizeof(SegPassSmem<VALS>);
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(seg_onesweep_kernel<VALS, SAFE>),
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pass_smem));
    for (int pass = 0; pass < kRadixPasses; ++pass) {
        seg_onesweep_kernel<VALS, SAFE><<<grid_of(L.rows, (size_t)kNumSMs * 2), kSegThreads, pass_smem, s>>>(
            in, out, tmp, vin, vout, vtmp, pass, ctl, lists.list[3], cap_large, prefix, hist, status[pass & 1],
            pass + 1 < kRadixPasses ? status[(pass + 1) & 1] : nullptr, order);
        B200_LAUNCH_CHECK();
    }
    seg_warp_kernel<VALS><<<grid_of(div_up(L.cap[0], kWarpKernelThreads / 32), (size_t)kNumSMs * 8), kWarpKernelThreads,
                            0, s>>>(in, out, vin, vout, ctl, lists.list[0], lists.cap[0], order);
    B200_LAUNCH_CHECK();
    B200_TRY((launch_small<kMed1Threads, kMed1Ipt, VALS, SAFE>(in, out, vin, vout, ctl, lists.list[1], L.cap[1], 1, order, 8, s)));
    B200_TRY((launch_small<kMed2Threads, kMed2Ipt, VALS, SAFE>(in, out, vin, vout, ctl, lists.list[2], L.cap[2], 2, order,
                                                               VALS ? 1 : 2, s)));
    return B200SORT_OK;
}

size_t segmented_workspace_bytes(size_t n, size_t num_segments) { return seg_layout(n, num_segments).bytes; }

int segmented_sort(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, const int32_t *v_in, int32_t *v_out,
                   int32_t *v_tmp, size_t n, const int32_t *d_offsets, size_t num_segments, void *d_ws,
                   cudaStream_t s, SignXor order) {
    if (num_segments == 0) return B200SORT_OK;
    const bool safe = !radix_atomic_order_ok();
    if (v_in == nullptr)
        return safe ? seg_sort_impl<0, 1>(d_in, d_out, d_tmp, nullptr, nullptr, nullptr, n, d_offsets, num_segments, d_ws, s, order)
                    : seg_sort_impl<0, 0>(d_in, d_out, d_tmp, nullptr, nullptr, nullptr, n, d_offsets, num_segments, d_ws, s, order);
    return safe ? seg_sort_impl<1, 1>(d_in, d_out, d_tmp, v_in, v_out, v_tmp, n, d_offsets, num_segments, d_ws, s, order)
                : seg_sort_impl<1, 0>(d_in, d_out, d_tmp, v_in, v_out, v_tmp, n, d_offsets, num_segments, d_ws, s, order);
}

int segmented_sort_indices(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, int64_t *idx_out, int32_t *tmp_idx,
                           size_t n, const int32_t *d_offsets, size_t num_segments, void *d_ws, cudaStream_t s,
                           SignXor order) {
    if (num_segments == 0) return B200SORT_OK;
    auto *idx32 = reinterpret_cast<int32_t *>(idx_out);
    return radix_atomic_order_ok()
               ? seg_sort_impl<kValsIdx, 0>(d_in, d_out, d_tmp, nullptr, idx32, tmp_idx, n, d_offsets, num_segments, d_ws, s, order)
               : seg_sort_impl<kValsIdx, 1>(d_in, d_out, d_tmp, nullptr, idx32, tmp_idx, n, d_offsets, num_segments, d_ws, s, order);
}

unsigned long long segmented_check_failures(unsigned long long *per_site) { return tu_check_failures(per_site); }

}  // namespace b200sort
