// segmented16.cu -- segmented sort of 16-bit keys: segment i = keys[offsets[i] .. offsets[i+1]) is sorted on its own
// in any order of b200sort_sort_keys16, keys only or with a 32-bit value (stable).  The structure is segmented.cu's
// (DESIGN section 4.2d) with two 8-bit passes over the 16-bit image instead of four over the 32-bit one; every call
// enqueues one memset and the same eight kernels whatever the number of segments (DESIGN section 4.2g).
//
//   g0  seg16_classify_kernel     clamps every segment to [0, n], routes it by length to a per-class list in the
//                                 workspace (class 0 is copied on the spot) and zeroes the histograms of the large ones
//   g1  seg16_tile_plan_kernel    one CTA: prefix of the large segments' tile counts = the global tile list
//   g2  seg16_hist_kernel         the two digit histograms of every large segment, privatised per CTA in shared memory
//   g3  seg16_onesweep_kernel x2  the stable passes over the tile list, look-back bounded by the segment's first tile;
//                                 in -> tmp, then tmp -> out
//   g4  seg16_warp_kernel         class 1: a warp per segment
//   g5  seg16_small_kernel x2     classes 2 and 3: a CTA per segment, both passes in shared memory
//
// The onesweep passes and the small-segment CTAs rank with lane-ordered shared-memory atomics like the 1-D kernels,
// behind the same self-test (radix_atomic_order_ok); SAFE = 1 is their ballot-ranked form.  Keys are read and
// written as 2-byte words, so a segment may begin at any 2-byte boundary.
#include "segmented16.cuh"
#include "radix.cuh"
#include "radix_digit.cuh"

namespace b200sort {

int radix_atomic_order_ok();       // radix.cu: the lane-order self-test's verdict for the current device

constexpr int kSeg16Passes = 2;

size_t segmented16_class_max(int c) {
    switch (c) {
        case 0: return kSeg16Max0;
        case 1: return kSeg16Max1;
        case 2: return kSeg16Max2;
        case 3: return kSeg16Max3;
        default: return 0;
    }
}

constexpr int kSeg16Warps = kSeg16Threads / 32;
constexpr int kWarp16SegMax = (int)kSeg16Max1;                // 128
constexpr int kWarp16SegIpt = kWarp16SegMax / 32;
constexpr int kWarp16KernelThreads = 256;
constexpr int kMed16aThreads = 256, kMed16aIpt = 4;           // class 2: 1024 slots
constexpr int kMed16bThreads = 512, kMed16bIpt = 16;          // class 3: 8192 slots
static_assert(kMed16aThreads * kMed16aIpt == (int)kSeg16Max2 && kMed16bThreads * kMed16bIpt == (int)kSeg16Max3, "");

// Head of the workspace, zeroed by one memset per call.
struct Seg16Control {
    uint32_t count[4];       // segments appended to the lists of classes 1, 2, 3 and 4 (large)
    uint32_t ticket[2];      // tile tickets of the two passes
    uint32_t tiles;          // tiles of the global list (g1)
    uint32_t pad[9];
};
constexpr size_t kSeg16ControlBytes = 256;

// Worst-case layout from (n, num_segments) alone, as segmented.cu's.
struct Seg16Layout {
    size_t cap[4];           // list capacities of classes 1..4
    size_t rows;             // status rows: tiles of the global list, at most n / tile + large segments
    size_t off_list[4], off_prefix, off_hist, off_status, bytes;
};
static Seg16Layout seg16_layout(size_t n, size_t S) {
    Seg16Layout L;
    for (int c = 0; c < 4; ++c) {
        const size_t most = n / (segmented16_class_max(c) + 1);
        L.cap[c] = S < most ? S : most;
    }
    L.rows = n / kSeg16Tile + L.cap[3];
    size_t o = kSeg16ControlBytes;
    for (int c = 0; c < 4; ++c) { L.off_list[c] = o; o = align_up(o + L.cap[c] * sizeof(uint2), 256); }
    L.off_prefix = o; o = align_up(o + (L.cap[3] + 1) * sizeof(uint32_t), 256);
    L.off_hist = o;   o = align_up(o + L.cap[3] * kSeg16Passes * kRadixBins * sizeof(uint32_t), 256);
    L.off_status = o; o += 2 * L.rows * kRadixBins * sizeof(uint32_t);
    L.bytes = o;
    return L;
}

struct Seg16Lists {
    uint2 *list[4];          // {begin, end} of the segments of classes 1..4
    uint32_t cap[4];
};

__device__ __forceinline__ uint32_t seg16_digit(uint32_t k, int pass, SignXor16 o) {
    return (image16(k, o) >> (pass * kRadixBits)) & (kRadixBins - 1);
}

// ---- g0 -------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
seg16_classify_kernel(const uint16_t *in, uint16_t *out, const int32_t *vin, int32_t *vout, uint32_t n,
                      const int32_t *offsets, uint32_t num_segments, Seg16Control *ctl, Seg16Lists lists, uint32_t *hist)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < num_segments; i += gridDim.x * blockDim.x) {
        const int32_t o0 = offsets[i], o1 = offsets[i + 1];
        const uint32_t b = o0 < 0 ? 0u : ((uint32_t)o0 > n ? n : (uint32_t)o0);
        const uint32_t e = o1 < (int32_t)b ? b : ((uint32_t)o1 > n ? n : (uint32_t)o1);
        const uint32_t len = e - b;
        if (len == 1 && in != out) out[b] = in[b];
        if (len == 1 && vin != nullptr && vin != vout) vout[b] = vin[b];
        // class c - 1; 4 = nothing to sort.  One atomicAdd per class and warp (segmented.cu).
        const int c = len <= kSeg16Max0 ? 4 : len <= kSeg16Max1 ? 0 : len <= kSeg16Max2 ? 1 : len <= kSeg16Max3 ? 2 : 3;
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
            uint4 *h = reinterpret_cast<uint4 *>(hist + (size_t)slot * kSeg16Passes * kRadixBins);
            for (int w = 0; w < kSeg16Passes * kRadixBins / 4; ++w) h[w] = make_uint4(0, 0, 0, 0);
        }
    }
}

// ---- g1 -------------------------------------------------------------------------------------------------------------
constexpr int kPlan16Threads = 1024;
__global__ void __launch_bounds__(kPlan16Threads)
seg16_tile_plan_kernel(Seg16Control *ctl, const uint2 *large, uint32_t cap, uint32_t *prefix, uint32_t max_tiles)
{
    __shared__ uint32_t s_warp[kPlan16Threads / 32];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t m = ctl->count[3] < cap ? ctl->count[3] : cap;
    const uint32_t per = (m + kPlan16Threads - 1) / kPlan16Threads;
    const uint32_t j0 = tid * per, j1 = (j0 + per < m) ? j0 + per : m;
    uint32_t sum = 0;
    for (uint32_t j = j0; j < j1; ++j) sum += (large[j].y - large[j].x + kSeg16Tile - 1) / kSeg16Tile;
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
        run += (large[j].y - large[j].x + kSeg16Tile - 1) / kSeg16Tile;
    }
    if (tid == kPlan16Threads - 1) {
        prefix[m] = run;
        B200_CHECK_AT(15, run <= max_tiles);
        ctl->tiles = run < max_tiles ? run : max_tiles;
    }
}

// The large segment that holds tile t of the global list: the last j with prefix[j] <= t.
__device__ __forceinline__ uint32_t seg16_of_tile(const uint32_t *prefix, uint32_t m, uint32_t t) {
    uint32_t lo = 0, hi = m;                   // prefix[lo] <= t < prefix[hi]
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (prefix[mid] <= t) lo = mid; else hi = mid;
    }
    return lo;
}

// ---- g2 -------------------------------------------------------------------------------------------------------------
// Each CTA counts a contiguous range of tiles into shared counters and flushes them to a segment's 2 x 256 counts when
// the range moves on to the next segment.  It also zeroes the status rows of the first pass.
__global__ void __launch_bounds__(kSeg16Threads)
seg16_hist_kernel(const uint16_t *in, const Seg16Control *ctl, const uint2 *large, uint32_t cap, const uint32_t *prefix,
                  uint32_t *hist, uint32_t *status0, SignXor16 order)
{
    __shared__ uint32_t s_hist[kSeg16Passes * kRadixBins];
    const uint32_t tid = threadIdx.x;
    const uint32_t m = ctl->count[3] < cap ? ctl->count[3] : cap;
    const uint32_t tiles = ctl->tiles;
    const uint32_t per = (tiles + gridDim.x - 1) / gridDim.x;
    const uint32_t t0 = blockIdx.x * per, t1 = (t0 + per < tiles) ? t0 + per : tiles;
    if (t0 >= t1) return;
    for (uint32_t i = tid; i < kSeg16Passes * kRadixBins; i += kSeg16Threads) s_hist[i] = 0;
    uint32_t j = seg16_of_tile(prefix, m, t0);
    auto flush = [&](uint32_t seg) {
        __syncthreads();
        for (uint32_t i = tid; i < kSeg16Passes * kRadixBins; i += kSeg16Threads) {
            const uint32_t c = s_hist[i];
            if (c) atomicAdd(hist + (size_t)seg * kSeg16Passes * kRadixBins + i, c);
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
        const uint32_t start = seg.x + (t - prefix[j]) * kSeg16Tile;
        const uint32_t valid = (seg.y - start < kSeg16Tile) ? seg.y - start : kSeg16Tile;
        for (uint32_t i = tid; i < valid; i += kSeg16Threads) {
            const uint32_t img = image16(in[start + i], order);
            atomicAdd(&s_hist[img & 0xFF], 1u);
            atomicAdd(&s_hist[kRadixBins + (img >> 8)], 1u);
        }
        if (tid < kRadixBins) status0[(size_t)t * kRadixBins + tid] = 0;
    }
    flush(j);
}

// ---- g3 -------------------------------------------------------------------------------------------------------------
template <int VALS>
struct Seg16PassSmem {
    uint32_t cnt[kSeg16Warps][kRadixBins];   // per-warp digit counts -> the warp's offset inside the digit's run
    int32_t vals[VALS ? kSeg16Tile : 1];     // the tile in digit order
    uint16_t keys[kSeg16Tile];
    uint32_t excl[kRadixBins];               // first tile-local position of each digit
    uint32_t dst[kRadixBins];                // segment-relative destination of tile-local position 0 of each digit
    uint32_t sums[2][8];
    uint32_t info[5];                        // ticket, segment begin, length, tile in segment, large-segment index
};

// One stable pass by the digit `pass` of the image over the tile list, as segmented.cu's seg_onesweep_kernel: tiles
// by ticket, {flag:2, count:30} status words, look-back over the earlier tiles OF ITS SEGMENT until an inclusive
// count, and key i of digit d goes to
//   segment begin + segment base[d] + (keys of digit d in earlier tiles of the segment) + tile-local rank.
// Slots past the segment's end are neither ranked nor staged.  Pass 0 reads in and writes tmp, pass 1 reads tmp and
// writes out, so out of place the input is only read.
template <int VALS, int SAFE>
__global__ void __launch_bounds__(kSeg16Threads, 2)
seg16_onesweep_kernel(const uint16_t *in, uint16_t *out, uint16_t *tmp, const int32_t *vin, int32_t *vout,
                      int32_t *vtmp, int pass, Seg16Control *ctl, const uint2 *large, uint32_t cap,
                      const uint32_t *prefix, const uint32_t *hist, uint32_t *status, uint32_t *status_next,
                      SignXor16 order)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Seg16PassSmem<VALS> &sm = *reinterpret_cast<Seg16PassSmem<VALS> *>(smem_raw);
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint16_t *src = pass == 0 ? in : tmp;
    uint16_t *dst = pass == 0 ? tmp : out;
    const int32_t *vsrc = pass == 0 ? vin : vtmp;
    int32_t *vdst = pass == 0 ? vtmp : vout;
    const uint32_t m = ctl->count[3] < cap ? ctl->count[3] : cap;
    const uint32_t tiles = ctl->tiles;
    uint32_t *wcnt = sm.cnt[warp];
    const uint32_t wofs = warp * (32 * kSeg16Ipt) + lane;

    for (;;) {
        if (tid == 0) {
            const uint32_t t = atomicAdd(&ctl->ticket[pass], 1u);
            sm.info[0] = t;
            if (t < tiles) {
                const uint32_t j = seg16_of_tile(prefix, m, t);
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
        const uint32_t start = k * kSeg16Tile;               // segment-relative
        const uint32_t valid = (len - start < kSeg16Tile) ? len - start : kSeg16Tile;

        // kr: the key in the low half, its rank among the warp's keys of its digit (< kSeg16Tile) in the high half
        uint32_t kr[kSeg16Ipt];
        int32_t val[VALS ? kSeg16Ipt : 1];
#pragma unroll
        for (int i = 0; i < kSeg16Ipt; ++i) {
            const uint32_t at = wofs + i * 32;                // warp-striped: tile order = memory order
            kr[i] = at < valid ? src[begin + start + at] : 0u;
            if constexpr (VALS != 0) val[i] = at < valid ? vsrc[begin + start + at] : 0;
        }
#pragma unroll
        for (int i = 0; i < kSeg16Ipt; ++i) {
            const bool ok = wofs + i * 32 < valid;           // the padding is not counted
            const uint32_t d = seg16_digit(kr[i], pass, order);
            uint32_t rank;
            if constexpr (SAFE != 0) {
                const uint32_t peers = __match_any_sync(0xffffffffu, ok ? d : kRadixBins);
                const uint32_t leader = __ffs(peers) - 1;
                uint32_t base = 0;
                if (ok && lane == leader) base = atomicAdd(wcnt + d, (uint32_t)__popc(peers));
                rank = __shfl_sync(0xffffffffu, base, leader) + __popc(peers & lanemask_lt());
            } else {
                rank = ok ? atomicAdd(wcnt + d, 1u) : 0u;
            }
            kr[i] |= rank << 16;
        }
        __syncthreads();                                       // warp counts final
        if (tid < kRadixBins) {
            uint32_t run = 0;
#pragma unroll
            for (int w = 0; w < kSeg16Warps; ++w) {
                const uint32_t c = sm.cnt[w][tid];
                sm.cnt[w][tid] = run;
                run += c;
            }
            uint32_t *row = status + (size_t)t * kRadixBins + tid;
            st_relaxed_gpu(row, (k == 0 ? kFlagIncl : kFlagLocal) | run);
            const uint32_t excl = scan256(run, sm.sums[0]);
            const uint32_t seg_base = scan256(hist[(size_t)j * kSeg16Passes * kRadixBins + pass * kRadixBins + tid],
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
        for (int i = 0; i < kSeg16Ipt; ++i) {
            if (wofs + i * 32 < valid) {
                const uint32_t key = kr[i] & 0xFFFFu;
                const uint32_t d = seg16_digit(key, pass, order);
                const uint32_t at = sm.excl[d] + wcnt[d] + (kr[i] >> 16);
                B200_CHECK_AT(1, at < kSeg16Tile);
                if (at < kSeg16Tile) {
                    sm.keys[at] = (uint16_t)key;
                    if constexpr (VALS != 0) sm.vals[at] = val[i];
                }
            }
        }
        __syncthreads();                                       // the tile is staged in digit order
        for (uint32_t i = tid; i < valid; i += kSeg16Threads) {
            const uint32_t kk = sm.keys[i];
            const uint32_t pos = sm.dst[seg16_digit(kk, pass, order)] + i;
            B200_CHECK_AT(15, pos < len);
            if (pos < len) {                                   // only malformed offsets fail this
                dst[begin + pos] = (uint16_t)kk;
                if constexpr (VALS != 0) vdst[begin + pos] = sm.vals[i];
            }
        }
        __syncthreads();                                       // shared memory free for the next tile
    }
}

// ---- g4 -------------------------------------------------------------------------------------------------------------
// Class 1: a warp per segment of 2..128 keys.  The rank of a key is the number of keys before it in (image, position)
// order, counted against the segment's images in shared memory: stable, no atomics, no padding.
template <int VALS>
__global__ void __launch_bounds__(kWarp16KernelThreads)
seg16_warp_kernel(const uint16_t *in, uint16_t *out, const int32_t *vin, int32_t *vout, const Seg16Control *ctl,
                  const uint2 *list, uint32_t cap, SignXor16 order)
{
    __shared__ uint32_t s_img[kWarp16KernelThreads / 32][kWarp16SegMax];
    const uint32_t lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint32_t count = ctl->count[0] < cap ? ctl->count[0] : cap;
    uint32_t *img_s = s_img[wib];
    for (uint32_t s = blockIdx.x * (kWarp16KernelThreads / 32) + wib; s < count;
         s += gridDim.x * (kWarp16KernelThreads / 32)) {
        const uint2 seg = list[s];
        const uint32_t len = seg.y - seg.x;
        uint32_t key[kWarp16SegIpt], img[kWarp16SegIpt], pos[kWarp16SegIpt];
        int32_t val[kWarp16SegIpt];
#pragma unroll
        for (int q = 0; q < kWarp16SegIpt; ++q) {
            const uint32_t i = lane + 32 * q;
            key[q] = i < len ? in[seg.x + i] : 0u;
            if constexpr (VALS != 0) val[q] = i < len ? vin[seg.x + i] : 0;
            img[q] = image16(key[q], order);
            pos[q] = 0;
            if (i < len) img_s[i] = img[q];
        }
        __syncwarp();                                          // every key read before any is written
        for (uint32_t i = 0; i < len; ++i) {
            const uint32_t v = img_s[i];
#pragma unroll
            for (int q = 0; q < kWarp16SegIpt; ++q) pos[q] += (v < img[q]) | ((v == img[q]) & (i < lane + 32 * q));
        }
#pragma unroll
        for (int q = 0; q < kWarp16SegIpt; ++q) {
            if (lane + 32 * q < len) {
                B200_CHECK_AT(15, pos[q] < len);
                out[seg.x + pos[q]] = (uint16_t)key[q];
                if constexpr (VALS != 0) vout[seg.x + pos[q]] = val[q];
            }
        }
        __syncwarp();                                          // img_s free for the warp's next segment
    }
}

// ---- g5 -------------------------------------------------------------------------------------------------------------
// Classes 2 and 3: one segment of n <= THREADS * IPT keys sorted in one CTA, radix_small_body's scheme on 16-bit
// images: the images sit in shared memory, each pass ranks the real keys with the warp's counters (slots past n are
// neither ranked nor moved), scans the 256 digits and scatters into the other buffer; values follow their keys.
// Shared memory: values [2][tile] (VALS), warp counters [warps][256], scan sums [8], images [2][tile].
constexpr size_t seg16_small_smem_bytes(int threads, int ipt, int vals) {
    return (size_t)2 * threads * ipt * (vals ? 4 : 0) + (size_t)(threads / 32) * kRadixBins * 4 + 32 +
           (size_t)2 * threads * ipt * 2;
}

template <int THREADS, int IPT, int VALS, int SAFE>
__device__ __forceinline__ void seg16_small_body(const uint16_t *in, uint16_t *out, uint32_t n, SignXor16 order,
                                                 const int32_t *vin, int32_t *vout)
{
    static_assert(THREADS >= kRadixBins && THREADS % 32 == 0, "the digit scan needs 256 threads");
    constexpr int kWarps = THREADS / 32;
    constexpr int kTile = THREADS * IPT;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    int32_t  *s_vbuf  = reinterpret_cast<int32_t *>(smem_raw);                         // [2][kTile] if VALS
    uint32_t *s_table = reinterpret_cast<uint32_t *>(s_vbuf + (VALS ? 2 * kTile : 0)); // [kWarps][256]
    uint32_t *s_sums  = s_table + kWarps * kRadixBins;                                 // [8]
    uint16_t *s_buf   = reinterpret_cast<uint16_t *>(s_sums + 8);                      // [2][kTile] images

    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t *wt = s_table + warp * kRadixBins;
    const uint32_t wofs = warp * (32 * IPT) + lane;

    for (uint32_t i = tid; i < n; i += THREADS) s_buf[i] = (uint16_t)image16(in[i], order);
    if constexpr (VALS != 0)
        for (uint32_t i = tid; i < n; i += THREADS) s_vbuf[i] = vin[i];
    __syncthreads();

    int cur = 0;
#pragma unroll 1
    for (int pass = 0; pass < kSeg16Passes; ++pass) {
        const int shift = pass * kRadixBits;
        const uint16_t *src = s_buf + cur * kTile;
        uint16_t *dst = s_buf + (cur ^ 1) * kTile;
        for (int j = lane; j < kRadixBins; j += 32) wt[j] = 0;
        __syncwarp();
        uint32_t img[IPT], rank[IPT];
#pragma unroll
        for (int i = 0; i < IPT; ++i) {
            const bool ok = wofs + i * 32 < n;
            img[i] = ok ? src[wofs + i * 32] : 0u;              // warp-striped: tile order = memory order
            const uint32_t d = (img[i] >> shift) & (kRadixBins - 1);
            if constexpr (SAFE != 0) {
                const uint32_t peers = __match_any_sync(0xffffffffu, ok ? d : kRadixBins);
                const uint32_t leader = __ffs(peers) - 1;
                uint32_t base = 0;
                if (ok && lane == leader) base = atomicAdd(wt + d, (uint32_t)__popc(peers));
                rank[i] = __shfl_sync(0xffffffffu, base, leader) + __popc(peers & lanemask_lt());
            } else {
                rank[i] = ok ? atomicAdd(wt + d, 1u) : 0u;
            }
        }
        __syncthreads();                                      // counts final, src fully read
        if (tid < kRadixBins) {
            uint32_t total = 0;
#pragma unroll
            for (int w = 0; w < kWarps; ++w) total += s_table[w * kRadixBins + tid];
            uint32_t run = scan256(total, s_sums);            // first position of this digit
#pragma unroll
            for (int w = 0; w < kWarps; ++w) {
                const uint32_t c = s_table[w * kRadixBins + tid];
                s_table[w * kRadixBins + tid] = run;
                run += c;
            }
        }
        __syncthreads();                                      // positions final
        const int32_t *vsrc = s_vbuf + cur * kTile;
        int32_t *vdst = s_vbuf + (cur ^ 1) * kTile;
#pragma unroll
        for (int i = 0; i < IPT; ++i) {
            const uint32_t at = wofs + i * 32;
            if (at >= n) continue;
            const uint32_t p = wt[(img[i] >> shift) & (kRadixBins - 1)] + rank[i];
            B200_CHECK_AT(8, p < (uint32_t)kTile);
            dst[p] = (uint16_t)img[i];
            if constexpr (VALS != 0) vdst[p] = vsrc[at];
        }
        __syncthreads();                                      // dst complete; the counters may be cleared
        cur ^= 1;
    }
    const SignXor16 inv = inverse16(order);
    const uint16_t *res = s_buf + cur * kTile;
    for (uint32_t i = tid; i < n; i += THREADS) out[i] = (uint16_t)image16(res[i], inv);
    if constexpr (VALS != 0) {
        const int32_t *vres = s_vbuf + cur * kTile;
        for (uint32_t i = tid; i < n; i += THREADS) vout[i] = vres[i];
    }
}

template <int THREADS, int IPT, int VALS, int SAFE>
__global__ void __launch_bounds__(THREADS)
seg16_small_kernel(const uint16_t *in, uint16_t *out, const int32_t *vin, int32_t *vout, const Seg16Control *ctl,
                   const uint2 *list, uint32_t cap, int c, SignXor16 order)
{
    const uint32_t count = ctl->count[c] < cap ? ctl->count[c] : cap;
    for (uint32_t s = blockIdx.x; s < count; s += gridDim.x) {
        const uint2 seg = list[s];
        seg16_small_body<THREADS, IPT, VALS, SAFE>(in + seg.x, out + seg.x, seg.y - seg.x, order,
                                                   VALS ? vin + seg.x : nullptr, VALS ? vout + seg.x : nullptr);
        __syncthreads();                                       // shared memory free for the next segment
    }
}

static unsigned seg16_grid(size_t want, size_t most) {
    const size_t g = want < most ? want : most;
    return (unsigned)(g < 1 ? 1 : g);
}

template <int THREADS, int IPT, int VALS, int SAFE>
static int launch_small16(const uint16_t *in, uint16_t *out, const int32_t *vin, int32_t *vout, const Seg16Control *ctl,
                          const uint2 *list, size_t cap, int c, SignXor16 order, unsigned per_sm, cudaStream_t s) {
    constexpr size_t smem = seg16_small_smem_bytes(THREADS, IPT, VALS);
    auto *fn = seg16_small_kernel<THREADS, IPT, VALS, SAFE>;
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(fn), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
    fn<<<seg16_grid(cap, (size_t)kNumSMs * per_sm), THREADS, smem, s>>>(in, out, vin, vout, ctl, list, (uint32_t)cap, c,
                                                                         order);
    B200_LAUNCH_CHECK();
    return B200SORT_OK;
}

template <int VALS, int SAFE>
static int seg16_sort_impl(const uint16_t *in, uint16_t *out, uint16_t *tmp, const int32_t *vin, int32_t *vout,
                           int32_t *vtmp, size_t n, const int32_t *offsets, size_t S, void *ws, cudaStream_t s,
                           SignXor16 order) {
    const Seg16Layout L = seg16_layout(n, S);
    auto *base = static_cast<unsigned char *>(ws);
    auto *ctl = reinterpret_cast<Seg16Control *>(base);
    Seg16Lists lists;
    for (int c = 0; c < 4; ++c) {
        lists.list[c] = reinterpret_cast<uint2 *>(base + L.off_list[c]);
        lists.cap[c] = (uint32_t)L.cap[c];
    }
    auto *prefix = reinterpret_cast<uint32_t *>(base + L.off_prefix);
    auto *hist = reinterpret_cast<uint32_t *>(base + L.off_hist);
    uint32_t *status[2] = {reinterpret_cast<uint32_t *>(base + L.off_status),
                           reinterpret_cast<uint32_t *>(base + L.off_status) + L.rows * kRadixBins};
    const uint32_t cap_large = (uint32_t)L.cap[3];

    B200_CUDA_TRY(cudaMemsetAsync(ctl, 0, sizeof(Seg16Control), s));
    seg16_classify_kernel<<<seg16_grid(div_up(S, 256), (size_t)kNumSMs * 8), 256, 0, s>>>(
        in, out, vin, vout, (uint32_t)n, offsets, (uint32_t)S, ctl, lists, hist);
    B200_LAUNCH_CHECK();
    seg16_tile_plan_kernel<<<1, kPlan16Threads, 0, s>>>(ctl, lists.list[3], cap_large, prefix, (uint32_t)L.rows);
    B200_LAUNCH_CHECK();
    seg16_hist_kernel<<<seg16_grid(L.rows, (size_t)kNumSMs * 4), kSeg16Threads, 0, s>>>(in, ctl, lists.list[3], cap_large,
                                                                                      prefix, hist, status[0], order);
    B200_LAUNCH_CHECK();
    constexpr size_t pass_smem = sizeof(Seg16PassSmem<VALS>);
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(seg16_onesweep_kernel<VALS, SAFE>),
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pass_smem));
    for (int pass = 0; pass < kSeg16Passes; ++pass) {
        seg16_onesweep_kernel<VALS, SAFE><<<seg16_grid(L.rows, (size_t)kNumSMs * 2), kSeg16Threads, pass_smem, s>>>(
            in, out, tmp, vin, vout, vtmp, pass, ctl, lists.list[3], cap_large, prefix, hist, status[pass],
            pass + 1 < kSeg16Passes ? status[pass + 1] : nullptr, order);
        B200_LAUNCH_CHECK();
    }
    seg16_warp_kernel<VALS><<<seg16_grid(div_up(L.cap[0], kWarp16KernelThreads / 32), (size_t)kNumSMs * 8),
                              kWarp16KernelThreads, 0, s>>>(in, out, vin, vout, ctl, lists.list[0], lists.cap[0], order);
    B200_LAUNCH_CHECK();
    B200_TRY((launch_small16<kMed16aThreads, kMed16aIpt, VALS, SAFE>(in, out, vin, vout, ctl, lists.list[1], L.cap[1], 1,
                                                                     order, 8, s)));
    B200_TRY((launch_small16<kMed16bThreads, kMed16bIpt, VALS, SAFE>(in, out, vin, vout, ctl, lists.list[2], L.cap[2], 2,
                                                                     order, VALS ? 2 : 4, s)));
    return B200SORT_OK;
}

size_t segmented16_workspace_bytes(size_t n, size_t num_segments) { return seg16_layout(n, num_segments).bytes; }

int segmented16_sort(const uint16_t *d_in, uint16_t *d_out, uint16_t *d_tmp, const int32_t *v_in, int32_t *v_out,
                     int32_t *v_tmp, size_t n, const int32_t *d_offsets, size_t num_segments, void *d_ws,
                     cudaStream_t s, SignXor16 order) {
    if (num_segments == 0) return B200SORT_OK;
    const bool safe = !radix_atomic_order_ok();
    if (v_in == nullptr)
        return safe ? seg16_sort_impl<0, 1>(d_in, d_out, d_tmp, nullptr, nullptr, nullptr, n, d_offsets, num_segments, d_ws, s, order)
                    : seg16_sort_impl<0, 0>(d_in, d_out, d_tmp, nullptr, nullptr, nullptr, n, d_offsets, num_segments, d_ws, s, order);
    return safe ? seg16_sort_impl<1, 1>(d_in, d_out, d_tmp, v_in, v_out, v_tmp, n, d_offsets, num_segments, d_ws, s, order)
                : seg16_sort_impl<1, 0>(d_in, d_out, d_tmp, v_in, v_out, v_tmp, n, d_offsets, num_segments, d_ws, s, order);
}

unsigned long long segmented16_check_failures(unsigned long long *per_site) { return tu_check_failures(per_site); }

}  // namespace b200sort
