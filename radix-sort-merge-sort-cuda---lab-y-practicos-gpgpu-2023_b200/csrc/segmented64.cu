// segmented64.cu -- segmented sort of 64-bit keys: segment i = keys[offsets[i] .. offsets[i+1]) is sorted on its own
// in any order of b200sort_sort_keys64, keys only or with a 32-bit value (stable).  The structure is segmented16.cu's
// (DESIGN section 4.2g) with the 8 digit passes of radix64.cu, and every pass that no segment needs is skipped; every
// call enqueues one memset and the same fifteen kernels whatever the number of segments and the data (DESIGN 4.2h).
//
//   g0  seg64_classify_kernel     clamps every segment to [0, n], routes it by length to a per-class list in the
//                                 workspace (class 0 is copied on the spot), records each large segment's first key
//                                 and zeroes its histograms
//   g1  seg64_tile_plan_kernel    one CTA: prefix of the large segments' tile counts = the global tile list
//   g2  seg64_hist_kernel         the 8 digit histograms of every large segment, privatised per CTA in shared memory,
//                                 and vary = OR of image(k) ^ image(first key of k's segment) over the large segments
//   g3  seg64_onesweep_kernel x8  the stable passes over the tile list, look-back bounded by the segment's first tile;
//                                 pass p runs iff byte p of vary is not zero, and derives its buffers from vary
//   g4  seg64_final_copy_kernel   the large segments' copy to out when the executed passes did not land there
//   g5  seg64_warp_kernel         class 1: a warp per segment
//   g6  seg64_small_kernel x2     classes 2 and 3: a CTA per segment, the passes its own keys need, in shared memory
//
// The onesweep passes and the small-segment CTAs rank with lane-ordered shared-memory atomics like the 1-D kernels,
// behind the same self-test (radix_atomic_order_ok); SAFE = 1 is their ballot-ranked form.  The digit helpers are
// copies of radix64.cu's (digit64, image64, key_of_last_image64), so that radix64.cu's kernels stay as they are.
#include "segmented64.cuh"
#include "radix.cuh"
#include "radix_digit.cuh"

namespace b200sort {

int radix_atomic_order_ok();       // radix.cu: the lane-order self-test's verdict for the current device

constexpr int kSeg64Passes = 8;

size_t segmented64_class_max(int c) {
    switch (c) {
        case 0: return kSeg64Max0;
        case 1: return kSeg64Max1;
        case 2: return kSeg64Max2;
        case 3: return kSeg64Max3;
        default: return 0;
    }
}

constexpr int kSeg64Warps = kSeg64Threads / 32;
constexpr int kWarp64SegMax = (int)kSeg64Max1;                // 128
constexpr int kWarp64SegIpt = kWarp64SegMax / 32;
constexpr int kWarp64KernelThreads = 256;
constexpr int kMed64aThreads = 256, kMed64aIpt = 4;           // class 2: 1024 slots
constexpr int kMed64bThreads = 512, kMed64bIpt = 16;          // class 3: 8192 slots
static_assert(kMed64aThreads * kMed64aIpt == (int)kSeg64Max2 && kMed64bThreads * kMed64bIpt == (int)kSeg64Max3, "");

// Head of the workspace, zeroed by one memset per call.
struct Seg64Control {
    uint32_t count[4];       // segments appended to the lists of classes 1, 2, 3 and 4 (large)
    uint32_t ticket[8];      // tile tickets of the 8 passes
    uint32_t tiles;          // tiles of the global list (g1)
    uint32_t vary[2];        // low and high word of the OR of image(k) ^ image(first key of k's large segment)
    uint32_t pad[1];
};
constexpr size_t kSeg64ControlBytes = 256;

// Worst-case layout from (n, num_segments) alone, as segmented16.cu's.
struct Seg64Layout {
    size_t cap[4];           // list capacities of classes 1..4
    size_t rows;             // status rows: tiles of the global list, at most n / tile + large segments
    size_t off_list[4], off_prefix, off_first, off_hist, off_status, bytes;
};
static Seg64Layout seg64_layout(size_t n, size_t S) {
    Seg64Layout L;
    for (int c = 0; c < 4; ++c) {
        const size_t most = n / (segmented64_class_max(c) + 1);
        L.cap[c] = S < most ? S : most;
    }
    L.rows = n / kSeg64Tile + L.cap[3];
    size_t o = kSeg64ControlBytes;
    for (int c = 0; c < 4; ++c) { L.off_list[c] = o; o = align_up(o + L.cap[c] * sizeof(uint2), 256); }
    L.off_prefix = o; o = align_up(o + (L.cap[3] + 1) * sizeof(uint32_t), 256);
    L.off_first = o;  o = align_up(o + L.cap[3] * sizeof(uint2), 256);
    L.off_hist = o;   o = align_up(o + L.cap[3] * kSeg64Passes * kRadixBins * sizeof(uint32_t), 256);
    L.off_status = o; o += 2 * L.rows * kRadixBins * sizeof(uint32_t);
    L.bytes = o;
    return L;
}

struct Seg64Lists {
    uint2 *list[4];          // {begin, end} of the segments of classes 1..4
    uint32_t cap[4];
};

// ---- digits (copies of radix64.cu's helpers) --------------------------------------------------------------------
__device__ __forceinline__ uint2 seg64_image(uint2 k, SignXor64 o) {
    const uint64_t m = (k.y >> 31) ? o.neg : o.pos;
    return make_uint2(k.x ^ (uint32_t)m, k.y ^ (uint32_t)(m >> 32));
}
__host__ __device__ __forceinline__ uint32_t seg64_half(uint64_t m, int pass) {
    return (uint32_t)(m >> (pass < 4 ? 0 : 32));
}
// The digit of pass p of a key's image; `flips` = flips_of(this pass's bytes of the neg and pos masks).
__device__ __forceinline__ uint32_t seg64_digit(uint2 k, int pass, uint32_t flips) {
    const uint32_t w = pass < 4 ? k.x : k.y;
    return ((w >> ((pass & 3) * kRadixBits)) ^ __byte_perm(flips, 0u, k.y >> 31)) & (kRadixBins - 1);
}
__device__ __forceinline__ uint32_t seg64_flips(SignXor64 o, int pass) {
    return flips_of(seg64_half(o.neg, pass), seg64_half(o.pos, pass), (pass & 3) * kRadixBits);
}
// Byte p of the 64-bit word {lo, hi}: zero iff every key agrees with its segment's first key in digit p.
__device__ __forceinline__ uint32_t seg64_byte(uint32_t lo, uint32_t hi, int pass) {
    return ((pass < 4 ? lo : hi) >> ((pass & 3) * kRadixBits)) & (kRadixBins - 1);
}

// The passes the onesweep class runs: bit p set iff some large segment has two keys that differ in digit p.
__device__ __forceinline__ uint32_t seg64_passes_run(const Seg64Control *ctl) {
    const uint32_t lo = ctl->vary[0], hi = ctl->vary[1];
    uint32_t m = 0;
#pragma unroll
    for (int p = 0; p < kSeg64Passes; ++p) m |= seg64_byte(lo, hi, p) ? 1u << p : 0u;
    return m;
}
// The buffer the j-th of `runs` executed passes writes, radix64.cu's plan: in place, tmp, out, tmp, ... (an odd count
// ends in tmp and needs the final copy); out of place, alternating so that the last one lands in out and the input
// is never written (no executed pass at all copies in -> out).
__device__ __forceinline__ uint32_t seg64_dst_sel(uint32_t j, uint32_t runs, uint32_t in_place) {
    if (in_place) return (j & 1) ? kSelOut : kSelTmp;
    return ((runs - 1 - j) & 1) ? kSelTmp : kSelOut;
}
template <typename T>
__device__ __forceinline__ T *seg64_buf(uint32_t sel, T *in, T *tmp, T *out) {
    return sel == kSelIn ? in : sel == kSelTmp ? tmp : out;
}

// ---- g0 -------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
seg64_classify_kernel(const uint2 *in, uint2 *out, const int32_t *vin, int32_t *vout, uint32_t n,
                      const int32_t *offsets, uint32_t num_segments, Seg64Control *ctl, Seg64Lists lists,
                      uint2 *first, uint32_t *hist)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < num_segments; i += gridDim.x * blockDim.x) {
        const int32_t o0 = offsets[i], o1 = offsets[i + 1];
        const uint32_t b = o0 < 0 ? 0u : ((uint32_t)o0 > n ? n : (uint32_t)o0);
        const uint32_t e = o1 < (int32_t)b ? b : ((uint32_t)o1 > n ? n : (uint32_t)o1);
        const uint32_t len = e - b;
        if (len == 1 && in != out) out[b] = in[b];
        if (len == 1 && vin != nullptr && vin != vout) vout[b] = vin[b];
        // class c - 1; 4 = nothing to sort.  One atomicAdd per class and warp (segmented.cu).
        const int c = len <= kSeg64Max0 ? 4 : len <= kSeg64Max1 ? 0 : len <= kSeg64Max2 ? 1 : len <= kSeg64Max3 ? 2 : 3;
        const uint32_t active = __activemask();
        const uint32_t peers = __match_any_sync(active, c);
        const uint32_t leader = __ffs(peers) - 1;
        uint32_t slot0 = 0;
        if (c < 4 && lane_id() == leader) slot0 = atomicAdd(&ctl->count[c], (uint32_t)__popc(peers));
        const uint32_t slot = __shfl_sync(active, slot0, leader) + __popc(peers & lanemask_lt());
        if (c == 4) continue;
        const uint32_t cap = c == 0 ? lists.cap[0] : c == 1 ? lists.cap[1] : c == 2 ? lists.cap[2] : lists.cap[3];
        uint2 *list = c == 0 ? lists.list[0] : c == 1 ? lists.list[1] : c == 2 ? lists.list[2] : lists.list[3];
        B200_CHECK_AT(15, slot < cap);
        if (slot >= cap) continue;                     // only with overlapping (malformed) segments
        list[slot] = make_uint2(b, e);
        if (c == 3) {
            first[slot] = in[b];                       // read before any pass can overwrite it (in place)
            uint4 *h = reinterpret_cast<uint4 *>(hist + (size_t)slot * kSeg64Passes * kRadixBins);
            for (int w = 0; w < kSeg64Passes * kRadixBins / 4; ++w) h[w] = make_uint4(0, 0, 0, 0);
        }
    }
}

// ---- g1 -------------------------------------------------------------------------------------------------------------
constexpr int kPlan64Threads = 1024;
__global__ void __launch_bounds__(kPlan64Threads)
seg64_tile_plan_kernel(Seg64Control *ctl, const uint2 *large, uint32_t cap, uint32_t *prefix, uint32_t max_tiles)
{
    __shared__ uint32_t s_warp[kPlan64Threads / 32];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t m = ctl->count[3] < cap ? ctl->count[3] : cap;
    const uint32_t per = (m + kPlan64Threads - 1) / kPlan64Threads;
    const uint32_t j0 = tid * per, j1 = (j0 + per < m) ? j0 + per : m;
    uint32_t sum = 0;
    for (uint32_t j = j0; j < j1; ++j) sum += (large[j].y - large[j].x + kSeg64Tile - 1) / kSeg64Tile;
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
        run += (large[j].y - large[j].x + kSeg64Tile - 1) / kSeg64Tile;
    }
    if (tid == kPlan64Threads - 1) {
        prefix[m] = run;
        B200_CHECK_AT(15, run <= max_tiles);
        ctl->tiles = run < max_tiles ? run : max_tiles;
    }
}

// The large segment that holds tile t of the global list: the last j with prefix[j] <= t.
__device__ __forceinline__ uint32_t seg64_of_tile(const uint32_t *prefix, uint32_t m, uint32_t t) {
    uint32_t lo = 0, hi = m;                   // prefix[lo] <= t < prefix[hi]
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (prefix[mid] <= t) lo = mid; else hi = mid;
    }
    return lo;
}

// ---- g2 -------------------------------------------------------------------------------------------------------------
// Each CTA counts a contiguous range of tiles into shared counters and flushes them to a segment's 8 x 256 counts when
// the range moves on to the next segment.  A key is counted in pass p only when its digit p differs from that of its
// segment's first key: the first key's digit gets no count (the pass kernel derives it as length - the others), so
// the digits every key shares, the common case of small ids in int64, cost no atomics on one hot counter.  The same
// XOR, ORed over every key, tells which passes run.  The CTA also zeroes the status rows of the first pass.
__global__ void __launch_bounds__(kSeg64Threads)
seg64_hist_kernel(const uint2 *in, Seg64Control *ctl, const uint2 *large, uint32_t cap, const uint32_t *prefix,
                  const uint2 *first, uint32_t *hist, uint32_t *status0, SignXor64 order)
{
    __shared__ uint32_t s_hist[kSeg64Passes * kRadixBins];
    const uint32_t tid = threadIdx.x;
    const uint32_t m = ctl->count[3] < cap ? ctl->count[3] : cap;
    const uint32_t tiles = ctl->tiles;
    const uint32_t per = (tiles + gridDim.x - 1) / gridDim.x;
    const uint32_t t0 = blockIdx.x * per, t1 = (t0 + per < tiles) ? t0 + per : tiles;
    if (t0 >= t1) return;
    for (uint32_t i = tid; i < kSeg64Passes * kRadixBins; i += kSeg64Threads) s_hist[i] = 0;
    uint32_t j = seg64_of_tile(prefix, m, t0);
    auto flush = [&](uint32_t seg) {
        __syncthreads();
        for (uint32_t i = tid; i < kSeg64Passes * kRadixBins; i += kSeg64Threads) {
            const uint32_t c = s_hist[i];
            if (c) atomicAdd(hist + (size_t)seg * kSeg64Passes * kRadixBins + i, c);
            s_hist[i] = 0;
        }
    };
    uint32_t vary_lo = 0, vary_hi = 0;
    __syncthreads();
    for (uint32_t t = t0; t < t1; ++t) {
        if (t >= prefix[j + 1]) {
            flush(j);
            while (t >= prefix[j + 1]) ++j;
            __syncthreads();
        }
        const uint2 seg = large[j];
        const uint2 ref = seg64_image(first[j], order);
        const uint32_t start = seg.x + (t - prefix[j]) * kSeg64Tile;
        const uint32_t valid = (seg.y - start < kSeg64Tile) ? seg.y - start : kSeg64Tile;
        for (uint32_t i = tid; i < valid; i += kSeg64Threads) {
            const uint2 img = seg64_image(in[start + i], order);
            const uint32_t xlo = img.x ^ ref.x, xhi = img.y ^ ref.y;
            vary_lo |= xlo;
            vary_hi |= xhi;
#pragma unroll
            for (int p = 0; p < kSeg64Passes; ++p)
                if (seg64_byte(xlo, xhi, p)) atomicAdd(&s_hist[p * kRadixBins + seg64_byte(img.x, img.y, p)], 1u);
        }
        if (tid < kRadixBins) status0[(size_t)t * kRadixBins + tid] = 0;
    }
    flush(j);
    vary_lo = __reduce_or_sync(0xffffffffu, vary_lo);
    vary_hi = __reduce_or_sync(0xffffffffu, vary_hi);
    if ((tid & 31) == 0) {
        if (vary_lo) atomicOr(&ctl->vary[0], vary_lo);
        if (vary_hi) atomicOr(&ctl->vary[1], vary_hi);
    }
}

// ---- g3 -------------------------------------------------------------------------------------------------------------
template <int VALS>
struct Seg64PassSmem {
    uint32_t cnt[kSeg64Warps][kRadixBins];   // per-warp digit counts -> the warp's offset inside the digit's run
    uint2 keys[kSeg64Tile];                  // the tile in digit order
    int32_t vals[VALS ? kSeg64Tile : 1];
    uint32_t excl[kRadixBins];               // first tile-local position of each digit
    uint32_t dst[kRadixBins];                // segment-relative destination of tile-local position 0 of each digit
    uint32_t sums[2][8];
    uint32_t info[5];                        // ticket, segment begin, length, tile in segment, large-segment index
};

// One stable pass by digit `pass` over the tile list, as segmented16.cu's seg16_onesweep_kernel: tiles by ticket,
// {flag:2, count:30} status words, look-back over the earlier tiles OF ITS SEGMENT until an inclusive count, and key i
// of digit d goes to
//   segment begin + segment base[d] + (keys of digit d in earlier tiles of the segment) + tile-local rank.
// Slots past the segment's end hold the key whose image is all ones (radix64.cu): digit 255, ranked after every real
// key of the tile, staged at the tile's end and never written; only the last tile of a segment has them, and no tile
// reads its status row.  A pass that no large segment needs only clears the next pass's status rows.
template <int VALS, int SAFE>
__global__ void __launch_bounds__(kSeg64Threads, 2)
seg64_onesweep_kernel(const uint2 *in, uint2 *out, uint2 *tmp, const int32_t *vin, int32_t *vout, int32_t *vtmp,
                      int pass, uint32_t in_place, Seg64Control *ctl, const uint2 *large, uint32_t cap,
                      const uint32_t *prefix, const uint2 *first, const uint32_t *hist, uint32_t *status,
                      uint32_t *status_next, SignXor64 order, uint2 pad_key)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Seg64PassSmem<VALS> &sm = *reinterpret_cast<Seg64PassSmem<VALS> *>(smem_raw);
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t tiles = ctl->tiles;
    const uint32_t run_mask = seg64_passes_run(ctl);
    if (!((run_mask >> pass) & 1u)) {                          // the identity on every large segment
        if (status_next != nullptr)
            for (uint32_t i = blockIdx.x * kSeg64Threads + tid; i < tiles * kRadixBins; i += gridDim.x * kSeg64Threads)
                status_next[i] = 0;
        return;
    }
    const uint32_t runs = __popc(run_mask), jx = __popc(run_mask & ((1u << pass) - 1u));
    const uint32_t src_sel = jx == 0 ? kSelIn : seg64_dst_sel(jx - 1, runs, in_place);
    const uint32_t dst_sel = seg64_dst_sel(jx, runs, in_place);
    const uint2 *src = seg64_buf<const uint2>(src_sel, in, tmp, out);
    uint2 *dst = seg64_buf<uint2>(dst_sel, nullptr, tmp, out);
    const int32_t *vsrc = seg64_buf<const int32_t>(src_sel, vin, vtmp, vout);
    int32_t *vdst = seg64_buf<int32_t>(dst_sel, nullptr, vtmp, vout);
    const uint32_t flips = seg64_flips(order, pass);
    const uint32_t m = ctl->count[3] < cap ? ctl->count[3] : cap;
    uint32_t *wcnt = sm.cnt[warp];
    const uint32_t wofs = warp * (32 * kSeg64Ipt) + lane;

    for (;;) {
        if (tid == 0) {
            const uint32_t t = atomicAdd(&ctl->ticket[pass], 1u);
            sm.info[0] = t;
            if (t < tiles) {
                const uint32_t j = seg64_of_tile(prefix, m, t);
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
        const uint32_t begin = sm.info[1], len = sm.info[2], k = sm.info[3];
        const uint32_t start = k * kSeg64Tile;               // segment-relative
        const uint32_t valid = (len - start < kSeg64Tile) ? len - start : kSeg64Tile;

        uint2 key[kSeg64Ipt];
        int32_t val[VALS ? kSeg64Ipt : 1];
        uint32_t rank[kSeg64Ipt];
#pragma unroll
        for (int i = 0; i < kSeg64Ipt; ++i) {
            const uint32_t at = wofs + i * 32;                // warp-striped: tile order = memory order
            key[i] = at < valid ? src[begin + start + at] : pad_key;
            if constexpr (VALS != 0) val[i] = at < valid ? vsrc[begin + start + at] : 0;
        }
#pragma unroll
        for (int i = 0; i < kSeg64Ipt; ++i) {
            const uint32_t d = seg64_digit(key[i], pass, flips);
            if constexpr (SAFE != 0) {
                const uint32_t peers = __match_any_sync(0xffffffffu, d);
                const uint32_t leader = __ffs(peers) - 1;
                uint32_t base = 0;
                if (lane == leader) base = atomicAdd(wcnt + d, (uint32_t)__popc(peers));
                rank[i] = __shfl_sync(0xffffffffu, base, leader) + __popc(peers & lanemask_lt());
            } else {
                rank[i] = atomicAdd(wcnt + d, 1u);
            }
        }
        __syncthreads();                                       // warp counts final
        if (tid < kRadixBins) {
            const uint32_t j = sm.info[4];
            uint32_t run = 0;
#pragma unroll
            for (int w = 0; w < kSeg64Warps; ++w) {
                const uint32_t c = sm.cnt[w][tid];
                sm.cnt[w][tid] = run;
                run += c;
            }
            uint32_t *row = status + (size_t)t * kRadixBins + tid;
            st_relaxed_gpu(row, (k == 0 ? kFlagIncl : kFlagLocal) | run);
            const uint32_t excl = scan256(run, sm.sums[0]);
            // the segment's counts leave out the digit of its first key: that one is length - the others
            uint32_t seg_base = scan256(hist[(size_t)j * kSeg64Passes * kRadixBins + pass * kRadixBins + tid],
                                        sm.sums[1]);
            uint32_t others = 0;
#pragma unroll
            for (int w = 0; w < kRadixBins / 32; ++w) others += sm.sums[1][w];
            if (tid > seg64_digit(first[j], pass, flips)) seg_base += len - others;
            uint32_t before = 0;                               // keys of this digit in the segment's earlier tiles
            if (k > 0) {
                for (const uint32_t *p = row - kRadixBins;; p -= kRadixBins) {
                    uint32_t w;
                    do { w = ld_relaxed_gpu(p); } while ((w & ~kValueMask) == 0);
                    before += w & kValueMask;
                    if (w & kFlagIncl) break;                  // the segment's first tile is always inclusive
                }
                // reaches 2^30 only when one digit holds all of a 2^30-key segment, a pass that is skipped
                st_relaxed_gpu(row, kFlagIncl | ((before + run) & kValueMask));
            }
            sm.excl[tid] = excl;
            sm.dst[tid] = seg_base + before - excl;
            if (status_next != nullptr) status_next[(size_t)t * kRadixBins + tid] = 0;
        }
        __syncthreads();                                       // offsets final
#pragma unroll
        for (int i = 0; i < kSeg64Ipt; ++i) {
            const uint32_t d = seg64_digit(key[i], pass, flips);
            const uint32_t at = sm.excl[d] + wcnt[d] + rank[i];
            B200_CHECK_AT(1, at < kSeg64Tile);
            if (at < kSeg64Tile) {
                sm.keys[at] = key[i];
                if constexpr (VALS != 0) sm.vals[at] = val[i];
            }
        }
        __syncthreads();                                       // the tile is staged in digit order
        for (uint32_t i = tid; i < valid; i += kSeg64Threads) {
            const uint2 kk = sm.keys[i];
            const uint32_t pos = sm.dst[seg64_digit(kk, pass, flips)] + i;
            B200_CHECK_AT(15, pos < len);
            if (pos < len) {                                   // only malformed offsets fail this
                dst[begin + pos] = kk;
                if constexpr (VALS != 0) vdst[begin + pos] = sm.vals[i];
            }
        }
        __syncthreads();                                       // shared memory free for the next tile
    }
}

// ---- g4 -------------------------------------------------------------------------------------------------------------
// The large segments' copy to out: in place after an odd number of executed passes (the result is in tmp), out of
// place when no pass ran (the input is the result).  The other classes write out themselves.
__global__ void __launch_bounds__(256)
seg64_final_copy_kernel(const uint2 *in, uint2 *out, const uint2 *tmp, const int32_t *vin, int32_t *vout,
                        const int32_t *vtmp, uint32_t in_place, const Seg64Control *ctl, const uint2 *large,
                        uint32_t cap, const uint32_t *prefix)
{
    const uint32_t runs = __popc(seg64_passes_run(ctl));
    const uint32_t sel = in_place ? ((runs & 1) ? kSelTmp : 0u) : (runs == 0 ? kSelIn : 0u);
    if (sel == 0) return;
    const uint2 *src = sel == kSelIn ? in : tmp;
    const int32_t *vsrc = sel == kSelIn ? vin : vtmp;
    const uint32_t m = ctl->count[3] < cap ? ctl->count[3] : cap;
    const uint32_t tiles = ctl->tiles;
    for (uint32_t t = blockIdx.x; t < tiles; t += gridDim.x) {
        const uint32_t j = seg64_of_tile(prefix, m, t);
        const uint2 seg = large[j];
        const uint32_t start = seg.x + (t - prefix[j]) * kSeg64Tile;
        const uint32_t valid = (seg.y - start < kSeg64Tile) ? seg.y - start : kSeg64Tile;
        for (uint32_t i = threadIdx.x; i < valid; i += blockDim.x) {
            out[start + i] = src[start + i];
            if (vsrc != nullptr) vout[start + i] = vsrc[start + i];
        }
    }
}

// ---- g5 -------------------------------------------------------------------------------------------------------------
// Class 1: a warp per segment of 2..128 keys.  The rank of a key is the number of keys before it in (image, position)
// order, counted against the segment's 64-bit images in shared memory: stable, no atomics, no padding.
template <int VALS>
__global__ void __launch_bounds__(kWarp64KernelThreads)
seg64_warp_kernel(const uint2 *in, uint2 *out, const int32_t *vin, int32_t *vout, const Seg64Control *ctl,
                  const uint2 *list, uint32_t cap, SignXor64 order)
{
    __shared__ unsigned long long s_img[kWarp64KernelThreads / 32][kWarp64SegMax];
    const uint32_t lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint32_t count = ctl->count[0] < cap ? ctl->count[0] : cap;
    unsigned long long *img_s = s_img[wib];
    for (uint32_t s = blockIdx.x * (kWarp64KernelThreads / 32) + wib; s < count;
         s += gridDim.x * (kWarp64KernelThreads / 32)) {
        const uint2 seg = list[s];
        const uint32_t len = seg.y - seg.x;
        uint2 key[kWarp64SegIpt];
        unsigned long long img[kWarp64SegIpt];
        uint32_t pos[kWarp64SegIpt];
        int32_t val[kWarp64SegIpt];
#pragma unroll
        for (int q = 0; q < kWarp64SegIpt; ++q) {
            const uint32_t i = lane + 32 * q;
            key[q] = i < len ? in[seg.x + i] : make_uint2(0, 0);
            if constexpr (VALS != 0) val[q] = i < len ? vin[seg.x + i] : 0;
            const uint2 m = seg64_image(key[q], order);
            img[q] = ((unsigned long long)m.y << 32) | m.x;
            pos[q] = 0;
            if (i < len) img_s[i] = img[q];
        }
        __syncwarp();                                          // every key read before any is written
        for (uint32_t i = 0; i < len; ++i) {
            const unsigned long long v = img_s[i];
#pragma unroll
            for (int q = 0; q < kWarp64SegIpt; ++q) pos[q] += (v < img[q]) | ((v == img[q]) & (i < lane + 32 * q));
        }
#pragma unroll
        for (int q = 0; q < kWarp64SegIpt; ++q) {
            if (lane + 32 * q < len) {
                B200_CHECK_AT(15, pos[q] < len);
                out[seg.x + pos[q]] = key[q];
                if constexpr (VALS != 0) vout[seg.x + pos[q]] = val[q];
            }
        }
        __syncwarp();                                          // img_s free for the warp's next segment
    }
}

// ---- g6 -------------------------------------------------------------------------------------------------------------
// Classes 2 and 3: one segment of n <= THREADS * IPT keys sorted in one CTA, seg16_small_body's scheme on 64-bit keys:
// the keys sit in shared memory, and the CTA ORs image(k) ^ image(first key) over them; each pass whose byte of that
// OR is not zero ranks the real keys with the warp's counters (slots past n are neither ranked nor moved), scans the
// 256 digits and scatters into the other buffer, values following their keys; the other passes are no swap at all.
// Shared memory: keys [2][tile], values [2][tile] (VALS), warp counters [warps][256], scan sums [8], warp ORs [warps].
constexpr size_t seg64_small_smem_bytes(int threads, int ipt, int vals) {
    return (size_t)2 * threads * ipt * 8 + (size_t)2 * threads * ipt * (vals ? 4 : 0) +
           (size_t)(threads / 32) * kRadixBins * 4 + 32 + (size_t)(threads / 32) * 8;
}

template <int THREADS, int IPT, int VALS, int SAFE>
__device__ __forceinline__ void seg64_small_body(const uint2 *in, uint2 *out, uint32_t n, SignXor64 order,
                                                 const int32_t *vin, int32_t *vout)
{
    static_assert(THREADS >= kRadixBins && THREADS % 32 == 0, "the digit scan needs 256 threads");
    constexpr int kWarps = THREADS / 32;
    constexpr int kTile = THREADS * IPT;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint2    *s_buf   = reinterpret_cast<uint2 *>(smem_raw);                             // [2][kTile] keys
    int32_t  *s_vbuf  = reinterpret_cast<int32_t *>(s_buf + 2 * kTile);                  // [2][kTile] if VALS
    uint32_t *s_table = reinterpret_cast<uint32_t *>(s_vbuf + (VALS ? 2 * kTile : 0));   // [kWarps][256]
    uint32_t *s_sums  = s_table + kWarps * kRadixBins;                                   // [8]
    uint2    *s_vary  = reinterpret_cast<uint2 *>(s_sums + 8);                           // [kWarps]

    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t *wt = s_table + warp * kRadixBins;
    const uint32_t wofs = warp * (32 * IPT) + lane;

    const uint2 ref = seg64_image(in[0], order);
    uint32_t vary_lo = 0, vary_hi = 0;
    for (uint32_t i = tid; i < n; i += THREADS) {
        const uint2 k = in[i];
        const uint2 img = seg64_image(k, order);
        vary_lo |= img.x ^ ref.x;
        vary_hi |= img.y ^ ref.y;
        s_buf[i] = k;
    }
    if constexpr (VALS != 0)
        for (uint32_t i = tid; i < n; i += THREADS) s_vbuf[i] = vin[i];
    vary_lo = __reduce_or_sync(0xffffffffu, vary_lo);
    vary_hi = __reduce_or_sync(0xffffffffu, vary_hi);
    if (lane == 0) s_vary[warp] = make_uint2(vary_lo, vary_hi);
    __syncthreads();
#pragma unroll
    for (int w = 0; w < kWarps; ++w) { vary_lo |= s_vary[w].x; vary_hi |= s_vary[w].y; }

    int cur = 0;
#pragma unroll 1
    for (int pass = 0; pass < kSeg64Passes; ++pass) {
        if (seg64_byte(vary_lo, vary_hi, pass) == 0) continue;   // every key of the segment has the same digit
        const uint32_t flips = seg64_flips(order, pass);
        const uint2 *src = s_buf + cur * kTile;
        uint2 *dst = s_buf + (cur ^ 1) * kTile;
        for (int j = lane; j < kRadixBins; j += 32) wt[j] = 0;
        __syncwarp();
        uint2 key[IPT];
        uint32_t rank[IPT];
#pragma unroll
        for (int i = 0; i < IPT; ++i) {
            const bool ok = wofs + i * 32 < n;
            key[i] = ok ? src[wofs + i * 32] : make_uint2(0, 0);  // warp-striped: tile order = memory order
            const uint32_t d = seg64_digit(key[i], pass, flips);
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
            const uint32_t p = wt[seg64_digit(key[i], pass, flips)] + rank[i];
            B200_CHECK_AT(8, p < (uint32_t)kTile);
            dst[p] = key[i];
            if constexpr (VALS != 0) vdst[p] = vsrc[at];
        }
        __syncthreads();                                      // dst complete; the counters may be cleared
        cur ^= 1;
    }
    const uint2 *res = s_buf + cur * kTile;
    for (uint32_t i = tid; i < n; i += THREADS) out[i] = res[i];
    if constexpr (VALS != 0) {
        const int32_t *vres = s_vbuf + cur * kTile;
        for (uint32_t i = tid; i < n; i += THREADS) vout[i] = vres[i];
    }
}

template <int THREADS, int IPT, int VALS, int SAFE>
__global__ void __launch_bounds__(THREADS)
seg64_small_kernel(const uint2 *in, uint2 *out, const int32_t *vin, int32_t *vout, const Seg64Control *ctl,
                   const uint2 *list, uint32_t cap, int c, SignXor64 order)
{
    const uint32_t count = ctl->count[c] < cap ? ctl->count[c] : cap;
    for (uint32_t s = blockIdx.x; s < count; s += gridDim.x) {
        const uint2 seg = list[s];
        seg64_small_body<THREADS, IPT, VALS, SAFE>(in + seg.x, out + seg.x, seg.y - seg.x, order,
                                                   VALS ? vin + seg.x : nullptr, VALS ? vout + seg.x : nullptr);
        __syncthreads();                                       // shared memory free for the next segment
    }
}

// ---- host side -------------------------------------------------------------------------------------------------------
static unsigned seg64_grid(size_t want, size_t most) {
    const size_t g = want < most ? want : most;
    return (unsigned)(g < 1 ? 1 : g);
}

// The key whose image is all ones: last in every order, digit 255 in every pass (radix64.cu's key_of_last_image64).
static uint2 seg64_pad_key(SignXor64 o) {
    const uint64_t a = ~0ull ^ o.neg, b = ~0ull ^ o.pos;
    const uint64_t k = (a >> 63) ? a : b;                 // whichever of the two maps back through its own mask
    return make_uint2((uint32_t)k, (uint32_t)(k >> 32));
}

template <int THREADS, int IPT, int VALS, int SAFE>
static int launch_small64(const uint2 *in, uint2 *out, const int32_t *vin, int32_t *vout, const Seg64Control *ctl,
                          const uint2 *list, size_t cap, int c, SignXor64 order, unsigned per_sm, cudaStream_t s) {
    constexpr size_t smem = seg64_small_smem_bytes(THREADS, IPT, VALS);
    auto *fn = seg64_small_kernel<THREADS, IPT, VALS, SAFE>;
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(fn), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
    fn<<<seg64_grid(cap, (size_t)kNumSMs * per_sm), THREADS, smem, s>>>(in, out, vin, vout, ctl, list, (uint32_t)cap, c,
                                                                         order);
    B200_LAUNCH_CHECK();
    return B200SORT_OK;
}

template <int VALS, int SAFE>
static int seg64_sort_impl(const uint2 *in, uint2 *out, uint2 *tmp, const int32_t *vin, int32_t *vout, int32_t *vtmp,
                           size_t n, const int32_t *offsets, size_t S, void *ws, cudaStream_t s, SignXor64 order) {
    const Seg64Layout L = seg64_layout(n, S);
    auto *base = static_cast<unsigned char *>(ws);
    auto *ctl = reinterpret_cast<Seg64Control *>(base);
    Seg64Lists lists;
    for (int c = 0; c < 4; ++c) {
        lists.list[c] = reinterpret_cast<uint2 *>(base + L.off_list[c]);
        lists.cap[c] = (uint32_t)L.cap[c];
    }
    auto *prefix = reinterpret_cast<uint32_t *>(base + L.off_prefix);
    auto *first = reinterpret_cast<uint2 *>(base + L.off_first);
    auto *hist = reinterpret_cast<uint32_t *>(base + L.off_hist);
    uint32_t *status[2] = {reinterpret_cast<uint32_t *>(base + L.off_status),
                           reinterpret_cast<uint32_t *>(base + L.off_status) + L.rows * kRadixBins};
    const uint32_t cap_large = (uint32_t)L.cap[3];
    const uint32_t in_place = in == out ? 1u : 0u;

    B200_CUDA_TRY(cudaMemsetAsync(ctl, 0, sizeof(Seg64Control), s));
    seg64_classify_kernel<<<seg64_grid(div_up(S, 256), (size_t)kNumSMs * 8), 256, 0, s>>>(
        in, out, vin, vout, (uint32_t)n, offsets, (uint32_t)S, ctl, lists, first, hist);
    B200_LAUNCH_CHECK();
    seg64_tile_plan_kernel<<<1, kPlan64Threads, 0, s>>>(ctl, lists.list[3], cap_large, prefix, (uint32_t)L.rows);
    B200_LAUNCH_CHECK();
    seg64_hist_kernel<<<seg64_grid(L.rows, (size_t)kNumSMs * 4), kSeg64Threads, 0, s>>>(
        in, ctl, lists.list[3], cap_large, prefix, first, hist, status[0], order);
    B200_LAUNCH_CHECK();
    constexpr size_t pass_smem = sizeof(Seg64PassSmem<VALS>);
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(seg64_onesweep_kernel<VALS, SAFE>),
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pass_smem));
    const uint2 pad = seg64_pad_key(order);
    for (int pass = 0; pass < kSeg64Passes; ++pass) {
        seg64_onesweep_kernel<VALS, SAFE><<<seg64_grid(L.rows, (size_t)kNumSMs * 2), kSeg64Threads, pass_smem, s>>>(
            in, out, tmp, vin, vout, vtmp, pass, in_place, ctl, lists.list[3], cap_large, prefix, first, hist,
            status[pass & 1], pass + 1 < kSeg64Passes ? status[(pass + 1) & 1] : nullptr, order, pad);
        B200_LAUNCH_CHECK();
    }
    seg64_final_copy_kernel<<<seg64_grid(L.rows, (size_t)kNumSMs * 8), 256, 0, s>>>(
        in, out, tmp, vin, vout, vtmp, in_place, ctl, lists.list[3], cap_large, prefix);
    B200_LAUNCH_CHECK();
    seg64_warp_kernel<VALS><<<seg64_grid(div_up(L.cap[0], kWarp64KernelThreads / 32), (size_t)kNumSMs * 8),
                              kWarp64KernelThreads, 0, s>>>(in, out, vin, vout, ctl, lists.list[0], lists.cap[0], order);
    B200_LAUNCH_CHECK();
    B200_TRY((launch_small64<kMed64aThreads, kMed64aIpt, VALS, SAFE>(in, out, vin, vout, ctl, lists.list[1], L.cap[1], 1,
                                                                     order, 8, s)));
    B200_TRY((launch_small64<kMed64bThreads, kMed64bIpt, VALS, SAFE>(in, out, vin, vout, ctl, lists.list[2], L.cap[2], 2,
                                                                     order, 1, s)));
    return B200SORT_OK;
}

size_t segmented64_workspace_bytes(size_t n, size_t num_segments) { return seg64_layout(n, num_segments).bytes; }

int segmented64_sort(const uint64_t *d_in, uint64_t *d_out, uint64_t *d_tmp, const int32_t *v_in, int32_t *v_out,
                     int32_t *v_tmp, size_t n, const int32_t *d_offsets, size_t num_segments, void *d_ws,
                     cudaStream_t s, SignXor64 order) {
    if (num_segments == 0) return B200SORT_OK;
    const bool safe = !radix_atomic_order_ok();
    const auto *in = reinterpret_cast<const uint2 *>(d_in);
    auto *out = reinterpret_cast<uint2 *>(d_out);
    auto *tmp = reinterpret_cast<uint2 *>(d_tmp);
    if (v_in == nullptr)
        return safe ? seg64_sort_impl<0, 1>(in, out, tmp, nullptr, nullptr, nullptr, n, d_offsets, num_segments, d_ws, s, order)
                    : seg64_sort_impl<0, 0>(in, out, tmp, nullptr, nullptr, nullptr, n, d_offsets, num_segments, d_ws, s, order);
    return safe ? seg64_sort_impl<1, 1>(in, out, tmp, v_in, v_out, v_tmp, n, d_offsets, num_segments, d_ws, s, order)
                : seg64_sort_impl<1, 0>(in, out, tmp, v_in, v_out, v_tmp, n, d_offsets, num_segments, d_ws, s, order);
}

unsigned long long segmented64_check_failures(unsigned long long *per_site) { return tu_check_failures(per_site); }

}  // namespace b200sort
