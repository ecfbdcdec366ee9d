// radix16.cu -- sorts of 16-bit keys (int16, uint16, float16, bfloat16; ascending or descending), DESIGN section 4.2f.
// A key has only 65536 bit patterns, and a keys-only sort's output is fixed by how often each pattern occurs, so
// keys are sorted by counting; key-value pairs need a stable scatter and take two radix passes of 8-bit digits.
//
//   r0  radix16_histogram_kernel<RUNS>  one read of the keys counts the 65536 images in packed 16-bit shared
//                                       counters (128 KiB) and writes one row of 65536 counts per CTA
//   r1  radix16_scan_kernel             one thread per image sums the rows and scans the counts in image order
//                                       (256 blocks of 256 images: block h holds the images of high byte h); its
//                                       last block writes the two passes' digit bases, the skip flags and the plan
//   keys only:
//   r2  radix16_fill_kernel             writes every pattern `count` times in image order, 16-byte stores; tiles
//                                       are output positions, so one pattern holding every key costs nothing extra
//   pairs:
//   r3  radix16_onesweep_kernel x2      the 64-bit sort's stable onesweep pass (radix64.cu) on 2-byte keys and
//                                       8192-key tiles: the low byte of the image, then the high byte
//   r4  radix16_final_copy_kernel       tmp -> out (or in -> out) when the plan did not land in out
//   with indices (DESIGN section 4.2j): r3 as radix16_onesweep_indices_kernel, whose values are made by the first
//   executed pass and stored as int64 by the last; r4 as radix16_final_indices_kernel, which also writes 0..n-1 when
//   both passes were skipped
//
// A call enqueues one memset and the same kernels whatever n (>= 2) and the data (3 for keys, 5 for pairs or indices),
// and the host never reads what the device computes: the sort is stream-ordered and can be captured in a CUDA graph.
#include "radix16.cuh"
#include "radix.cuh"
#include "radix_digit.cuh"

#include <stdlib.h>

namespace b200sort {

int radix_atomic_order_ok();       // radix.cu: the lane-order self-test's verdict for the current device
int radix_skip_enabled();          // radix.cu: b200sort_radix_set_skip

constexpr uint32_t kImages16 = 1u << 16;
constexpr uint32_t kScan16Blocks = kImages16 / kRadixBins;   // 256

// Head of the workspace.  The first kR16ZeroBytes are zeroed by one memset per call; the rest is written before it
// is read.  The per-CTA count rows and the status rows of the passes follow.
struct R16Control {
    uint32_t over[kImages16];                 // repairs of wrapped 16-bit shared counters, mod 2^32 (global atomics)
    uint32_t hist_lo[kRadixBins];             // pass 0 digit counts: low byte of the image (global atomics)
    uint32_t ticket[2];                       // tile tickets of each pass
    uint32_t scan_blocks_done;                // last-block detection in the scan kernel
    uint32_t pad0[5];
    // ---- not zeroed ----
    uint32_t incl[kImages16];                 // inclusive scan of the counts inside each block of 256 images
    uint32_t hist_hi[kScan16Blocks];          // pass 1 digit counts: keys per high byte of the image
    uint32_t base[2][kRadixBins];             // exclusive scans of hist_lo, hist_hi; base[1][h] + incl[j] = end of j
    uint32_t skip[2];                         // 1 = one digit value holds every key: the pass is the identity
    uint32_t src_sel[2];                      // buffer pass p reads : kSelIn / kSelTmp / kSelOut
    uint32_t dst_sel[2];                      // buffer pass p writes: kSelTmp / kSelOut
    uint32_t final_copy;                      // 0 none, else copy from that kSel* buffer to out
};
constexpr size_t kR16ZeroBytes = offsetof(R16Control, incl);
constexpr size_t kR16ControlBytes = (sizeof(R16Control) + 255) / 256 * 256;

// ---- r0 -------------------------------------------------------------------------------------------------------------
// 65536 32-bit counters would need 256 KiB, more than a CTA can have.  Image j counts in half (j & 1) of shared word
// j >> 1.  A counter that wraps past 0xFFFF is repaired in ctl->over from the atomic's return value: +65536 for the
// image, and when the low half wrapped, -1 for the neighbour that received its carry (+65536 more if that carry
// wrapped the neighbour too).  Every wrap is seen by exactly the one atomic that caused it, so the row plus `over`
// is exact.  RUNS = 1 adds a run of equal images among a thread's 8 keys with one atomic (sorted and constant inputs
// otherwise put 32 lanes on one address); RUNS = 0 adds every key on its own.
constexpr int kH16Threads = 1024;
constexpr int kH16Unroll = 4;                               // 128-bit loads (8 keys each) in flight per thread
constexpr size_t kH16SmemBytes = kImages16 * 2;             // 128 KiB

__device__ __forceinline__ void h16_add(uint32_t *sh, uint32_t img, uint32_t run, R16Control *ctl) {
    const uint32_t s = (img & 1) * 16, inc = run << s;
    const uint32_t old = atomicAdd(sh + (img >> 1), inc);
    if (((old >> s) & 0xffffu) + run > 0xffffu) {
        atomicAdd(&ctl->over[img], 65536u);
        if (s == 0) {
            atomicAdd(&ctl->over[img ^ 1], 0xffffffffu);
            if (old > 0xffffffffu - inc) atomicAdd(&ctl->over[img ^ 1], 65536u);
        }
    }
}

template <int RUNS>
__device__ __forceinline__ void h16_add8(uint32_t *sh, uint4 w, SignXor16 o, R16Control *ctl) {
    const uint32_t img[8] = {image16(w.x & 0xffffu, o), image16(w.x >> 16, o), image16(w.y & 0xffffu, o),
                             image16(w.y >> 16, o),     image16(w.z & 0xffffu, o), image16(w.z >> 16, o),
                             image16(w.w & 0xffffu, o), image16(w.w >> 16, o)};
    if constexpr (RUNS != 0) {
        uint32_t run = 1;
#pragma unroll
        for (int i = 0; i < 7; ++i) {
            if (img[i + 1] == img[i]) { ++run; }
            else { h16_add(sh, img[i], run, ctl); run = 1; }
        }
        h16_add(sh, img[7], run, ctl);
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) h16_add(sh, img[i], 1, ctl);
    }
}

template <int RUNS>
__global__ void __launch_bounds__(kH16Threads, 1)
radix16_histogram_kernel(const uint16_t *__restrict__ keys, uint32_t n, uint32_t *part, R16Control *ctl,
                         uint32_t *status_to_zero, size_t status_words, SignXor16 order)
{
    extern __shared__ __align__(16) uint32_t sh[];
    const uint32_t tid = threadIdx.x;
    for (uint32_t i = tid; i < kImages16 / 8; i += kH16Threads) reinterpret_cast<uint4 *>(sh)[i] = make_uint4(0, 0, 0, 0);
    {   // the status rows of the first pass (pairs)
        uint4 *z = reinterpret_cast<uint4 *>(status_to_zero);
        for (size_t i = (size_t)blockIdx.x * kH16Threads + tid; i < status_words / 4; i += (size_t)gridDim.x * kH16Threads)
            z[i] = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();

    // keys are 2-byte aligned: up to 7 keys before the first 16-byte boundary, up to 7 after the last
    const uint32_t to_line = ((16u - (uint32_t)(reinterpret_cast<uintptr_t>(keys) & 15)) & 15u) >> 1;
    const uint32_t head = to_line < n ? to_line : n;
    const uint32_t nvec = (n - head) >> 3;
    const uint4 *v = reinterpret_cast<const uint4 *>(keys + head);
    constexpr uint32_t kChunk = kH16Threads * kH16Unroll;
    for (uint32_t base = blockIdx.x * kChunk; base < nvec; base += gridDim.x * kChunk) {
        uint4 r[kH16Unroll];
        bool ok[kH16Unroll];
#pragma unroll
        for (int u = 0; u < kH16Unroll; ++u) {
            const uint32_t idx = base + u * kH16Threads + tid;
            ok[u] = idx < nvec;
            if (ok[u]) r[u] = __ldcs(v + idx);
        }
#pragma unroll
        for (int u = 0; u < kH16Unroll; ++u)
            if (ok[u]) h16_add8<RUNS>(sh, r[u], order, ctl);
    }
    if (blockIdx.x == 0) {
        const uint32_t tail = head + nvec * 8;
        if (tid < head) h16_add(sh, image16(keys[tid], order), 1, ctl);
        else if (tid >= 8 && tid - 8 < n - tail) h16_add(sh, image16(keys[tail + tid - 8], order), 1, ctl);
    }
    __syncthreads();
    uint4 *row = reinterpret_cast<uint4 *>(part + (size_t)blockIdx.x * kImages16);
    for (uint32_t i = tid; i < kImages16 / 4; i += kH16Threads) {
        const uint2 w = reinterpret_cast<const uint2 *>(sh)[i];
        row[i] = make_uint4(w.x & 0xffffu, w.x >> 16, w.y & 0xffffu, w.y >> 16);
    }
}

// ---- r1 -------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kRadixBins)
radix16_scan_kernel(const uint32_t *part, uint32_t rows, uint32_t n, R16Control *ctl, uint32_t skip_enabled,
                    uint32_t in_place)
{
    __shared__ uint32_t s_sums[2][8];
    __shared__ uint32_t s_skip[2];
    __shared__ uint32_t s_is_last;
    const uint32_t tid = threadIdx.x, img = blockIdx.x * kRadixBins + tid;
    uint32_t c = ctl->over[img];
#pragma unroll 8
    for (uint32_t r = 0; r < rows; ++r) c += __ldcs(part + (size_t)r * kImages16 + img);
    const uint32_t incl = scan256(c, s_sums[0]) + c;
    ctl->incl[img] = incl;
    if (c) atomicAdd(&ctl->hist_lo[tid], c);
    if (tid == kRadixBins - 1) ctl->hist_hi[blockIdx.x] = incl;

    // the last block to finish: digit bases, skippable passes, the buffer plan
    __threadfence();
    __syncthreads();
    if (tid == 0) s_is_last = (atomicAdd(&ctl->scan_blocks_done, 1u) == gridDim.x - 1) ? 1u : 0u;
    if (tid < 2) s_skip[tid] = 0;
    __syncthreads();
    if (!s_is_last) return;
    __threadfence();
    const uint32_t lo = __ldcg(&ctl->hist_lo[tid]), hi = __ldcg(&ctl->hist_hi[tid]);
    ctl->base[0][tid] = scan256(lo, s_sums[0]);
    ctl->base[1][tid] = scan256(hi, s_sums[1]);
    if (skip_enabled && lo == n) s_skip[0] = 1;
    if (skip_enabled && hi == n) s_skip[1] = 1;
    __syncthreads();
    // radix64.cu's plan with two passes: executed pass j reads what executed pass j-1 wrote (the input for j = 0).
    // In place, writes alternate tmp, out; one executed pass leaves the result in tmp for the final copy.  Out of
    // place, the last executed pass lands in out and the input is never written; no executed pass copies in -> out.
    if (tid == 0) {
        const uint32_t executed = (s_skip[0] ? 0u : 1u) + (s_skip[1] ? 0u : 1u);
        uint32_t j = 0, cur = kSelIn;
        for (int p = 0; p < 2; ++p) {
            ctl->skip[p] = s_skip[p];
            ctl->src_sel[p] = cur;
            uint32_t dst = cur;
            if (!s_skip[p]) {
                if (in_place) dst = (j % 2 == 0) ? kSelTmp : kSelOut;
                else          dst = ((executed - 1 - j) % 2 == 0) ? kSelOut : kSelTmp;
                ++j;
                cur = dst;
            }
            ctl->dst_sel[p] = dst;
        }
        uint32_t final_copy = 0;
        if (in_place) { if (cur == kSelTmp) final_copy = kSelTmp; }
        else          { if (executed == 0) final_copy = kSelIn; }
        ctl->final_copy = final_copy;
    }
}

// Image j fills output positions [start16(j), end16(j)).
__device__ __forceinline__ uint32_t end16(const R16Control *ctl, uint32_t j) {
    return ctl->base[1][j >> 8] + ctl->incl[j];
}
__device__ __forceinline__ uint32_t start16(const R16Control *ctl, uint32_t j) {
    return (j & (kRadixBins - 1)) ? end16(ctl, j - 1) : ctl->base[1][j >> 8];
}

// ---- r2 -------------------------------------------------------------------------------------------------------------
// Output position p sits at line position p + off, where off is the output's key offset from a 16-byte boundary;
// tile t is line positions [t * kF16Tile, (t + 1) * kF16Tile).  The CTA finds the images of its first and last
// position (two rounds of loads: the 256 block ends, then the 256 image ends of the block), marks in shared memory
// the first position of every non-empty image between them, and a running maximum over the tile gives each position
// its image.  The work per tile is its positions plus the empty images it passes, at most 65536 over all tiles.
constexpr int kF16Threads = 512;
constexpr int kF16Rounds = 2;
constexpr uint32_t kF16Tile = kF16Threads * 8 * kF16Rounds;   // 8192 positions

__global__ void __launch_bounds__(kF16Threads)
radix16_fill_kernel(uint16_t *out, uint32_t n, const R16Control *ctl, SignXor16 inv)
{
    __shared__ __align__(16) uint16_t s_mark[kF16Tile];    // image whose run starts here, else 0
    __shared__ uint32_t s_warp[kF16Threads / 32];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int r = 0; r < kF16Rounds; ++r) reinterpret_cast<uint4 *>(s_mark)[r * kF16Threads + tid] = make_uint4(0, 0, 0, 0);
    const uint32_t off = (uint32_t)(reinterpret_cast<uintptr_t>(out) & 15) >> 1;
    uint16_t *const line = out - off;
    const uint32_t v0 = blockIdx.x * kF16Tile;
    const uint32_t first = v0 > off ? v0 - off : 0;
    const uint32_t last = (v0 + kF16Tile < off + n ? v0 + kF16Tile : off + n) - off - 1;

    // the image of p is the number of images that end at or before p: threads 0..255 find it for `first`,
    // threads 256..511 for `last`, one byte at a time
    const uint32_t h = tid & (kRadixBins - 1);
    const uint32_t block_end = h + 1 < kRadixBins ? ctl->base[1][h + 1] : n;
    const uint32_t hf = __syncthreads_count(tid < kRadixBins && block_end <= first);
    const uint32_t hl = __syncthreads_count(tid >= kRadixBins && block_end <= last);
    const uint32_t hp = tid < kRadixBins ? hf : hl;
    const uint32_t e = ctl->base[1][hp] + ctl->incl[hp * kRadixBins + h];
    const uint32_t j_first = hf * kRadixBins + __syncthreads_count(tid < kRadixBins && e <= first);
    const uint32_t j_last = hl * kRadixBins + __syncthreads_count(tid >= kRadixBins && e <= last);

    for (uint32_t j = j_first + 1 + tid; j <= j_last; j += kF16Threads) {
        const uint32_t s = start16(ctl, j);
        if (end16(ctl, j) > s) {
            const uint32_t at = s + off - v0;
            B200_CHECK_AT(1, at < kF16Tile);
            if (at < kF16Tile) s_mark[at] = (uint16_t)j;
        }
    }
    __syncthreads();

    uint32_t carry = j_first;
#pragma unroll
    for (int r = 0; r < kF16Rounds; ++r) {
        const uint32_t c = r * kF16Threads + tid;               // this thread's 8 line positions
        const uint4 mk = reinterpret_cast<const uint4 *>(s_mark)[c];
        uint32_t m[8] = {mk.x & 0xffffu, mk.x >> 16, mk.y & 0xffffu, mk.y >> 16,
                         mk.z & 0xffffu, mk.z >> 16, mk.w & 0xffffu, mk.w >> 16};
#pragma unroll
        for (int i = 1; i < 8; ++i) m[i] = max(m[i], m[i - 1]);
        uint32_t x = m[7];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= (uint32_t)o) x = max(x, y);
        }
        if (lane == 31) s_warp[warp] = x;
        __syncthreads();
        uint32_t before = carry, total = carry;
#pragma unroll
        for (int w = 0; w < kF16Threads / 32; ++w) {
            const uint32_t t = s_warp[w];
            if (w < (int)warp) before = max(before, t);
            total = max(total, t);
        }
        const uint32_t prev = __shfl_up_sync(0xffffffffu, x, 1);
        if (lane > 0) before = max(before, prev);
        carry = total;
        __syncthreads();                                         // s_warp is free for the next round

        uint32_t k[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) k[i] = image16(max(before, m[i]), inv) & 0xffffu;
        const uint32_t v = v0 + 8 * c;
        if (v >= off && v + 8 <= off + n) {
            B200_CHECK_AT(2, v + 8 - off <= n);
            *reinterpret_cast<uint4 *>(line + v) = make_uint4(k[0] | k[1] << 16, k[2] | k[3] << 16,
                                                              k[4] | k[5] << 16, k[6] | k[7] << 16);
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (v + i >= off && v + i < off + n) line[v + i] = (uint16_t)k[i];
        }
    }
}

// ---- r3 -------------------------------------------------------------------------------------------------------------
constexpr int kP16Threads = 512;
constexpr int kP16Warps = kP16Threads / 32;
#ifdef B200SORT_EXPERIMENTS
constexpr uint32_t kP16MinTile = kP16Threads * 8;          // the workspace also serves the 4096-key shape
#endif

template <int IPT>
struct R16PassSmem {
    uint32_t cnt[kP16Warps][kRadixBins];   // per-warp digit counts -> the warp's offset inside the digit's run
    int32_t vals[kP16Threads * IPT];       // the tile in digit order
    uint16_t keys[kP16Threads * IPT];
    uint32_t excl[kRadixBins];             // first tile-local position of each digit
    uint32_t dst[kRadixBins];              // destination of tile-local position 0 of each digit
    uint32_t sums[8];
    uint32_t ticket;
};

template <typename T>
__device__ __forceinline__ T *sel_buf16(uint32_t sel, T *in, T *tmp, T *out) {
    return sel == kSelIn ? in : sel == kSelTmp ? tmp : out;
}

__device__ __forceinline__ uint32_t digit16(uint32_t k, int pass, SignXor16 o) {
    return (image16(k, o) >> (pass * kRadixBits)) & (kRadixBins - 1);
}

// radix64_onesweep_kernel on 2-byte keys (see there): tickets, {flag:2, count:30} look-back, ranks from lane-ordered
// shared atomics (SAFE = 1: the ballot form), staging in digit order.  Slots past n in the last tile hold the key
// whose image is 0xFFFF: digit 255 in both passes, ranked after every real key, staged at the end, never written.
// IDX = 1: the values are the keys' input positions (b200sort_radix_sort_indices_keys16).  vin and vout are unused,
// vtmp holds n int32 positions between the two passes and idx_out is the int64 index output.  The first executed pass
// (pass 0, or pass 1 when pass 0 is skipped) makes the positions instead of loading them; the last executed pass
// (pass 1, or pass 0 when pass 1 is skipped) stores them as int64 into idx_out; only when both passes execute does pass
// 0 write them as int32 into vtmp for pass 1.  The index output is never read, so unlike the keys it does not follow
// src_sel / dst_sel: an in-place sort with one executed pass still stores its indices directly.
template <int IPT, int SAFE, int IDX>
__device__ __forceinline__ void
radix16_onesweep_body(const uint16_t *in, uint16_t *out, uint16_t *tmp, const int32_t *vin, int32_t *vout,
                      int32_t *vtmp, uint32_t n, int pass, R16Control *ctl, uint32_t *status, uint32_t *status_next,
                      SignXor16 order, uint32_t pad_key, int64_t *idx_out)
{
    constexpr uint32_t kTile = kP16Threads * IPT;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    R16PassSmem<IPT> &sm = *reinterpret_cast<R16PassSmem<IPT> *>(smem_raw);
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t tiles = (n + kTile - 1) / kTile;
    if (ctl->skip[pass]) {                                     // the identity: only the next pass's rows need clearing
        if (status_next != nullptr)
            for (uint32_t i = blockIdx.x * kP16Threads + tid; i < tiles * kRadixBins; i += gridDim.x * kP16Threads)
                status_next[i] = 0;
        return;
    }
    const uint16_t *src = sel_buf16<const uint16_t>(ctl->src_sel[pass], in, tmp, out);
    uint16_t *dst = sel_buf16<uint16_t>(ctl->dst_sel[pass], nullptr, tmp, out);
    const int32_t *vsrc = sel_buf16<const int32_t>(ctl->src_sel[pass], vin, vtmp, vout);
    int32_t *vdst = sel_buf16<int32_t>(ctl->dst_sel[pass], nullptr, vtmp, vout);
    bool make = false, wide = false;                            // IDX: first / last executed pass
    if constexpr (IDX != 0) {
        make = pass == 0 || ctl->skip[0] != 0;
        wide = pass == 1 || ctl->skip[1] != 0;
    }
    const uint32_t *base = ctl->base[pass];
    uint32_t *wcnt = sm.cnt[warp];
    const uint32_t wofs = warp * (32 * IPT) + lane;

    for (;;) {
        if (tid == 0) sm.ticket = atomicAdd(&ctl->ticket[pass], 1u);
        for (int d = lane; d < kRadixBins; d += 32) wcnt[d] = 0;
        __syncthreads();
        const uint32_t t = sm.ticket;
        if (t >= tiles) return;
        const uint32_t start = t * kTile;
        const uint32_t valid = (n - start < kTile) ? n - start : kTile;

        uint32_t key[IPT];
        int32_t val[IPT];
        uint32_t rank[IPT];
#pragma unroll
        for (int i = 0; i < IPT; ++i) {
            const uint32_t at = wofs + i * 32;                   // warp-striped: tile order = memory order
            key[i] = at < valid ? src[start + at] : pad_key;
            if constexpr (IDX != 0) val[i] = make ? (int32_t)(start + at) : (at < valid ? vtmp[start + at] : 0);
            else val[i] = at < valid ? vsrc[start + at] : 0;
        }
#pragma unroll
        for (int i = 0; i < IPT; ++i) {
            const uint32_t d = digit16(key[i], pass, order);
            if constexpr (SAFE != 0) {
                const uint32_t peers = __match_any_sync(0xffffffffu, d);
                const uint32_t leader = __ffs(peers) - 1;
                uint32_t first = 0;
                if (lane == leader) first = atomicAdd(wcnt + d, (uint32_t)__popc(peers));
                rank[i] = __shfl_sync(0xffffffffu, first, leader) + __popc(peers & lanemask_lt());
            } else {
                rank[i] = atomicAdd(wcnt + d, 1u);
            }
        }
        __syncthreads();                                         // warp counts final
        if (tid < kRadixBins) {
            uint32_t run = 0;
#pragma unroll
            for (int w = 0; w < kP16Warps; ++w) {
                const uint32_t c = sm.cnt[w][tid];
                sm.cnt[w][tid] = run;
                run += c;
            }
            uint32_t *row = status + (size_t)t * kRadixBins + tid;
            st_relaxed_gpu(row, (t == 0 ? kFlagIncl : kFlagLocal) | run);
            const uint32_t excl = scan256(run, sm.sums);
            uint32_t before = 0;                                 // keys of this digit in the earlier tiles
            if (t > 0) {
                for (const uint32_t *p = row - kRadixBins;; p -= kRadixBins) {
                    uint32_t w;
                    do { w = ld_relaxed_gpu(p); } while ((w & ~kValueMask) == 0);
                    before += w & kValueMask;
                    if (w & kFlagIncl) break;                    // tile 0 is always inclusive
                }
                // below n <= 2^30 except for the padded count of the last tile, which no tile reads
                st_relaxed_gpu(row, kFlagIncl | ((before + run) & kValueMask));
            }
            sm.excl[tid] = excl;
            sm.dst[tid] = base[tid] + before - excl;
            if (status_next != nullptr) status_next[(size_t)t * kRadixBins + tid] = 0;
        }
        __syncthreads();                                         // offsets final
#pragma unroll
        for (int i = 0; i < IPT; ++i) {
            const uint32_t d = digit16(key[i], pass, order);
            const uint32_t at = sm.excl[d] + wcnt[d] + rank[i];
            B200_CHECK_AT(1, at < kTile);
            if (at < kTile) {
                sm.keys[at] = (uint16_t)key[i];
                sm.vals[at] = val[i];
            }
        }
        __syncthreads();                                         // the tile is staged in digit order
        for (uint32_t i = tid; i < valid; i += kP16Threads) {
            const uint32_t k = sm.keys[i];
            const uint32_t pos = sm.dst[digit16(k, pass, order)] + i;
            B200_CHECK_AT(2, pos < n);
            if (pos < n) {
                dst[pos] = (uint16_t)k;
                if constexpr (IDX != 0) {
                    if (wide) {
                        B200_CHECK((reinterpret_cast<uintptr_t>(idx_out) & 7) == 0);
                        idx_out[pos] = sm.vals[i];
                    } else {
                        vtmp[pos] = sm.vals[i];
                    }
                } else {
                    vdst[pos] = sm.vals[i];
                }
            }
        }
        __syncthreads();                                         // shared memory free for the next tile
    }
}

template <int IPT, int SAFE>
__global__ void __launch_bounds__(kP16Threads, IPT <= 16 ? 2 : 1)
radix16_onesweep_kernel(const uint16_t *in, uint16_t *out, uint16_t *tmp, const int32_t *vin, int32_t *vout,
                        int32_t *vtmp, uint32_t n, int pass, R16Control *ctl, uint32_t *status, uint32_t *status_next,
                        SignXor16 order, uint32_t pad_key)
{
    radix16_onesweep_body<IPT, SAFE, 0>(in, out, tmp, vin, vout, vtmp, n, pass, ctl, status, status_next, order,
                                        pad_key, nullptr);
}

// The pass of the sort with indices (IDX above): tmp_idx holds n int32, idx_out is the int64 index output.
template <int IPT, int SAFE>
__global__ void __launch_bounds__(kP16Threads, IPT <= 16 ? 2 : 1)
radix16_onesweep_indices_kernel(const uint16_t *in, uint16_t *out, uint16_t *tmp, int32_t *tmp_idx, int64_t *idx_out,
                                uint32_t n, int pass, R16Control *ctl, uint32_t *status, uint32_t *status_next,
                                SignXor16 order, uint32_t pad_key)
{
    radix16_onesweep_body<IPT, SAFE, 1>(in, out, tmp, nullptr, nullptr, tmp_idx, n, pass, ctl, status, status_next,
                                        order, pad_key, idx_out);
}

// ---- r4 -------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
radix16_final_copy_kernel(const uint16_t *in, uint16_t *out, const uint16_t *tmp, const int32_t *vin, int32_t *vout,
                          const int32_t *vtmp, uint32_t n, const R16Control *ctl)
{
    const uint32_t sel = ctl->final_copy;
    if (sel == 0) return;
    const uint16_t *src = sel == kSelIn ? in : tmp;
    const int32_t *vsrc = sel == kSelIn ? vin : vtmp;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        out[i] = src[i];
        vout[i] = vsrc[i];
    }
}

// The final step of the sort with indices, in place of the final copy.  Keys: the final copy's plan.  Indices: with
// both passes skipped (one bit pattern holds every key) the sort is the identity and they are 0..n-1; otherwise the
// last executed pass has stored them.
__global__ void __launch_bounds__(256)
radix16_final_indices_kernel(const uint16_t *in, uint16_t *out, const uint16_t *tmp, int64_t *idx_out, uint32_t n,
                             const R16Control *ctl)
{
    const uint32_t sel = ctl->final_copy;
    const bool identity = ctl->skip[0] != 0 && ctl->skip[1] != 0;
    if (sel == 0 && !identity) return;
    const uint16_t *src = sel == kSelIn ? in : tmp;
    B200_CHECK((reinterpret_cast<uintptr_t>(idx_out) & 7) == 0);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        if (sel != 0) out[i] = src[i];
        if (identity) idx_out[i] = i;
    }
}

// ---- host side -------------------------------------------------------------------------------------------------------
// The shipped shapes; make EXPERIMENTS=1 also compiles the ones they were measured against (DESIGN 4.2f), chosen
// with B200SORT_R16_HIST_RUNS=0 and B200SORT_R16_IPT=8 or 32.
constexpr int kH16Runs = 1;
constexpr int kP16Ipt = 16;
#ifndef B200SORT_EXPERIMENTS
constexpr uint32_t kP16MinTile = kP16Threads * kP16Ipt;
#endif

static int r16_env(const char *name, int dflt) {
#ifdef B200SORT_EXPERIMENTS
    const char *e = getenv(name);
    return e != nullptr ? atoi(e) : dflt;
#else
    (void)name;
    return dflt;
#endif
}

static size_t h16_grid(size_t n) {
    const size_t chunks = div_up(n / 8 + 1, (size_t)kH16Threads * kH16Unroll);
    return chunks < (size_t)kNumSMs ? chunks : (size_t)kNumSMs;
}
static size_t r16_rows(size_t n) { return div_up(n > 0 ? n : 1, (size_t)kP16MinTile); }

size_t radix16_workspace_bytes(size_t n) {
    return kR16ControlBytes + h16_grid(n) * kImages16 * sizeof(uint32_t) + 2 * r16_rows(n) * kRadixBins * sizeof(uint32_t);
}

template <int RUNS>
static int launch_histogram(const uint16_t *in, uint32_t n, uint32_t *part, unsigned grid, R16Control *ctl,
                            uint32_t *status, size_t status_words, SignXor16 order, cudaStream_t s) {
    auto *fn = radix16_histogram_kernel<RUNS>;
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(fn), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)kH16SmemBytes));
    fn<<<grid, kH16Threads, kH16SmemBytes, s>>>(in, n, part, ctl, status, status_words, order);
    B200_LAUNCH_CHECK();
    return B200SORT_OK;
}

template <int IPT, int SAFE>
static int launch_passes(const uint16_t *in, uint16_t *out, uint16_t *tmp, const int32_t *vin, int32_t *vout,
                         int32_t *vtmp, uint32_t n, R16Control *ctl, uint32_t *const *status, SignXor16 order,
                         cudaStream_t s) {
    constexpr size_t smem = sizeof(R16PassSmem<IPT>);
    auto *fn = radix16_onesweep_kernel<IPT, SAFE>;
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(fn), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
    const size_t tiles = div_up(n, (size_t)kP16Threads * IPT);
    const size_t per_sm = IPT <= 16 ? 2 : 1;
    const unsigned grid = (unsigned)(tiles < per_sm * kNumSMs ? tiles : per_sm * kNumSMs);
    const uint32_t pad = image16(0xffffu, inverse16(order));    // the key whose image is 0xFFFF
    for (int pass = 0; pass < 2; ++pass) {
        fn<<<grid, kP16Threads, smem, s>>>(in, out, tmp, vin, vout, vtmp, n, pass, ctl, status[pass],
                                           pass == 0 ? status[1] : nullptr, order, pad);
        B200_LAUNCH_CHECK();
    }
    return B200SORT_OK;
}

template <int SAFE>
static int launch_passes_ipt(int ipt, const uint16_t *in, uint16_t *out, uint16_t *tmp, const int32_t *vin,
                             int32_t *vout, int32_t *vtmp, uint32_t n, R16Control *ctl, uint32_t *const *status,
                             SignXor16 order, cudaStream_t s) {
#ifdef B200SORT_EXPERIMENTS
    if (ipt == 8) return launch_passes<8, SAFE>(in, out, tmp, vin, vout, vtmp, n, ctl, status, order, s);
    if (ipt == 32) return launch_passes<32, SAFE>(in, out, tmp, vin, vout, vtmp, n, ctl, status, order, s);
#endif
    (void)ipt;
    return launch_passes<kP16Ipt, SAFE>(in, out, tmp, vin, vout, vtmp, n, ctl, status, order, s);
}

int radix16_sort(const uint16_t *d_in, uint16_t *d_out, uint16_t *d_tmp, const int32_t *v_in, int32_t *v_out,
                 int32_t *v_tmp, size_t n, void *d_ws, size_t ws_bytes, cudaStream_t s, SignXor16 order) {
    const bool pairs = v_in != nullptr;
    if (n == 0) return B200SORT_OK;
    if (n == 1) {
        if (d_in != d_out) B200_CUDA_TRY(cudaMemcpyAsync(d_out, d_in, sizeof(uint16_t), cudaMemcpyDeviceToDevice, s));
        if (pairs && v_in != v_out)
            B200_CUDA_TRY(cudaMemcpyAsync(v_out, v_in, sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
        return B200SORT_OK;
    }
    if (d_ws == nullptr || (reinterpret_cast<uintptr_t>(d_ws) & 255) != 0 || ws_bytes < radix16_workspace_bytes(n))
        return B200SORT_ERR_WORKSPACE;
    const int skip = radix_skip_enabled();
    // The passes' status words carry 30-bit counts; a digit count reaches 2^30 only when n = 2^30 and one digit value
    // holds every key, which is the case pass skipping removes.  The counting sort has no such words.
    if (pairs && n >= ((size_t)1 << 30) && !skip) return B200SORT_ERR_INVALID;
    const bool safe = pairs && !radix_atomic_order_ok();
    auto *ctl = static_cast<R16Control *>(d_ws);
    const size_t hgrid = h16_grid(n), rows = r16_rows(n);
    uint32_t *part = reinterpret_cast<uint32_t *>(static_cast<unsigned char *>(d_ws) + kR16ControlBytes);
    uint32_t *status[2];
    status[0] = part + hgrid * kImages16;
    status[1] = status[0] + rows * kRadixBins;
    const uint32_t n32 = (uint32_t)n;
    const size_t status_words = pairs ? rows * kRadixBins : 0;

    B200_CUDA_TRY(cudaMemsetAsync(ctl, 0, kR16ZeroBytes, s));
#ifdef B200SORT_EXPERIMENTS
    if (r16_env("B200SORT_R16_HIST_RUNS", kH16Runs) == 0)
        B200_TRY(launch_histogram<0>(d_in, n32, part, (unsigned)hgrid, ctl, status[0], status_words, order, s));
    else
#endif
        B200_TRY(launch_histogram<kH16Runs>(d_in, n32, part, (unsigned)hgrid, ctl, status[0], status_words, order, s));
    radix16_scan_kernel<<<kScan16Blocks, kRadixBins, 0, s>>>(part, (uint32_t)hgrid, n32, ctl, (uint32_t)skip,
                                                             d_in == d_out ? 1u : 0u);
    B200_LAUNCH_CHECK();
    if (!pairs) {
        const size_t off = (reinterpret_cast<uintptr_t>(d_out) & 15) >> 1;
        radix16_fill_kernel<<<(unsigned)div_up(off + n, (size_t)kF16Tile), kF16Threads, 0, s>>>(d_out, n32, ctl,
                                                                                            inverse16(order));
        B200_LAUNCH_CHECK();
        return B200SORT_OK;
    }
    const int ipt = r16_env("B200SORT_R16_IPT", kP16Ipt);
    if (safe) B200_TRY(launch_passes_ipt<1>(ipt, d_in, d_out, d_tmp, v_in, v_out, v_tmp, n32, ctl, status, order, s));
    else      B200_TRY(launch_passes_ipt<0>(ipt, d_in, d_out, d_tmp, v_in, v_out, v_tmp, n32, ctl, status, order, s));
    const size_t blocks = div_up(n, 256);
    radix16_final_copy_kernel<<<(unsigned)(blocks < (size_t)kNumSMs * 8 ? blocks : (size_t)kNumSMs * 8), 256, 0, s>>>(
        d_in, d_out, d_tmp, v_in, v_out, v_tmp, n32, ctl);
    B200_LAUNCH_CHECK();
    return B200SORT_OK;
}

// ---- sort with indices -------------------------------------------------------------------------------------------
// The pairs pipeline with the values made on the device: memset, histogram, scan, two passes, one final kernel.
template <int SAFE>
static int launch_indices_passes(const uint16_t *in, uint16_t *out, uint16_t *tmp, int32_t *tmp_idx, int64_t *idx_out,
                                 uint32_t n, R16Control *ctl, uint32_t *const *status, SignXor16 order, cudaStream_t s) {
    constexpr size_t smem = sizeof(R16PassSmem<kP16Ipt>);
    auto *fn = radix16_onesweep_indices_kernel<kP16Ipt, SAFE>;
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(fn), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
    const size_t tiles = div_up(n, (size_t)kP16Threads * kP16Ipt);
    const unsigned grid = (unsigned)(tiles < 2 * (size_t)kNumSMs ? tiles : 2 * (size_t)kNumSMs);
    const uint32_t pad = image16(0xffffu, inverse16(order));
    for (int pass = 0; pass < 2; ++pass) {
        fn<<<grid, kP16Threads, smem, s>>>(in, out, tmp, tmp_idx, idx_out, n, pass, ctl, status[pass],
                                           pass == 0 ? status[1] : nullptr, order, pad);
        B200_LAUNCH_CHECK();
    }
    return B200SORT_OK;
}

int radix16_sort_indices(const uint16_t *d_in, uint16_t *d_out, uint16_t *d_tmp, int64_t *idx_out, int32_t *tmp_idx,
                         size_t n, void *d_ws, size_t ws_bytes, cudaStream_t s, SignXor16 order) {
    if (n == 0) return B200SORT_OK;
    if (n == 1) {
        if (d_in != d_out) B200_CUDA_TRY(cudaMemcpyAsync(d_out, d_in, sizeof(uint16_t), cudaMemcpyDeviceToDevice, s));
        B200_CUDA_TRY(cudaMemsetAsync(idx_out, 0, sizeof(int64_t), s));
        return B200SORT_OK;
    }
    if (d_ws == nullptr || (reinterpret_cast<uintptr_t>(d_ws) & 255) != 0 || ws_bytes < radix16_workspace_bytes(n))
        return B200SORT_ERR_WORKSPACE;
    const int skip = radix_skip_enabled();
    if (n >= ((size_t)1 << 30) && !skip) return B200SORT_ERR_INVALID;   // the 30-bit status counts, see radix16_sort
    const bool safe = !radix_atomic_order_ok();
    auto *ctl = static_cast<R16Control *>(d_ws);
    const size_t hgrid = h16_grid(n), rows = r16_rows(n);
    uint32_t *part = reinterpret_cast<uint32_t *>(static_cast<unsigned char *>(d_ws) + kR16ControlBytes);
    uint32_t *status[2];
    status[0] = part + hgrid * kImages16;
    status[1] = status[0] + rows * kRadixBins;
    const uint32_t n32 = (uint32_t)n;

    B200_CUDA_TRY(cudaMemsetAsync(ctl, 0, kR16ZeroBytes, s));
    B200_TRY(launch_histogram<kH16Runs>(d_in, n32, part, (unsigned)hgrid, ctl, status[0], rows * kRadixBins, order, s));
    radix16_scan_kernel<<<kScan16Blocks, kRadixBins, 0, s>>>(part, (uint32_t)hgrid, n32, ctl, (uint32_t)skip,
                                                             d_in == d_out ? 1u : 0u);
    B200_LAUNCH_CHECK();
    if (safe) B200_TRY(launch_indices_passes<1>(d_in, d_out, d_tmp, tmp_idx, idx_out, n32, ctl, status, order, s));
    else      B200_TRY(launch_indices_passes<0>(d_in, d_out, d_tmp, tmp_idx, idx_out, n32, ctl, status, order, s));
    const size_t blocks = div_up(n, 256);
    radix16_final_indices_kernel<<<(unsigned)(blocks < (size_t)kNumSMs * 8 ? blocks : (size_t)kNumSMs * 8), 256, 0, s>>>(
        d_in, d_out, d_tmp, idx_out, n32, ctl);
    B200_LAUNCH_CHECK();
    return B200SORT_OK;
}

unsigned long long radix16_check_failures(unsigned long long *per_site) { return tu_check_failures(per_site); }

}  // namespace b200sort
