// radix64.cu -- stable LSD radix sort of 64-bit keys (int64, uint64, float64; ascending or descending), keys only or
// with a 32-bit value, in 8 passes of 8-bit digits of the key's image (DESIGN section 4.2e).
//
//   r0  radix64_histogram_kernel   one read of the keys builds the 8 digit histograms of the images; its last block
//                                  writes the exclusive bases and the plan: which passes are skipped (one bin holds
//                                  every key) and which buffer each executed pass reads and writes
//   r1  radix64_onesweep_kernel x8 persistent CTAs draw 4096-key tiles by ticket, rank by digit, look back over the
//                                  earlier tiles' {flag:2, count:30} status words, stage the tile in digit order in
//                                  shared memory and write it out coalesced; a skipped pass only clears the next
//                                  pass's status rows
//   r2  radix64_final_copy_kernel  tmp -> out (or in -> out) when the plan did not land in out
//
// Every call enqueues one memset and these ten kernels whatever the data, and the host never reads what the device
// computes: the sort is stream-ordered and can be captured in a CUDA graph.  The passes rank with lane-ordered
// shared-memory atomics behind the 1-D sort's self-test (radix_atomic_order_ok); SAFE = 1 is the ballot-ranked form.
#include "radix64.cuh"
#include "radix.cuh"
#include "radix_digit.cuh"

namespace b200sort {

int radix_atomic_order_ok();       // radix.cu: the lane-order self-test's verdict for the current device
int radix_skip_enabled();          // radix.cu: b200sort_radix_set_skip

constexpr int kR64Passes = 8;
constexpr int kR64Threads = 512;
constexpr int kR64Ipt = 8;
constexpr uint32_t kR64Tile = kR64Threads * kR64Ipt;    // 4096 keys per tile
constexpr int kR64Warps = kR64Threads / 32;

// Head of the workspace.  The first kR64ZeroBytes are zeroed by one memset per call; the rest is written by the
// histogram kernel's last block before any pass reads it.
struct R64Control {
    uint32_t hist[kR64Passes][kRadixBins];    // digit counts of the images (global atomics)
    uint32_t ticket[kR64Passes];              // tile tickets of each pass
    uint32_t hist_blocks_done;                // last-block detection in the histogram kernel
    uint32_t pad0[7];
    // ---- not zeroed ----
    uint32_t base[kR64Passes][kRadixBins];    // exclusive scan of hist[p]
    uint32_t skip[kR64Passes];                // 1 = one bin holds every key: the pass is the identity
    uint32_t src_sel[kR64Passes];             // buffer pass p reads : kSelIn / kSelTmp / kSelOut
    uint32_t dst_sel[kR64Passes];             // buffer pass p writes: kSelTmp / kSelOut
    uint32_t final_copy;                      // 0 none, else copy from that kSel* buffer to out
};
constexpr size_t kR64ZeroBytes = offsetof(R64Control, base);
constexpr size_t kR64ControlBytes = (sizeof(R64Control) + 255) / 256 * 256;

// The digit of pass p of a key's image: from the low word for p < 4, the high word for p >= 4; the sign that picks
// the mask is always bit 63.  `flips` (flips_of) holds this pass's byte of the pos mask in byte 0 and of the neg mask
// in byte 1, as in the 32-bit generic kernels.
__device__ __forceinline__ uint32_t digit64(uint2 k, int pass, uint32_t flips) {
    const uint32_t w = pass < 4 ? k.x : k.y;
    return ((w >> ((pass & 3) * kRadixBits)) ^ __byte_perm(flips, 0u, k.y >> 31)) & (kRadixBins - 1);
}
__host__ __device__ __forceinline__ uint32_t half_of(uint64_t m, int pass) { return (uint32_t)(m >> (pass < 4 ? 0 : 32)); }

// ---- r0 -------------------------------------------------------------------------------------------------------------
// The 32-bit histogram's lane-private 16-bit counters (radix_hist.cuh) for 8 places: counter (place p, digit d, lane l)
// lives in half (p & 1) of word ((p >> 1) * 256 + d) * 32 + l, 128 KiB in all.  Lane l only ever touches bank l, so
// no two lanes of one atomic instruction meet whatever the data.  That budget allows one CTA per SM, so the CTA has
// 1024 threads to keep enough loads in flight; one thread per word row in the flush.
constexpr int kH64Threads = 1024;
constexpr int kH64Unroll = 4;                               // 128-bit loads (2 keys each) in flight per thread
constexpr int kH64SmemWords = (kR64Passes / 2) * kRadixBins * 32;
constexpr size_t kH64SmemBytes = (size_t)kH64SmemWords * 4;   // 128 KiB
constexpr int kH64FlushIters = 128;   // 128 iters * (4 loads * 2 keys) * 32 warps = 32768 hits per lane column
static_assert(kH64Threads == (kR64Passes / 2) * kRadixBins, "one thread per word row");

__device__ __forceinline__ void h64_add(uint32_t col_s, uint2 img) {
#define B200_H64_RED(W, SEL, OFS, INC)                                                                              \
    asm volatile("red.shared.add.u32 [%0+" #OFS "], " #INC ";" :: "r"(col_s + (__byte_perm(W, 0u, SEL) << 7)) : "memory")
    B200_H64_RED(img.x, 0x4440u, 0, 1);
    B200_H64_RED(img.x, 0x4441u, 0, 65536);
    B200_H64_RED(img.x, 0x4442u, 32768, 1);
    B200_H64_RED(img.x, 0x4443u, 32768, 65536);
    B200_H64_RED(img.y, 0x4440u, 65536, 1);
    B200_H64_RED(img.y, 0x4441u, 65536, 65536);
    B200_H64_RED(img.y, 0x4442u, 98304, 1);
    B200_H64_RED(img.y, 0x4443u, 98304, 65536);
#undef B200_H64_RED
}

__device__ __forceinline__ void h64_flush(uint32_t *sh, R64Control *ctl, uint32_t tid) {
    __syncthreads();
    uint32_t lo = 0, hi = 0;
#pragma unroll
    for (uint32_t l = 0; l < 32; ++l) {
        const uint32_t idx = tid * 32 + ((l + tid) & 31);     // rotate: conflict-free across threads
        const uint32_t v = sh[idx];
        sh[idx] = 0;
        lo += v & 0xffffu;
        hi += v >> 16;
    }
    const uint32_t pp = tid >> kRadixBits, d = tid & (kRadixBins - 1);
    if (lo) atomicAdd(&ctl->hist[2 * pp][d], lo);
    if (hi) atomicAdd(&ctl->hist[2 * pp + 1][d], hi);
    __syncthreads();
}

__device__ __forceinline__ uint2 image64(uint2 k, SignXor64 o) {
    const uint64_t m = (k.y >> 31) ? o.neg : o.pos;
    return make_uint2(k.x ^ (uint32_t)m, k.y ^ (uint32_t)(m >> 32));
}

__global__ void __launch_bounds__(kH64Threads, 1)
radix64_histogram_kernel(const uint2 *__restrict__ keys, uint32_t n, R64Control *ctl, uint32_t *status_to_zero,
                         size_t status_words, uint32_t skip_enabled, uint32_t in_place, SignXor64 order)
{
    extern __shared__ __align__(16) uint32_t sh[];
    __shared__ uint32_t s_sums[kR64Passes][kRadixBins / 32];
    __shared__ uint32_t s_skip[kR64Passes];
    __shared__ uint32_t s_is_last;
    const uint32_t tid = threadIdx.x;
    {
        uint4 *z = reinterpret_cast<uint4 *>(sh);
        for (uint32_t i = tid; i < kH64SmemWords / 4; i += kH64Threads) z[i] = make_uint4(0, 0, 0, 0);
    }
    {   // the status rows of the first pass
        uint4 *z = reinterpret_cast<uint4 *>(status_to_zero);
        for (size_t i = (size_t)blockIdx.x * kH64Threads + tid; i < status_words / 4; i += (size_t)gridDim.x * kH64Threads)
            z[i] = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();
    const uint32_t col = (uint32_t)__cvta_generic_to_shared(sh + (tid & 31));

    // keys are 8-byte aligned: at most one key before the first 16-byte boundary, at most one after the last
    const uint32_t head = ((reinterpret_cast<uintptr_t>(keys) & 15) != 0 && n > 0) ? 1u : 0u;
    const uint32_t npairs = (n - head) / 2;
    const uint4 *v = reinterpret_cast<const uint4 *>(keys + head);
    constexpr uint32_t kChunk = kH64Threads * kH64Unroll;
    int iters = 0;
    for (uint32_t base = blockIdx.x * kChunk; base < npairs; base += gridDim.x * kChunk) {
        uint4 r[kH64Unroll];
        bool ok[kH64Unroll];
#pragma unroll
        for (int u = 0; u < kH64Unroll; ++u) {
            const uint32_t idx = base + u * kH64Threads + tid;
            ok[u] = idx < npairs;
            if (ok[u]) r[u] = __ldcs(v + idx);
        }
#pragma unroll
        for (int u = 0; u < kH64Unroll; ++u) {
            if (ok[u]) {
                h64_add(col, image64(make_uint2(r[u].x, r[u].y), order));
                h64_add(col, image64(make_uint2(r[u].z, r[u].w), order));
            }
        }
        if (++iters == kH64FlushIters) { h64_flush(sh, ctl, tid); iters = 0; }
    }
    if (blockIdx.x == 0 && tid == 0) {
        if (head) h64_add(col, image64(keys[0], order));
        if (head + 2 * npairs < n) h64_add(col, image64(keys[n - 1], order));
    }
    h64_flush(sh, ctl, tid);

    // the last block to finish: bases, skippable passes, the buffer plan
    __threadfence();
    __syncthreads();
    if (tid == 0) s_is_last = (atomicAdd(&ctl->hist_blocks_done, 1u) == gridDim.x - 1) ? 1u : 0u;
    if (tid < kR64Passes) s_skip[tid] = 0;
    __syncthreads();
    if (!s_is_last) return;
    __threadfence();
    if (tid < kRadixBins) {
        for (int p = 0; p < kR64Passes; ++p) {
            const uint32_t c = __ldcg(&ctl->hist[p][tid]);
            ctl->base[p][tid] = scan256(c, s_sums[p]);
            if (skip_enabled && c == n) s_skip[p] = 1;
        }
    }
    __syncthreads();
    // Executed pass j reads what executed pass j-1 wrote (the input for j = 0).  In place, writes alternate tmp, out,
    // tmp, ...; an odd count leaves the result in tmp for the final copy.  Out of place, writes alternate so that the
    // last executed pass lands in out and the input is never written; no executed pass at all copies in -> out.
    if (tid == 0) {
        uint32_t executed = 0;
        for (int p = 0; p < kR64Passes; ++p) executed += s_skip[p] ? 0u : 1u;
        uint32_t j = 0, cur = kSelIn;
        for (int p = 0; p < kR64Passes; ++p) {
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

// ---- r1 -------------------------------------------------------------------------------------------------------------
template <int VALS>
struct R64PassSmem {
    uint32_t cnt[kR64Warps][kRadixBins];   // per-warp digit counts -> the warp's offset inside the digit's run
    uint2 keys[kR64Tile];                  // the tile in digit order
    int32_t vals[VALS ? kR64Tile : 1];
    uint32_t excl[kRadixBins];             // first tile-local position of each digit
    uint32_t dst[kRadixBins];              // destination of tile-local position 0 of each digit
    uint32_t sums[8];
    uint32_t ticket;
};

template <typename T>
__device__ __forceinline__ T *sel_buf(uint32_t sel, T *in, T *tmp, T *out) {
    return sel == kSelIn ? in : sel == kSelTmp ? tmp : out;
}

// One stable pass by digit `pass`.  Tile t publishes its digit counts (kFlagIncl for tile 0, else kFlagLocal), walks
// back over the earlier tiles until an inclusive count, and sends its key i of digit d to
//   base[d] + (keys of digit d in earlier tiles) + (rank of the key among the tile's keys of digit d).
// Slots past n in the last tile hold the key whose image is all ones: digit 255 in every pass, ranked after every
// real key of the tile, so they are staged at the tile's end and never written.
template <int VALS, int SAFE>
__global__ void __launch_bounds__(kR64Threads, 2)
radix64_onesweep_kernel(const uint2 *in, uint2 *out, uint2 *tmp, const int32_t *vin, int32_t *vout, int32_t *vtmp,
                        uint32_t n, int pass, R64Control *ctl, uint32_t *status, uint32_t *status_next, SignXor64 order,
                        uint2 pad_key)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    R64PassSmem<VALS> &sm = *reinterpret_cast<R64PassSmem<VALS> *>(smem_raw);
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t tiles = (n + kR64Tile - 1) / kR64Tile;
    if (ctl->skip[pass]) {                                     // the identity: only the next pass's rows need clearing
        if (status_next != nullptr)
            for (uint32_t i = blockIdx.x * kR64Threads + tid; i < tiles * kRadixBins; i += gridDim.x * kR64Threads)
                status_next[i] = 0;
        return;
    }
    const uint32_t flips = flips_of(half_of(order.neg, pass), half_of(order.pos, pass), (pass & 3) * kRadixBits);
    const uint2 *src = sel_buf<const uint2>(ctl->src_sel[pass], in, tmp, out);
    uint2 *dst = sel_buf<uint2>(ctl->dst_sel[pass], nullptr, tmp, out);
    const int32_t *vsrc = sel_buf<const int32_t>(ctl->src_sel[pass], vin, vtmp, vout);
    int32_t *vdst = sel_buf<int32_t>(ctl->dst_sel[pass], nullptr, vtmp, vout);
    const uint32_t *base = ctl->base[pass];
    uint32_t *wcnt = sm.cnt[warp];
    const uint32_t wofs = warp * (32 * kR64Ipt) + lane;

    for (;;) {
        if (tid == 0) sm.ticket = atomicAdd(&ctl->ticket[pass], 1u);
        for (int d = lane; d < kRadixBins; d += 32) wcnt[d] = 0;
        __syncthreads();
        const uint32_t t = sm.ticket;
        if (t >= tiles) return;
        const uint32_t start = t * kR64Tile;
        const uint32_t valid = (n - start < kR64Tile) ? n - start : kR64Tile;

        uint2 key[kR64Ipt];
        int32_t val[VALS ? kR64Ipt : 1];
        uint32_t rank[kR64Ipt];
#pragma unroll
        for (int i = 0; i < kR64Ipt; ++i) {
            const uint32_t at = wofs + i * 32;                   // warp-striped: tile order = memory order
            key[i] = at < valid ? src[start + at] : pad_key;
            if constexpr (VALS != 0) val[i] = at < valid ? vsrc[start + at] : 0;
        }
#pragma unroll
        for (int i = 0; i < kR64Ipt; ++i) {
            const uint32_t d = digit64(key[i], pass, flips);
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
            for (int w = 0; w < kR64Warps; ++w) {
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
        for (int i = 0; i < kR64Ipt; ++i) {
            const uint32_t d = digit64(key[i], pass, flips);
            const uint32_t at = sm.excl[d] + wcnt[d] + rank[i];
            B200_CHECK_AT(1, at < kR64Tile);
            if (at < kR64Tile) {
                sm.keys[at] = key[i];
                if constexpr (VALS != 0) sm.vals[at] = val[i];
            }
        }
        __syncthreads();                                         // the tile is staged in digit order
        for (uint32_t i = tid; i < valid; i += kR64Threads) {
            const uint2 k = sm.keys[i];
            const uint32_t pos = sm.dst[digit64(k, pass, flips)] + i;
            B200_CHECK_AT(2, pos < n);
            if (pos < n) {
                dst[pos] = k;
                if constexpr (VALS != 0) vdst[pos] = sm.vals[i];
            }
        }
        __syncthreads();                                         // shared memory free for the next tile
    }
}

// ---- r2 -------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
radix64_final_copy_kernel(const uint2 *in, uint2 *out, const uint2 *tmp, const int32_t *vin, int32_t *vout,
                          const int32_t *vtmp, uint32_t n, const R64Control *ctl)
{
    const uint32_t sel = ctl->final_copy;
    if (sel == 0) return;
    const uint2 *src = sel == kSelIn ? in : tmp;
    const int32_t *vsrc = sel == kSelIn ? vin : vtmp;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        out[i] = src[i];
        if (vsrc != nullptr) vout[i] = vsrc[i];
    }
}

// ---- host side -------------------------------------------------------------------------------------------------------
static size_t r64_rows(size_t n) { return div_up(n > 0 ? n : 1, (size_t)kR64Tile); }

size_t radix64_workspace_bytes(size_t n) {
    return kR64ControlBytes + 2 * r64_rows(n) * kRadixBins * sizeof(uint32_t);
}

// The key whose image is all ones: last in every order, digit 255 in every pass.
static uint2 key_of_last_image64(SignXor64 o) {
    const uint64_t a = ~0ull ^ o.neg, b = ~0ull ^ o.pos;
    const uint64_t k = (a >> 63) ? a : b;                 // whichever of the two maps back through its own mask
    return make_uint2((uint32_t)k, (uint32_t)(k >> 32));
}

template <int VALS, int SAFE>
static int launch_passes(const uint2 *in, uint2 *out, uint2 *tmp, const int32_t *vin, int32_t *vout, int32_t *vtmp,
                         uint32_t n, R64Control *ctl, uint32_t *const *status, SignXor64 order, cudaStream_t s) {
    constexpr size_t smem = sizeof(R64PassSmem<VALS>);
    auto *fn = radix64_onesweep_kernel<VALS, SAFE>;
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(fn), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
    const size_t tiles = div_up(n, (size_t)kR64Tile);
    const unsigned grid = (unsigned)(tiles < 2u * kNumSMs ? tiles : 2u * kNumSMs);
    const uint2 pad = key_of_last_image64(order);
    for (int pass = 0; pass < kR64Passes; ++pass) {
        fn<<<grid, kR64Threads, smem, s>>>(in, out, tmp, vin, vout, vtmp, n, pass, ctl, status[pass & 1],
                                           pass + 1 < kR64Passes ? status[(pass + 1) & 1] : nullptr, order, pad);
        B200_LAUNCH_CHECK();
    }
    return B200SORT_OK;
}

int radix64_sort(const uint64_t *d_in, uint64_t *d_out, uint64_t *d_tmp, const int32_t *v_in, int32_t *v_out,
                 int32_t *v_tmp, size_t n, void *d_ws, size_t ws_bytes, cudaStream_t s, SignXor64 order) {
    if (n == 0) return B200SORT_OK;
    if (n == 1) {
        if (d_in != d_out) B200_CUDA_TRY(cudaMemcpyAsync(d_out, d_in, sizeof(uint64_t), cudaMemcpyDeviceToDevice, s));
        if (v_in != v_out) B200_CUDA_TRY(cudaMemcpyAsync(v_out, v_in, sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
        return B200SORT_OK;
    }
    if (d_ws == nullptr || (reinterpret_cast<uintptr_t>(d_ws) & 255) != 0 || ws_bytes < radix64_workspace_bytes(n))
        return B200SORT_ERR_WORKSPACE;
    const int skip = radix_skip_enabled();
    // Status words carry 30-bit counts; a digit count reaches 2^30 only when n = 2^30 and one bin holds every key,
    // which is the case pass skipping removes (as in the 32-bit sort).
    if (n >= ((size_t)1 << 30) && !skip) return B200SORT_ERR_INVALID;
    const bool safe = !radix_atomic_order_ok();
    auto *ctl = static_cast<R64Control *>(d_ws);
    const size_t rows = r64_rows(n);
    uint32_t *status[2];
    status[0] = reinterpret_cast<uint32_t *>(static_cast<unsigned char *>(d_ws) + kR64ControlBytes);
    status[1] = status[0] + rows * kRadixBins;
    const auto *in = reinterpret_cast<const uint2 *>(d_in);
    auto *out = reinterpret_cast<uint2 *>(d_out);
    auto *tmp = reinterpret_cast<uint2 *>(d_tmp);
    const uint32_t n32 = (uint32_t)n;

    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(radix64_histogram_kernel),
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kH64SmemBytes));
    B200_CUDA_TRY(cudaMemsetAsync(ctl, 0, kR64ZeroBytes, s));
    const size_t chunks = div_up(n / 2 + 1, (size_t)kH64Threads * kH64Unroll);
    const unsigned hgrid = (unsigned)(chunks < (size_t)kNumSMs ? chunks : (size_t)kNumSMs);
    radix64_histogram_kernel<<<hgrid, kH64Threads, kH64SmemBytes, s>>>(in, n32, ctl, status[0], rows * kRadixBins,
                                                                       (uint32_t)skip, d_in == d_out ? 1u : 0u, order);
    B200_LAUNCH_CHECK();
    if (v_in == nullptr)
        B200_TRY((safe ? launch_passes<0, 1>(in, out, tmp, nullptr, nullptr, nullptr, n32, ctl, status, order, s)
                       : launch_passes<0, 0>(in, out, tmp, nullptr, nullptr, nullptr, n32, ctl, status, order, s)));
    else
        B200_TRY((safe ? launch_passes<1, 1>(in, out, tmp, v_in, v_out, v_tmp, n32, ctl, status, order, s)
                       : launch_passes<1, 0>(in, out, tmp, v_in, v_out, v_tmp, n32, ctl, status, order, s)));
    const size_t blocks = div_up(n, 256);
    radix64_final_copy_kernel<<<(unsigned)(blocks < (size_t)kNumSMs * 8 ? blocks : (size_t)kNumSMs * 8), 256, 0, s>>>(
        in, out, tmp, v_in, v_out, v_tmp, n32, ctl);
    B200_LAUNCH_CHECK();
    return B200SORT_OK;
}

unsigned long long radix64_check_failures(unsigned long long *per_site) { return tu_check_failures(per_site); }

}  // namespace b200sort
