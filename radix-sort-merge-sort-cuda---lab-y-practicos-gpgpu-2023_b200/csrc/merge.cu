// merge.cu -- merge sort of int32 keys for sm_100a.
//
// Replaces the lab's merge stages (SRM/lab.cu:192-197 orderedJoin, :209-270 separators_kernel,
// :272-300 merge_segments_kernel) with
//
//   k3  block_sort_kernel        one CTA sorts a tile of kBlockTile keys: a bitonic network on the
//                                K keys each thread holds in registers, then log2(threads) rounds
//                                of merge-path merging through shared memory.          8 B/key
//   k4  merge_partition_kernel   one thread per output-tile boundary: diagonal binary search over
//                                the two runs in global memory (replaces the separator ranking,
//                                no 1024-thread / 48 KiB limit, no tail window).       O(n/T log n)
//   k5  merge_pass_kernel        one CTA per output tile: stages its A- and B-slice in shared
//                                memory, every thread merge-path-searches its K outputs and
//                                merges them serially, coalesced store.                8 B/key
//
// Ties take from A first (the reference's rule, SRM/lab.cu:163-170); for keys-only data it is
// invisible in the output but it keeps the partition consistent between k4 and k5.
#include "merge.cuh"

#include <atomic>

namespace b200sort {

constexpr int kSortThreads = 256;
constexpr int kSortK       = 16;
constexpr int kSortTile    = kSortThreads * kSortK;   // 4096

// Shared-memory index skew: one pad word per 32 so that "thread t, item k" (stride K) and
// "item j, thread t" (stride 1) are both conflict-free.
__device__ __forceinline__ uint32_t pad(uint32_t i) { return i + (i >> 5); }
// + K + 1: the serial merge reads one element ahead and, past the end of a ragged tile, up to K on.
constexpr int kSortSmemWords = (kSortTile + kSortK + 1) + ((kSortTile + kSortK + 1) >> 5) + 1;

// 256-bit global accesses (sm_100+): a thread that owns 16 consecutive keys moves them as two full
// 32-byte sectors.  (128-bit accesses at a 64-byte lane stride write half sectors and cost twice the
// load/store-pipe wavefronts: measured slower than staging through shared memory.)
__device__ __forceinline__ void st_stream_v8(int32_t *p, const int32_t *k) {
    asm volatile("st.global.L1::no_allocate.v8.s32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 :: "l"(p), "r"(k[0]), "r"(k[1]), "r"(k[2]), "r"(k[3]), "r"(k[4]), "r"(k[5]), "r"(k[6]), "r"(k[7])
                 : "memory");
}
__device__ __forceinline__ void ld_stream_v8(const int32_t *p, int32_t *k) {
    asm volatile("ld.global.L1::no_allocate.v8.s32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(k[0]), "=r"(k[1]), "=r"(k[2]), "=r"(k[3]), "=r"(k[4]), "=r"(k[5]), "=r"(k[6]), "=r"(k[7])
                 : "l"(p) : "memory");
}

__device__ __forceinline__ void cas(int32_t &a, int32_t &b, bool ascending) {
    const bool sw = ascending ? (a > b) : (a < b);
    const int32_t x = sw ? b : a, y = sw ? a : b;
    a = x; b = y;
}

// Bitonic sorting network over K registers (all indices are compile-time after unrolling).
template <int K>
__device__ __forceinline__ void thread_bitonic_sort(int32_t (&key)[K]) {
#pragma unroll
    for (int k = 2; k <= K; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
#pragma unroll
            for (int i = 0; i < K; ++i) {
                const int l = i ^ j;
                if (l > i) cas(key[i], key[l], (i & k) == 0);
            }
        }
    }
}

// Number of A elements among the first `diag` outputs of merge(A, B), A before equal B.
// A = s[a_base .. a_base+la), B = s[b_base .. b_base+lb), padded indexing.
__device__ __forceinline__ uint32_t merge_path_smem(const int32_t *s, uint32_t a_base, uint32_t la,
                                                    uint32_t b_base, uint32_t lb, uint32_t diag) {
    uint32_t lo = diag > lb ? diag - lb : 0, hi = diag < la ? diag : la;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        const int32_t a = s[pad(a_base + mid)];
        const int32_t b = s[pad(b_base + diag - 1 - mid)];
        if (a <= b) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// Serial merge of K outputs starting at (a_ptr, b_ptr); absolute padded-index pointers.
template <int K>
__device__ __forceinline__ void serial_merge(const int32_t *s, uint32_t a_ptr, uint32_t a_end,
                                             uint32_t b_ptr, uint32_t b_end, int32_t (&out)[K]) {
    int32_t a_val = s[pad(a_ptr)], b_val = s[pad(b_ptr)];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const bool take_a = (b_ptr >= b_end) || (a_ptr < a_end && a_val <= b_val);
        out[k] = take_a ? a_val : b_val;
        if (take_a) { ++a_ptr; a_val = s[pad(a_ptr)]; }
        else        { ++b_ptr; b_val = s[pad(b_ptr)]; }
    }
}

// ------------------------------------------------------------------------------------------------
// k3
// ------------------------------------------------------------------------------------------------
// 32 sorted runs of K keys (one per lane, in registers) -> one sorted run of 32 * K keys in blocked
// order (lane l ends with elements [l*K, l*K + K)), by bitonic merging: no shared memory, no searches.
// Element index i = lane * K + k.  Merging two sorted halves of a block of m = lanes * K elements:
// first i meets m - 1 - i  (= lane ^ (lanes - 1), register K - 1 - k), the smaller stays low; then
// the half-cleaners i ^ j for j = m/4 ... K across lanes (shuffles) and j = K/2 ... 1 in registers.
// (ncu of the block sort with all rounds in shared memory: load/store pipe 92 % busy, 7 wavefronts
// per 32 keys and round; a shuffle stage is one.)
template <int K>
__device__ __forceinline__ void warp_bitonic_merge_rounds(int32_t (&key)[K], uint32_t lane) {
    constexpr uint32_t full = 0xffffffffu;
#pragma unroll
    for (int lanes = 2; lanes <= 32; lanes <<= 1) {
        {
            const bool low = (lane & (lanes >> 1)) == 0;
#pragma unroll
            for (int k = 0; k < K / 2; ++k) {
                const int32_t a = key[k], b = key[K - 1 - k];
                const int32_t pb = __shfl_xor_sync(full, b, lanes - 1);   // partner's key[K-1-k] meets my key[k]
                const int32_t pa = __shfl_xor_sync(full, a, lanes - 1);   // partner's key[k] meets my key[K-1-k]
                key[k] = low ? min(a, pb) : max(a, pb);
                key[K - 1 - k] = low ? min(b, pa) : max(b, pa);
            }
        }
#pragma unroll
        for (int j = lanes >> 2; j >= 1; j >>= 1) {
            const bool low = (lane & j) == 0;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const int32_t v = __shfl_xor_sync(full, key[k], j);
                key[k] = low ? min(key[k], v) : max(key[k], v);
            }
        }
#pragma unroll
        for (int j = K >> 1; j >= 1; j >>= 1) {
#pragma unroll
            for (int k = 0; k < K; ++k) {
                if ((k & j) == 0) {
                    const int32_t a = min(key[k], key[k | j]), b = max(key[k], key[k | j]);
                    key[k] = a; key[k | j] = b;
                }
            }
        }
    }
}

// THREADS = 256: 4096-key tiles; THREADS = 512: 8192-key tiles (one more round in shared memory, one
// global merge pass less).  Full, 32-byte-aligned tiles are loaded and stored with 256-bit accesses
// straight from / to the 16 consecutive keys a thread owns.
// WARPNET: the rounds 16 -> 512 run as a bitonic network over the warp's registers.
// KEYS (block_sort_keys_kernel): every key is loaded as sign_xor(k, ld) and stored as sign_xor(k, st).
template <int THREADS, int WARPNET, int KEYS>
__device__ __forceinline__ void block_sort_body(const int32_t *in, int32_t *out, size_t n, SignXor ld, SignXor st)
{
    constexpr int kTile = THREADS * kSortK;
    constexpr int kWords = (kTile + kSortK + 1) + ((kTile + kSortK + 1) >> 5) + 1;
    __shared__ int32_t s[kWords];
    const uint32_t tid = threadIdx.x;
    const size_t tile_base = (size_t)blockIdx.x * kTile;
    const uint32_t valid = (n - tile_base < (size_t)kTile) ? (uint32_t)(n - tile_base) : (uint32_t)kTile;
    const bool direct = valid == (uint32_t)kTile &&
                        ((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & 31) == 0;

    int32_t key[kSortK];
    if (direct) {
        const int32_t *src = in + tile_base + (size_t)tid * kSortK;
#pragma unroll
        for (int q = 0; q < kSortK / 8; ++q) ld_stream_v8(src + 8 * q, key + 8 * q);
        if (KEYS) {
#pragma unroll
            for (int k = 0; k < kSortK; ++k) key[k] = (int32_t)sign_xor((uint32_t)key[k], ld.neg, ld.pos);
        }
        if (tid == 0) s[pad(kTile)] = 0x7FFFFFFF;
    } else {
        // coalesced load; the tail is padded with INT_MAX, which sorts last
#pragma unroll
        for (int j = 0; j < kSortK; ++j) {
            const uint32_t i = j * THREADS + tid;
            s[pad(i)] = (i < valid) ? (KEYS ? (int32_t)sign_xor((uint32_t)ld_stream(in + tile_base + i), ld.neg, ld.pos)
                                            : ld_stream(in + tile_base + i))
                                    : 0x7FFFFFFF;
        }
        if (tid == 0) s[pad(kTile)] = 0x7FFFFFFF;
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kSortK; ++k) key[k] = s[pad(tid * kSortK + k)];
        __syncthreads();
    }
    thread_bitonic_sort<kSortK>(key);
    if (WARPNET) warp_bitonic_merge_rounds<kSortK>(key, tid & 31);

    // merge rounds: sorted runs of len -> 2*len
#pragma unroll 1
    for (uint32_t len = WARPNET ? 32 * kSortK : kSortK; len < (uint32_t)kTile; len <<= 1) {
#pragma unroll
        for (int k = 0; k < kSortK; ++k) s[pad(tid * kSortK + k)] = key[k];
        __syncthreads();
        const uint32_t first = tid * kSortK;
        const uint32_t start = first & ~(2 * len - 1);
        const uint32_t diag = first - start;
        const uint32_t ai = merge_path_smem(s, start, len, start + len, len, diag);
        serial_merge<kSortK>(s, start + ai, start + len, start + len + (diag - ai), start + 2 * len, key);
        __syncthreads();
    }

    if (KEYS) {
#pragma unroll
        for (int k = 0; k < kSortK; ++k) key[k] = (int32_t)sign_xor((uint32_t)key[k], st.neg, st.pos);
    }
    if (direct) {
        int32_t *dst = out + tile_base + (size_t)tid * kSortK;
#pragma unroll
        for (int q = 0; q < kSortK / 8; ++q) st_stream_v8(dst + 8 * q, key + 8 * q);
        return;
    }
#pragma unroll
    for (int k = 0; k < kSortK; ++k) s[pad(tid * kSortK + k)] = key[k];
    __syncthreads();
#pragma unroll
    for (int j = 0; j < kSortK; ++j) {
        const uint32_t i = j * THREADS + tid;
        if (i < valid) st_stream(out + tile_base + i, s[pad(i)]);
    }
}

template <int THREADS, int WARPNET>
__global__ void __launch_bounds__(THREADS)
block_sort_kernel(const int32_t *in, int32_t *out, size_t n)
{
    block_sort_body<THREADS, WARPNET, 0>(in, out, n, SignXor{0, 0}, SignXor{0, 0});
}
template <int THREADS, int WARPNET>
__global__ void __launch_bounds__(THREADS)
block_sort_keys_kernel(const int32_t *in, int32_t *out, size_t n, SignXor ld, SignXor st)
{
    block_sort_body<THREADS, WARPNET, 1>(in, out, n, ld, st);
}

// ------------------------------------------------------------------------------------------------
// k3-lab: the assignment's staged tile sort (parts a-c of SRM/letra.pdf p.3), kept as a third way to
// produce sorted 4096-key tiles:
//   stage 1  every warp sorts 32-key groups with the LSD "split" primitive, one bit per iteration
//            (SRM/lab.cu:47-87).  The exclusive scan of the flags (SRM/lab.cu:11-41, 15 shuffles) is
//            one __ballot_sync + two __popc; bit 31 is split with inverted sense so that the order
//            is signed; the loop exits as soon as the group is sorted (SRM/lab.cu:61).
//   stage 2  rank merges of neighbouring runs 32 -> 64 -> ... -> 4096 in shared memory: every key
//            binary-searches the sibling run (SRM/lab.cu:102-132) and lands at own index + rank,
//            A before equal B's (SRM/lab.cu:144-182, :192-197) -- here up to 4096 per block, not 512.
// Stage 3 (runs longer than a block, SRM/lab.cu:209-300) is the merge-path pair k4/k5 below.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kSortThreads)
lab_tile_sort_kernel(const int32_t *in, int32_t *out, size_t n)
{
    __shared__ int32_t buf[2][kSortTile];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const size_t tile_base = (size_t)blockIdx.x * kSortTile;
    const uint32_t valid = (n - tile_base < (size_t)kSortTile) ? (uint32_t)(n - tile_base) : (uint32_t)kSortTile;
    const uint32_t lt = lanemask_lt();

    // stage 1: each warp takes groups warp, warp+8, ... of 32 consecutive keys
    for (uint32_t g = warp; g < kSortTile / 32; g += kSortThreads / 32) {
        const uint32_t i = g * 32 + lane;
        int32_t key = (i < valid) ? ld_stream(in + tile_base + i) : 0x7FFFFFFF;     // padding sorts last
        int32_t *swap = buf[0] + g * 32;
        for (int bit = 0; bit < 32; ++bit) {
            int32_t prev = __shfl_up_sync(0xffffffffu, key, 1);
            if (lane == 0) prev = key;
            if (__all_sync(0xffffffffu, prev <= key)) break;                        // sorted: done
            const bool set = (static_cast<uint32_t>(key) >> bit) & 1u;
            const bool first = (bit == 31) ? set : !set;                            // who goes in front
            const uint32_t front = __ballot_sync(0xffffffffu, first);
            const uint32_t f = __popc(front & lt);                                  // exclusive scan of the flags
            const uint32_t dst = first ? f : lane - f + __popc(front);              // the split rule
            swap[dst] = key;
            __syncwarp();
            key = swap[lane];
            __syncwarp();
        }
        swap[lane] = key;
    }
    __syncthreads();

    // stage 2: rank merges, ping-pong between the two buffers
    int cur = 0;
    for (uint32_t len = 32; len < (uint32_t)kSortTile; len <<= 1) {
        const int32_t *src = buf[cur];
        int32_t *dst = buf[cur ^ 1];
#pragma unroll 4
        for (uint32_t i = tid; i < (uint32_t)kSortTile; i += kSortThreads) {
            const uint32_t pair = i & ~(2 * len - 1);
            const bool from_b = (i & len) != 0;
            const int32_t x = src[i];
            const int32_t *other = src + pair + (from_b ? 0 : len);
            // rank of x in the sibling run: lower bound for A's keys, upper bound for B's keys
            uint32_t lo = 0, hi = len;
            while (lo < hi) {
                const uint32_t mid = (lo + hi) >> 1;
                const int32_t y = other[mid];
                const bool down = from_b ? (x < y) : (x <= y);
                if (down) hi = mid; else lo = mid + 1;
            }
            dst[pair + (i & (len - 1)) + lo] = x;
        }
        __syncthreads();
        cur ^= 1;
    }
    for (uint32_t i = tid; i < valid; i += kSortThreads) st_stream(out + tile_base + i, buf[cur][i]);
}

// ------------------------------------------------------------------------------------------------
// k4
// ------------------------------------------------------------------------------------------------
struct PairGeom { size_t base; size_t la; size_t lb; };
__device__ __forceinline__ PairGeom pair_of(size_t g, size_t n, size_t run) {
    PairGeom p;
    p.base = g / (2 * run) * (2 * run);
    const size_t rest = n - p.base;
    p.la = rest < run ? rest : run;
    p.lb = rest - p.la < run ? rest - p.la : run;
    return p;
}

__global__ void __launch_bounds__(128)
merge_partition_kernel(const int32_t *__restrict__ in, size_t n, size_t run, uint32_t *splits,
                       size_t num_tiles)
{
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= num_tiles) {
        if (t == num_tiles) splits[t] = 0;   // sentinel, never read as a start
        return;
    }
    const size_t g = t * kSortTile;
    const PairGeom p = pair_of(g, n, run);
    const size_t diag = g - p.base;          // < la + lb because g < n
    const int32_t *a = in + p.base, *b = a + p.la;
    size_t lo = diag > p.lb ? diag - p.lb : 0, hi = diag < p.la ? diag : p.la;
    while (lo < hi) {
        const size_t mid = (lo + hi) >> 1;
        if (__ldg(a + mid) <= __ldg(b + diag - 1 - mid)) lo = mid + 1; else hi = mid;
    }
    splits[t] = (uint32_t)lo;
}

// ------------------------------------------------------------------------------------------------
// k5
// ------------------------------------------------------------------------------------------------
// Persistent: a CTA walks over output tiles blockIdx, blockIdx + grid, ... and loads the NEXT tile's
// slices into registers before it merges the current one, so the two dependent global round trips
// of a tile (split points, then keys) overlap with the merging of the tile before it.  (ncu of the
// one-tile-per-CTA version: long-scoreboard stall 18.5 of 27 cycles per issue.)
struct MergeTileGeom {
    const int32_t *a, *b;      // this tile's slices of the two runs
    uint32_t na, nb;           // their lengths; na + nb = keys the tile produces
};
// sp0 / sp1 = splits[t] / splits[t + 1] (loaded an iteration ahead by the caller)
__device__ __forceinline__ MergeTileGeom merge_tile_geom(const int32_t *in, size_t n, size_t run,
                                                         uint32_t sp0, uint32_t sp1, size_t t) {
    const size_t g0 = t * kSortTile;
    const PairGeom p = pair_of(g0, n, run);
    const size_t diag0 = g0 - p.base;
    const size_t pair_len = p.la + p.lb;
    const size_t diag1 = diag0 + kSortTile < pair_len ? diag0 + kSortTile : pair_len;
    const size_t a0 = sp0;
    const size_t b0 = diag0 - a0;
    const size_t a1 = (diag1 == pair_len) ? p.la : (size_t)sp1;
    const size_t b1 = diag1 - a1;
    MergeTileGeom g;
    g.a = in + p.base + a0;
    g.b = in + p.base + p.la + b0;
    g.na = (uint32_t)(a1 - a0);
    g.nb = (uint32_t)(b1 - b0);
    return g;
}

// KEYS (merge_pass_keys_kernel): every key is stored as sign_xor(k, st).
template <int KEYS>
__device__ __forceinline__ void
merge_pass_body(const int32_t *__restrict__ in, int32_t *__restrict__ out, size_t n, size_t run,
                const uint32_t *__restrict__ splits, size_t t_begin, size_t tiles, SignXor st)
{
    __shared__ int32_t s[kSortSmemWords];
    const uint32_t tid = threadIdx.x;
    size_t t = t_begin + blockIdx.x;
    if (t >= tiles) return;

    int32_t next_keys[kSortK];
    MergeTileGeom geo = merge_tile_geom(in, n, run, __ldg(splits + t), __ldg(splits + t + 1), t);
    // split points of the tile after this one (splits has tiles + 1 entries; the last is a sentinel)
    uint32_t sp0 = 0, sp1 = 0;
    if (t + gridDim.x < tiles) { sp0 = __ldg(splits + t + gridDim.x); sp1 = __ldg(splits + t + gridDim.x + 1); }
    auto fetch = [&](const MergeTileGeom &g) {
        const uint32_t total = g.na + g.nb;
#pragma unroll
        for (int j = 0; j < kSortK; ++j) {
            const uint32_t i = j * kSortThreads + tid;
            int32_t v = 0x7FFFFFFF;
            if (i < g.na) v = ld_stream(g.a + i);
            else if (i < total) v = ld_stream(g.b + (i - g.na));
            next_keys[j] = v;
        }
    };
    fetch(geo);
    for (;;) {
        const uint32_t na = geo.na, nb = geo.nb, total = na + nb;
        const size_t g0 = t * kSortTile;
#pragma unroll
        for (int j = 0; j < kSortK; ++j) s[pad(j * kSortThreads + tid)] = next_keys[j];
        if (tid == 0) s[pad(kSortTile)] = 0x7FFFFFFF;
        __syncthreads();

        // the next tile's loads go out now and land while this tile is merged
        const size_t t_next = t + gridDim.x;
        const bool more = t_next < tiles;
        if (more) {
            geo = merge_tile_geom(in, n, run, sp0, sp1, t_next);
            fetch(geo);
            const size_t t_after = t_next + gridDim.x;       // and the split points one tile further on
            if (t_after < tiles) { sp0 = __ldg(splits + t_after); sp1 = __ldg(splits + t_after + 1); }
        }

        const uint32_t first = tid * kSortK;
        const uint32_t diag = first < total ? first : total;
        const uint32_t ai = merge_path_smem(s, 0, na, na, nb, diag);
        int32_t key[kSortK];
        serial_merge<kSortK>(s, ai, na, na + (diag - ai), total, key);
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kSortK; ++k) s[pad(first + k)] = key[k];
        __syncthreads();
#pragma unroll
        for (int j = 0; j < kSortK; ++j) {
            const uint32_t i = j * kSortThreads + tid;
            if (i < total) st_stream(out + g0 + i, KEYS ? (int32_t)sign_xor((uint32_t)s[pad(i)], st.neg, st.pos) : s[pad(i)]);
        }
        if (!more) break;
        t = t_next;
        __syncthreads();                                   // the staging area is reused
    }
}

__global__ void __launch_bounds__(kSortThreads, 4)
merge_pass_kernel(const int32_t *__restrict__ in, int32_t *__restrict__ out, size_t n, size_t run,
                  const uint32_t *__restrict__ splits, size_t t_begin, size_t tiles /* = end of the range */)
{
    merge_pass_body<0>(in, out, n, run, splits, t_begin, tiles, SignXor{0, 0});
}
__global__ void __launch_bounds__(kSortThreads, 4)
merge_pass_keys_kernel(const int32_t *__restrict__ in, int32_t *__restrict__ out, size_t n, size_t run,
                       const uint32_t *__restrict__ splits, size_t t_begin, size_t tiles, SignXor st)
{
    merge_pass_body<1>(in, out, n, run, splits, t_begin, tiles, st);
}

// ------------------------------------------------------------------------------------------------
// k5' (default): the same pass with far fewer instructions per key
// ------------------------------------------------------------------------------------------------
// What ncu showed for k5 (profiles/r01_merge.md): ~50 warp instructions per 32 keys at 1.4 IPC and four
// barriers per tile; nothing else is near a limit (HBM 32 %, shared-memory pipe 40 %).  Here
//   * each slice is followed by a gap of kGap slots whose first kSortK + 1 hold sentinels (INT_MAX),
//     so the serial merge needs no bounds tests: out = min(a, b), one compare, one load.  A sentinel
//     can only be taken in place of a key that is itself INT_MAX, and then every key still to come
//     is INT_MAX too, so the values are exact.  kGap = 32 keeps the padded address of "element i of
//     the tile" a per-thread constant plus a compile-time offset (+33 words if it belongs to B);
//   * every thread ends with 16 CONSECUTIVE outputs in registers and stores them as two 256-bit
//     stores straight to global memory -- no second trip through shared memory, no barriers for it;
//   * the staging area is double-buffered: one barrier per tile;
//   * run lengths that are powers of two (every pass of merge_sort) take shifts, not 64-bit divisions.
constexpr int kGap = 32;
constexpr int kPass2Logical = kSortTile + 2 * kGap;
constexpr int kPass2Words = kPass2Logical + (kPass2Logical >> 5) + 1;
static_assert(kGap % 32 == 0 && kGap >= kSortK + 1, "see the staging stores");

// A = s[0 .. na), B = s[b_base .. b_base + nb) (logical indices, padded on access).
__device__ __forceinline__ uint32_t merge_path_gap(const int32_t *s, uint32_t na, uint32_t b_base,
                                                   uint32_t nb, uint32_t diag) {
    uint32_t lo = diag > nb ? diag - nb : 0, hi = diag < na ? diag : na;
    const uint32_t b_last = b_base + diag - 1;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        const int32_t a = s[pad(mid)];
        const int32_t b = s[pad(b_last - mid)];
        if (a <= b) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// K outputs from (a_ptr, b_ptr); both runs end in at least K + 1 sentinels.
template <int K>
__device__ __forceinline__ void serial_merge_sentinel(const int32_t *s, uint32_t a_ptr, uint32_t b_ptr,
                                                      int32_t (&out)[K]) {
    int32_t a_val = s[pad(a_ptr)], b_val = s[pad(b_ptr)];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const bool take_a = a_val <= b_val;                // ties: A first (SRM/lab.cu:163-170)
        out[k] = take_a ? a_val : b_val;
        const uint32_t nxt = (take_a ? a_ptr : b_ptr) + 1;
        const int32_t v = s[pad(nxt)];
        a_ptr = take_a ? nxt : a_ptr;  a_val = take_a ? v : a_val;
        b_ptr = take_a ? b_ptr : nxt;  b_val = take_a ? b_val : v;
    }
}

// The tile's two slices as 32-bit element offsets into `in` (n <= B200SORT_MAX_N = 2^30).
// pair_shift >= 0: 2 * run == 1 << pair_shift (shifts instead of 64-bit divisions).
struct MergeTileGeom32 { uint32_t oa, ob, na, nb; };
__device__ __forceinline__ MergeTileGeom32 merge_tile_geom32(const int32_t *in, size_t n, size_t run, int pair_shift,
                                                             uint32_t sp0, uint32_t sp1, size_t t) {
    MergeTileGeom32 g;
    if (pair_shift < 0) {
        const MergeTileGeom w = merge_tile_geom(in, n, run, sp0, sp1, t);
        g.oa = (uint32_t)(w.a - in); g.ob = (uint32_t)(w.b - in); g.na = w.na; g.nb = w.nb;
        return g;
    }
    const uint32_t n32 = (uint32_t)n, run32 = (uint32_t)run;
    const uint32_t g0 = (uint32_t)t * kSortTile;
    const uint32_t base = (g0 >> pair_shift) << pair_shift;
    const uint32_t rest = n32 - base;
    const uint32_t la = rest < run32 ? rest : run32;
    const uint32_t lb = rest - la < run32 ? rest - la : run32;
    const uint32_t diag0 = g0 - base;
    const uint32_t pair_len = la + lb;
    const uint32_t diag1 = diag0 + kSortTile < pair_len ? diag0 + kSortTile : pair_len;
    const uint32_t a1 = (diag1 == pair_len) ? la : sp1;
    g.oa = base + sp0;
    g.ob = base + la + (diag0 - sp0);
    g.na = a1 - sp0;
    g.nb = (diag1 - a1) - (diag0 - sp0);
    return g;
}

// MINB: CTAs per SM the register allocation is held to (4: 64 registers, 5: 48, 6: 40).
// KEYS (merge_pass2_keys_kernel): every key is stored as sign_xor(k, st).
template <int KEYS>
__device__ __forceinline__ void
merge_pass2_body(const int32_t *__restrict__ in, int32_t *__restrict__ out, size_t n, size_t run, int pair_shift,
                 const uint32_t *__restrict__ splits, size_t t_begin, size_t tiles, SignXor st)
{
    __shared__ int32_t s2[2][kPass2Words];
    const uint32_t tid = threadIdx.x;
    size_t t = t_begin + blockIdx.x;
    if (t >= tiles) return;
    const bool out_aligned = (reinterpret_cast<uintptr_t>(out) & 31) == 0;
    const uint32_t padtid = pad(tid);

    int32_t next_keys[kSortK];
    MergeTileGeom32 geo = merge_tile_geom32(in, n, run, pair_shift, __ldg(splits + t), __ldg(splits + t + 1), t);
    uint32_t sp0 = 0, sp1 = 0;
    if (t + gridDim.x < tiles) { sp0 = __ldg(splits + t + gridDim.x); sp1 = __ldg(splits + t + gridDim.x + 1); }
    auto fetch = [&](const MergeTileGeom32 &g) {
        const uint32_t total = g.na + g.nb;
        const uint32_t ia = g.oa + tid;                        // element i of the tile is in[ia + i - tid] ...
        const uint32_t ib = g.ob + tid - g.na;                 // ... or in[ib + i - tid] once i >= na  (ob >= na)
#pragma unroll
        for (int j = 0; j < kSortK; ++j) {
            const uint32_t i = j * kSortThreads + tid;
            const int32_t *src = in + ((i < g.na) ? ia : ib);
            next_keys[j] = (i < total) ? ld_stream(src + j * kSortThreads) : 0x7FFFFFFF;
        }
    };
    fetch(geo);
    int buf = 0;
    for (;;) {
        int32_t *s = s2[buf];
        const uint32_t na = geo.na, nb = geo.nb, total = na + nb;
        const size_t g0 = t * kSortTile;
        // element i = j * 256 + tid sits at pad(i) = pad(tid) + j * 264, B's elements kGap slots further
        // on: pad(i + 32) = pad(i) + 33
        {
            int32_t *sa = s + padtid, *sb = sa + kGap + kGap / 32;
#pragma unroll
            for (int j = 0; j < kSortK; ++j) {
                const uint32_t i = j * kSortThreads + tid;
                int32_t *dst = (i < na) ? sa : sb;
                dst[j * (kSortThreads + kSortThreads / 32)] = next_keys[j];
            }
        }
        if (tid <= kSortK) s[pad(na + tid)] = 0x7FFFFFFF;                                        // after A
        else if (tid >= 32 && tid <= 32 + kSortK) s[pad(total + kGap + (tid - 32))] = 0x7FFFFFFF;   // after B
        __syncthreads();    // the only barrier of the tile: the other buffer was last read a tile ago

        // the next tile's loads go out now and land while this tile is merged
        const size_t t_next = t + gridDim.x;
        const bool more = t_next < tiles;
        if (more) {
            geo = merge_tile_geom32(in, n, run, pair_shift, sp0, sp1, t_next);
            fetch(geo);
            const size_t t_after = t_next + gridDim.x;
            if (t_after < tiles) { sp0 = __ldg(splits + t_after); sp1 = __ldg(splits + t_after + 1); }
        }

        const uint32_t first = tid * kSortK;
        const uint32_t diag = first < total ? first : total;
        const uint32_t ai = merge_path_gap(s, na, na + kGap, nb, diag);
        int32_t key[kSortK];
        serial_merge_sentinel<kSortK>(s, ai, na + kGap + (diag - ai), key);
        if (KEYS) {
#pragma unroll
            for (int k = 0; k < kSortK; ++k) key[k] = (int32_t)sign_xor((uint32_t)key[k], st.neg, st.pos);
        }
        int32_t *dst = out + g0 + first;
        if (total == (uint32_t)kSortTile && out_aligned) {
#pragma unroll
            for (int q = 0; q < kSortK / 8; ++q) st_stream_v8(dst + 8 * q, key + 8 * q);
        } else {
#pragma unroll
            for (int k = 0; k < kSortK; ++k)
                if (first + k < total) st_stream(dst + k, key[k]);
        }
        if (!more) break;
        t = t_next;
        buf ^= 1;
    }
}

template <int MINB>
__global__ void __launch_bounds__(kSortThreads, MINB)
merge_pass2_kernel(const int32_t *__restrict__ in, int32_t *__restrict__ out, size_t n, size_t run,
                   int pair_shift, const uint32_t *__restrict__ splits, size_t t_begin,
                   size_t tiles /* = end of the range */)
{
    merge_pass2_body<0>(in, out, n, run, pair_shift, splits, t_begin, tiles, SignXor{0, 0});
}
template <int MINB>
__global__ void __launch_bounds__(kSortThreads, MINB)
merge_pass2_keys_kernel(const int32_t *__restrict__ in, int32_t *__restrict__ out, size_t n, size_t run,
                        int pair_shift, const uint32_t *__restrict__ splits, size_t t_begin, size_t tiles, SignXor st)
{
    merge_pass2_body<1>(in, out, n, run, pair_shift, splits, t_begin, tiles, st);
}

// ================================================================================================
// host side
// ================================================================================================
// bit 0: merge pass = k5 (staged output, bounds-tested serial merge) instead of k5'
// bit 1: block sort tiles of 4096 keys (256 threads) instead of 8192 (512 threads)
// bit 2: block sort with every round in shared memory (no warp-register bitonic rounds)
// bits 3-4: k5' with 4 + k CTAs per SM (k = 0, 1, 2)
// The shipped library compiles variants 0 (default) and 1 (the staged-store pass, kept for A/B); the other 22
// were measured in round 1 (profiles/r01_merge_variants.txt) and need make EXPERIMENTS=1.
#ifdef B200SORT_EXPERIMENTS
constexpr int kMergeVariants = 24;
#else
constexpr int kMergeVariants = 2;
#endif
static std::atomic<int> g_merge_variant{0};
int merge_set_variant(int v) {
    if (v < 0 || v >= kMergeVariants) return B200SORT_ERR_INVALID;
    g_merge_variant.store(v);
    return B200SORT_OK;
}
int merge_num_variants() { return kMergeVariants; }
const char *merge_variant_name(int v) {
    static const char *names[24] = {
        "block8192_warpnet_pass2_sentinel_direct_store", "block8192_warpnet_pass1_staged_store",
        "block4096_warpnet_pass2_sentinel_direct_store", "block4096_warpnet_pass1_staged_store",
        "block8192_smemrounds_pass2_sentinel_direct_store", "block8192_smemrounds_pass1_staged_store",
        "block4096_smemrounds_pass2_sentinel_direct_store", "block4096_smemrounds_pass1_staged_store",
        "block8192_warpnet_pass2_5ctas", "(8|1)", "block4096_warpnet_pass2_5ctas", "(10|1)",
        "block8192_smemrounds_pass2_5ctas", "(12|1)", "block4096_smemrounds_pass2_5ctas", "(14|1)",
        "block8192_warpnet_pass2_6ctas", "(16|1)", "block4096_warpnet_pass2_6ctas", "(18|1)",
        "block8192_smemrounds_pass2_6ctas", "(20|1)", "block4096_smemrounds_pass2_6ctas", "(22|1)"};
    return (v >= 0 && v < 24) ? names[v] : nullptr;
}

size_t merge_block_tile() { return (g_merge_variant.load() & 2) ? kSortTile : 2 * kSortTile; }
size_t merge_tile() { return kSortTile; }

size_t merge_workspace_bytes(size_t n) {
    return align_up((div_up(n > 0 ? n : 1, kSortTile) + 2) * sizeof(uint32_t), 256);
}

int merge_block_sort(const int32_t *d_in, int32_t *d_out, size_t n, cudaStream_t s, bool lab_stages) {
    if (n == 0) return B200SORT_OK;
    if (lab_stages)
        lab_tile_sort_kernel<<<(unsigned)div_up(n, kSortTile), kSortThreads, 0, s>>>(d_in, d_out, n);
    else {
        const bool small = merge_block_tile() == (size_t)kSortTile, net = (g_merge_variant.load() & 4) == 0;
        const unsigned g1 = (unsigned)div_up(n, kSortTile), g2 = (unsigned)div_up(n, 2 * kSortTile);
#ifdef B200SORT_EXPERIMENTS
        if (small && net)       block_sort_kernel<kSortThreads, 1><<<g1, kSortThreads, 0, s>>>(d_in, d_out, n);
        else if (small)         block_sort_kernel<kSortThreads, 0><<<g1, kSortThreads, 0, s>>>(d_in, d_out, n);
        else if (!net)          block_sort_kernel<2 * kSortThreads, 0><<<g2, 2 * kSortThreads, 0, s>>>(d_in, d_out, n);
        else
#endif
        { (void)small; (void)net; (void)g1;
          block_sort_kernel<2 * kSortThreads, 1><<<g2, 2 * kSortThreads, 0, s>>>(d_in, d_out, n); }
    }
    B200_LAUNCH_CHECK();
    return B200SORT_OK;
}

int merge_partition(const int32_t *d_in, size_t n, size_t run, uint32_t *d_splits, cudaStream_t s) {
    if (n == 0) return B200SORT_OK;
    if (run == 0 || run % kSortTile != 0) return B200SORT_ERR_INVALID;
    const size_t tiles = div_up(n, kSortTile);
    merge_partition_kernel<<<(unsigned)div_up(tiles + 1, 128), 128, 0, s>>>(d_in, n, run, d_splits, tiles);
    B200_LAUNCH_CHECK();
    return B200SORT_OK;
}

int merge_pass_range(const int32_t *d_in, int32_t *d_out, size_t n, size_t run, const uint32_t *d_splits,
                     size_t tile_begin, size_t tile_end, cudaStream_t s, const SignXor *st) {
    if (n == 0) return B200SORT_OK;
    if (run == 0 || run % kSortTile != 0) return B200SORT_ERR_INVALID;
    const size_t tiles = div_up(n, kSortTile);
    if (tile_end > tiles) tile_end = tiles;
    if (tile_begin >= tile_end) return B200SORT_OK;
    const size_t count = tile_end - tile_begin;
    const int variant = g_merge_variant.load();
    const int per_sm = (variant & 1) ? 4 : 4 + ((variant >> 3) & 3);   // persistent: 4..6 CTAs of 256 threads per SM
    const size_t slots = (size_t)kNumSMs * per_sm;
    const unsigned grid = (unsigned)(count < slots ? count : slots);
    if ((variant & 1) == 0)
    {
        int pair_shift = -1;                                   // 2 * run a power of two: shifts instead of divisions
        if ((run & (run - 1)) == 0) { pair_shift = 1; while (((size_t)1 << pair_shift) < 2 * run) ++pair_shift; }
        if (st != nullptr)
            merge_pass2_keys_kernel<4><<<grid, kSortThreads, 0, s>>>(d_in, d_out, n, run, pair_shift, d_splits, tile_begin,
                                                                    tile_end, *st);
        else
#ifdef B200SORT_EXPERIMENTS
        if (per_sm == 5)      merge_pass2_kernel<5><<<grid, kSortThreads, 0, s>>>(d_in, d_out, n, run, pair_shift, d_splits, tile_begin, tile_end);
        else if (per_sm == 6) merge_pass2_kernel<6><<<grid, kSortThreads, 0, s>>>(d_in, d_out, n, run, pair_shift, d_splits, tile_begin, tile_end);
        else
#endif
        merge_pass2_kernel<4><<<grid, kSortThreads, 0, s>>>(d_in, d_out, n, run, pair_shift, d_splits, tile_begin, tile_end);
    }
    else if (st != nullptr)
        merge_pass_keys_kernel<<<grid, kSortThreads, 0, s>>>(d_in, d_out, n, run, d_splits, tile_begin, tile_end, *st);
    else
        merge_pass_kernel<<<grid, kSortThreads, 0, s>>>(d_in, d_out, n, run, d_splits, tile_begin, tile_end);
    B200_LAUNCH_CHECK();
    return B200SORT_OK;
}

int merge_pass(const int32_t *d_in, int32_t *d_out, size_t n, size_t run, const uint32_t *d_splits,
               cudaStream_t s) {
    return merge_pass_range(d_in, d_out, n, run, d_splits, 0, div_up(n, kSortTile), s);
}

namespace {
int merge_sort_impl(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, size_t n, void *d_ws,
                    size_t ws_bytes, cudaStream_t s, float *ms, bool lab_stages, const SignXor *order) {
    if (ms) ms[0] = ms[1] = ms[2] = 0.f;
    if (n == 0) return B200SORT_OK;
    if (n == 1) {
        if (d_in != d_out) B200_CUDA_TRY(cudaMemcpyAsync(d_out, d_in, sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
        return B200SORT_OK;
    }
    if (d_ws == nullptr || ws_bytes < merge_workspace_bytes(n)) return B200SORT_ERR_WORKSPACE;
    auto *splits = static_cast<uint32_t *>(d_ws);
    const size_t first_run = lab_stages ? (size_t)kSortTile : merge_block_tile();
    int passes = 0;
    for (size_t run = first_run; run < n; run *= 2) ++passes;
    // Land the final pass in d_out: the block sort (which may run in place) writes to whichever
    // buffer makes that so.  d_in is only ever read by the block sort.
    int32_t *src = (passes % 2 == 0) ? d_out : d_tmp;
    int32_t *dst = (passes % 2 == 0) ? d_tmp : d_out;
    struct Events {
        cudaEvent_t e[3] = {nullptr, nullptr, nullptr};
        ~Events() { for (auto &x : e) if (x) cudaEventDestroy(x); }
    } events;
    cudaEvent_t (&ev)[3] = events.e;
    if (ms) {
        for (auto &e : ev) B200_CUDA_TRY(cudaEventCreate(&e));
        B200_CUDA_TRY(cudaEventRecord(ev[0], s));
    }
    // order: the block sort maps every key to image ^ 0x80000000 (a signed-comparable int32), the passes sort those
    // with the int32 kernels, and the last kernel maps them back: d_tmp and d_out are scratch until then
    SignXor to_signed{}, to_key{}, identity{0u, 0u};
    if (order != nullptr) {
        const SignXor inv = image_inverse(*order);
        to_signed = SignXor{order->neg ^ 0x80000000u, order->pos ^ 0x80000000u};
        to_key = SignXor{inv.pos ^ 0x80000000u, inv.neg ^ 0x80000000u};     // keyed on the image's top bit = !(sign)
    }
    if (order != nullptr) {
        block_sort_keys_kernel<2 * kSortThreads, 1><<<(unsigned)div_up(n, 2 * kSortTile), 2 * kSortThreads, 0, s>>>(
            d_in, src, n, to_signed, passes == 0 ? to_key : identity);
        B200_LAUNCH_CHECK();
    } else {
        B200_TRY(merge_block_sort(d_in, src, n, s, lab_stages));
    }
    if (ms) B200_CUDA_TRY(cudaEventRecord(ev[1], s));
    int pass = 0;
    for (size_t run = first_run; run < n; run *= 2, ++pass) {
        B200_TRY(merge_partition(src, n, run, splits, s));
        B200_TRY(merge_pass_range(src, dst, n, run, splits, 0, div_up(n, kSortTile), s,
                                  (order != nullptr && pass == passes - 1) ? &to_key : nullptr));
        int32_t *t = src; src = dst; dst = t;
    }
    if (ms) {
        B200_CUDA_TRY(cudaEventRecord(ev[2], s));
        B200_CUDA_TRY(cudaEventSynchronize(ev[2]));
        B200_CUDA_TRY(cudaEventElapsedTime(&ms[0], ev[0], ev[1]));   // block sort
        B200_CUDA_TRY(cudaEventElapsedTime(&ms[1], ev[1], ev[2]));   // all merge passes
        ms[2] = (float)passes;
    }
    return B200SORT_OK;
}
}  // namespace

int merge_sort(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, size_t n, void *d_ws,
               size_t ws_bytes, cudaStream_t s, float *ms, bool lab_stages) {
    return merge_sort_impl(d_in, d_out, d_tmp, n, d_ws, ws_bytes, s, ms, lab_stages, nullptr);
}

int merge_sort_keys(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, size_t n, void *d_ws,
                    size_t ws_bytes, cudaStream_t s, SignXor order) {
    // the generic kernels exist for the shipped shapes only (8192-key block sort, variants 0 and 1)
    if (n > 1 && g_merge_variant.load() > 1) return B200SORT_ERR_INVALID;
    return merge_sort_impl(d_in, d_out, d_tmp, n, d_ws, ws_bytes, s, nullptr, false, &order);
}

}  // namespace b200sort
