// dist.cu -- one-box multi-GPU sort: the device kernels and the host planner (north_star (c)).
//
// No reference counterpart (the lab is single-GPU, SRM/run.sh:11).  One process per GPU; the
// collectives (counts all-gather / all-reduce, optional NCCL all-to-all) are the caller's
// plumbing (torch.distributed in <pkg>/dist.py).  This file provides
//
//   dist_histogram_kernel   2^bits-bin histogram of the top `bits` bits of key ^ 0x80000000
//                           (the MSD-digit partition histogram).                    4 B/key
//   dist_plan               pure host function: contiguous bin ranges -> ranks, balanced on the
//                           global counts; per-rank send / receive counts and the offset of this
//                           rank's block inside every destination's receive buffer.
//   dist_partition_kernel   multisplit of the local keys by destination rank, staged through
//                           shared memory so that every destination receives coalesced runs.
//                           The destination table holds device-visible base pointers: local
//                           pointers (then an NCCL all-to-all moves the blocks) or peer-mapped
//                           pointers (then the scatter IS the exchange: the stores travel over
//                           NVLink while the kernel is still partitioning).   4 B/key read + 4 B/key
//                           written (locally or on the peers).
//
// The order of keys inside a destination block is irrelevant (a full local sort follows), so the
// multisplit is unstable and ranks keys with plain shared-memory atomicAdd.  (Measured alternative:
// peeling the warp's destinations off one at a time -- one ballot and one atomic per destination
// present -- was slower at 2 GPUs, 1.31 against 1.06 ms: the shuffles cost more than the conflicts.)
#include "dist.cuh"

#include <cstdlib>
#include <cstring>
#include <vector>

namespace b200sort {

constexpr int kDistThreads = 512;
constexpr int kDistIpt = 16;

constexpr int kDistMaxWorld = 16;

// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kDistThreads)
dist_histogram_kernel(const int32_t *__restrict__ keys, size_t n, int bits, unsigned long long *hist)
{
    extern __shared__ uint32_t sh[];                   // 2^bits counters
    const uint32_t nbins = 1u << bits;
    const uint32_t tid = threadIdx.x;
    for (uint32_t i = tid; i < nbins; i += kDistThreads) sh[i] = 0;
    __syncthreads();
    const int shift = 32 - bits;

    size_t head = ((16 - (reinterpret_cast<uintptr_t>(keys) & 15)) & 15) / 4;
    if (head > n) head = n;
    const size_t nvec = (n - head) / 4;
    const size_t tail_start = head + nvec * 4;
    const int4 *v = reinterpret_cast<const int4 *>(keys + head);
    // a block handles at most 2^32 / (its share) keys; counters are 32-bit and n <= 2^30
    for (size_t i = (size_t)blockIdx.x * kDistThreads + tid; i < nvec; i += (size_t)gridDim.x * kDistThreads) {
        const int4 r = ld_stream_v4(v + i);
        atomicAdd(&sh[key_bits(r.x) >> shift], 1u);
        atomicAdd(&sh[key_bits(r.y) >> shift], 1u);
        atomicAdd(&sh[key_bits(r.z) >> shift], 1u);
        atomicAdd(&sh[key_bits(r.w) >> shift], 1u);
    }
    if (blockIdx.x == 0) {
        for (size_t i = tid; i < head; i += kDistThreads) atomicAdd(&sh[key_bits(keys[i]) >> shift], 1u);
        for (size_t i = tail_start + tid; i < n; i += kDistThreads) atomicAdd(&sh[key_bits(keys[i]) >> shift], 1u);
    }
    __syncthreads();
    for (uint32_t i = tid; i < nbins; i += kDistThreads)
        if (sh[i]) atomicAdd(&hist[i], (unsigned long long)sh[i]);
}

// ------------------------------------------------------------------------------------------------
struct DistPartitionArgs {
    int32_t *dst_base[kDistMaxWorld];                  // receive buffer of every rank
    unsigned long long dst_offset[kDistMaxWorld];      // where this rank's block starts in it (host plan)
    const DistPlanDev *plan;                           // non-null: offsets (and the error flag) come from the device plan
    unsigned int *src_hist;                            // HIST: [world][4][256] digit counts of what this rank sends where
};

// Staging area: the tile's keys grouped by destination, with up to 3 pad slots in front of every
// group so that (slot index - index in the destination buffer) is a multiple of 4.  A 16-byte
// aligned vector of the staging area then maps to a 16-byte aligned vector of the destination, and
// the interior of every group leaves with 128-bit stores (4x fewer store instructions and 512-byte
// instead of 128-byte NVLink writes per warp); only group heads and tails use 32-bit stores.


__device__ __forceinline__ void st_stream_v4(int32_t *p, int4 v) {
    asm volatile("st.global.L1::no_allocate.v4.s32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// TMA: the interior of every destination group (whole 16-byte chunks: the staging is co-aligned) leaves with ONE
// bulk copy shared -> global per destination and tile (cp.async.bulk.global.shared::cta; the destination may be
// a peer-mapped buffer: the copy then crosses NVLink in large posted writes); group heads and tails (<= 3 + 3
// words) by ordinary stores.
// HIST: the four 8-bit digit histograms the destination's local sort needs are counted HERE, per destination, in
// shared memory (4 atomics per key that hide under the NVLink-bound transfer) and added to args.src_hist when the CTA
// is done; a reduce-scatter over the ranks then hands every rank the histogram of exactly the keys it received, and
// its local sort skips its own histogram kernel (0.31 ms at 2^28 keys).
template <int THREADS, int OCC, int TMA = 0, int HIST = 0>
__global__ void __launch_bounds__(THREADS, OCC)
dist_partition_kernel(const int32_t *__restrict__ keys, size_t n, int bits, int world,
                      const int *__restrict__ bin_owner, DistPartitionArgs args,
                      unsigned long long *cursor /* [world], zeroed */)
{
    constexpr int kTile = THREADS * kDistIpt;
    constexpr int kSlots = kTile + 4 * kDistMaxWorld;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    int32_t *s_keys = reinterpret_cast<int32_t *>(smem_raw);                  // [kSlots]
    uint8_t *s_dest = reinterpret_cast<uint8_t *>(s_keys + kSlots);       // [kSlots], 0xFF = pad
    uint32_t *s_cnt = reinterpret_cast<uint32_t *>(s_dest + kSlots);      // [kDistMaxWorld]
    uint32_t *s_start = s_cnt + kDistMaxWorld;                                // [kDistMaxWorld + 2]
    unsigned long long *s_gbase = reinterpret_cast<unsigned long long *>(s_start + kDistMaxWorld + 2);
    uint8_t *s_owner = reinterpret_cast<uint8_t *>(s_gbase + kDistMaxWorld);  // [2^bits]
    uint32_t *s_hist = reinterpret_cast<uint32_t *>(s_owner + ((size_t)1 << bits));   // HIST: [world][4][256]

    const uint32_t tid = threadIdx.x;
    const uint32_t nbins = 1u << bits;
    const int shift = 32 - bits;
    if (args.plan != nullptr && args.plan->error) return;     // some receive buffer is too small: nobody writes
    for (uint32_t i = tid; i < nbins; i += THREADS) s_owner[i] = (uint8_t)bin_owner[i];
    if (HIST) for (uint32_t i = tid; i < (uint32_t)world * 1024u; i += THREADS) s_hist[i] = 0;

    const size_t tiles = (n + kTile - 1) / kTile;
    for (size_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const size_t base = tile * kTile;
        const uint32_t valid = (n - base < (size_t)kTile) ? (uint32_t)(n - base) : (uint32_t)kTile;
        if (tid < kDistMaxWorld) s_cnt[tid] = 0;
        if (!TMA)
            for (uint32_t i = tid; i < kSlots / 16; i += THREADS)     // every slot starts as a pad
                reinterpret_cast<uint4 *>(s_dest)[i] = make_uint4(~0u, ~0u, ~0u, ~0u);
        if (TMA) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // my bulk copies have read the staging area
        __syncthreads();                               // also: s_owner ready, previous tile drained

        int32_t key[kDistIpt];
        uint32_t slot[kDistIpt];                       // (dest << 16) | rank inside the tile's dest group
#pragma unroll
        for (int i = 0; i < kDistIpt; ++i) {
            const uint32_t p = i * THREADS + tid;
            if (p < valid) key[i] = ld_stream(keys + base + p);
        }
#pragma unroll
        for (int i = 0; i < kDistIpt; ++i) {
            const uint32_t p = i * THREADS + tid;
            if (p < valid) {
                const uint32_t kb = key_bits(key[i]);
                const uint32_t d = s_owner[kb >> shift];
                slot[i] = (d << 16) | atomicAdd(&s_cnt[d], 1u);
                if (HIST) {
                    uint32_t *h = s_hist + d * 1024u;
                    atomicAdd(h + (kb & 255u), 1u);
                    atomicAdd(h + 256u + ((kb >> 8) & 255u), 1u);
                    atomicAdd(h + 512u + ((kb >> 16) & 255u), 1u);     // the top byte's histogram follows from the bin counts
                }
            }
        }
        __syncthreads();
        if (tid < (uint32_t)world)                     // reserve this tile's share of every destination
            s_gbase[tid] = (args.plan != nullptr ? args.plan->dst_offset[tid] : args.dst_offset[tid]) +
                           (s_cnt[tid] ? atomicAdd(&cursor[tid], (unsigned long long)s_cnt[tid]) : 0ull);
        __syncthreads();
        if (tid == 0) {
            uint32_t run = 0;
            for (int d = 0; d < world; ++d) {
                run += ((uint32_t)s_gbase[d] - run) & 3u;          // co-align staging and destination
                s_start[d] = run;
                run += s_cnt[d];
            }
            s_start[world] = run;
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < kDistIpt; ++i) {
            const uint32_t p = i * THREADS + tid;
            if (p < valid) {
                const uint32_t d = slot[i] >> 16;
                const uint32_t q = s_start[d] + (slot[i] & 0xffffu);
                B200_CHECK_AT(9, q < (uint32_t)kSlots && d < (uint32_t)world);
                s_keys[q] = key[i];
                if (!TMA) s_dest[q] = (uint8_t)d;
            }
        }
        if (TMA) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncthreads();
            if (tid < (uint32_t)world) {
                const uint32_t start = s_start[tid], c = s_cnt[tid];
                int32_t *dst = args.dst_base[tid] + s_gbase[tid];            // element 0 of this tile's group
                uint32_t head = (4u - ((uint32_t)s_gbase[tid] & 3u)) & 3u;
                if (head > c) head = c;
                const uint32_t body = (c - head) & ~3u;
                B200_CHECK_AT(10, body == 0 || (((start + head) & 3u) == 0 && ((s_gbase[tid] + head) & 3ull) == 0));   // 16-byte aligned on both sides
                if (body > 0)
                    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                                 :: "l"(dst + head), "r"((uint32_t)__cvta_generic_to_shared(s_keys + start + head)), "r"(body * 4u) : "memory");
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                for (uint32_t e = 0; e < head; ++e) st_stream(dst + e, s_keys[start + e]);
                for (uint32_t e = head + body; e < c; ++e) st_stream(dst + e, s_keys[start + e]);
            }
            continue;                                  // the loop head waits for the copies and synchronises
        }
        __syncthreads();
        const uint32_t vectors = (s_start[world] + 3) / 4;
        for (uint32_t v = tid; v < vectors; v += THREADS) {
            const uint32_t d4 = reinterpret_cast<const uint32_t *>(s_dest)[v];
            if (d4 == 0xFFFFFFFFu) continue;
            const uint32_t d0 = d4 & 0xFFu;
            if (d4 == d0 * 0x01010101u) {
                const int4 k = reinterpret_cast<const int4 *>(s_keys)[v];
                st_stream_v4(args.dst_base[d0] + s_gbase[d0] + (4 * v - s_start[d0]), k);
            } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const uint32_t d = (d4 >> (8 * e)) & 0xFFu;
                    if (d != 0xFFu)
                        st_stream(args.dst_base[d] + s_gbase[d] + (4 * v + e - s_start[d]), s_keys[4 * v + e]);
                }
            }
        }
        __syncthreads();                               // the staging area is reused by the next tile
    }
    if (TMA) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    if (HIST) {
        __syncthreads();
        for (uint32_t i = tid; i < (uint32_t)world * 1024u; i += THREADS)
            if (s_hist[i]) atomicAdd(&args.src_hist[i], s_hist[i]);
    }
}

// ------------------------------------------------------------------------------------------------
// The planner.  Rank k's range ends at the bin boundary closest to k/world of the keys; exact integer
// arithmetic, one function for the host planner (dist_plan) and the device planner (dist_plan_kernel), so that
// they agree bit for bit.  cum[b] = keys in bins < b (cum[nbins] = total).
__host__ __device__ inline uint32_t plan_boundary(const unsigned long long *cum, uint32_t nbins, uint32_t world, uint32_t k) {
    const unsigned long long total = cum[nbins];
    uint32_t lo = 0, hi = nbins;                       // first b with cum[b] * world >= total * k
    while (lo < hi) {
        const uint32_t mid = (lo + hi) / 2;
        if (cum[mid] * world >= total * k) hi = mid; else lo = mid + 1;
    }
    if (lo > 0) {
        // the bin that straddles the target goes to the NEXT rank if more than half of it lies beyond the target
        const unsigned long long c0 = cum[lo - 1], g = cum[lo] - cum[lo - 1];
        if (c0 > 0 && (2 * c0 + g) * world > 2 * total * k && (c0 + g) * world > total * k) return lo - 1;
    }
    return lo;
}

__global__ void __launch_bounds__(1024)
dist_plan_kernel(const unsigned long long *__restrict__ all_hist, uint32_t world, uint32_t rank, uint32_t nbins,
                 unsigned long long cap, int *bin_owner, DistPlanDev *plan, unsigned long long *cum /* [nbins + 1] */)
{
    __shared__ unsigned long long s_part[32];
    __shared__ uint32_t s_bound[kDistMaxWorld + 1];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // exclusive prefix sums of the global bin counts: every thread owns nbins / 1024 consecutive bins
    const uint32_t per = (nbins + 1023) / 1024;
    const uint32_t b0 = tid * per;
    unsigned long long local = 0;
    for (uint32_t j = 0; j < per && b0 + j < nbins; ++j)
        for (uint32_t r = 0; r < world; ++r) local += all_hist[(size_t)r * nbins + b0 + j];
    unsigned long long x = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= (uint32_t)o) x += y;
    }
    if (lane == 31) s_part[warp] = x;
    __syncthreads();
    if (warp == 0) {
        unsigned long long w = s_part[lane], z = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long y = __shfl_up_sync(0xffffffffu, z, o);
            if (lane >= (uint32_t)o) z += y;
        }
        s_part[lane] = z - w;                          // exclusive over the warps
    }
    __syncthreads();
    unsigned long long run = x - local + s_part[warp];
    for (uint32_t j = 0; j < per && b0 + j < nbins; ++j) {
        cum[b0 + j] = run;
        for (uint32_t r = 0; r < world; ++r) run += all_hist[(size_t)r * nbins + b0 + j];
    }
    if (tid == 1023 || (b0 < nbins && b0 + per >= nbins)) cum[nbins] = run;   // the thread that owns the last bin
    __threadfence_block();
    __syncthreads();
    if (tid <= world) s_bound[tid] = (tid == 0) ? 0u : (tid == world) ? nbins : plan_boundary(cum, nbins, world, tid);
    __syncthreads();
    for (uint32_t b = tid; b < nbins; b += 1024) {
        uint32_t o = 0;
        for (uint32_t k = 1; k < world; ++k) o += (s_bound[k] <= b) ? 1u : 0u;
        bin_owner[b] = (int)o;
    }
    if (tid < 256) {                                   // top-byte histogram of this rank's range: bins t*2^(bits-8) .. of byte t
        const uint32_t per_byte = nbins >> 8, lo = s_bound[rank], hi = s_bound[rank + 1];
        uint32_t c = 0;
        if (per_byte > 0) {
            const uint32_t a = tid * per_byte > lo ? tid * per_byte : lo;
            const uint32_t b = (tid + 1) * per_byte < hi ? (tid + 1) * per_byte : hi;
            if (b > a) c = (uint32_t)(cum[b] - cum[a]);
        }
        plan->top_hist[tid] = c;
    }
    if (tid < world) {
        const unsigned long long rc = cum[s_bound[tid + 1]] - cum[s_bound[tid]];
        plan->recv_count[tid] = rc;
        if (tid == rank) plan->m = (unsigned int)rc;
        if (rc > cap) plan->error = 1u;                // host zeroes the record before the kernel
    }
    // this rank's block inside every destination: keys of the earlier ranks in that destination's range
    for (uint32_t pair = warp; pair < (rank + 1) * world; pair += 32) {
        const uint32_t src = pair / world, o = pair % world;
        unsigned long long acc = 0;
        for (uint32_t b = s_bound[o] + lane; b < s_bound[o + 1]; b += 32) acc += all_hist[(size_t)src * nbins + b];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
        if (lane == 0) {
            if (src == rank) plan->send_count[o] = acc;
            else atomicAdd(&plan->dst_offset[o], acc);
        }
    }
}

// ================================================================================================
// the destination cursors, then (device planner) the prefix sums of the global bin counts
unsigned long long dist_check_failures(unsigned long long *per_site) { return tu_check_failures(per_site); }
size_t dist_workspace_bytes(size_t, int bits) { return 256 + (((size_t)1 << bits) + 1) * sizeof(unsigned long long); }

static size_t partition_smem(int bits, int threads, int hist_world = 0) {
    const size_t slots = (size_t)threads * kDistIpt + 4 * kDistMaxWorld;
    return slots * 4 + slots + (kDistMaxWorld * 2 + 2) * 4 + kDistMaxWorld * 8 + ((size_t)1 << bits) + 16 + (size_t)hist_world * 4096;
}

int dist_histogram(const int32_t *d_keys, size_t n, int bits, unsigned long long *d_hist, cudaStream_t s) {
    if (bits < B200SORT_DIST_BITS_MIN || bits > B200SORT_DIST_BITS_MAX) return B200SORT_ERR_INVALID;
    const size_t nbins = (size_t)1 << bits;
    B200_CUDA_TRY(cudaMemsetAsync(d_hist, 0, nbins * sizeof(unsigned long long), s));
    if (n == 0) return B200SORT_OK;
    const size_t want = div_up(div_up(n, 4), (size_t)kDistThreads * 4);
    const unsigned grid = (unsigned)(want < (size_t)kNumSMs * 3 ? (want ? want : 1) : (size_t)kNumSMs * 3);
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(dist_histogram_kernel),
                                       cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)(((size_t)1 << B200SORT_DIST_BITS_MAX) * sizeof(uint32_t))));
    dist_histogram_kernel<<<grid, kDistThreads, nbins * sizeof(uint32_t), s>>>(d_keys, n, bits, d_hist);
    B200_LAUNCH_CHECK();
    return B200SORT_OK;
}

int dist_plan(const unsigned long long *all_hist, int world, int rank, int bits, int *bin_owner,
              unsigned long long *recv_count, unsigned long long *send_count,
              unsigned long long *dst_offset) {
    if (all_hist == nullptr || bin_owner == nullptr || world < 1 || world > kDistMaxWorld || rank < 0 ||
        rank >= world || bits < B200SORT_DIST_BITS_MIN || bits > B200SORT_DIST_BITS_MAX)
        return B200SORT_ERR_INVALID;
    const size_t nbins = (size_t)1 << bits;
    std::vector<unsigned long long> global(nbins, 0), cum(nbins + 1, 0);
    for (int r = 0; r < world; ++r)
        for (size_t b = 0; b < nbins; ++b) { global[b] += all_hist[(size_t)r * nbins + b]; }
    for (size_t b = 0; b < nbins; ++b) cum[b + 1] = cum[b] + global[b];

    // Contiguous bin ranges: rank r ends at the bin boundary closest to (r+1)/world of the keys (plan_boundary, the
    // function the device planner uses).  Owners are non-decreasing in the bin index, so the concatenation of the
    // ranks' sorted outputs is globally sorted and signed order is kept (bins index key ^ 0x80000000).
    {
        size_t b = 0;
        for (int k = 1; k <= world; ++k) {
            const size_t end = (k == world) ? nbins : plan_boundary(cum.data(), (uint32_t)nbins, (uint32_t)world, (uint32_t)k);
            for (; b < end; ++b) bin_owner[b] = k - 1;
        }
    }
    if (recv_count) std::memset(recv_count, 0, sizeof(unsigned long long) * world);
    if (send_count) std::memset(send_count, 0, sizeof(unsigned long long) * world);
    if (dst_offset) std::memset(dst_offset, 0, sizeof(unsigned long long) * world);
    for (size_t b = 0; b < nbins; ++b) {
        const int o = bin_owner[b];
        if (recv_count) recv_count[o] += global[b];
        if (send_count) send_count[o] += all_hist[(size_t)rank * nbins + b];
        if (dst_offset)
            for (int s = 0; s < rank; ++s) dst_offset[o] += all_hist[(size_t)s * nbins + b];
    }
    return B200SORT_OK;
}

static int partition_launch(const int32_t *d_keys, size_t n, int bits, int world, int32_t *const *h_dst_base,
                            const int *d_bin_owner, const unsigned long long *h_dst_offset, const DistPlanDev *d_plan,
                            void *d_ws, size_t ws_bytes, cudaStream_t s, unsigned int *d_src_hist = nullptr) {
    if (bits < B200SORT_DIST_BITS_MIN || bits > B200SORT_DIST_BITS_MAX || world < 1 || world > kDistMaxWorld ||
        h_dst_base == nullptr || (h_dst_offset == nullptr && d_plan == nullptr) || d_bin_owner == nullptr)
        return B200SORT_ERR_INVALID;
    // Below 8 bits a bin spans more than one top-byte value, so the plan record cannot give row 3 (top_hist stays zero)
    // and source histograms would hand the local sort a wrong top-byte row.
    if (d_src_hist != nullptr && bits < 8) return B200SORT_ERR_INVALID;
    if (d_ws == nullptr || ws_bytes < 256) return B200SORT_ERR_WORKSPACE;
    for (int r = 0; r < world; ++r)       // 128-bit stores / bulk copies into the destinations
        if (reinterpret_cast<uintptr_t>(h_dst_base[r]) & 15) return B200SORT_ERR_INVALID;
    // every call overwrites the source histograms, n == 0 included: a rank that sends nothing contributes zeros
    if (d_src_hist != nullptr)
        B200_CUDA_TRY(cudaMemsetAsync(d_src_hist, 0, (size_t)world * 1024 * sizeof(unsigned int), s));
    if (n == 0) return B200SORT_OK;
    DistPartitionArgs args;
    std::memset(&args, 0, sizeof args);
    for (int r = 0; r < world; ++r) { args.dst_base[r] = h_dst_base[r]; args.dst_offset[r] = h_dst_offset ? h_dst_offset[r] : 0; }
    args.plan = d_plan;
    args.src_hist = d_src_hist;
    if (d_src_hist != nullptr) {                       // histograms ride along: the bulk-copy shape only
        B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(dist_partition_kernel<512, 2, 1, 1>),
                                           cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)partition_smem(B200SORT_DIST_BITS_MAX, 512, kDistMaxWorld)));
        auto *cur = static_cast<unsigned long long *>(d_ws);
        B200_CUDA_TRY(cudaMemsetAsync(cur, 0, sizeof(unsigned long long) * kDistMaxWorld, s));
        const size_t t = div_up(n, (size_t)512 * kDistIpt);
        const unsigned g = (unsigned)(t < (size_t)kNumSMs * 2 ? t : (size_t)kNumSMs * 2);
        dist_partition_kernel<512, 2, 1, 1><<<g, 512, partition_smem(bits, 512, world), s>>>(d_keys, n, bits, world, d_bin_owner, args, cur);
        B200_LAUNCH_CHECK();
        return B200SORT_OK;
    }
    // Compiled shapes: 512 threads x 2 CTAs/SM (8192-key tiles), write-out by bulk copies (default) or by 128-bit
    // stores (B200SORT_DIST_TMA=0); 256 threads x 4 CTAs/SM with stores (B200SORT_DIST_SHAPE=1).
    static const int shape = [] { const char *e = getenv("B200SORT_DIST_SHAPE"); return (e && e[0] == '1') ? 1 : 0; }();
    static const int tma = [] { const char *e = getenv("B200SORT_DIST_TMA"); return (e && e[0] == '0') ? 0 : 1; }();
    // function attributes are per device: set before every launch
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(dist_partition_kernel<512, 2, 0>),
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)partition_smem(B200SORT_DIST_BITS_MAX, 512)));
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(dist_partition_kernel<512, 2, 1>),
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)partition_smem(B200SORT_DIST_BITS_MAX, 512)));
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(dist_partition_kernel<256, 4, 0>),
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)partition_smem(B200SORT_DIST_BITS_MAX, 256)));
    auto *cursor = static_cast<unsigned long long *>(d_ws);
    B200_CUDA_TRY(cudaMemsetAsync(cursor, 0, sizeof(unsigned long long) * kDistMaxWorld, s));
    if (shape == 0) {
        const size_t tiles = div_up(n, (size_t)512 * kDistIpt);
        const unsigned grid = (unsigned)(tiles < (size_t)kNumSMs * 2 ? tiles : (size_t)kNumSMs * 2);
        if (tma) dist_partition_kernel<512, 2, 1><<<grid, 512, partition_smem(bits, 512), s>>>(d_keys, n, bits, world, d_bin_owner, args, cursor);
        else     dist_partition_kernel<512, 2, 0><<<grid, 512, partition_smem(bits, 512), s>>>(d_keys, n, bits, world, d_bin_owner, args, cursor);
    } else {
        const size_t tiles = div_up(n, (size_t)256 * kDistIpt);
        const unsigned grid = (unsigned)(tiles < (size_t)kNumSMs * 4 ? tiles : (size_t)kNumSMs * 4);
        dist_partition_kernel<256, 4, 0><<<grid, 256, partition_smem(bits, 256), s>>>(d_keys, n, bits, world, d_bin_owner, args, cursor);
    }
    B200_LAUNCH_CHECK();
    return B200SORT_OK;
}

int dist_partition(const int32_t *d_keys, size_t n, int bits, int world, int32_t *const *h_dst_base,
                   const int *d_bin_owner, const unsigned long long *h_dst_offset, void *d_ws,
                   size_t ws_bytes, cudaStream_t s) {
    if (h_dst_offset == nullptr) return B200SORT_ERR_INVALID;
    return partition_launch(d_keys, n, bits, world, h_dst_base, d_bin_owner, h_dst_offset, nullptr, d_ws, ws_bytes, s);
}

int dist_partition_planned(const int32_t *d_keys, size_t n, int bits, int world, int32_t *const *h_dst_base,
                           const int *d_bin_owner, const void *d_plan, unsigned int *d_src_hist, void *d_ws, size_t ws_bytes,
                           cudaStream_t s) {
    if (d_plan == nullptr) return B200SORT_ERR_INVALID;
    return partition_launch(d_keys, n, bits, world, h_dst_base, d_bin_owner, nullptr, static_cast<const DistPlanDev *>(d_plan),
                            d_ws, ws_bytes, s, d_src_hist);
}

int dist_plan_device(const unsigned long long *d_all_hist, int world, int rank, int bits, unsigned long long cap,
                     int *d_bin_owner, void *d_plan, void *d_ws, size_t ws_bytes, cudaStream_t s) {
    if (d_all_hist == nullptr || d_bin_owner == nullptr || d_plan == nullptr || world < 1 || world > kDistMaxWorld ||
        rank < 0 || rank >= world || bits < B200SORT_DIST_BITS_MIN || bits > B200SORT_DIST_BITS_MAX)
        return B200SORT_ERR_INVALID;
    if (d_ws == nullptr || ws_bytes < dist_workspace_bytes(0, bits)) return B200SORT_ERR_WORKSPACE;
    B200_CUDA_TRY(cudaMemsetAsync(d_plan, 0, sizeof(DistPlanDev), s));
    auto *cum = reinterpret_cast<unsigned long long *>(static_cast<unsigned char *>(d_ws) + 256);
    dist_plan_kernel<<<1, 1024, 0, s>>>(d_all_hist, (uint32_t)world, (uint32_t)rank, 1u << bits, cap, d_bin_owner,
                                        static_cast<DistPlanDev *>(d_plan), cum);
    B200_LAUNCH_CHECK();
    return B200SORT_OK;
}

}  // namespace b200sort
