// radix_pipelined.cuh -- k2', k2'': the pass as a persistent, software-pipelined CTA (included by radix.cu).
#pragma once
#include "radix_tile.cuh"
#include "radix_async.cuh"

namespace b200sort {

// ================================================================================================
// k2': the same pass as a PERSISTENT, software-pipelined CTA
// ================================================================================================
// One CTA per SM slot loops over tiles (tickets).  14 worker warps load / rank / stage / write the
// keys; 2 chain warps own everything that talks to other tiles (publish the tile's digit counts,
// decoupled look-back with 128-bit status loads, publish the inclusive counts, global offsets).
// The workers never wait for the chain on the tile they are ranking: tile i is written out only
// after tile i+1 has been ranked and staged (double-buffered staging area), and the global loads
// of tile i+1 are in flight while tile i-1 is being written.  So neither the look-back latency
// nor the load latency sits on the workers' critical path.
constexpr int kPPWorkerWarps = 14;
constexpr int kPPWorkers = kPPWorkerWarps * 32;      // 448
constexpr int kPPThreads = 512;
constexpr int kPPChain = kPPThreads - kPPWorkers;    // 64 threads, 4 digits each
constexpr uint32_t kPPPoison = 0xFFFFFFFFu;
constexpr int kPPWindow = 8;                         // status rows in flight per chain thread
enum { kBarW = 1, kBarA = 2, kBarTotals = 3, kBarTstart = 5, kBarGofs = 7 };   // +buffer for the last three

__device__ __forceinline__ void bar_arrive(int id, int count) {
    asm volatile("bar.arrive %0, %1;" :: "r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ uint4 ld_relaxed_gpu_v4(const uint32_t *p) {
    uint4 v;
    asm volatile("ld.relaxed.gpu.global.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_gpu_v4(uint32_t *p, uint4 v) {
    asm volatile("st.relaxed.gpu.global.v4.u32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// Two-level look-back.  Tiles are grouped kPPGroup at a time.  A tile's prefix is
//   (sum of the totals of the earlier GROUPS) + (sum of the totals of the earlier tiles of ITS group).
// Both sums are walks over status rows whose partial values do not depend on any other walk (a
// tile's own total, a group's own total), so no tile waits for a long serial chain: the inclusive
// front only has to advance one GROUP per round trip.  (With one level the front must advance one
// tile per round trip times the window, which is what bounded the pass: ~35 tiles start per
// microsecond and a status round trip through L2 takes ~0.4 us.)
constexpr int kPPGroup = kLookGroup;

// Walk back over status rows: row at distance d (1 <= d <= max_dist) is `first - (d-1)*256`; each
// thread handles four digits with 128-bit loads, W rows in flight.  Flags: 0 not published yet
// (poll again), kFlagLocal partial (keep walking), kFlagIncl inclusive (stop).  Rows beyond
// max_dist count as inclusive zero.  acc[k] += everything taken.
template <int W>
__device__ __forceinline__ void chain_walk(const uint32_t *first, uint32_t max_dist, uint32_t (&acc)[4]) {
    uint32_t need[4] = {1, 1, 1, 1};
    bool done[4] = {false, false, false, false};
    uint32_t back = 1;
    for (;;) {
        uint4 win[W];
#pragma unroll
        for (int j = 0; j < W; ++j)
            win[j] = (back + j <= max_dist) ? ld_relaxed_gpu_v4(first - (size_t)(back + j - 1) * kRadixBins)
                                            : make_uint4(kFlagIncl, kFlagIncl, kFlagIncl, kFlagIncl);
#pragma unroll
        for (int j = 0; j < W; ++j) {
            const uint32_t w4[4] = {win[j].x, win[j].y, win[j].z, win[j].w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (!done[k] && need[k] == back + j) {
                    const uint32_t f = w4[k] & ~kValueMask;
                    if (f != 0) {
                        acc[k] += w4[k] & kValueMask;
                        need[k] += 1;
                        done[k] = (f == kFlagIncl);
                    }
                }
            }
        }
        if (done[0] && done[1] && done[2] && done[3]) break;
        uint32_t nb = 0xFFFFFFFFu;
#pragma unroll
        for (int k = 0; k < 4; ++k) if (!done[k] && need[k] < nb) nb = need[k];
        back = nb;
    }
}

template <int IPT>
struct PipelinedShape {
    static constexpr int kTile = kPPWorkers * IPT;
    static constexpr size_t kSmemBytes =
        (size_t)kPPWorkerWarps * kRadixBins * 4     // per-warp digit counters -> positions
        + (size_t)2 * kTile * 4                     // two staging buffers
        + (size_t)3 * 2 * kRadixBins * 4            // gofs, total, tstart, double-buffered
        + 128;                                      // warp sums, tickets, tile ids
};

template <int IPT>
__global__ void __launch_bounds__(kPPThreads, 2)
radix_onesweep_pipelined_kernel(const int32_t *in_buf, int32_t *out_buf, int32_t *tmp_buf, size_t n,
                                int pass, RadixControl *ctl, uint32_t *status_cur, uint32_t *status_next,
                                int follow_plan)
{
    constexpr int kTile = PipelinedShape<IPT>::kTile;
    static_assert(IPT % 2 == 0 && 32 * IPT < 65536, "ranks are packed in pairs");

    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint32_t *s_table  = reinterpret_cast<uint32_t *>(smem_raw);                     // [14][256]
    int32_t  *s_keys   = reinterpret_cast<int32_t *>(s_table + kPPWorkerWarps * kRadixBins);   // [2][kTile]
    uint32_t *s_gofs   = reinterpret_cast<uint32_t *>(s_keys + 2 * kTile);           // [2][256]
    uint32_t *s_total  = s_gofs + 2 * kRadixBins;                                    // [2][256]
    uint32_t *s_tstart = s_total + 2 * kRadixBins;                                   // [2][256]
    uint32_t *s_misc   = s_tstart + 2 * kRadixBins;     // [0..7] warp sums, [8..9] next ticket, [10..11] tile id

    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const size_t tiles = (n + kTile - 1) / kTile;

    const int32_t *in = in_buf;
    int32_t *out = out_buf;
    if (follow_plan) {
        if (ctl->skip[pass]) {
            const size_t rows = tiles + (tiles + kPPGroup - 1) / kPPGroup;       // tile rows + group rows
            if (status_next != nullptr)
                for (size_t row = blockIdx.x; row < rows; row += gridDim.x)
                    if (tid < kRadixBins) status_next[row * kRadixBins + tid] = 0;
            return;
        }
        const uint32_t ss = ctl->src_sel[pass], ds = ctl->dst_sel[pass];
        in = (ss == kSelIn) ? in_buf : (ss == kSelTmp) ? tmp_buf : out_buf;
        out = (ds == kSelTmp) ? tmp_buf : out_buf;
    }
    const int shift = pass * kRadixBits;
    const uint32_t flip = (pass == kRadixPasses - 1) ? 0x80u : 0u;

    if (warp >= kPPWorkerWarps) {
        // ======================== chain warps ========================
        const uint32_t c4 = (tid - kPPWorkers) * 4;                 // my four digits
        const uint4 base4 = *reinterpret_cast<const uint4 *>(&ctl->base[pass][c4]);
        int b = 0;
        for (;;) {
            bar_sync(kBarTotals + b, kRadixBins + kPPChain);
            const uint32_t tile = s_misc[10 + b];
            if (tile == kPPPoison) break;
            const uint4 tot = *reinterpret_cast<const uint4 *>(s_total + b * kRadixBins + c4);
            const uint32_t group = tile / kPPGroup, r = tile % kPPGroup;
            const bool last_of_group = (r == kPPGroup - 1) || ((size_t)tile + 1 == tiles);
            uint32_t *row = status_cur + (size_t)tile * kRadixBins + c4;                 // tile rows
            uint32_t *grow = status_cur + (tiles + group) * kRadixBins + c4;             // group rows follow
            const uint32_t flag0 = (r == 0) ? kFlagIncl : kFlagLocal;                    // inclusive WITHIN the group
            st_relaxed_gpu_v4(row, make_uint4(flag0 | tot.x, flag0 | tot.y, flag0 | tot.z, flag0 | tot.w));
            if (status_next != nullptr) {
                *reinterpret_cast<uint4 *>(status_next + (size_t)tile * kRadixBins + c4) = make_uint4(0, 0, 0, 0);
                if (last_of_group)
                    *reinterpret_cast<uint4 *>(status_next + (tiles + group) * kRadixBins + c4) = make_uint4(0, 0, 0, 0);
            }
            // level 1: earlier tiles of my group
            uint32_t prev[4] = {0, 0, 0, 0};
            if (r > 0) {
                chain_walk<kPPWindow>(row - kRadixBins, r, prev);
                st_relaxed_gpu_v4(row, make_uint4(kFlagIncl | (prev[0] + tot.x), kFlagIncl | (prev[1] + tot.y),
                                                  kFlagIncl | (prev[2] + tot.z), kFlagIncl | (prev[3] + tot.w)));
            }
            // level 2: earlier groups (the last tile of a group owns the group's row)
            const uint32_t gflag = (group == 0) ? kFlagIncl : kFlagLocal;
            const uint4 gtot = make_uint4(prev[0] + tot.x, prev[1] + tot.y, prev[2] + tot.z, prev[3] + tot.w);
            if (last_of_group)
                st_relaxed_gpu_v4(grow, make_uint4(gflag | gtot.x, gflag | gtot.y, gflag | gtot.z, gflag | gtot.w));
            if (group > 0) {
                uint32_t gprev[4] = {0, 0, 0, 0};
                chain_walk<kPPWindow>(grow - kRadixBins, group, gprev);
                if (last_of_group)
                    st_relaxed_gpu_v4(grow, make_uint4(kFlagIncl | ((gprev[0] + gtot.x) & kValueMask),
                                                       kFlagIncl | ((gprev[1] + gtot.y) & kValueMask),
                                                       kFlagIncl | ((gprev[2] + gtot.z) & kValueMask),
                                                       kFlagIncl | ((gprev[3] + gtot.w) & kValueMask)));
#pragma unroll
                for (int k = 0; k < 4; ++k) prev[k] += gprev[k];
            }
            __syncwarp();
            bar_sync(kBarTstart + b, kRadixBins + kPPChain);
            const uint4 ts = *reinterpret_cast<const uint4 *>(s_tstart + b * kRadixBins + c4);
            *reinterpret_cast<uint4 *>(s_gofs + b * kRadixBins + c4) =
                make_uint4(base4.x + prev[0] - ts.x, base4.y + prev[1] - ts.y,
                           base4.z + prev[2] - ts.z, base4.w + prev[3] - ts.w);
            __threadfence_block();
            bar_arrive(kBarGofs + b, kPPThreads);
            b ^= 1;
        }
        return;
    }

    // ============================ worker warps ============================
    uint32_t *wt = s_table + warp * kRadixBins;
    {
        uint4 *z = reinterpret_cast<uint4 *>(wt);
#pragma unroll
        for (int j = lane; j < kRadixBins / 4; j += 32) z[j] = make_uint4(0, 0, 0, 0);
    }
    if (tid == 0) s_misc[8] = atomicAdd(&ctl->ticket[pass], 1u);
    bar_sync(kBarW, kPPWorkers);
    uint32_t tile = s_misc[8];
    uint32_t prev_tile = kPPPoison;
    const uint32_t wofs = warp * (32 * IPT) + lane;

    int32_t key[IPT];
    auto load_tile = [&](uint32_t t) {
        const size_t tile_base = (size_t)t * kTile;
        const uint32_t valid = (n - tile_base < (size_t)kTile) ? (uint32_t)(n - tile_base) : (uint32_t)kTile;
        const int32_t *src = in + tile_base + wofs;
        if (valid == (uint32_t)kTile) {
#pragma unroll
            for (int i = 0; i < IPT; ++i) key[i] = ld_stream(src + i * 32);
        } else {
#pragma unroll
            for (int i = 0; i < IPT; ++i)
                key[i] = (wofs + i * 32 < valid) ? ld_stream(src + i * 32) : 0x7FFFFFFF;
        }
    };
    auto write_tile = [&](uint32_t t, int buf) {
        const size_t tile_base = (size_t)t * kTile;
        const uint32_t valid = (n - tile_base < (size_t)kTile) ? (uint32_t)(n - tile_base) : (uint32_t)kTile;
        const int32_t *sk = s_keys + buf * kTile;
        const uint32_t *go = s_gofs + buf * kRadixBins;
        if (valid == (uint32_t)kTile) {
#pragma unroll
            for (int j = 0; j < IPT; ++j) {
                const uint32_t p = tid + j * kPPWorkers;
                const int32_t k = sk[p];
                st_stream(out + (size_t)(uint32_t)(go[digit_of(k, shift, flip)] + p), k);
            }
        } else {
#pragma unroll
            for (int j = 0; j < IPT; ++j) {
                const uint32_t p = tid + j * kPPWorkers;
                if (p < valid) {
                    const int32_t k = sk[p];
                    st_stream(out + (size_t)(uint32_t)(go[digit_of(k, shift, flip)] + p), k);
                }
            }
        }
    };

    if (tile < tiles) load_tile(tile);
    int b = 0;
    uint32_t iter = 0;
    while (tile < tiles) {
        // ---- rank: one shared-memory atomicAdd per key (lane-ordered; see the self-test) ----------
        uint32_t rank2[IPT / 2];
#pragma unroll
        for (int i = 0; i < IPT; ++i) {
            const uint32_t r = atomicAdd(wt + digit_of(key[i], shift, flip), 1u);
            rank2[i / 2] = (i & 1) ? (rank2[i / 2] | (r << 16)) : r;
        }
        bar_sync(kBarW, kPPWorkers);
        // next ticket (everybody has read the slot being overwritten: that read precedes this barrier)
        if (tid == 0) s_misc[8 + ((iter + 1) & 1)] = atomicAdd(&ctl->ticket[pass], 1u);

        // ---- threads 0..255, thread = digit: totals -> chain; scan; counts -> positions ----------
        if (tid < kRadixBins) {
            uint32_t total = 0;
#pragma unroll
            for (int w = 0; w < kPPWorkerWarps; ++w) total += s_table[w * kRadixBins + tid];
            s_total[b * kRadixBins + tid] = total;
            if (tid == 0) s_misc[10 + b] = tile;
            __threadfence_block();
            bar_arrive(kBarTotals + b, kRadixBins + kPPChain);
            uint32_t x = total;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
                if (lane >= (uint32_t)o) x += y;
            }
            if (lane == 31) s_misc[warp] = x;
            bar_sync(kBarA, kRadixBins);
            uint32_t add = 0;
#pragma unroll
            for (int w = 0; w < kRadixBins / 32; ++w) add += (w < (int)warp) ? s_misc[w] : 0u;
            const uint32_t tile_start = x - total + add;
            uint32_t run = tile_start;
#pragma unroll
            for (int w = 0; w < kPPWorkerWarps; ++w) {
                const uint32_t c = s_table[w * kRadixBins + tid];
                s_table[w * kRadixBins + tid] = run;
                run += c;
            }
            s_tstart[b * kRadixBins + tid] = tile_start;
            __threadfence_block();
            bar_arrive(kBarTstart + b, kRadixBins + kPPChain);
        }
        bar_sync(kBarW, kPPWorkers);                       // positions are final
        const uint32_t next = s_misc[8 + ((iter + 1) & 1)];

        // ---- stage this tile's keys in digit order ----------------------------------------------------
        {
            int32_t *sk = s_keys + b * kTile;
#pragma unroll
            for (int i = 0; i < IPT; ++i) {
                const uint32_t r = (i & 1) ? (rank2[i / 2] >> 16) : (rank2[i / 2] & 0xffffu);
                sk[wt[digit_of(key[i], shift, flip)] + r] = key[i];
            }
        }
        __syncwarp();
        {
            uint4 *z = reinterpret_cast<uint4 *>(wt);      // my warp's counters, for the next tile
#pragma unroll
            for (int j = lane; j < kRadixBins / 4; j += 32) z[j] = make_uint4(0, 0, 0, 0);
        }
        __syncwarp();

        // ---- loads of the next tile go out now and land while the previous tile is written ----
        if (next < tiles) load_tile(next);
        if (prev_tile != kPPPoison) {
            bar_sync(kBarGofs + (b ^ 1), kPPThreads);      // the chain finished tile i-1 long ago
            write_tile(prev_tile, b ^ 1);
        }
        prev_tile = tile;
        tile = next;
        b ^= 1;
        ++iter;
    }
    if (prev_tile != kPPPoison) {
        bar_sync(kBarW, kPPWorkers);                       // the last tile is fully staged
        bar_sync(kBarGofs + (b ^ 1), kPPThreads);
        write_tile(prev_tile, b ^ 1);
    }
    if (tid < kRadixBins) {                                // release the chain warps
        if (tid == 0) s_misc[10 + b] = kPPPoison;
        __threadfence_block();
        bar_arrive(kBarTotals + b, kRadixBins + kPPChain);
    }
}

// ================================================================================================
// k2'': persistent CTA, every warp a worker, DELAYED two-level look-back
// ================================================================================================
// What the phase probe showed (profiles/r01_phase_timing.txt): a tile needs the counts of the tiles
// that started a few hundred nanoseconds before it, and those are often not published yet --
// the look-back does not wait for a long chain but for STRAGGLERS among its ~32 nearest
// predecessors, 4-5 us of a 9 us tile lifetime, with the SM's registers and shared memory held idle.
// Here the CTA does not wait: it publishes tile i's counts, then ranks and stages tile i+1, and only
// then resolves tile i's prefix -- by which time every straggler has long published -- and writes
// tile i out.  The two-level rows make that possible: a tile's own total and a group's own total do
// not depend on anybody's look-back, so delaying one's OWN prefix delays nobody else.  Only the last
// tile of each group sums its group right away (1 tile in 32 waits for stragglers).
//   tile row  : kFlagLocal = the tile's digit counts, kFlagIncl = inclusive within its group
//   group row : kFlagLocal = the group's digit counts, kFlagIncl = inclusive over all groups
// SPLIT: the previous tile's two look-back walks run concurrently, one per thread group (see below).
// PACK : two warps share one row of digit counters, 16 bits each (8 rows instead of 16): half the
//        shared-memory traffic of the digit phase and of the zeroing.
// KV   : every key carries a 32-bit value through the pass (sort-by-key; SURVEY section 8(f)-4): the
//        values are loaded, staged and written beside the keys, so the staging area doubles.
// PFW1 / PFW2: status rows of the previous tile's look-back that ONE thread fetches into shared memory with two bulk
// loads (TMA) underneath the ranking: the nearest PFW1 tile rows of its group and the nearest PFW2 group rows.
constexpr int kPfw1 = 12, kPfw2 = 6;                 // 18 KB: what is left of 2 x 113 KB per SM beside the 10240-key tile
template <int IPT, int PACK = 0, int KV = 0, int PFW = 0>
struct Pipelined2Shape {
    static constexpr int kThreads = 512;
    static constexpr int kTile = kThreads * IPT;
    static constexpr int kRows = PACK ? 8 : 16;
    static constexpr size_t kSmemBytes =
        (size_t)kRows * kRadixBins * 4              // per-warp digit counters -> positions
        + (size_t)(KV ? 4 : 2) * kTile * 4          // two staging buffers (keys; KV: and two for the values)
        + (size_t)(2 + 1 + 2 + 1) * kRadixBins * 4  // gofs[2], total, tstart[2], previous tile's group prefix
        + 128
        + (PFW ? (size_t)(kPfw1 + kPfw2) * kRadixBins * 4 : 0);
};

// EG   : the last tile of a group makes its GROUP row inclusive at once (it walks the earlier group rows
//        right after publishing the group's own total) instead of one iteration later, so that every other
//        tile's walk over the group rows ends at the first row it reads.
// OVL  : no CTA barrier between the digit phase and the staging.  Group A stages as soon as ITS positions
//        are final; group B walks the previous tile's tile rows, sends the first window of group-row loads
//        off, stages while they fly, then finishes the walk.  One CTA barrier before the write-out.
// SAFE : rank with eight __ballot_sync per key and ONE atomic per distinct digit of the warp instruction (documented
//        behaviour only) instead of one atomic per key (which needs same-address lanes to be resolved in lane order).
// DEVN : the key count is read from the control block (written by the histogram kernel from a device pointer,
//        radix_sort_devn) instead of the kernel argument.  A separate instantiation: as a run-time switch it cost
//        the default kernel 64 bytes of spills and 4 % (0.696 -> 0.726 ms per pass).
// KEYS = 1: any key order (RadixControl::key_neg / key_pos / key_pad); 0: int32 ascending.
template <int IPT, int TIMING, int SPLIT, int PACK, int KV, int EG = 0, int OVL = 0, int LATE = 0, int SAFE = 0, int PFW = 0, int DEVN = 0,
          int KEYS = 0>
__device__ __forceinline__ void
radix_onesweep_pipelined2_body(const int32_t *in_buf, int32_t *out_buf, int32_t *tmp_buf, size_t n,
                               int pass, RadixControl *ctl, uint32_t *status_cur, uint32_t *status_next,
                               int follow_plan, const int32_t *in_vals, int32_t *out_vals, int32_t *tmp_vals)
{
    constexpr int kThreads = 512;
    constexpr int kTile = Pipelined2Shape<IPT, PACK, KV>::kTile;
    constexpr int kRows = Pipelined2Shape<IPT, PACK, KV>::kRows;
    constexpr int W = 8;                                      // status rows in flight per thread
    static_assert(IPT % 2 == 0 && 32 * IPT < 65536, "ranks are packed in pairs");
    static_assert(kTile + 64 < 65536, "PACK keeps 16-bit positions");
    static_assert(!(OVL && SPLIT), "OVL restructures the unsplit resolve");
    static_assert(!PFW || (!SPLIT && !OVL && !EG), "the prefetched look-back is written for the unsplit resolve");

    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint32_t *s_table  = reinterpret_cast<uint32_t *>(smem_raw);                      // [kRows][256]
    int32_t  *s_keys   = reinterpret_cast<int32_t *>(s_table + kRows * kRadixBins);   // [2][kTile]
    int32_t  *s_vals   = s_keys + 2 * kTile;                                          // KV: [2][kTile]
    uint32_t *s_gofs   = reinterpret_cast<uint32_t *>(s_keys + (KV ? 4 : 2) * kTile); // [2][256]
    uint32_t *s_total  = s_gofs + 2 * kRadixBins;                                     // [256]
    uint32_t *s_tstart = s_total + kRadixBins;                                        // [2][256]
    uint32_t *s_g2     = s_tstart + 2 * kRadixBins;           // [256] SPLIT: previous tile's prefix over earlier groups
    uint32_t *s_misc   = s_g2 + kRadixBins;                   // [0..7] warp sums, [8..9] tickets, [16..17] mbarrier
    uint32_t *s_win1   = s_misc + 32;                         // PFW: [kPfw1][256] nearest tile rows, [kPfw2][256] group rows
    uint32_t *s_win2   = s_win1 + kPfw1 * kRadixBins;

    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // The tile count (and, DEVN, the key count produced on the device: radix_sort_devn) lives in shared memory and is
    // re-read where it is needed: held in registers it pushed the kernel over its 64 (16 to 64 bytes of spills).
    if (tid == 0) {
        const uint32_t n32 = DEVN ? ctl->n_dev : (uint32_t)n;
        s_misc[20] = n32;
        s_misc[21] = (uint32_t)(((size_t)n32 + kTile - 1) / kTile);
        if (KEYS && SAFE) s_misc[22] = flips_of(ctl->key_neg, ctl->key_pos, pass * kRadixBits);
    }
    __syncthreads();
    auto n_f = [&]() -> size_t { return DEVN ? (size_t)reinterpret_cast<volatile uint32_t *>(s_misc)[20] : n; };
    auto tiles_f = [&]() -> size_t { return (size_t)reinterpret_cast<volatile uint32_t *>(s_misc)[21]; };

    const int32_t *in = in_buf;
    int32_t *out = out_buf;
    const int32_t *vin = in_vals;
    int32_t *vout = out_vals;
    if (follow_plan) {
        if (ctl->skip[pass]) {
            const size_t rows = tiles_f() + (tiles_f() + kLookGroup - 1) / kLookGroup;
            if (status_next != nullptr)
                for (size_t row = blockIdx.x; row < rows; row += gridDim.x)
                    if (tid < kRadixBins) status_next[row * kRadixBins + tid] = 0;
            return;
        }
        const uint32_t ss = ctl->src_sel[pass], ds = ctl->dst_sel[pass];
        in = (ss == kSelIn) ? in_buf : (ss == kSelTmp) ? tmp_buf : out_buf;
        out = (ds == kSelTmp) ? tmp_buf : out_buf;
        if (KV) {                                             // the values follow the keys' plan
            vin = (ss == kSelIn) ? in_vals : (ss == kSelTmp) ? tmp_vals : out_vals;
            vout = (ds == kSelTmp) ? tmp_vals : out_vals;
        }
    }
    const int shift = pass * kRadixBits;
    const uint32_t flip = (pass == kRadixPasses - 1) ? 0x80u : 0u;
    // the ballot-ranked shape (SAFE) already spills for int32: there the order's bytes are re-read from shared memory
    // (s_misc[22]) at every use instead of taking a register
    const uint32_t flips = (KEYS && !SAFE) ? flips_of(ctl->key_neg, ctl->key_pos, shift) : 0u;
    auto dig = [&](int32_t k) -> uint32_t {
        if (!KEYS) return digit_of(k, shift, flip);
        return digit_of_image(k, shift, SAFE ? reinterpret_cast<volatile uint32_t *>(s_misc)[22] : flips);
    };
    const uint32_t lt = lanemask_lt();
    const bool in_a = tid < kRadixBins;                       // warps 0..7 : thread = digit
    const bool in_b = !in_a;                                  // warps 8..15: thread - 256 = digit
    const uint32_t bd = tid - kRadixBins;
    // my warp's counters: a row of its own, or (PACK) one 16-bit half of the row it shares with warp ^ 1
    uint32_t *wt = s_table + (PACK ? (warp >> 1) : warp) * kRadixBins;
    const uint32_t sh = PACK ? (warp & 1) * 16 : 0;
    const uint32_t wofs = warp * (32 * IPT) + lane;
    auto my_half = [&](uint32_t word) -> uint32_t { return PACK ? ((word >> sh) & 0xffffu) : word; };
    auto zero_counters = [&]() {
        uint4 *z = reinterpret_cast<uint4 *>(wt);
        if (PACK) {
            z[(warp & 1) * 32 + lane] = make_uint4(0, 0, 0, 0);      // each warp of the pair clears half the row
        } else {
#pragma unroll
            for (int j = lane; j < kRadixBins / 4; j += 32) z[j] = make_uint4(0, 0, 0, 0);
        }
    };
    auto pair_bar = [&]() { bar_sync(3 + (warp >> 1), 64); };     // the two warps that share a counter row

    int32_t key[IPT];
    int32_t val[KV ? IPT : 1];
    auto load_tile = [&](uint32_t t) {
        const size_t tile_base = (size_t)t * kTile;
        const uint32_t valid = (n_f() - tile_base < (size_t)kTile) ? (uint32_t)(n_f() - tile_base) : (uint32_t)kTile;
        const int32_t *src = in + tile_base + wofs;
        if (valid == (uint32_t)kTile) {
#pragma unroll
            for (int i = 0; i < IPT; ++i) key[i] = ld_stream(src + i * 32);
        } else {
#pragma unroll
            for (int i = 0; i < IPT; ++i)
                key[i] = (wofs + i * 32 < valid) ? ld_stream(src + i * 32) : (KEYS ? (int32_t)ctl->key_pad : 0x7FFFFFFF);
        }
        if (KV) {
            const int32_t *vsrc = vin + tile_base + wofs;
#pragma unroll
            for (int i = 0; i < (KV ? IPT : 0); ++i)
                val[i] = (wofs + i * 32 < valid) ? ld_stream(vsrc + i * 32) : 0;
        }
    };
    auto write_tile = [&](uint32_t t, int buf) {
        const size_t tile_base = (size_t)t * kTile;
        const uint32_t valid = (n_f() - tile_base < (size_t)kTile) ? (uint32_t)(n_f() - tile_base) : (uint32_t)kTile;
        const int32_t *sk = s_keys + buf * kTile;
        const int32_t *sv = s_vals + buf * kTile;
        const uint32_t *go = s_gofs + buf * kRadixBins;
        if (valid == (uint32_t)kTile) {
#pragma unroll
            for (int j = 0; j < IPT; ++j) {
                const uint32_t p = tid + j * kThreads;
                const int32_t k = sk[p];
                const size_t dst = (size_t)(uint32_t)(go[dig(k)] + p);
                B200_CHECK_AT(2, dst < n_f());
                st_stream(out + dst, k);
                if (KV) st_stream(vout + dst, sv[p]);
            }
        } else {
#pragma unroll
            for (int j = 0; j < IPT; ++j) {
                const uint32_t p = tid + j * kThreads;
                if (p < valid) {
                    const int32_t k = sk[p];
                    const size_t dst = (size_t)(uint32_t)(go[dig(k)] + p);
                    B200_CHECK_AT(2, dst < n_f());
                    st_stream(out + dst, k);
                    if (KV) st_stream(vout + dst, sv[p]);
                }
            }
        }
    };

    // group B's memory of the previous tile (the one whose prefix is resolved one iteration late)
    uint32_t digit_base = in_b ? ctl->base[pass][bd] : 0u;
    uint32_t p_total = 0, p_in = 0;                           // its count of my digit; in-group prefix if known
    bool p_in_known = false;
    uint32_t p_g = 0;                                         // EG: its prefix over the earlier groups, if known
    bool p_g_known = false;
    // PFW: rows of the previous tile's look-back fetched by bulk load (issued when the iteration begins)
    const uint32_t pf_mbar = smem_u32(&s_misc[16]);
    uint32_t pf_have1 = 0, pf_have2 = 0, pf_parity = 0;
    auto prefetch_rows = [&](uint32_t pt) {                   // every thread computes the counts, one thread issues
        const uint32_t group = pt / kLookGroup, r = pt % kLookGroup;
        const bool last_of_group = (r == kLookGroup - 1) || ((size_t)pt + 1 == tiles_f());
        pf_have1 = last_of_group ? 0u : (r < (uint32_t)kPfw1 ? r : (uint32_t)kPfw1);
        pf_have2 = group < (uint32_t)kPfw2 ? group : (uint32_t)kPfw2;
        if (tid == kRadixBins && pf_have1 + pf_have2 > 0) {
            fence_proxy_async_smem();
            mbar_expect_tx(pf_mbar, (pf_have1 + pf_have2) * kRadixBins * 4);
            if (pf_have1) bulk_load(smem_u32(s_win1), status_cur + ((size_t)pt - pf_have1) * kRadixBins, pf_have1 * kRadixBins * 4, pf_mbar);
            if (pf_have2) bulk_load(smem_u32(s_win2), status_cur + (tiles_f() + group - pf_have2) * kRadixBins, pf_have2 * kRadixBins * 4, pf_mbar);
        }
    };
    // !SPLIT: the previous tile's look-back, run by group B alone: fills s_gofs[buf].
    auto resolve_prev = [&](uint32_t pt, int buf) {
        const uint32_t group = pt / kLookGroup, r = pt % kLookGroup;
        const bool last_of_group = (r == kLookGroup - 1) || ((size_t)pt + 1 == tiles_f());
        uint32_t *row = status_cur + (size_t)pt * kRadixBins + bd;
        uint32_t *grow = status_cur + (tiles_f() + group) * kRadixBins + bd;
        if (PFW && pf_have1 + pf_have2 > 0) { mbar_wait(pf_mbar, pf_parity); pf_parity ^= 1; }   // the fetched rows have landed
        uint32_t inprev = p_in;
        if (!p_in_known) {
            inprev = (r > 0) ? (PFW ? walk_back_prefetched<W>(s_win1 + bd, pf_have1, row - kRadixBins, r)
                                    : walk_back<W>(row - kRadixBins, r)) : 0u;
            if (r > 0) st_relaxed_gpu(row, kFlagIncl | (inprev + p_total));   // shortens later walks
        }
        uint32_t gprev = 0;
        if (group > 0) {
            if (EG && p_g_known) {
                gprev = p_g;                                  // summed (and published) when the tile was published
            } else {
                gprev = PFW ? walk_back_prefetched<W>(s_win2 + bd, pf_have2, grow - kRadixBins, group)
                            : walk_back<W>(grow - kRadixBins, group);
                if (last_of_group) st_relaxed_gpu(grow, kFlagIncl | ((gprev + inprev + p_total) & kValueMask));
            }
        }
        // the run lies inside the array (the last tile's count of digit 255 includes its padding slots)
        B200_CHECK_AT(3, (size_t)digit_base + inprev + gprev + (((size_t)pt + 1 == tiles_f()) ? 0u : p_total) <= n_f());
        s_gofs[buf * kRadixBins + bd] = digit_base + inprev + gprev - s_tstart[buf * kRadixBins + bd];
    };
    // SPLIT: the two walks are given to the two groups and started before anything else in the digit
    // phase, because a dependent global round trip costs ~2500 cycles in this kernel (it queues behind
    // the shared-memory traffic of both CTAs on the SM):
    //   group A (thread = digit) loads the first window of GROUP rows, does its digit work while the
    //           loads are in flight, finishes the walk and leaves the prefix in s_g2;
    //   group B (thread = digit) walks the TILE rows of the previous tile's group, then publishes this
    //           tile's counts, and after SYNC2 combines both prefixes into s_gofs[buf].
    constexpr int W1 = 12, W2 = 8;               // (16, 8) and (8, 8) spill; this pair does not
    uint32_t win2[W2];
    auto level2_load = [&](uint32_t pt, uint32_t dg) {
        const uint32_t group = pt / kLookGroup;
        const uint32_t *first = status_cur + (tiles_f() + group) * kRadixBins + dg - kRadixBins;
#pragma unroll
        for (int j = 0; j < W2; ++j)
            win2[j] = ((uint32_t)(j + 1) <= group) ? ld_relaxed_gpu(first - (size_t)j * kRadixBins) : kFlagIncl;
    };
    auto level2_finish = [&](uint32_t pt, uint32_t dg) -> uint32_t {
        const uint32_t group = pt / kLookGroup;
        const uint32_t *first = status_cur + (tiles_f() + group) * kRadixBins + dg - kRadixBins;
        uint32_t acc = 0, back = 1;
        bool have = true;
        for (;;) {
            if (!have) {
#pragma unroll
                for (int j = 0; j < W2; ++j)
                    win2[j] = (back + j <= group) ? ld_relaxed_gpu(first - (size_t)(back + j - 1) * kRadixBins) : kFlagIncl;
            }
            have = false;
            bool done = false;
            uint32_t used = 0;
#pragma unroll
            for (int j = 0; j < W2; ++j) {
                if (!done && used == (uint32_t)j) {
                    const uint32_t f = win2[j] & ~kValueMask;
                    if (f != 0) { acc += win2[j] & kValueMask; used = j + 1; done = (f == kFlagIncl); }
                }
            }
            if (done) break;
            back += used;
        }
        return acc;
    };
    auto level1 = [&](uint32_t pt) -> uint32_t {       // group B
        if (p_in_known) return p_in;                 // the last tile of a group summed its group when it published
        const uint32_t r = pt % kLookGroup;
        uint32_t *row = status_cur + (size_t)pt * kRadixBins + bd;
        const uint32_t in = (r > 0) ? walk_back<W1>(row - kRadixBins, r) : 0u;
        if (r > 0) st_relaxed_gpu(row, kFlagIncl | (in + p_total));        // shortens later walks
        return in;
    };
    auto combine_prev = [&](uint32_t pt, int buf, uint32_t q_total, uint32_t q_in) {   // group B, after A's level2_finish
        const uint32_t group = pt / kLookGroup;
        const bool last = (pt % kLookGroup == kLookGroup - 1) || ((size_t)pt + 1 == tiles_f());
        const uint32_t gprev = s_g2[bd];
        if (last && group > 0)
            st_relaxed_gpu(status_cur + (tiles_f() + group) * kRadixBins + bd, kFlagIncl | ((gprev + q_in + q_total) & kValueMask));
        s_gofs[buf * kRadixBins + bd] = digit_base + q_in + gprev - s_tstart[buf * kRadixBins + bd];
    };

    zero_counters();
    if (tid == 0) {
        s_misc[8] = atomicAdd(&ctl->ticket[pass], 1u);
        if (PFW) { mbar_init(pf_mbar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    }
    __syncthreads();
    uint32_t tile = s_misc[8];
    uint32_t prev_tile = 0xFFFFFFFFu;
    if (tile < tiles_f()) load_tile(tile);
    int b = 0;
    uint32_t iter = 0;

    while (tile < tiles_f()) {
        const uint32_t dbg_tile = tile;
        if (TIMING) { asm volatile("" :: "r"(key[0]), "r"(key[IPT - 1])); }
        B200_STAMP(0);                                        // this tile's keys are in registers
        if (PFW) { pf_have1 = pf_have2 = 0; if (prev_tile != 0xFFFFFFFFu) prefetch_rows(prev_tile); }
        if (PACK) pair_bar();                                 // my partner has cleared its half of our counter row
        // ---- rank: one shared-memory atomicAdd per key (lane-ordered; see the self-test) ----------
        uint32_t rank2[IPT / 2];
        {
            const uint32_t d0 = dig(key[0]);
            const uint32_t agree = __ballot_sync(0xffffffffu, d0 == __shfl_sync(0xffffffffu, d0, 0));
            // hot digit of the pass (the histogram kernel found one value holding > 1/8 of the keys), else
            // a locally hot one (a quarter of the warp's first keys agree with lane 0's: sorted input)
            const uint32_t hot_word = follow_plan ? ctl->hot[pass] : 0u;
            const bool hot = hot_word != 0 || __popc(agree) >= 8;
            if (SAFE) {
#pragma unroll
                for (int i = 0; i < IPT; ++i) {
                    const uint32_t d = dig(key[i]);
                    uint32_t peers = 0xffffffffu;                 // lanes of this instruction that hold my digit
#pragma unroll
                    for (int bit = 0; bit < kRadixBits; ++bit) {
                        const bool one = (d >> bit) & 1u;
                        const uint32_t vote = __ballot_sync(0xffffffffu, one);
                        peers &= one ? vote : ~vote;
                    }
                    const uint32_t lower = peers & lt;
                    uint32_t before = 0;
                    if (lower == 0) before = my_half(atomicAdd(wt + d, (uint32_t)__popc(peers) << sh));   // one lane per digit
                    before = __shfl_sync(0xffffffffu, before, __ffs(peers) - 1);
                    const uint32_t r = before + __popc(lower);
                    rank2[i / 2] = (i & 1) ? (rank2[i / 2] | (r << 16)) : r;
                }
            } else if (!hot) {
#pragma unroll
                for (int i = 0; i < IPT; ++i) {
                    const uint32_t r = my_half(atomicAdd(wt + dig(key[i]), 1u << sh));
                    rank2[i / 2] = (i & 1) ? (rank2[i / 2] | (r << 16)) : r;
                }
            } else {
                // the lanes that hold the hot digit are ranked with one ballot and ONE atomic (by their first
                // lane); the others take the atomic as usual
#pragma unroll
                for (int i = 0; i < IPT; ++i) {
                    const uint32_t d = dig(key[i]);
                    const uint32_t hd = hot_word ? hot_word - 1u : __shfl_sync(0xffffffffu, d, 0);
                    const bool same = (d == hd);
                    const uint32_t sm = __ballot_sync(0xffffffffu, same);
                    const uint32_t leader = (uint32_t)(__ffs(sm) - 1) & 31u;
                    uint32_t r = 0;
                    if (!same || lane == leader) r = my_half(atomicAdd(wt + d, (same ? (uint32_t)__popc(sm) : 1u) << sh));
                    const uint32_t r0 = __shfl_sync(0xffffffffu, r, leader);
                    if (same) r = r0 + __popc(sm & lt);
                    rank2[i / 2] = (i & 1) ? (rank2[i / 2] | (r << 16)) : r;
                }
            }
        }
        if (TIMING) { asm volatile("" :: "r"(rank2[0]), "r"(rank2[IPT / 2 - 1])); }
        B200_STAMP(1);                                        // ranked
        __syncthreads();                                      // SYNC1: counts are final
        B200_STAMP(2);
        if (!LATE && tid == 0) s_misc[8 + ((iter + 1) & 1)] = atomicAdd(&ctl->ticket[pass], 1u);

        const bool have_prev = prev_tile != 0xFFFFFFFFu;
        uint32_t q_total_keep = 0, q_in_keep = 0;             // SPLIT, group B: the previous tile's count and in-group prefix
        uint32_t o_total = 0, o_in = 0, o_g = 0;              // OVL, group B: the same, and its prefix over the groups
        bool o_g_known = false;
        if (in_a) {
            if (SPLIT && have_prev && prev_tile / kLookGroup > 0) level2_load(prev_tile, tid);
            // thread = digit: tile totals -> group B; exclusive scan; warp counts -> positions
            uint32_t total = 0;
#pragma unroll
            for (int w = 0; w < kRows; ++w) {
                const uint32_t c = s_table[w * kRadixBins + tid];
                total += PACK ? (c & 0xffffu) + (c >> 16) : c;
            }
            s_total[tid] = total;
            __threadfence_block();
            bar_arrive(2, 512);
            uint32_t x = total;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
                if (lane >= (uint32_t)o) x += y;
            }
            if (lane == 31) s_misc[warp] = x;
            bar_sync(1, kRadixBins);
            uint32_t add = 0;
#pragma unroll
            for (int w = 0; w < kRadixBins / 32; ++w) add += (w < (int)warp) ? s_misc[w] : 0u;
            const uint32_t tile_start = x - total + add;
            uint32_t run = tile_start;
#pragma unroll
            for (int w = 0; w < kRows; ++w) {
                const uint32_t c = s_table[w * kRadixBins + tid];
                if (PACK) {                                   // warp 2w's keys first, then warp 2w+1's
                    const uint32_t lo = c & 0xffffu;
                    s_table[w * kRadixBins + tid] = run | ((run + lo) << 16);
                    run += lo + (c >> 16);
                } else {
                    s_table[w * kRadixBins + tid] = run;
                    run += c;
                }
            }
            s_tstart[b * kRadixBins + tid] = tile_start;
            if (SPLIT && have_prev) s_g2[tid] = (prev_tile / kLookGroup > 0) ? level2_finish(prev_tile, tid) : 0u;
            if (OVL) {                                        // positions final: group B may stage; so may group A
                __threadfence_block();
                bar_arrive(11, 512);
                bar_sync(12, kRadixBins);
            }
            B200_STAMP(3);                                    // group A done
        } else {
            if (SPLIT) {
                // the previous tile's in-group prefix first (it needs nothing from this tile) ...
                q_total_keep = p_total;
                if (have_prev) q_in_keep = level1(prev_tile);
                B200_STAMP(11);                               // previous tile: level-1 prefix known
            }
            // ... publish this tile's counts ...
            bar_sync(2, 512);
            const uint32_t total = s_total[bd];
            const uint32_t group = tile / kLookGroup, r = tile % kLookGroup;
            const bool last_of_group = (r == kLookGroup - 1) || ((size_t)tile + 1 == tiles_f());
            uint32_t *row = status_cur + (size_t)tile * kRadixBins + bd;
            st_relaxed_gpu(row, (r == 0 ? kFlagIncl : kFlagLocal) | total);
            if (status_next != nullptr) {
                status_next[(size_t)tile * kRadixBins + bd] = 0;
                if (last_of_group) status_next[(tiles_f() + group) * kRadixBins + bd] = 0;
            }
            B200_STAMP(10);                                   // published
            if (!SPLIT && !OVL) {
                // ... resolve the PREVIOUS tile's prefix (everything it needs was published long ago) ...
                if (have_prev) resolve_prev(prev_tile, b ^ 1);
                B200_STAMP(11);                               // previous tile resolved
            }
            if (OVL && have_prev) {
                // ... the previous tile's in-group prefix now, the first window of its group rows sent off ...
                o_total = p_total;
                o_in = level1(prev_tile);
                o_g_known = EG && p_g_known;
                o_g = p_g;
                if (prev_tile / kLookGroup > 0 && !o_g_known) level2_load(prev_tile, bd);
                B200_STAMP(11);
            }
            // ... and, for the last tile of a group only, sum the group now so that nobody after
            // it has to wait an iteration for the group's total
            p_total = total;
            p_in_known = false;
            p_g_known = false;
            if (last_of_group) {
                p_in = (r > 0) ? walk_back<W>(row - kRadixBins, r) : 0u;
                p_in_known = true;
                if (r > 0) st_relaxed_gpu(row, kFlagIncl | (p_in + total));
                uint32_t *grow = status_cur + (tiles_f() + group) * kRadixBins + bd;
                st_relaxed_gpu(grow, (group == 0 ? kFlagIncl : kFlagLocal) | (p_in + total));
                if (EG && !SPLIT && group > 0) {
                    // every row this walk waits for is published by a running CTA before that CTA waits for
                    // anything (its group's own total first, then its walk), so the walk terminates
                    p_g = walk_back<W>(grow - kRadixBins, group);
                    p_g_known = true;
                    st_relaxed_gpu(grow, kFlagIncl | ((p_g + p_in + total) & kValueMask));
                }
            }
            __syncwarp();
            // LATE: the next tile's ticket is drawn AFTER the look-back (the one phase whose length varies), so that
            // from ticket to publication every tile takes the same time and tiles_f() are published in ticket order
            if (LATE && tid == kRadixBins) {
                const uint32_t t_next = atomicAdd(&ctl->ticket[pass], 1u);
                s_misc[8 + ((iter + 1) & 1)] = t_next;
                // ... and the tile some CTA will draw half a round of tickets from now is sent for (TMA prefetch into L2):
                // the loads an SM can have in flight are bounded by the L1 its CTAs' shared memory leaves (60 KB here),
                // so how long a load is in flight -- HBM or L2 -- bounds how fast the keys come in
                const size_t t_far = (size_t)t_next + gridDim.x / 2;
                if (t_far < tiles_f()) {
                    const size_t left = (n_f() - t_far * kTile) * 4;
                    const uint32_t bytes = (uint32_t)((left < (size_t)kTile * 4 ? left : (size_t)kTile * 4) & ~(size_t)15);
                    if (bytes > 0) {
                        bulk_prefetch_l2(reinterpret_cast<const void *>(reinterpret_cast<uintptr_t>(in + t_far * kTile) & ~(uintptr_t)15), bytes);
                        if (KV) bulk_prefetch_l2(reinterpret_cast<const void *>(reinterpret_cast<uintptr_t>(vin + t_far * kTile) & ~(uintptr_t)15), bytes);
                    }
                }
            }
            if (OVL) bar_sync(11, 512);                       // group A's positions are final
            B200_STAMP(3);                                    // group B done
        }
        if (!OVL) __syncthreads();                            // SYNC2: positions final; previous tile: offsets (SPLIT: both prefixes) known
        if (SPLIT && in_b && have_prev) combine_prev(prev_tile, b ^ 1, q_total_keep, q_in_keep);
        B200_STAMP(4);
        const uint32_t next = s_misc[8 + ((iter + 1) & 1)];

        // ---- stage this tile's keys in digit order ----------------------------------------------------
        {
            int32_t *sk = s_keys + b * kTile;
            int32_t *sv = s_vals + b * kTile;
#pragma unroll
            for (int i = 0; i < IPT; ++i) {
                const uint32_t r = (i & 1) ? (rank2[i / 2] >> 16) : (rank2[i / 2] & 0xffffu);
                const uint32_t pos = my_half(wt[dig(key[i])]) + r;
                B200_CHECK_AT(1, pos < (uint32_t)kTile);
                sk[pos] = key[i];
                if (KV) sv[pos] = val[KV ? i : 0];
            }
        }
        // the counters are cleared for the next tile once nobody reads positions from them any more
        if (PACK && !SPLIT) pair_bar(); else __syncwarp();
        if (!(PACK && SPLIT)) { zero_counters(); __syncwarp(); }
        B200_STAMP(5);                                        // staged
        // ---- the next tile's loads go out now and land while the previous tile is written --------
        if (next < tiles_f()) load_tile(next);
        B200_STAMP(6);
        if (SPLIT) {
            __syncthreads();                                  // SYNC3: the previous tile's offsets are in s_gofs
            if (PACK) zero_counters();
        }
        if (OVL) {
            if (in_b && have_prev) {                          // finish the previous tile's walk over the group rows
                const uint32_t pg = prev_tile / kLookGroup;
                const bool plast = (prev_tile % kLookGroup == kLookGroup - 1) || ((size_t)prev_tile + 1 == tiles_f());
                uint32_t gprev = 0;
                if (pg > 0) {
                    if (o_g_known) gprev = o_g;
                    else {
                        gprev = level2_finish(prev_tile, bd);
                        if (plast) st_relaxed_gpu(status_cur + (tiles_f() + pg) * kRadixBins + bd,
                                                  kFlagIncl | ((gprev + o_in + o_total) & kValueMask));
                    }
                }
                s_gofs[(b ^ 1) * kRadixBins + bd] = digit_base + o_in + gprev - s_tstart[(b ^ 1) * kRadixBins + bd];
            }
            __syncthreads();                                  // the previous tile's offsets are in s_gofs
        }
        if (have_prev) write_tile(prev_tile, b ^ 1);
        B200_STAMP(7);                                        // previous tile written
        if (TIMING && g_phase_dbg != nullptr && lane == 0 && (warp == 0 || warp == 8))
            g_phase_dbg[((size_t)dbg_tile * 2 + (warp >> 3)) * 16 + 9] = tile;
        prev_tile = tile;
        tile = next;
        b ^= 1;
        ++iter;
    }
    // ---- drain: the last tile is staged, its prefix is still to be resolved ----------------------------
    if (prev_tile != 0xFFFFFFFFu) {
        __syncthreads();
        if (SPLIT) {
            uint32_t q_in = 0;
            if (in_a) { if (prev_tile / kLookGroup > 0) { level2_load(prev_tile, tid); s_g2[tid] = level2_finish(prev_tile, tid); } else s_g2[tid] = 0; }
            else q_in = level1(prev_tile);
            __syncthreads();
            if (in_b) combine_prev(prev_tile, b ^ 1, p_total, q_in);
        } else {
            if (PFW) pf_have1 = pf_have2 = 0;                 // nothing was fetched for the last tile
            if (in_b) resolve_prev(prev_tile, b ^ 1);
        }
        __syncthreads();
        write_tile(prev_tile, b ^ 1);
    }
}

// MINB: CTAs per SM the register allocation is held to (3 with tiles of <= 6144 keys: 40 registers).
template <int IPT, int TIMING = 0, int SPLIT = 0, int PACK = 0, int MINB = 2, int EG = 0, int OVL = 0, int LATE = 0, int SAFE = 0, int PFW = 0, int DEVN = 0,
          int KEYS = 0>
__global__ void __launch_bounds__(512, MINB)
radix_onesweep_pipelined2_kernel(const int32_t *in_buf, int32_t *out_buf, int32_t *tmp_buf, size_t n,
                                 int pass, RadixControl *ctl, uint32_t *status_cur, uint32_t *status_next,
                                 int follow_plan)
{
    radix_onesweep_pipelined2_body<IPT, TIMING, SPLIT, PACK, 0, EG, OVL, LATE, SAFE, PFW, DEVN, KEYS>(in_buf, out_buf, tmp_buf, n, pass, ctl, status_cur,
                                                                status_next, follow_plan, nullptr, nullptr, nullptr);
}

// Sort-by-key: the same pass with a 32-bit value riding along with every key.
template <int IPT, int SAFE = 0, int KEYS = 0>
__global__ void __launch_bounds__(512, 2)
radix_onesweep_pairs_kernel(const int32_t *in_buf, int32_t *out_buf, int32_t *tmp_buf, size_t n,
                            int pass, RadixControl *ctl, uint32_t *status_cur, uint32_t *status_next,
                            int follow_plan, const int32_t *in_vals, int32_t *out_vals, int32_t *tmp_vals)
{
    radix_onesweep_pipelined2_body<IPT, 0, 0, 1, 1, 0, 0, 1, SAFE, 0, 0, KEYS>(in_buf, out_buf, tmp_buf, n, pass, ctl, status_cur,
                                                    status_next, follow_plan, in_vals, out_vals, tmp_vals);
}

}  // namespace b200sort
