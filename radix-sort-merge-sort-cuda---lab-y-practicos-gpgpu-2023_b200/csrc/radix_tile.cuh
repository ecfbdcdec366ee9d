// radix_tile.cuh -- k2: one onesweep pass, one tile per CTA; shared look-back helpers (included by radix.cu).
#pragma once
#include "radix.cuh"
#include "radix_digit.cuh"

#include <cooperative_groups.h>

namespace cg = cooperative_groups;

namespace b200sort {

// ================================================================================================
// k2: one onesweep pass
// ================================================================================================

// How a warp finds, for each of its 32 current keys, the lanes holding the same digit:
//   kRankMatch   __match_any_sync (one MATCH instruction; runs on the ADU pipe)
//   kRankBallot  eight __ballot_sync, one per digit bit (VOTE + LOP3, no shared memory)
//   kRankAtomic  atomicOr of the lane bit into a per-warp {peer mask, count} table in shared memory
//   kRankAdd     EXPERIMENT: plain atomicAdd, stable only if the hardware resolves same-address
//                lanes of one instruction in lane order (undocumented)
enum RankMode { kRankMatch = 0, kRankBallot = 1, kRankAtomic = 2, kRankAdd = 3 };

template <int WARPS, int IPT, int MODE>
struct OnesweepShape {
    static constexpr int kThreads = WARPS * 32;
    static constexpr int kTile    = kThreads * IPT;
    static constexpr int kTableWords = (MODE == kRankAtomic) ? 2 : 1;   // words per (warp, digit)
    static constexpr size_t kSmemBytes =
        (size_t)WARPS * kRadixBins * 4 * kTableWords   // per-warp digit counters -> offsets
        + (size_t)kTile * 4                            // keys staged in digit order
        + (size_t)kRadixBins * 4 * 4                   // global offset, tile total, tile start, chain prefix
        + 64;                                          // warp sums, tile id
};

// ---- two-level look-back ---------------------------------------------------------------------------
// Measured with the phase probe (tools/phase_timing.py): with one level the look-back takes 4.7 us of
// a 9 us tile lifetime.  The inclusive front can only advance (window / L2 round trip) = 8 / 0.26 us
// = 31 tiles per microsecond, which is exactly the rate the pass ran at: the chain, not the SMs,
// set the speed.  With two levels tiles are grouped kLookGroup at a time and a tile's prefix is
//   (totals of the earlier GROUPS) + (totals of the earlier tiles of ITS group);
// both are walks over rows whose partial values (a tile's own total, a group's own total) do not
// depend on any other walk, so nobody waits for a long serial chain.
constexpr int kLookGroup = 32;

// Walk back over status rows for one digit: the row at distance d (1 <= d <= max_dist) is
// first - (d-1)*256.  Flags: 0 not published (poll again), kFlagLocal partial (keep walking),
// kFlagIncl inclusive (stop).  Rows beyond max_dist count as inclusive zero.
template <int W>
__device__ __forceinline__ uint32_t walk_back(const uint32_t *first, uint32_t max_dist) {
    uint32_t acc = 0, back = 1;
    for (;;) {
        uint32_t win[W];
#pragma unroll
        for (int j = 0; j < W; ++j)
            win[j] = (back + j <= max_dist) ? ld_relaxed_gpu(first - (size_t)(back + j - 1) * kRadixBins) : kFlagIncl;
        bool done = false;
        uint32_t used = 0;
#pragma unroll
        for (int j = 0; j < W; ++j) {
            if (!done && used == (uint32_t)j) {
                const uint32_t f = win[j] & ~kValueMask;
                if (f != 0) {
                    acc += win[j] & kValueMask;
                    used = j + 1;
                    done = (f == kFlagIncl);
                }
            }
        }
        if (done) return acc;
        back += used;
    }
}

// CL > 1: the CTAs of a thread-block cluster take CL consecutive tiles and act as ONE link of the
// look-back chain: tile totals are exchanged through distributed shared memory, the last CTA of
// the cluster publishes / looks back for all of them and hands the result to its peers.  The
// chain then has CL times fewer links, which is what bounds the pass once ranking is cheap.
__device__ __forceinline__ void cluster_arrive() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_wait() {
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// Phase-timing probe (TIMING variants only): lane 0 of warp 0 (group A) and of warp 8 (group B)
// stamp clock64() at the phase boundaries into g_phase_dbg[tile][2][16].
__device__ long long *g_phase_dbg = nullptr;
#define B200_STAMP(slot)                                                                  \
    do {                                                                                  \
        if (TIMING && g_phase_dbg != nullptr && lane == 0 && (warp == 0 || warp == 8))    \
            g_phase_dbg[((size_t)dbg_tile * 2 + (warp >> 3)) * 16 + (slot)] = clock64();  \
    } while (0)

// PF > 0: after issuing its own loads a CTA prefetches into L2 the tile PF tickets ahead (the
// tile some CTA will pick up about one CTA-lifetime later), so that tile's loads hit L2.
// BSF: group B stages its keys before consuming the look-back window instead of after.
// TL: two-level look-back (tile rows + group rows, see walk_back below); implies BSF.
template <int WARPS, int IPT, int MIN_BLOCKS, int MODE, int CL, int PF = 0, int BSF = 0, int TIMING = 0, int TL = 0>
__global__ void __launch_bounds__(WARPS * 32, MIN_BLOCKS)
radix_onesweep_kernel(const int32_t *in_buf, int32_t *out_buf, int32_t *tmp_buf, size_t n, int pass,
                      RadixControl *ctl, uint32_t *status_cur, uint32_t *status_next,
                      int follow_plan)
{
    using Shape = OnesweepShape<WARPS, IPT, MODE>;
    constexpr int kThreads = Shape::kThreads;
    constexpr int kTile    = Shape::kTile;
    constexpr int TW       = Shape::kTableWords;
    static_assert(WARPS >= kRadixBins / 32, "need one thread per digit");

    extern __shared__ __align__(16) unsigned char smem_raw[];
    // [WARPS][256] entries of TW words.  Entry word TW-1 is the running count, later the offset
    // of (warp, digit) inside the staged tile; with kRankAtomic word 0 is the peer mask.
    uint32_t *s_table = reinterpret_cast<uint32_t *>(smem_raw);
    int32_t  *s_keys  = reinterpret_cast<int32_t *>(s_table + WARPS * kRadixBins * TW);
    uint32_t *s_gofs  = reinterpret_cast<uint32_t *>(s_keys + kTile);             // [256]
    uint32_t *s_misc  = s_gofs + kRadixBins;                                      // [16]

    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t dbg_tile = blockIdx.x;
    B200_STAMP(0);

    // follow_plan: buffers and skipping come from the plan the histogram kernel wrote.
    const int32_t *in = in_buf;
    int32_t *out = out_buf;
    if (follow_plan) {
        if (ctl->skip[pass]) {
            // Identity pass.  Still hand the next pass a clean status buffer.
            if (status_next != nullptr && tid < kRadixBins && blockIdx.x % CL == 0)
                status_next[(size_t)(blockIdx.x / CL) * kRadixBins + tid] = 0;
            if (TL && status_next != nullptr && tid < kRadixBins && blockIdx.x % kLookGroup == 0)
                status_next[((n + kTile - 1) / kTile + blockIdx.x / kLookGroup) * kRadixBins + tid] = 0;
            return;
        }
        const uint32_t ss = ctl->src_sel[pass], ds = ctl->dst_sel[pass];
        in = (ss == kSelIn) ? in_buf : (ss == kSelTmp) ? tmp_buf : out_buf;
        out = (ds == kSelTmp) ? tmp_buf : out_buf;
    }

    // Tiles are handed out by ticket so that a tile only ever waits on tiles already running.
    uint32_t crank = 0;                                      // my rank inside the cluster
    if (CL > 1) {
        cg::cluster_group cluster = cg::this_cluster();
        crank = cluster.block_rank();
        if (crank == 0 && tid == 0) {
            const uint32_t t = atomicAdd(&ctl->ticket[pass], 1u);
            for (int q = 0; q < CL; ++q) cluster.map_shared_rank(s_misc, q)[8] = t;
        }
    } else {
        if (tid == 0) s_misc[8] = atomicAdd(&ctl->ticket[pass], 1u);
    }
    {
        uint4 *z = reinterpret_cast<uint4 *>(s_table + warp * kRadixBins * TW);
#pragma unroll
        for (int j = lane; j < kRadixBins * TW / 4; j += 32) z[j] = make_uint4(0, 0, 0, 0);
    }
    if (CL > 1) { cluster_arrive(); cluster_wait(); } else __syncthreads();
    const uint32_t link = s_misc[8];                         // my link of the look-back chain
    const uint32_t tile = link * CL + crank;
    B200_STAMP(1);
    const size_t tile_base = (size_t)tile * kTile;
    const uint32_t valid = (tile_base >= n) ? 0u
                         : (n - tile_base < (size_t)kTile) ? (uint32_t)(n - tile_base) : (uint32_t)kTile;
    const int shift = pass * kRadixBits;
    const uint32_t flip = (pass == kRadixPasses - 1) ? 0x80u : 0u;

    // ---- load, warp-striped: item i of lane l is key warp*32*IPT + i*32 + l of the tile ---------
    int32_t key[IPT];
    {
        const uint32_t wofs = warp * (32 * IPT) + lane;
        const int32_t *src = in + tile_base + wofs;
        if (valid == (uint32_t)kTile) {
#pragma unroll
            for (int i = 0; i < IPT; ++i) key[i] = ld_stream(src + i * 32);
        } else {
#pragma unroll
            for (int i = 0; i < IPT; ++i)
                key[i] = (wofs + i * 32 < valid) ? ld_stream(src + i * 32) : 0x7FFFFFFF;  // sorts last
        }
    }
    if (PF > 0) {
        constexpr uint32_t kLines = (uint32_t)kTile * 4 / 128;
        const size_t ahead = ((size_t)tile + PF) * kTile + (size_t)tid * 32;
        if (tid < kLines && ahead + 32 <= n)
            asm volatile("prefetch.global.L2 [%0];" :: "l"(in + ahead));
        if (kLines > (uint32_t)kThreads && tid + kThreads < kLines && ahead + (size_t)kThreads * 32 + 32 <= n)
            asm volatile("prefetch.global.L2 [%0];" :: "l"(in + ahead + (size_t)kThreads * 32));
    }

    if (TIMING) { asm volatile("" :: "r"(key[0]), "r"(key[IPT - 1])); B200_STAMP(2); }   // loads have landed
    // ---- rank inside the warp: earlier keys of this warp with my digit ----------------------------
    // (two 16-bit ranks per register: a warp holds at most 32*IPT < 65536 keys)
    static_assert(IPT % 2 == 0 && 32 * IPT < 65536, "ranks are packed in pairs");
    uint32_t rank2[IPT / 2];
    {
        uint32_t *wt = s_table + warp * kRadixBins * TW;
        const uint32_t lt = lanemask_lt();
        // "hot" = some digit value is frequent: globally (the histogram kernel saw one bin with more
        // than 1/8 of the keys) or in this warp's part of the tile (sorted / clustered input: a
        // quarter of the lanes agree with lane 0 on the first key).  Warp-uniform.
        bool hot = false;
        if (MODE == kRankAdd) {
            const uint32_t d0 = digit_of(key[0], shift, flip);
            const uint32_t agree = __ballot_sync(0xffffffffu, d0 == __shfl_sync(0xffffffffu, d0, 0));
            hot = (follow_plan && ctl->hot[pass] != 0) || __popc(agree) >= 8;
        }
        if (MODE == kRankAdd && !hot) {
            // the common case, kept free of any per-key branch
#pragma unroll
            for (int i = 0; i < IPT; ++i) {
                const uint32_t r = atomicAdd(wt + digit_of(key[i], shift, flip), 1u);
                rank2[i / 2] = (i & 1) ? (rank2[i / 2] | (r << 16)) : r;
            }
        } else {
#pragma unroll
        for (int i = 0; i < IPT; ++i) {
            const uint32_t d = digit_of(key[i], shift, flip);
            if (MODE == kRankAdd) {
                // A digit value is frequent: same-address atomics would serialise.  The lanes that
                // share lane 0's digit are ranked with one ballot and ONE atomic.
                const bool same = (d == __shfl_sync(0xffffffffu, d, 0));
                const uint32_t sm = __ballot_sync(0xffffffffu, same);
                uint32_t r = 0;
                if (!same || lane == 0) r = atomicAdd(wt + d, lane == 0 ? (uint32_t)__popc(sm) : 1u);
                const uint32_t r0 = __shfl_sync(0xffffffffu, r, 0);
                if (same) r = r0 + __popc(sm & lt);
                rank2[i / 2] = (i & 1) ? (rank2[i / 2] | (r << 16)) : r;
            } else if (MODE == kRankAtomic) {
                atomicOr(wt + 2 * d, 1u << lane);
                __syncwarp();
                const uint2 e = *reinterpret_cast<const uint2 *>(wt + 2 * d);   // {peers, count}
                const uint32_t lower = e.x & lt;
                const uint32_t r = e.y + __popc(lower);
                rank2[i / 2] = (i & 1) ? (rank2[i / 2] | (r << 16)) : r;
                __syncwarp();
                if (lower == 0)                                                   // lowest peer
                    *reinterpret_cast<uint2 *>(wt + 2 * d) = make_uint2(0u, e.y + __popc(e.x));
                __syncwarp();
            } else {
                uint32_t peers;
                if (MODE == kRankMatch) {
                    peers = __match_any_sync(0xffffffffu, d);
                } else {
                    peers = 0xffffffffu;
#pragma unroll
                    for (int b = 0; b < kRadixBits; ++b) {
                        const bool bit = (d >> b) & 1u;
                        const uint32_t vote = __ballot_sync(0xffffffffu, bit);
                        peers &= bit ? vote : ~vote;
                    }
                }
                const uint32_t lower = peers & lt;
                uint32_t before = 0;
                if (lower == 0) before = atomicAdd(wt + d, (uint32_t)__popc(peers));   // one lane per digit
                before = __shfl_sync(0xffffffffu, before, __ffs(peers) - 1);
                const uint32_t r = before + __popc(lower);
                rank2[i / 2] = (i & 1) ? (rank2[i / 2] | (r << 16)) : r;
            }
        }
        }
    }
    if (TIMING) { asm volatile("" :: "r"(rank2[0]), "r"(rank2[IPT / 2 - 1])); B200_STAMP(3); }   // ranked
    __syncthreads();
    B200_STAMP(4);

    // ---- per digit, two thread groups working side by side --------------------------------------
    //   group A (threads 0..255, thread = digit): tile totals, exclusive scan over the digits,
    //           warp counts -> positions inside the staged tile;
    //   group B (threads 256..511, thread - 256 = digit; the same threads as A when the CTA has
    //           fewer than 16 warps): publish the tile total, decoupled look-back over the
    //           predecessor tiles with kLookWindow status words in flight per thread, publish the
    //           inclusive count, global offset of the digit.
    // Status words only ever move 0 -> local -> inclusive, so a stale (prefetched) read is safe.
    // Named barriers: 1 = inside group A; 2 = "totals are in shared memory" (A arrives, B waits);
    //                 3 = "positions are final" (A arrives, B waits).
    constexpr bool kSplit = (WARPS >= 16);
    constexpr int kLookWindow = (CL == 1 && IPT <= 16) ? 16 : 8;
    uint32_t *s_total = s_misc + 16;                         // [256]
    uint32_t *s_tstart = s_total + kRadixBins;               // [256]
    uint32_t *s_prev = s_tstart + kRadixBins;                // [256] (clusters: written by the looker)

    const bool in_a = tid < kRadixBins;
    const bool in_b = kSplit ? (tid >= kRadixBins && tid < 2 * kRadixBins) : in_a;
    const uint32_t bd = kSplit ? tid - kRadixBins : tid;     // group B's digit
    const uint32_t *look = status_cur + (size_t)link * kRadixBins + bd;   // my digit in my link's row
    const bool looker = (CL == 1) || (crank == CL - 1);      // the CTA that talks to the chain

    uint32_t win[kLookWindow];
    uint32_t digit_base = 0;                                 // global start of my digit (group B)
    if (in_b) digit_base = ctl->base[pass][bd];              // fetched early: it is off the critical path
    if (kSplit && in_b && looker && !TL) {
        // first window, issued before anything else so that it overlaps group A's work
#pragma unroll
        for (int j = 0; j < kLookWindow; ++j)
            win[j] = (link >= (uint32_t)(j + 1)) ? ld_relaxed_gpu(look - (size_t)(j + 1) * kRadixBins)
                                                 : kFlagIncl;            // before link 0: inclusive 0
    }
    if (in_a) {
        uint32_t total = 0;
#pragma unroll
        for (int w = 0; w < WARPS; ++w) total += s_table[(w * kRadixBins + tid) * TW + (TW - 1)];
        s_total[tid] = total;
        if (CL > 1) cluster_arrive();                        // #1: my totals are in shared memory
        if (kSplit) { __threadfence_block(); asm volatile("bar.arrive 2, 512;" ::: "memory"); }
        uint32_t x = total;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= (uint32_t)o) x += y;
        }
        if (lane == 31) s_misc[warp] = x;
        asm volatile("bar.sync 1, 256;" ::: "memory");
        uint32_t add = 0;
#pragma unroll
        for (int w = 0; w < kRadixBins / 32; ++w) add += (w < (int)warp) ? s_misc[w] : 0u;
        const uint32_t tile_start = x - total + add;
        uint32_t run = tile_start;
#pragma unroll
        for (int w = 0; w < WARPS; ++w) {
            uint32_t *e = s_table + (w * kRadixBins + tid) * TW + (TW - 1);
            const uint32_t c = *e;
            *e = run;
            run += c;
        }
        s_tstart[tid] = tile_start;
        if (kSplit) { __threadfence_block(); asm volatile("bar.arrive 3, %0;" :: "n"(WARPS * 32) : "memory"); }
        asm volatile("bar.sync 1, 256;" ::: "memory");      // every (warp, digit) position is final
        if (CL > 1) { cluster_wait(); cluster_arrive(); }    // finish #1; #2: nothing to announce
        B200_STAMP(5);                                       // group A done
    }
    if (CL > 1 && !in_a && !in_b) { cluster_arrive(); cluster_wait(); cluster_arrive(); }
    if (kSplit && !in_a && !in_b) asm volatile("bar.sync 3, %0;" :: "n"(WARPS * 32) : "memory");   // warps 16..: wait for the positions
    if (in_b) {
        if (kSplit) asm volatile("bar.sync 2, 512;" ::: "memory");
        uint32_t total = s_total[bd];                        // my tile; becomes my link's total
        uint32_t before = 0;                                 // same digit in earlier tiles of my link
        if (CL > 1) {
            if (kSplit) cluster_arrive();                    // #1 (group A arrived for itself)
            cluster_wait();                                  // every CTA's totals are readable
            cg::cluster_group cluster = cg::this_cluster();
            uint32_t rest = 0;
#pragma unroll
            for (int q = 0; q < CL; ++q) {
                if (looker ? (q < CL - 1) : (q < (int)crank)) {
                    const uint32_t c = cluster.map_shared_rank(s_total, q)[bd];
                    if (q < (int)crank) before += c;
                    rest += c;
                }
            }
            if (looker) total += rest;
        }
        uint32_t prev = 0;
        if (TL) {
            static_assert(!TL || (CL == 1 && WARPS >= 16), "two-level look-back: split CTAs without clusters");
            const size_t num_tiles = (n + kTile - 1) / kTile;
            const uint32_t group = tile / kLookGroup, r = tile % kLookGroup;
            const bool last_of_group = (r == kLookGroup - 1) || ((size_t)tile + 1 == num_tiles);
            uint32_t *row = status_cur + (size_t)tile * kRadixBins + bd;                   // tile rows ...
            uint32_t *grow = status_cur + (num_tiles + group) * kRadixBins + bd;           // ... then group rows
            st_relaxed_gpu(row, (r == 0 ? kFlagIncl : kFlagLocal) | total);               // inclusive WITHIN the group
            if (status_next != nullptr) {
                status_next[(size_t)tile * kRadixBins + bd] = 0;
                if (last_of_group) status_next[(num_tiles + group) * kRadixBins + bd] = 0;
            }
            // stage my keys now (positions are final once group A says so): that frees their
            // registers for the windows below and overlaps with the predecessors' publishing
            asm volatile("bar.sync 3, %0;" :: "n"(WARPS * 32) : "memory");
#pragma unroll
            for (int i = 0; i < IPT; ++i) {
                const uint32_t d = digit_of(key[i], shift, flip);
                const uint32_t rk = (i & 1) ? (rank2[i / 2] >> 16) : (rank2[i / 2] & 0xffffu);
                s_keys[s_table[(warp * kRadixBins + d) * TW + (TW - 1)] + rk] = key[i];
            }
            B200_STAMP(10);                                  // staged, walks start
            uint32_t inprev = 0;
            if (r > 0) {
                inprev = walk_back<16>(row - kRadixBins, r);
                st_relaxed_gpu(row, kFlagIncl | (inprev + total));
            }
            B200_STAMP(11);                                  // level 1 done
            const uint32_t gtot = inprev + total;
            if (last_of_group) st_relaxed_gpu(grow, (group == 0 ? kFlagIncl : kFlagLocal) | gtot);
            uint32_t gprev = 0;
            if (group > 0) {
                gprev = walk_back<16>(grow - kRadixBins, group);
                if (last_of_group) st_relaxed_gpu(grow, kFlagIncl | ((gprev + gtot) & kValueMask));
            }
            prev = inprev + gprev;
            B200_STAMP(12);                                  // level 2 done
        }
        if (!TL && looker) {
            st_relaxed_gpu(const_cast<uint32_t *>(look), (link == 0 ? kFlagIncl : kFlagLocal) | total);
            if (status_next != nullptr) status_next[(size_t)link * kRadixBins + bd] = 0;
        }
        if (!TL && BSF && kSplit && CL == 1) {
            // positions are final as soon as group A says so: stage my keys while the prefetched
            // status words are still in flight
            asm volatile("bar.sync 3, %0;" :: "n"(WARPS * 32) : "memory");
#pragma unroll
            for (int i = 0; i < IPT; ++i) {
                const uint32_t d = digit_of(key[i], shift, flip);
                const uint32_t r = (i & 1) ? (rank2[i / 2] >> 16) : (rank2[i / 2] & 0xffffu);
                s_keys[s_table[(warp * kRadixBins + d) * TW + (TW - 1)] + r] = key[i];
            }
        }
        if (!TL && looker) {
            if (link > 0) {
                uint32_t back = 1;                           // distance of the window's first link
                bool have = kSplit;                          // window already loaded?
                for (;;) {
                    if (!have) {
#pragma unroll
                        for (int j = 0; j < kLookWindow; ++j)
                            win[j] = (link >= back + j) ? ld_relaxed_gpu(look - (size_t)(back + j) * kRadixBins)
                                                        : kFlagIncl;
                    }
                    have = false;
                    bool done = false;
                    uint32_t used = 0;
#pragma unroll
                    for (int j = 0; j < kLookWindow; ++j) {
                        if (!done && used == (uint32_t)j) {
                            const uint32_t f = win[j] & ~kValueMask;
                            if (f != 0) {                    // published: take it
                                prev += win[j] & kValueMask;
                                used = j + 1;
                                done = (f == kFlagIncl);
                            }
                        }
                    }
                    if (done) break;
                    back += used;                            // re-poll from the first unpublished link
                }
                st_relaxed_gpu(const_cast<uint32_t *>(look), kFlagIncl | ((prev + total) & kValueMask));
            }
            if (CL > 1) {                                    // hand the chain prefix to my peers
                cg::cluster_group cluster = cg::this_cluster();
#pragma unroll
                for (int q = 0; q < CL - 1; ++q) cluster.map_shared_rank(s_prev, q)[bd] = prev;
            }
        }
        __syncwarp();                                        // the look-back loop diverges per digit
        if (CL > 1) {
            cluster_arrive();                                // #2: the prefix is in everybody's memory
            cluster_wait();
            if (!looker) prev = s_prev[bd];
        }
        if (kSplit && !((BSF || TL) && CL == 1)) asm volatile("bar.sync 3, %0;" :: "n"(WARPS * 32) : "memory");
        s_gofs[bd] = digit_base + prev + before - s_tstart[bd];
        B200_STAMP(5);                                       // group B done (look-back finished)
    }
    // Positions must be final before anybody stages keys: group A knows (its barrier 1), group B
    // knows (barrier 3); a CTA that is not split simply synchronises.
    static_assert(CL == 1 || WARPS == 16, "clustered shapes are exactly groups A and B");
    if (!kSplit) __syncthreads();

    // ---- stage the keys in shared memory in digit order ---------------------------------------------
    if (!((BSF || TL) && kSplit && CL == 1 && in_b)) {
#pragma unroll
        for (int i = 0; i < IPT; ++i) {
            const uint32_t d = digit_of(key[i], shift, flip);
            const uint32_t r = (i & 1) ? (rank2[i / 2] >> 16) : (rank2[i / 2] & 0xffffu);
            s_keys[s_table[(warp * kRadixBins + d) * TW + (TW - 1)] + r] = key[i];
        }
    }
    if (CL > 1 && !in_b) cluster_wait();                     // finish #2 (group B already did)
    B200_STAMP(6);                                           // staged
    __syncthreads();
    B200_STAMP(7);

    // ---- scatter: consecutive threads write consecutive addresses inside each digit run -----------
    if (valid == (uint32_t)kTile) {
#pragma unroll
        for (int j = 0; j < IPT; ++j) {
            const uint32_t p = tid + j * kThreads;
            const int32_t k = s_keys[p];
            st_stream(out + (size_t)(uint32_t)(s_gofs[digit_of(k, shift, flip)] + p), k);
        }
    } else {
#pragma unroll
        for (int j = 0; j < IPT; ++j) {
            const uint32_t p = tid + j * kThreads;
            if (p < valid) {
                const int32_t k = s_keys[p];
                st_stream(out + (size_t)(uint32_t)(s_gofs[digit_of(k, shift, flip)] + p), k);
            }
        }
    }
    B200_STAMP(8);
    if (TIMING && g_phase_dbg != nullptr && lane == 0 && (warp == 0 || warp == 8))
        g_phase_dbg[((size_t)dbg_tile * 2 + (warp >> 3)) * 16 + 9] = tile;
}


}  // namespace b200sort
