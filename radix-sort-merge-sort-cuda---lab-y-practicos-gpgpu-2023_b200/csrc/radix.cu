// radix.cu -- onesweep LSD radix sort of int32 keys for sm_100a.
//
// Replaces the lab's radix stage (SRM/lab.cu:11-87: exlusiveScan + radix_sort_kernel, one bit per
// iteration on 32-key warp tiles) with a full 4-pass, 8-bit-digit least-significant-digit sort:
//
//   k1  radix_histogram_kernel (radix_hist.cuh)   ONE read of the keys (128-bit loads) builds all four
//        digit histograms; its last block turns them into exclusive bases, decides which passes are
//        skippable, flags hot digits, plans the buffers and zeroes the first status buffer.   4 B/key
//   k2  one pass, 8 B/key, in several compiled families (b200sort_radix_set_variant picks a shape):
//        radix_onesweep_tma3_kernel (radix_tma3.cuh)  DEFAULT from 2^23 keys on: persistent CTAs, 16384-key
//              tiles, keys parked in tensor memory, positions from a second shared-memory atomicAdd,
//              write-out by TMA bulk copies, tiles prefetched into L2 by the TMA unit;
//        radix_onesweep_pipelined2_kernel (radix_pipelined.cuh)  the default below 2^23 keys: persistent
//              CTAs, every warp a worker, one shared-memory atomicAdd per key as the rank (16-bit
//              counters, two warps per row), delayed two-level decoupled look-back, double-buffered
//              staging, coalesced scatter by the load/store pipe;
//        radix_onesweep_kernel (radix_tile.cuh)  one tile per CTA; rank by MATCH / ballots /
//              atomicOr table / atomicAdd; one- or two-level look-back; optional clusters;
//        radix_onesweep_pipelined_kernel (radix_pipelined.cuh)  14 worker warps + 2 chain warps.
//   k3  radix_final_copy_kernel, radix_atomic_order_selftest_kernel (radix_misc.cuh)
//   k0  radix_small_kernel (radix_small.cuh)  n <= 8192: all four passes in one CTA, one launch
// This file is the host side: the shape table, workspace layout, launches.
//
// Signed order: digits are taken from key ^ 0x80000000 (only the top digit changes).  Any other key order
// (b200sort_sort_keys): digits of the key's image k ^ (k < 0 ? key_neg : key_pos), by a second, generic instantiation
// of the histogram, the small-array kernel and the shipped pass kernels (DESIGN section 4.2c).
// Stability of every pass is what makes LSD correct: inside a tile the order is (warp, item,
// lane) and keys are loaded warp-striped so that this is memory order.
#include "radix.cuh"
#include "radix_hist.cuh"
#include "radix_tile.cuh"
#include "radix_pipelined.cuh"
#include "radix_tma.cuh"
#include "radix_tma2.cuh"
#include "radix_tma3.cuh"
#include "radix_misc.cuh"
#include "radix_small.cuh"

#include <atomic>
#include <cstdlib>
#include <mutex>

namespace b200sort {

// k0 (radix_small.cuh): int32 ascending and any other key order
__global__ void __launch_bounds__(kSmallThreads, 1)
radix_small_kernel(const int32_t *in, int32_t *out, uint32_t n)
{
    radix_small_body<0>(in, out, n, SignXor{0x80000000u, 0x80000000u});
}
__global__ void __launch_bounds__(kSmallThreads, 1)
radix_small_keys_kernel(const int32_t *in, int32_t *out, uint32_t n, SignXor order)
{
    radix_small_body<1>(in, out, n, order);
}

// ================================================================================================
// host side
// ================================================================================================
namespace {

using OnesweepFn = void (*)(const int32_t *, int32_t *, int32_t *, size_t, int, RadixControl *,
                            uint32_t *, uint32_t *, int);

struct Variant {
    const char *name;
    int mode;
    int cluster;       // CTAs per cluster (1 = none); 0 marks the persistent pipelined kernel (2 CTAs per SM),
                       // -k the same with k CTAs per SM
    int two_level;     // status rows: one per tile plus one per group of kLookGroup tiles
    int threads;
    int tile;
    size_t smem;
    OnesweepFn fn;
    OnesweepFn fn_devn = nullptr;   // the same shape reading the key count from the control block (radix_sort_devn)
    OnesweepFn fn_key = nullptr;    // the same shape for any key order (RadixControl::key_*; b200sort_sort_keys)
};

#define B200_VARIANT(W, I, B, M, C)                                                                 \
    { "warps" #W "_ipt" #I "_occ" #B "_" #M "_cl" #C, M, C, 0, OnesweepShape<W, I, M>::kThreads,      \
      OnesweepShape<W, I, M>::kTile, OnesweepShape<W, I, M>::kSmemBytes,                            \
      radix_onesweep_kernel<W, I, B, M, C> }

#define B200_VARIANT_X(W, I, B, M, C, P, S)                                                         \
    { "warps" #W "_ipt" #I "_occ" #B "_" #M "_cl" #C "_pf" #P "_bsf" #S, M, C, 0, OnesweepShape<W, I, M>::kThreads, \
      OnesweepShape<W, I, M>::kTile, OnesweepShape<W, I, M>::kSmemBytes,                            \
      radix_onesweep_kernel<W, I, B, M, C, P, S> }

#define B200_VARIANT_T(W, I, B, M, C, P, S, L)                                                       \
    { "TIMING_warps" #W "_ipt" #I "_" #M "_pf" #P "_tl" #L, M, C, L, OnesweepShape<W, I, M>::kThreads,  \
      OnesweepShape<W, I, M>::kTile, OnesweepShape<W, I, M>::kSmemBytes,                            \
      radix_onesweep_kernel<W, I, B, M, C, P, S, 1, L> }

#define B200_VARIANT_TL(W, I, B, M, P)                                                              \
    { "warps" #W "_ipt" #I "_occ" #B "_" #M "_pf" #P "_twolevel", M, 1, 1, OnesweepShape<W, I, M>::kThreads, \
      OnesweepShape<W, I, M>::kTile, OnesweepShape<W, I, M>::kSmemBytes,                            \
      radix_onesweep_kernel<W, I, B, M, 1, P, 1, 0, 1> }

#define B200_PP_VARIANT(I)                                                                          \
    { "pipelined_14w_ipt" #I "_kRankAdd", kRankAdd, 0, 1, kPPThreads, PipelinedShape<I>::kTile,     \
      PipelinedShape<I>::kSmemBytes, radix_onesweep_pipelined_kernel<I> }

#define B200_PP2_VARIANT(I)                                                                         \
    { "pipelined2_16w_ipt" #I "_kRankAdd_delayed_twolevel", kRankAdd, 0, 1, 512,                    \
      Pipelined2Shape<I>::kTile, Pipelined2Shape<I>::kSmemBytes, radix_onesweep_pipelined2_kernel<I> }

#define B200_PP2X_VARIANT(I, S, P)                                                                  \
    { "pipelined2_16w_ipt" #I "_kRankAdd_split" #S "_pack" #P, kRankAdd, 0, 1, 512, Pipelined2Shape<I, P>::kTile, \
      Pipelined2Shape<I, P>::kSmemBytes, radix_onesweep_pipelined2_kernel<I, 0, S, P> }

const Variant kVariants[] = {
    // ---- the shipped shapes ------------------------------------------------------------------------------------
    { "tma3_16w_2x16_kRankAdd_tmem_keys_bulk_store_a_counts_b_resolves", kRankAdd, 0, 1, kT2Threads, kT2Tile, kT3SmemBytes,
      radix_onesweep_tma3_kernel<0, 0, 0, 1>, radix_onesweep_tma3_kernel<0, 1, 0, 1>,
      radix_onesweep_tma3_kernel<0, 0, 0, 1, 1> },   //  0: DEFAULT: persistent CTAs,
                                               //     16384-key tiles, keys parked in tensor memory, positions from a second
                                               //     shared atomic, write-out by TMA bulk copies, one half of the CTA counts
                                               //     and publishes while the other writes out and resolves, the next tiles
                                               //     prefetched into L2 by the TMA unit.  As the default CONFIGURATION
                                               //     (radix_sort_impl) arrays below 2^23 keys run shape 1.
    { "pipelined2_16w_ipt20_kRankAdd_pack1_late_ticket", kRankAdd, 0, 1, 512, Pipelined2Shape<20, 1>::kTile,
      Pipelined2Shape<20, 1>::kSmemBytes, radix_onesweep_pipelined2_kernel<20, 0, 0, 1, 2, 0, 0, 1>,
      radix_onesweep_pipelined2_kernel<20, 0, 0, 1, 2, 0, 0, 1, 0, 0, 1>,
      radix_onesweep_pipelined2_kernel<20, 0, 0, 1, 2, 0, 0, 1, 0, 0, 0, 1> },   //  1: the ALTERNATE: 10240-key tiles,
                                               //     delayed two-level look-back, 16-bit counters (two warps per row),
                                               //     ticket drawn after the look-back, write-out by the load/store pipe
    { "pipelined2_16w_ipt20_kRankBallot_pack1_late_ticket", kRankBallot, 0, 1, 512, Pipelined2Shape<20, 1>::kTile,
      Pipelined2Shape<20, 1>::kSmemBytes, radix_onesweep_pipelined2_kernel<20, 0, 0, 1, 2, 0, 0, 1, 1>,
      radix_onesweep_pipelined2_kernel<20, 0, 0, 1, 2, 0, 0, 1, 1, 0, 1>,
      radix_onesweep_pipelined2_kernel<20, 0, 0, 1, 2, 0, 0, 1, 1, 0, 0, 1> },   //  2: the documented-
                                               //     behaviour fallback: shape 1 ranked by ballots
    { "tma3_16w_2x16_kRankAdd_tmem_keys_bulk_store_a_counts_b_resolves_any_size", kRankAdd, 0, 1, kT2Threads, kT2Tile,
      kT3SmemBytes, radix_onesweep_tma3_kernel<0, 0, 0, 1>, radix_onesweep_tma3_kernel<0, 1, 0, 1>,
      radix_onesweep_tma3_kernel<0, 0, 0, 1, 1> },   //  3: shape 0
                                               //     whatever the size
#ifdef B200SORT_EXPERIMENTS
    // ---- every other shape measured in rounds 1-2 (profiles/r0*_onesweep_variants.md): make EXPERIMENTS=1 ----------
    // (the phase-timing twins, the earlier TMA kernels, round 1's default and round 1's fallback come first)
    { "TIMING_tma3_16w_2x16", kRankAdd, 0, 1, kT2Threads, kT2Tile, kT3SmemBytes, radix_onesweep_tma3_kernel<1> },
    { "tma3_16w_2x16_kRankAdd_in_step", kRankAdd, 0, 1, kT2Threads, kT2Tile, kT3SmemBytes, radix_onesweep_tma3_kernel<0, 0, 1> },
    { "TIMING_tma3i_16w_2x16", kRankAdd, 0, 1, kT2Threads, kT2Tile, kT3SmemBytes, radix_onesweep_tma3_kernel<1, 0, 1> },
    { "tma3_16w_2x16_kRankAdd_out_of_step", kRankAdd, 0, 1, kT2Threads, kT2Tile, kT3SmemBytes, radix_onesweep_tma3_kernel<0> },
    { "TIMING_tma3a_16w_2x16", kRankAdd, 0, 1, kT2Threads, kT2Tile, kT3SmemBytes, radix_onesweep_tma3_kernel<1, 0, 0, 1> },
    { "tma_16w_ipt20_kRankAdd_tmem_parked_bulk_store", kRankAdd, 0, 1, kTmaThreads, kTmaTile, kTmaSmemBytes,
      radix_onesweep_tma_kernel<0> },          //     keys + ranks parked in tensor memory, late co-aligned staging, TMA write-out
    { "tma2_16w_2x16_kRankAdd_tmem_keys_second_atomic_bulk_store", kRankAdd, 0, 1, kT2Threads, kT2Tile, kT2SmemBytes,
      radix_onesweep_tma2_kernel<0>, radix_onesweep_tma2_kernel<0, 1> },   //     16384-key tiles, keys only in tensor memory,
                                               //     positions by a second atomic, TMA write-out, all warps in step
    { "TIMING_tma2_16w_2x16", kRankAdd, 0, 1, kT2Threads, kT2Tile, kT2SmemBytes, radix_onesweep_tma2_kernel<1> },
    { "TIMING_tma_16w_ipt20", kRankAdd, 0, 1, kTmaThreads, kTmaTile, kTmaSmemBytes, radix_onesweep_tma_kernel<1> },   //  3
    { "TIMING_pipelined2_ipt20_pack", kRankAdd, 0, 1, 512, Pipelined2Shape<20, 1>::kTile,
      Pipelined2Shape<20, 1>::kSmemBytes, radix_onesweep_pipelined2_kernel<20, 1, 0, 1, 2, 0, 0, 1> },   //  4
    B200_PP2X_VARIANT(20, 0, 1),               //  5: variant 0 with the ticket drawn before the look-back (round 1's default)
    B200_VARIANT(16, 16, 2, kRankBallot, 1),   //  6: one tile per CTA, ballot-ranked (round 1's fallback)
    { "pipelined2_16w_ipt22_kRankAdd_pack1_late_ticket", kRankAdd, 0, 1, 512, Pipelined2Shape<22, 1>::kTile,
      Pipelined2Shape<22, 1>::kSmemBytes, radix_onesweep_pipelined2_kernel<22, 0, 0, 1, 2, 0, 0, 1> },   //  7: 11264-key tiles
    { "pipelined2_16w_ipt24_kRankAdd_pack1_late_ticket", kRankAdd, 0, 1, 512, Pipelined2Shape<24, 1>::kTile,
      Pipelined2Shape<24, 1>::kSmemBytes, radix_onesweep_pipelined2_kernel<24, 0, 0, 1, 2, 0, 0, 1> },   //  8: 12288-key tiles
    { "pipelined2_16w_ipt20_kRankAdd_pack1_late_ticket_prefetch", kRankAdd, 0, 1, 512, Pipelined2Shape<20, 1, 0, 1>::kTile,
      Pipelined2Shape<20, 1, 0, 1>::kSmemBytes, radix_onesweep_pipelined2_kernel<20, 0, 0, 1, 2, 0, 0, 1, 0, 1> },   //  7: + the
                                               //     previous tile's look-back rows fetched by bulk load under the ranking
    { "TIMING_pipelined2_prefetch", kRankAdd, 0, 1, 512, Pipelined2Shape<20, 1, 0, 1>::kTile,
      Pipelined2Shape<20, 1, 0, 1>::kSmemBytes, radix_onesweep_pipelined2_kernel<20, 1, 0, 1, 2, 0, 0, 1, 0, 1> },   //  8
    // ---- round 1's table (its default, B200_PP2X_VARIANT(20, 0, 1), and its fallback are listed above) ----
    B200_VARIANT(16, 18, 2, kRankAdd, 1),      //  1: 9216
    B200_VARIANT(16, 16, 2, kRankAdd, 1),      //  2: 8192
    B200_VARIANT(8, 24, 3, kRankAdd, 1),       //  3: 6144, 256 threads
    B200_VARIANT(8, 16, 4, kRankAdd, 1),       //  4: 4096, 4 CTAs/SM
    B200_VARIANT(16, 16, 2, kRankAtomic, 1),   //  6
    B200_VARIANT(16, 16, 2, kRankMatch, 1),    //  7
    B200_VARIANT(8, 24, 3, kRankBallot, 1),    //  8
    B200_VARIANT(8, 8, 6, kRankBallot, 1),     //  9: 2048-key tiles
    B200_VARIANT(12, 16, 3, kRankAdd, 1),      // 10: 6144, 384 threads
    B200_VARIANT(16, 12, 2, kRankAdd, 1),      // 11: 6144, 512 threads
    B200_VARIANT(16, 16, 2, kRankAdd, 2),      // 12: clusters of 2 / 4 / 8 CTAs = one chain link
    B200_VARIANT(16, 16, 2, kRankAdd, 4),      // 13
    B200_VARIANT(16, 16, 2, kRankAdd, 8),      // 14
    B200_VARIANT(16, 18, 2, kRankAdd, 4),      // 15
    B200_VARIANT(16, 20, 2, kRankAdd, 4),      // 16
    B200_VARIANT(16, 20, 2, kRankAdd, 8),      // 17
    B200_VARIANT(16, 16, 2, kRankBallot, 4),   // 18
    B200_PP_VARIANT(20),                       // 19: persistent pipelined, 448 x 20 = 8960-key tiles
    B200_PP_VARIANT(16),                       // 20: 7168
    B200_PP_VARIANT(24),                       // 21: 10752
    B200_PP_VARIANT(18),                       // 22: 8064
    B200_VARIANT(32, 10, 2, kRankAdd, 1),      // 23: 1024 threads x 10 keys, 2 CTAs/SM = full occupancy, 32 regs
    B200_VARIANT(32, 8, 2, kRankAdd, 1),       // 24: 8192
    B200_VARIANT(32, 12, 1, kRankAdd, 1),      // 25: 12288, 1 CTA/SM
    B200_VARIANT(24, 12, 2, kRankAdd, 1),      // 26: 768 threads x 12 = 9216, 2 CTAs/SM (42 regs)
    B200_VARIANT_X(16, 20, 2, kRankAdd, 1, 296, 0),   // 27: default shape + L2 prefetch one CTA-lifetime ahead
    B200_VARIANT_X(16, 20, 2, kRankAdd, 1, 0, 1),     // 28: default shape, group B stages before the look-back
    B200_VARIANT_X(16, 20, 2, kRankAdd, 1, 296, 1),   // 29: both
    B200_VARIANT_X(16, 20, 2, kRankAdd, 1, 592, 1),   // 30: both, two lifetimes ahead
    B200_VARIANT_X(16, 16, 2, kRankAdd, 1, 296, 1),   // 31: 8192-key tiles, both
    B200_VARIANT_T(16, 20, 2, kRankAdd, 1, 296, 0, 0),   // 32: variant 27 with the phase-timing probe
    B200_VARIANT_TL(16, 20, 2, kRankAdd, 296),        // 33: two-level look-back, 10240-key tiles
    B200_VARIANT_TL(16, 20, 2, kRankAdd, 0),          // 34: same without the L2 prefetch
    B200_VARIANT_TL(16, 16, 2, kRankAdd, 296),        // 35: 8192
    B200_VARIANT_TL(16, 18, 2, kRankAdd, 296),        // 36: 9216
    B200_VARIANT_TL(16, 22, 2, kRankAdd, 296),        // 37: 11264
    B200_VARIANT_TL(16, 24, 2, kRankAdd, 296),        // 38: 12288
    B200_VARIANT_T(16, 20, 2, kRankAdd, 1, 296, 1, 1),   // 39: variant 33 with the phase-timing probe
    B200_PP2_VARIANT(20),                             // 40: persistent, delayed two-level look-back, 10240
    B200_PP2_VARIANT(16),                             // 41: 8192
    B200_VARIANT(16, 20, 2, kRankAdd, 1),             // 42: one tile per CTA, 10240-key tiles (round-1 default until PP2)
    B200_PP2_VARIANT(22),                             // 43: 11264
    { "TIMING_pipelined2_ipt18", kRankAdd, 0, 1, 512, Pipelined2Shape<18>::kTile,
      Pipelined2Shape<18>::kSmemBytes, radix_onesweep_pipelined2_kernel<18, 1> },   // 44
    B200_PP2X_VARIANT(18, 1, 0),                      // 45: the previous tile's two look-back walks split over the groups
    B200_PP2X_VARIANT(18, 0, 1),                      // 46: 16-bit counters, two warps per row
    B200_PP2X_VARIANT(18, 1, 1),                      // 47: both
    B200_PP2X_VARIANT(20, 1, 1),                      // 48: both, 10240-key tiles
    B200_PP2X_VARIANT(16, 1, 1),                      // 49: both, 8192-key tiles
    B200_PP2_VARIANT(18),                             // 50: the default until the packed counters (0.728 ms/pass)
    B200_PP2X_VARIANT(22, 0, 1),                      // 51: 11264
    B200_PP2X_VARIANT(24, 0, 1),                      // 52: 12288
    { "pipelined2_16w_ipt12_kRankAdd_pack1_3ctas", kRankAdd, -3, 1, 512, Pipelined2Shape<12, 1>::kTile,
      Pipelined2Shape<12, 1>::kSmemBytes, radix_onesweep_pipelined2_kernel<12, 0, 0, 1, 3> },   // 53: 3 CTAs per SM, 6144
    { "pipelined2_16w_ipt10_kRankAdd_pack1_3ctas", kRankAdd, -3, 1, 512, Pipelined2Shape<10, 1>::kTile,
      Pipelined2Shape<10, 1>::kSmemBytes, radix_onesweep_pipelined2_kernel<10, 0, 0, 1, 3> },   // 54: 5120
    { "pipelined2_16w_ipt20_kRankAdd_pack1_earlygroup", kRankAdd, 0, 1, 512, Pipelined2Shape<20, 1>::kTile,
      Pipelined2Shape<20, 1>::kSmemBytes, radix_onesweep_pipelined2_kernel<20, 0, 0, 1, 2, 1> },   // 55: group rows
                                                      //     made inclusive by their last tile at once
    { "pipelined2_16w_ipt18_kRankAdd_pack1_earlygroup", kRankAdd, 0, 1, 512, Pipelined2Shape<18, 1>::kTile,
      Pipelined2Shape<18, 1>::kSmemBytes, radix_onesweep_pipelined2_kernel<18, 0, 0, 1, 2, 1> },   // 56
    { "pipelined2_16w_ipt20_kRankAdd_pack1_overlap", kRankAdd, 0, 1, 512, Pipelined2Shape<20, 1>::kTile,
      Pipelined2Shape<20, 1>::kSmemBytes, radix_onesweep_pipelined2_kernel<20, 0, 0, 1, 2, 0, 1> },   // 57: no barrier
                                                      //     between digit phase and staging; B stages under its status loads
    { "pipelined2_16w_ipt18_kRankAdd_pack1_overlap", kRankAdd, 0, 1, 512, Pipelined2Shape<18, 1>::kTile,
      Pipelined2Shape<18, 1>::kSmemBytes, radix_onesweep_pipelined2_kernel<18, 0, 0, 1, 2, 0, 1> },   // 58
#endif
};
constexpr int kFallbackVariant = 2;
constexpr int kSmallTileVariant = 1;
// Below this many keys the default configuration runs shape 1: its smaller tiles fill the machine earlier
// (profiles/r02_size_sweep.txt: 0.146 against 0.144 ms at 2^22, 0.290 against 0.273 ms at 2^24).
constexpr size_t kDefaultMinKeys = (size_t)1 << 23;
constexpr int kNumVariants = sizeof(kVariants) / sizeof(kVariants[0]);

std::atomic<int> g_variant{0};
// Verdict of the lane-order self-test PER DEVICE: -1 unknown, 0 failed (or B200SORT_RANK_SAFE=1), 1 passed.
constexpr int kMaxDevices = 64;
std::atomic<int> g_atomic_order[kMaxDevices];
std::mutex g_selftest_mu;
struct AtomicOrderInit { AtomicOrderInit() { for (auto &a : g_atomic_order) a.store(-1); } } g_atomic_order_init;

// The self-test's flag word: one per device, as every __device__ variable is, so the test allocates nothing.
__device__ uint32_t g_selftest_bad;

// Runs the self-test on the current device unless its verdict is cached.  Called from b200sort_device_check()
// (the explicit init) and, as a fallback, lazily from the first sort on a device: it launches on a private stream and
// BLOCKS.  It may run while this thread or another one captures a CUDA graph (a first sort inside torch.cuda.graph):
// it switches this thread to the relaxed capture mode for the test, so the capture neither forbids nor sees its calls,
// and it allocates and frees nothing.  Only a verdict read back from the kernel is cached; if a CUDA call fails, the
// caller runs the ballot-ranked shape and the next call tries again.
int atomic_order_ok() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) { cudaGetLastError(); return 0; }
    int v = g_atomic_order[dev].load(std::memory_order_acquire);
    if (v >= 0) return v;
    std::lock_guard<std::mutex> lock(g_selftest_mu);
    v = g_atomic_order[dev].load(std::memory_order_acquire);
    if (v >= 0) return v;
    const char *env = getenv("B200SORT_RANK_SAFE");
    if (env != nullptr && env[0] == '1') { g_atomic_order[dev].store(0); return 0; }
    cudaStreamCaptureMode mode = cudaStreamCaptureModeRelaxed;
    if (cudaThreadExchangeStreamCaptureMode(&mode) != cudaSuccess) { cudaGetLastError(); return 0; }
    uint32_t *d_bad = nullptr, h_bad = 1;
    cudaStream_t st = nullptr;
    bool ok = cudaGetSymbolAddress(reinterpret_cast<void **>(&d_bad), g_selftest_bad) == cudaSuccess &&
              cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) == cudaSuccess &&
              cudaMemsetAsync(d_bad, 0, sizeof(uint32_t), st) == cudaSuccess;
    if (ok) {
        radix_atomic_order_selftest_kernel<<<kNumSMs * 2, 512, 0, st>>>(d_bad);
        ++g_launch_count;
        ok = cudaGetLastError() == cudaSuccess &&
             cudaMemcpyAsync(&h_bad, d_bad, sizeof(uint32_t), cudaMemcpyDeviceToHost, st) == cudaSuccess &&
             cudaStreamSynchronize(st) == cudaSuccess;
    }
    if (st) cudaStreamDestroy(st);
    cudaThreadExchangeStreamCaptureMode(&mode);                  // the caller's mode again
    if (!ok) { cudaGetLastError(); return 0; }                  // no verdict: the safe shape, for this call only
    v = (h_bad == 0) ? 1 : 0;
    g_atomic_order[dev].store(v, std::memory_order_release);
    return v;
}

// The variant to launch: the selected one, unless it needs lane-ordered atomics and this device
// failed (or was told to skip) the self-test.
int effective_variant();
std::atomic<int> g_skip_enabled{1};
// one-CTA sort for n <= 8192: B200SORT_RADIX_SMALL=0 in the environment or any explicit
// b200sort_radix_set_variant call other than 0 switches it off (sweeps and the all-shapes test must reach
// the shape they selected)
const bool g_small_env_on = [] { const char *e = getenv("B200SORT_RADIX_SMALL"); return !(e && e[0] == '0'); }();
std::atomic<int> g_small_enabled{g_small_env_on ? 1 : 0};
// Function attributes are per device, so they are set before every launch instead of once per process
// (the call costs well under a microsecond).
int ensure_smem_attr(int v, bool keys = false) {
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(keys ? kVariants[v].fn_key : kVariants[v].fn),
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kVariants[v].smem));
    return B200SORT_OK;
}
int ensure_hist_attr(bool keys = false) {
    B200_CUDA_TRY(cudaFuncSetAttribute(keys ? reinterpret_cast<const void *>(radix_histogram_keys_kernel)
                                            : reinterpret_cast<const void *>(radix_histogram_kernel),
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kHistSmemBytes));
    return B200SORT_OK;
}

// status rows a pass needs: one per tile, plus (pipelined kernel) one per group of tiles
size_t status_rows(const Variant &var, size_t tiles) {
    return var.two_level ? tiles + div_up(tiles, (size_t)kLookGroup) : tiles;
}

int launch_onesweep(const Variant &var, size_t tiles, cudaStream_t s, const int32_t *in, int32_t *out,
                    int32_t *tmp, size_t n, int pass, RadixControl *ctl, uint32_t *cur, uint32_t *next,
                    int follow_plan, bool devn = false, bool keys = false) {
    if (devn && (var.fn_devn == nullptr || var.cluster != 0)) return B200SORT_ERR_INVALID;
    if (keys && (var.fn_key == nullptr || var.cluster != 0)) return B200SORT_ERR_INVALID;
    if (var.cluster <= 0) {          // persistent: one CTA per resident slot, tiles by ticket
        const unsigned slots = (var.cluster == 0 ? 2u : (unsigned)(-var.cluster)) * kNumSMs;
        const unsigned grid = (unsigned)(tiles < slots ? tiles : slots);
        (devn ? var.fn_devn : keys ? var.fn_key : var.fn)<<<grid, var.threads, var.smem, s>>>(in, out, tmp, n, pass, ctl, cur,
                                                                                            next, follow_plan);
        B200_LAUNCH_CHECK();
        return B200SORT_OK;
    }
    const unsigned grid = (unsigned)(div_up(tiles, (size_t)var.cluster) * var.cluster);
    if (var.cluster == 1) {
        var.fn<<<grid, var.threads, var.smem, s>>>(in, out, tmp, n, pass, ctl, cur, next, follow_plan);
    } else {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(grid, 1, 1);
        cfg.blockDim = dim3((unsigned)var.threads, 1, 1);
        cfg.dynamicSmemBytes = var.smem;
        cfg.stream = s;
        cudaLaunchAttribute attr;
        attr.id = cudaLaunchAttributeClusterDimension;
        attr.val.clusterDim.x = (unsigned)var.cluster;
        attr.val.clusterDim.y = 1;
        attr.val.clusterDim.z = 1;
        cfg.attrs = &attr;
        cfg.numAttrs = 1;
        B200_CUDA_TRY(cudaLaunchKernelEx(&cfg, var.fn, in, out, tmp, n, pass, ctl, cur, next, follow_plan));
    }
    B200_LAUNCH_CHECK();
    return B200SORT_OK;
}

int hist_grid(size_t n) {
    const size_t chunks = div_up(div_up(n, 4), (size_t)kHistThreads * kHistUnroll);
    size_t g = chunks < (size_t)kNumSMs * kHistBlocksPerSM ? chunks : (size_t)kNumSMs * kHistBlocksPerSM;
    return (int)(g < 1 ? 1 : g);
}

}  // namespace

namespace {
int effective_variant() {
    const int v = g_variant.load();
    if (kVariants[v].mode == kRankAdd && !atomic_order_ok()) return kFallbackVariant;
    return v;
}
}  // namespace

int radix_set_phase_debug(long long *d_buf) {
    B200_CUDA_TRY(cudaMemcpyToSymbol(g_phase_dbg, &d_buf, sizeof d_buf));
    return B200SORT_OK;
}
int radix_atomic_order_ok() { return atomic_order_ok(); }
unsigned long long radix_check_failures(unsigned long long *per_site) { return tu_check_failures(per_site); }
int radix_num_variants() { return kNumVariants; }
const char *radix_variant_name(int v) { return (v >= 0 && v < kNumVariants) ? kVariants[v].name : nullptr; }
int radix_set_variant(int v) {
    if (v < 0 || v >= kNumVariants) return B200SORT_ERR_INVALID;
    g_variant.store(v);
    g_small_enabled.store((v == 0 && g_small_env_on) ? 1 : 0);        // 0 = the default configuration
    return B200SORT_OK;
}
void radix_set_skip(int enabled) { g_skip_enabled.store(enabled ? 1 : 0); }
int radix_skip_enabled() { return g_skip_enabled.load(); }
size_t radix_current_tile() { return (size_t)kVariants[g_variant.load()].tile; }
const char *radix_effective_variant_name() { return kVariants[effective_variant()].name; }

size_t radix_workspace_bytes(size_t n) {
    const size_t tiles = div_up(n > 0 ? n : 1, kRadixMinTile);
    const size_t rows = tiles + div_up(tiles, (size_t)kPPGroup) + 1;
    return kRadixControlBytes + 2 * rows * kRadixBins * sizeof(uint32_t);
}

int radix_histogram(const int32_t *d_keys, size_t n, uint32_t *d_hist, cudaStream_t s) {
    // Standalone histogram (unit tests, per-kernel timing): d_hist doubles as the control block's
    // histogram area, so a scratch control block is not needed -- the kernel is given a control
    // block that lives in a small static device allocation.
    RadixControl *scratch = nullptr;
    B200_CUDA_TRY(cudaMallocAsync(reinterpret_cast<void **>(&scratch), kRadixControlBytes, s));
    int rc = ensure_hist_attr();
    if (rc == B200SORT_OK) rc = record_cuda(cudaMemsetAsync(scratch, 0, kRadixZeroBytes, s));
    if (rc == B200SORT_OK && n > 0) {
        radix_histogram_kernel<<<hist_grid(n), kHistThreads, kHistSmemBytes, s>>>(d_keys, n, scratch, nullptr, 0, 0, 0);
        ++g_launch_count;
        rc = record_cuda(cudaGetLastError());
    }
    if (rc == B200SORT_OK)
        rc = record_cuda(cudaMemcpyAsync(d_hist, scratch->hist, sizeof(uint32_t) * kRadixPasses * kRadixBins,
                                         cudaMemcpyDeviceToDevice, s));
    cudaFreeAsync(scratch, s);
    return rc;
}

static int check_ws(void *d_ws, size_t ws_bytes, size_t n) {
    if (d_ws == nullptr || (reinterpret_cast<uintptr_t>(d_ws) & 255) != 0) return B200SORT_ERR_WORKSPACE;
    if (ws_bytes < radix_workspace_bytes(n)) return B200SORT_ERR_WORKSPACE;
    return B200SORT_OK;
}

int radix_single_pass(const int32_t *d_in, int32_t *d_out, size_t n, int pass, void *d_ws,
                      size_t ws_bytes, cudaStream_t s) {
    if (pass < 0 || pass >= kRadixPasses) return B200SORT_ERR_INVALID;
    if (n == 0) return B200SORT_OK;
    B200_TRY(check_ws(d_ws, ws_bytes, n));
    const int v = effective_variant();
    B200_TRY(ensure_smem_attr(v));
    B200_TRY(ensure_hist_attr());
    const Variant &var = kVariants[v];
    auto *ctl = static_cast<RadixControl *>(d_ws);
    auto *status0 = reinterpret_cast<uint32_t *>(static_cast<unsigned char *>(d_ws) + kRadixControlBytes);
    const size_t tiles = div_up(n, (size_t)var.tile);
    B200_CUDA_TRY(cudaMemsetAsync(ctl, 0, kRadixZeroBytes, s));
    radix_histogram_kernel<<<hist_grid(n), kHistThreads, kHistSmemBytes, s>>>(d_in, n, ctl, status0,
                                                                 status_rows(var, tiles) * kRadixBins, 0, 0);
    B200_LAUNCH_CHECK();
    B200_TRY(launch_onesweep(var, tiles, s, d_in, d_out, nullptr, n, pass, ctl, status0, nullptr, 0));
    return B200SORT_OK;
}

namespace {

struct StepTimer {
    cudaStream_t s;
    float *ms;
    cudaEvent_t ev[8] = {};
    int n = 0;
    ~StepTimer() { for (auto &e : ev) if (e) cudaEventDestroy(e); }
    int begin() {
        if (!ms) return B200SORT_OK;
        for (auto &e : ev) B200_CUDA_TRY(cudaEventCreate(&e));
        return mark();
    }
    int mark() {
        if (!ms) return B200SORT_OK;
        B200_CUDA_TRY(cudaEventRecord(ev[n++], s));
        return B200SORT_OK;
    }
    int finish() {
        if (!ms) return B200SORT_OK;
        B200_CUDA_TRY(cudaEventSynchronize(ev[n - 1]));
        for (int i = 0; i + 1 < n; ++i) B200_CUDA_TRY(cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]));
        return B200SORT_OK;
    }
};

int radix_sort_impl(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, size_t n, void *d_ws,
                    size_t ws_bytes, cudaStream_t s, float *ms, const uint32_t *d_n = nullptr,
                    const uint32_t *d_hist = nullptr, const SignXor *order = nullptr) {
    // d_n != nullptr: n is an upper bound (grids, status rows), the kernels read the key count from *d_n;
    // d_hist != nullptr (with d_n): the four digit histograms exist already, the histogram kernel is not run;
    // order != nullptr (not with d_n): any key order, by the generic instantiations
    if (ms) for (int i = 0; i < 6; ++i) ms[i] = 0.f;
    if (n == 0) return B200SORT_OK;
    if (n == 1 && d_n == nullptr) {
        if (d_in != d_out) B200_CUDA_TRY(cudaMemcpyAsync(d_out, d_in, sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
        return B200SORT_OK;
    }
    B200_TRY(check_ws(d_ws, ws_bytes, n));
    // Status words carry 30-bit counts.  A digit count reaches 2^30 only if n = 2^30 and one bin holds every key,
    // which is exactly the case pass skipping removes: with skipping switched off that size is refused.
    if (n >= ((size_t)1 << 30) && !g_skip_enabled.load()) return B200SORT_ERR_INVALID;
    // k0: up to 8192 keys are sorted by one CTA in one launch (untimed calls only: the timed form reports
    // the pipeline's kernels).  Same lane-ordered atomic rank as the pass kernel, same gate.
    if (ms == nullptr && d_n == nullptr && n <= (size_t)kSmallTile && g_small_enabled.load() && atomic_order_ok()) {
        if (order != nullptr) {
            B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(radix_small_keys_kernel),
                                               cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmallSmemBytes));
            radix_small_keys_kernel<<<1, kSmallThreads, kSmallSmemBytes, s>>>(d_in, d_out, (uint32_t)n, *order);
        } else {
            B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(radix_small_kernel),
                                               cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmallSmemBytes));
            radix_small_kernel<<<1, kSmallThreads, kSmallSmemBytes, s>>>(d_in, d_out, (uint32_t)n);
        }
        B200_LAUNCH_CHECK();
        return B200SORT_OK;
    }
    int v = effective_variant();
    if (d_n != nullptr && kVariants[v].fn_devn == nullptr) v = atomic_order_ok() ? 0 : kFallbackVariant;
    if (v == 0 && n < kDefaultMinKeys) v = kSmallTileVariant;
    const bool keys = order != nullptr;
    if (keys && (d_n != nullptr || kVariants[v].fn_key == nullptr)) return B200SORT_ERR_INVALID;   // an experiment shape
    B200_TRY(ensure_smem_attr(v, keys));
    if (d_n != nullptr)
        B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(kVariants[v].fn_devn),
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kVariants[v].smem));
    B200_TRY(ensure_hist_attr(keys));
    const Variant &var = kVariants[v];
    auto *ctl = static_cast<RadixControl *>(d_ws);
    const size_t tiles = div_up(n, (size_t)var.tile);
    const size_t rows = status_rows(var, tiles);
    uint32_t *status[2];
    status[0] = reinterpret_cast<uint32_t *>(static_cast<unsigned char *>(d_ws) + kRadixControlBytes);
    status[1] = status[0] + rows * kRadixBins;
    const int skip = g_skip_enabled.load();
    const uint32_t in_place = (d_in == d_out) ? 1u : 0u;
    StepTimer timer{s, ms};

    B200_CUDA_TRY(cudaMemsetAsync(ctl, 0, kRadixZeroBytes, s));
    B200_TRY(timer.begin());
    if (d_hist != nullptr) {
        B200_CUDA_TRY(cudaMemsetAsync(status[0], 0, rows * kRadixBins * sizeof(uint32_t), s));
        radix_plan_kernel<<<1, kHistThreads, 0, s>>>(d_hist, d_n, ctl, (uint32_t)skip, in_place);
    } else if (keys) {
        radix_histogram_keys_kernel<<<hist_grid(n), kHistThreads, kHistSmemBytes, s>>>(d_in, n, ctl, status[0],
                                                                                       rows * kRadixBins, (uint32_t)skip,
                                                                                       in_place, *order);
    } else {
        radix_histogram_kernel<<<hist_grid(n), kHistThreads, kHistSmemBytes, s>>>(d_in, n, ctl, status[0], rows * kRadixBins,
                                                                     (uint32_t)skip, in_place, d_n);
    }
    B200_LAUNCH_CHECK();
    B200_TRY(timer.mark());
    for (int pass = 0; pass < kRadixPasses; ++pass) {
        uint32_t *cur = status[pass & 1];
        uint32_t *next = (pass + 1 < kRadixPasses) ? status[(pass + 1) & 1] : nullptr;
        B200_TRY(launch_onesweep(var, tiles, s, d_in, d_out, d_tmp, n, pass, ctl, cur, next, 1, d_n != nullptr, keys));
        B200_TRY(timer.mark());
    }
    if (skip) {
        // Only the plan (on the device) knows whether a final copy is needed; the kernel exits at
        // once when it is not.  With skipping off the pass count is always even / lands in out.
        const size_t blocks = div_up(div_up(n, 4), 256);
        const unsigned grid = (unsigned)(blocks < (size_t)kNumSMs * 8 ? blocks : (size_t)kNumSMs * 8);
        radix_final_copy_kernel<<<grid, 256, 0, s>>>(d_in, d_out, d_tmp, n, ctl, d_n ? 1u : 0u);
        B200_LAUNCH_CHECK();
    }
    B200_TRY(timer.mark());
    return timer.finish();
}

}  // namespace

int radix_sort(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, size_t n, void *d_ws,
               size_t ws_bytes, cudaStream_t s, const SignXor *order) {
    return radix_sort_impl(d_in, d_out, d_tmp, n, d_ws, ws_bytes, s, nullptr, nullptr, nullptr, order);
}

int radix_sort_devn(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, size_t n_max, const uint32_t *d_n,
                    const uint32_t *d_hist, void *d_ws, size_t ws_bytes, cudaStream_t s) {
    if (d_n == nullptr) return B200SORT_ERR_INVALID;
    return radix_sort_impl(d_in, d_out, d_tmp, n_max, d_ws, ws_bytes, s, nullptr, d_n, d_hist);
}

// ---- sort-by-key (SURVEY section 8(f)-4) ----------------------------------------------------------------
// The same four stable passes with a 32-bit value carried beside every key: 16 B/key per pass.
// The packed-counter persistent kernel with 512 x 10 = 5120-key tiles (the values
// take the registers and the shared memory the larger key-only tile uses).  Stable, because every
// pass is (that is what makes LSD correct in the first place): equal keys keep their input order,
// the A-before-B rule of SRM/lab.cu:163-170 carried through the whole sort.
// Pairs per thread: 10 (default) or 12 (B200SORT_PAIRS_IPT=12, for A/B).
template <int IPT, int SAFE, int KEYS = 0>
int launch_pairs_passes(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, const int32_t *v_in, int32_t *v_out,
                        int32_t *v_tmp, size_t n, RadixControl *ctl, uint32_t *const *status, cudaStream_t s) {
    constexpr size_t smem = Pipelined2Shape<IPT, 1, 1>::kSmemBytes;
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(radix_onesweep_pairs_kernel<IPT, SAFE, KEYS>),
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const size_t tiles = div_up(n, (size_t)Pipelined2Shape<IPT, 1, 1>::kTile);
    const unsigned slots = 2u * kNumSMs;
    const unsigned grid = (unsigned)(tiles < slots ? tiles : slots);
    for (int pass = 0; pass < kRadixPasses; ++pass) {
        uint32_t *cur = status[pass & 1];
        uint32_t *next = (pass + 1 < kRadixPasses) ? status[(pass + 1) & 1] : nullptr;
        radix_onesweep_pairs_kernel<IPT, SAFE, KEYS><<<grid, 512, smem, s>>>(d_in, d_out, d_tmp, n, pass, ctl, cur, next, 1,
                                                                      v_in, v_out, v_tmp);
        B200_LAUNCH_CHECK();
    }
    return B200SORT_OK;
}
int pairs_ipt() {
#ifdef B200SORT_EXPERIMENTS
    static const int v = [] { const char *e = getenv("B200SORT_PAIRS_IPT"); return (e && atoi(e) == 12) ? 12 : 10; }();
#else
    static const int v = 10;
#endif
    return v;
}
size_t radix_pairs_tile() { return 512u * (size_t)(atomic_order_ok() ? pairs_ipt() : 10); }

int radix_sort_pairs(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, const int32_t *v_in, int32_t *v_out,
                     int32_t *v_tmp, size_t n, void *d_ws, size_t ws_bytes, cudaStream_t s, const SignXor *order) {
    if (n == 0) return B200SORT_OK;
    if (n == 1) {
        if (d_in != d_out) B200_CUDA_TRY(cudaMemcpyAsync(d_out, d_in, sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
        if (v_in != v_out) B200_CUDA_TRY(cudaMemcpyAsync(v_out, v_in, sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
        return B200SORT_OK;
    }
    if ((d_in == d_out) != (v_in == v_out)) return B200SORT_ERR_INVALID;   // the plan is shared by keys and values
    B200_TRY(check_ws(d_ws, ws_bytes, n));
    if (n >= ((size_t)1 << 30) && !g_skip_enabled.load()) return B200SORT_ERR_INVALID;   // see radix_sort_impl
    const bool safe = !atomic_order_ok();                                  // then the ballot-ranked shape runs
    const bool keys = order != nullptr;
    if (keys && !safe && pairs_ipt() != 10) return B200SORT_ERR_INVALID;   // the generic pairs kernel has 5120-key tiles
    B200_TRY(ensure_hist_attr(keys));
    auto *ctl = static_cast<RadixControl *>(d_ws);
    const size_t tiles = div_up(n, 512u * (size_t)(safe ? 10 : pairs_ipt()));   // radix_pairs_tile(), from the
    const size_t rows = tiles + div_up(tiles, (size_t)kLookGroup);             // verdict this call runs on
    uint32_t *status[2];
    status[0] = reinterpret_cast<uint32_t *>(static_cast<unsigned char *>(d_ws) + kRadixControlBytes);
    status[1] = status[0] + rows * kRadixBins;
    const int skip = g_skip_enabled.load();
    const uint32_t in_place = (d_in == d_out) ? 1u : 0u;

    B200_CUDA_TRY(cudaMemsetAsync(ctl, 0, kRadixZeroBytes, s));
    if (keys)
        radix_histogram_keys_kernel<<<hist_grid(n), kHistThreads, kHistSmemBytes, s>>>(d_in, n, ctl, status[0],
                                                                                       rows * kRadixBins, (uint32_t)skip,
                                                                                       in_place, *order);
    else
        radix_histogram_kernel<<<hist_grid(n), kHistThreads, kHistSmemBytes, s>>>(d_in, n, ctl, status[0], rows * kRadixBins,
                                                                     (uint32_t)skip, in_place);
    B200_LAUNCH_CHECK();
    if (keys && safe)           B200_TRY((launch_pairs_passes<10, 1, 1>(d_in, d_out, d_tmp, v_in, v_out, v_tmp, n, ctl, status, s)));
    else if (keys)              B200_TRY((launch_pairs_passes<10, 0, 1>(d_in, d_out, d_tmp, v_in, v_out, v_tmp, n, ctl, status, s)));
    else if (safe)              B200_TRY((launch_pairs_passes<10, 1>(d_in, d_out, d_tmp, v_in, v_out, v_tmp, n, ctl, status, s)));
#ifdef B200SORT_EXPERIMENTS
    else if (pairs_ipt() == 12) B200_TRY((launch_pairs_passes<12, 0>(d_in, d_out, d_tmp, v_in, v_out, v_tmp, n, ctl, status, s)));
#endif
    else                        B200_TRY((launch_pairs_passes<10, 0>(d_in, d_out, d_tmp, v_in, v_out, v_tmp, n, ctl, status, s)));
    if (skip) {
        const size_t blocks = div_up(div_up(n, 4), 256);
        const unsigned g2 = (unsigned)(blocks < (size_t)kNumSMs * 8 ? blocks : (size_t)kNumSMs * 8);
        radix_final_copy_kernel<<<g2, 256, 0, s>>>(d_in, d_out, d_tmp, n, ctl);
        B200_LAUNCH_CHECK();
        radix_final_copy_kernel<<<g2, 256, 0, s>>>(v_in, v_out, v_tmp, n, ctl);
        B200_LAUNCH_CHECK();
    }
    return B200SORT_OK;
}

// ---- sort with indices ------------------------------------------------------------------------------------------
// The generic pairs pipeline with the values made on the device: histogram, four passes, one final kernel.  The
// indices never travel as an input, and travel as int64 only when they are stored for the last time.
template <int SAFE>
int launch_indices_passes(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, int32_t *idx_out32, int32_t *tmp_idx,
                          size_t n, RadixControl *ctl, uint32_t *const *status, cudaStream_t s) {
    constexpr size_t smem = Pipelined2Shape<10, 1, 1>::kSmemBytes;
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(radix_onesweep_indices_kernel<10, SAFE>),
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const size_t tiles = div_up(n, (size_t)Pipelined2Shape<10, 1, 1>::kTile);
    const unsigned slots = 2u * kNumSMs;
    const unsigned grid = (unsigned)(tiles < slots ? tiles : slots);
    for (int pass = 0; pass < kRadixPasses; ++pass) {
        uint32_t *cur = status[pass & 1];
        uint32_t *next = (pass + 1 < kRadixPasses) ? status[(pass + 1) & 1] : nullptr;
        radix_onesweep_indices_kernel<10, SAFE><<<grid, 512, smem, s>>>(d_in, d_out, d_tmp, n, pass, ctl, cur, next, 1,
                                                                       idx_out32, tmp_idx);
        B200_LAUNCH_CHECK();
    }
    return B200SORT_OK;
}

int radix_sort_indices(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, int64_t *idx_out, int32_t *tmp_idx, size_t n,
                       void *d_ws, size_t ws_bytes, cudaStream_t s, const SignXor &order) {
    if (n == 0) return B200SORT_OK;
    if (n == 1) {
        if (d_in != d_out) B200_CUDA_TRY(cudaMemcpyAsync(d_out, d_in, sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
        B200_CUDA_TRY(cudaMemsetAsync(idx_out, 0, sizeof(int64_t), s));
        return B200SORT_OK;
    }
    B200_TRY(check_ws(d_ws, ws_bytes, n));
    if (n >= ((size_t)1 << 30) && !g_skip_enabled.load()) return B200SORT_ERR_INVALID;   // see radix_sort_impl
    const bool safe = !atomic_order_ok();
    B200_TRY(ensure_hist_attr(true));
    auto *ctl = static_cast<RadixControl *>(d_ws);
    const size_t tiles = div_up(n, (size_t)Pipelined2Shape<10, 1, 1>::kTile);
    const size_t rows = tiles + div_up(tiles, (size_t)kLookGroup);
    uint32_t *status[2];
    status[0] = reinterpret_cast<uint32_t *>(static_cast<unsigned char *>(d_ws) + kRadixControlBytes);
    status[1] = status[0] + rows * kRadixBins;
    const int skip = g_skip_enabled.load();
    const uint32_t in_place = (d_in == d_out) ? 1u : 0u;
    auto *idx32 = reinterpret_cast<int32_t *>(idx_out);

    B200_CUDA_TRY(cudaMemsetAsync(ctl, 0, kRadixZeroBytes, s));
    radix_histogram_keys_kernel<<<hist_grid(n), kHistThreads, kHistSmemBytes, s>>>(d_in, n, ctl, status[0], rows * kRadixBins,
                                                                                   (uint32_t)skip, in_place, order);
    B200_LAUNCH_CHECK();
    if (safe) B200_TRY(launch_indices_passes<1>(d_in, d_out, d_tmp, idx32, tmp_idx, n, ctl, status, s));
    else      B200_TRY(launch_indices_passes<0>(d_in, d_out, d_tmp, idx32, tmp_idx, n, ctl, status, s));
    if (skip) {
        // With skipping off all four passes run, and the fourth stores the int64 indices into out.
        const size_t blocks = div_up(n, 256);
        const unsigned g2 = (unsigned)(blocks < (size_t)kNumSMs * 8 ? blocks : (size_t)kNumSMs * 8);
        radix_final_indices_kernel<<<g2, 256, 0, s>>>(d_in, d_out, d_tmp, idx_out, tmp_idx, n, ctl);
        B200_LAUNCH_CHECK();
    }
    return B200SORT_OK;
}

int radix_sort_timed(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, size_t n, void *d_ws,
                     size_t ws_bytes, cudaStream_t s, float *ms) {
    return radix_sort_impl(d_in, d_out, d_tmp, n, d_ws, ws_bytes, s, ms);
}

}  // namespace b200sort
