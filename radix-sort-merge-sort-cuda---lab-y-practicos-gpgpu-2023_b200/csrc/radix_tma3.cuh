// radix_tma3.cuh -- k2: one onesweep pass, 16384-key tiles, the two halves of the CTA on different jobs (included by
// radix.cu).
//
// Replaces the lab's radix stage (SRM/lab.cu:47-87 radix_sort_kernel + :11-41 exlusiveScan) like the other pass
// kernels.  Same data path as radix_tma2.cuh (keys parked in tensor memory, positions from a second shared-memory
// atomicAdd, write-out by TMA bulk copies), another schedule.  There every warp walks R -> D -> S -> W in step, and
// during D -- the previous tile's look-back sums and staging layout: dependent shared-memory reads that only half the
// CTA works on -- the load/store pipe idles.  Here the halves do different things at the same time, so that the
// pipe-heavy counting of one overlaps the latency-bound write-out and look-back of the other (t = the tile counted in
// this iteration, p = the tile counted an iteration ago).  The shipped schedule (ACOUNT):
//
//            group A (warps 0..7)                         group B (warps 8..15)
//      W     request batch 0 of the next tile             thread = digit: bulk copy of every run of p (16-byte aligned
//                                                          interior) + its <= 3 + 3 edge words; request t's look-back rows
//      R|D   count + park its keys of tile t AND those    D  prefix of tile p from the fetched rows; the first staged
//            of warp w + 8 (same tensor-memory lanes)        word of every run is added to p's counters
//      P     publish t, draw the next ticket, prefetch
//            the tile half a round ahead into L2, turn
//            t's counters into positions inside the
//            runs, lay out t's staging slots
//   -- L --  (B arrives, A waits: p's positions are final; nobody still reads the staging area) ------------------
//      S     stage its keys of p                          stage its keys of p (parked by warp w - 8)
//   -- Y --  (everybody: p is staged, the ticket is drawn) ------------------------------------------------------
//
// A tile is published ~9 k cycles after the barrier Y that precedes its counting and resolved ~17 k cycles later, so
// its predecessors -- ticketed a few hundred cycles before it -- are in when the look-back reads their rows.  Two
// earlier schedules are kept as template flags for `make experiments`: every half counts its own keys, out of step
// (ACOUNT = 0, INSTEP = 0: the tile is published at the END of the iteration and resolved ~5 k cycles later, so the
// look-back waits for stragglers: 0.606 ms against 0.580) and the same in step (INSTEP: 0.613 ms).
#pragma once
#include "radix_tma2.cuh"

namespace b200sort {

// Every digit run gets a staging slot of whole 16-byte chunks with four words to spare, so that wherever its first
// destination word falls mod 4 the run can start at the co-aligned word of the slot: the slots then depend on the
// tile's COUNTS only and are laid out when the tile is published, off the look-back's critical path.
constexpr int kT3StageWords = kT2Tile + kRadixBins * 7 + 64;
constexpr int kT3Group = 4;                                     // shared-memory atomics a thread issues back to back
constexpr int kT3Win1 = 10;                                     // nearest earlier tile rows of the group ...
constexpr int kT3Win2 = 7;                                      // ... and nearest group rows that fit beside the tile
constexpr size_t kT3SmemBytes =
    (size_t)kT3StageWords * 4
    + (size_t)2 * kT2Rows * kRadixBins * 4       // digit counters -> positions, this tile's and the previous tile's
    + (size_t)8 * kRadixBins * 4                 // x2: run {start | length, destination}; tile counts | slot; in-group prefix
    + (size_t)(kT3Win1 + kT3Win2) * kRadixBins * 4
    + 256;
static_assert(kT3SmemBytes <= 115712, "two CTAs per SM");

// The look-back sum over status rows of which the nearest `have` (<= ROWS) sit in shared memory in memory order
// (win[(have - d) * 256] = the row at distance d, for my digit).  All of them are loaded at once: a dependent
// shared-memory round trip is what the resolving threads pay most for while the other warps keep the pipe busy.
template <int ROWS>
__device__ __forceinline__ void load_window(const uint32_t *win, uint32_t have, uint32_t (&w)[ROWS]) {
    const uint32_t *nearest = win + (size_t)(have - 1) * kRadixBins;
#pragma unroll
    for (int j = 0; j < ROWS; ++j) w[j] = ((uint32_t)j < have) ? nearest[-j * kRadixBins] : 0u;
}
template <int ROWS, int W>
__device__ __forceinline__ uint32_t sum_window(const uint32_t (&w)[ROWS], uint32_t have, const uint32_t *first, uint32_t max_dist) {
    uint32_t acc = 0;
#pragma unroll
    for (int j = 0; j < ROWS; ++j) {
        if ((uint32_t)j < have) {
            uint32_t x = w[j];
            while ((x & ~kValueMask) == 0) x = ld_relaxed_gpu(first - (size_t)j * kRadixBins);   // fetched before it was published
            acc += x & kValueMask;
            if ((x & ~kValueMask) == kFlagIncl) return acc;
        }
    }
    if (max_dist > have) acc += walk_back<W>(first - (size_t)have * kRadixBins, max_dist - have);
    return acc;
}

// KEYS = 1: any key order (RadixControl::key_neg / key_pos / key_pad); 0: int32 ascending.
template <int TIMING, int DEVN = 0, int INSTEP = 0, int ACOUNT = 0, int KEYS = 0>
__device__ __forceinline__ void
radix_onesweep_tma3_body(const int32_t *in_buf, int32_t *out_buf, int32_t *tmp_buf, size_t n, int pass,
                         RadixControl *ctl, uint32_t *status_cur, uint32_t *status_next, int follow_plan)
{
    constexpr int kTile = kT2Tile;
    constexpr int kRows = kT2Rows;
    constexpr uint32_t kNone = 0xFFFFFFFFu;

    extern __shared__ __align__(128) unsigned char smem_tma3[];
    int32_t  *s_stage  = reinterpret_cast<int32_t *>(smem_tma3);                         // [kT3StageWords]
    uint32_t *s_table  = reinterpret_cast<uint32_t *>(s_stage + kT3StageWords);          // [2][kRows][256]
    uint2    *s_rg     = reinterpret_cast<uint2 *>(s_table + 2 * kRows * kRadixBins);    // [2][256] {first staged word | keys to
                                                                 //           write << 16, first destination word} of the run
    uint32_t *s_ptot   = reinterpret_cast<uint32_t *>(s_rg + 2 * kRadixBins);            // [2][256] the published tile's digit count
                                                                 //           | its slot's first word << 16
    uint32_t *s_pin    = s_ptot + 2 * kRadixBins;                // [2][256] in-group prefix, if the tile summed its group
    uint32_t *s_win1   = s_pin + 2 * kRadixBins;                     // [kT3Win1][256] tile rows before the published tile
    uint32_t *s_win2   = s_win1 + kT3Win1 * kRadixBins;          // [kT3Win2][256] group rows before its group
    uint32_t *s_misc   = s_win2 + kT3Win2 * kRadixBins;          // [0..7] warp sums, [8] ticket, [10] tmem base, [16..17] mbarrier,
                                                                 // [20] key count, [21] tile count
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    const int32_t *in = in_buf;
    int32_t *out = out_buf;
    if (follow_plan) {
        if (ctl->skip[pass]) {
            const size_t n_now = DEVN ? (size_t)ctl->n_dev : n;
            const size_t tl = (n_now + kTile - 1) / kTile;
            const size_t rows = tl + (tl + kLookGroup - 1) / kLookGroup;
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
    const uint32_t flips = KEYS ? flips_of(ctl->key_neg, ctl->key_pos, shift) : 0u;
    auto dig = [&](int32_t k) -> uint32_t { return KEYS ? digit_of_image(k, shift, flips) : digit_of(k, shift, flip); };
    const uint32_t lt = lanemask_lt();
    const bool in_a = tid < kRadixBins;                          // warps 0..7 : thread = digit
    const uint32_t bd = tid - kRadixBins;                        // warps 8..15: thread - 256 = digit
    const uint32_t sh = (warp & 1) * 16;
    // word offset of `out` inside its 16-byte chunk: word g of the array is word g + gmis of the aligned base
    const uint32_t gmis = (uint32_t)((reinterpret_cast<uintptr_t>(out) >> 2) & 3u);
    int32_t *out_al = out - gmis;
    const uint32_t stage_s = smem_u32(s_stage);
    auto pair_bar = [&]() { bar_sync(3 + (warp >> 1), 64); };    // the two warps that share a counter row

    // ---- tensor memory: 256 columns; this warp owns lanes 32*(warp%4).., columns (warp/4)*64 + half*32 + batch*16.. --
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     :: "r"(smem_u32(&s_misc[10])), "n"(kT2TmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    {
        uint4 *z = reinterpret_cast<uint4 *>(s_table);
        for (uint32_t i = tid; i < 2 * kRows * kRadixBins / 4; i += kT2Threads) z[i] = make_uint4(0, 0, 0, 0);
    }
    const uint32_t mbar = smem_u32(&s_misc[16]);
    if (tid == 0) {
        s_misc[8] = atomicAdd(&ctl->ticket[pass], 1u);
        mbar_init(mbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        // the key count and the tile count live in shared memory (re-read where needed: registers are scarce)
        const uint32_t n32 = DEVN ? ctl->n_dev : (uint32_t)n;
        s_misc[20] = n32;
        s_misc[21] = (uint32_t)(((size_t)n32 + kTile - 1) / kTile);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    auto n_f = [&]() -> size_t { return DEVN ? (size_t)reinterpret_cast<volatile uint32_t *>(s_misc)[20] : n; };
    auto tiles_f = [&]() -> size_t { return (size_t)reinterpret_cast<volatile uint32_t *>(s_misc)[21]; };
    const uint32_t tmem_base = s_misc[10];
    const uint32_t tmem_warp = tmem_base + (((warp & 3u) * 32u) << 16) + (warp >> 2) * 64u;

    int32_t ka[kT2Batch], kb[kT2Batch];                          // batch 0 / batch 1 of the tile being counted
    auto load_batch_of = [&](uint32_t t, uint32_t wsel, int batch, int32_t (&k)[kT2Batch]) {   // warp wsel's slice
        const size_t tile_base = (size_t)t * kTile;
        const size_t n_now = n_f();
        const uint32_t valid = (n_now - tile_base < (size_t)kTile) ? (uint32_t)(n_now - tile_base) : (uint32_t)kTile;
        const uint32_t o = wsel * (32 * kT2Ipt) + lane + batch * (32 * kT2Batch);
        const int32_t *src = in + tile_base + o;
        if (valid == (uint32_t)kTile) {
#pragma unroll
            for (int i = 0; i < kT2Batch; ++i) k[i] = ld_stream(src + i * 32);
        } else {
#pragma unroll
            for (int i = 0; i < kT2Batch; ++i)
                k[i] = (o + i * 32 < valid) ? ld_stream(src + i * 32) : (KEYS ? (int32_t)ctl->key_pad : 0x7FFFFFFF);
        }
    };
    auto load_batch = [&](uint32_t t, int batch, int32_t (&k)[kT2Batch]) { load_batch_of(t, warp, batch, k); };
    // one shared-memory atomicAdd per key on the warp's half of its counter row.  COUNT: the result is not used (rank
    // phase); otherwise it is the key's staged position, and the key goes there.  A hot digit (the histogram kernel
    // found one value holding > 1/8 of the keys, or a quarter of the warp's first keys agree with lane 0's) is handled
    // with one ballot and ONE atomic per instruction, so skewed / sorted inputs do not serialise on one address.
    auto sweep = [&](const int32_t (&k)[kT2Batch], uint32_t *wt, bool count_only) {
        const uint32_t d0 = dig(k[0]);
        const uint32_t agree = __ballot_sync(0xffffffffu, d0 == __shfl_sync(0xffffffffu, d0, 0));
        const uint32_t hot_word = follow_plan ? ctl->hot[pass] : 0u;
        const bool hot = hot_word != 0 || __popc(agree) >= 8;
        if (!hot) {
            // A thread keeps at most 2 x kT3Group atomics in flight.  Shared-memory instructions queue in order: with
            // all 16 of a batch outstanding in every counting / staging warp, the queue is ~1.5 k cycles deep and
            // the other half of the CTA pays that for every dependent read of its look-back; the pipe itself is as
            // busy with a shallow queue.  Staging: group g's stores wait for its positions and are issued behind
            // group g+1's atomics (a store between two atomics orders them: the compiler cannot know that the staging
            // area and the counters do not alias).  Counting: the address of group g+2's first atomic formally
            // depends on the last result of group g (bit 31 of a 16 + 16 bit counter word is never set).
            uint32_t pos[kT2Batch];
#pragma unroll
            for (int i = 0; i < kT2Batch; ++i) {
                uint32_t d = dig(k[i]);
                if (count_only && i >= 2 * kT3Group && i % kT3Group == 0) d += pos[i - kT3Group - 1] >> 31;
                pos[i] = atomicAdd(wt + d, 1u << sh);
                if (!count_only && i >= kT3Group && i % kT3Group == kT3Group - 1) {
#pragma unroll
                    for (int j = i - 2 * kT3Group + 1; j <= i - kT3Group; ++j) {
                        const uint32_t q = (pos[j] >> sh) & 0xffffu;
                        B200_CHECK_AT(11, q < (uint32_t)kT3StageWords);
                        s_stage[q] = k[j];
                    }
                }
            }
            if (!count_only) {
#pragma unroll
                for (int j = kT2Batch - kT3Group; j < kT2Batch; ++j) {
                    const uint32_t q = (pos[j] >> sh) & 0xffffu;
                    B200_CHECK_AT(11, q < (uint32_t)kT3StageWords);
                    s_stage[q] = k[j];
                }
            }
        } else {
#pragma unroll
            for (int i = 0; i < kT2Batch; ++i) {
                const uint32_t d = dig(k[i]);
                const uint32_t hd = hot_word ? hot_word - 1u : __shfl_sync(0xffffffffu, d, 0);
                const bool same = (d == hd);
                const uint32_t sm = __ballot_sync(0xffffffffu, same);
                const uint32_t leader = (uint32_t)(__ffs(sm) - 1) & 31u;
                uint32_t r = 0;
                if (!same || lane == leader)
                    r = (atomicAdd(wt + d, (same ? (uint32_t)__popc(sm) : 1u) << sh) >> sh) & 0xffffu;
                const uint32_t r0 = __shfl_sync(0xffffffffu, r, leader);
                if (same) r = r0 + __popc(sm & lt);
                if (!count_only) {
                    B200_CHECK_AT(11, r < (uint32_t)kT3StageWords);
                    s_stage[r] = k[i];
                }
            }
        }
    };

    // R: count `tile`'s keys of this warp and park them in tensor memory
    auto count_and_park = [&](uint32_t t, uint32_t cb, uint32_t *tab_cur) {
        load_batch(t, 1, kb);                                    // lands while batch 0 is counted
        uint32_t *wt = tab_cur + (warp >> 1) * kRadixBins;
        sweep(ka, wt, true);
        tmem_st16(tmem_warp + cb * 32u, ka);
        sweep(kb, wt, true);
        tmem_st16(tmem_warp + cb * 32u + 16u, kb);
    };
    // ACOUNT: group A's warp w counts and parks its own keys AND those of warp w + 8 (same lane quadrant of tensor
    // memory, the columns of w + 8; the counters of w + 8: row (w >> 1) + 4, the same half), so that the tile can be
    // published without waiting for group B.  Two register sets, four batches, every load one batch ahead.
    auto count_and_park_both = [&](uint32_t t, uint32_t cb, uint32_t *tab_cur) {
        uint32_t *wt = tab_cur + (warp >> 1) * kRadixBins;
        const uint32_t tm = tmem_warp + cb * 32u;
        load_batch(t, 1, kb);
        sweep(ka, wt, true);
        tmem_st16(tm, ka);
        tmem_wait_st();                                          // (not needed for the registers; measured: 0.580 ms with
        load_batch_of(t, warp + 8, 0, ka);                       //  the two waits, 0.590 without -- they pace the warp)
        sweep(kb, wt, true);
        tmem_st16(tm + 16u, kb);
        tmem_wait_st();
        load_batch_of(t, warp + 8, 1, kb);
        sweep(ka, wt + 4 * kRadixBins, true);
        tmem_st16(tm + 128u, ka);
        sweep(kb, wt + 4 * kRadixBins, true);
        tmem_st16(tm + 128u + 16u, kb);
        tmem_wait_st();
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");   // warp w + 8 reads them an iteration from now
    };
    // S: stage the previous tile's keys of this warp: keys come back from tensor memory, positions from the second atomic
    auto stage_own = [&](uint32_t cb, uint32_t *tab_prev) {
        const uint32_t tp = tmem_warp + (cb ^ 1) * 32u;
        uint32_t *wt = tab_prev + (warp >> 1) * kRadixBins;
        tmem_wait_st();
#pragma unroll
        for (int batch = 0; batch < 2; ++batch) {
            uint32_t u0[8], u1[8];
            tmem_ld8(tp + batch * 16, u0);
            tmem_ld8(tp + batch * 16 + 8, u1);
            tmem_wait_ld();
            int32_t k[kT2Batch];
#pragma unroll
            for (int i = 0; i < 8; ++i) { k[i] = (int32_t)u0[i]; k[8 + i] = (int32_t)u1[i]; }
            sweep(k, wt, false);
        }
        // the counters are cleared for the tile after next once the pair takes no more positions from them
        pair_bar();
        reinterpret_cast<uint4 *>(tab_prev + (warp >> 1) * kRadixBins)[(warp & 1) * 32 + lane] = make_uint4(0, 0, 0, 0);
        fence_proxy_async_smem();                                // staged keys -> visible to the bulk copies
    };

    auto window_rows = [&](uint32_t p, uint32_t &h1, uint32_t &h2) {      // look-back rows of tile p the TMA unit fetches
        const uint32_t group = p / kLookGroup, r = p % kLookGroup;
        const bool last_of_group = (r == kLookGroup - 1) || ((size_t)p + 1 == tiles_f());
        h1 = last_of_group ? 0u : (r < (uint32_t)kT3Win1 ? r : (uint32_t)kT3Win1);
        h2 = group < (uint32_t)kT3Win2 ? group : (uint32_t)kT3Win2;
    };

    uint32_t tile = s_misc[8];
    uint32_t prev_tile = kNone;
    uint32_t win_parity = 0;
    __syncthreads();                                             // s_misc[8] is rewritten inside the loop
    if (tile < tiles_f()) load_batch(tile, 0, ka);
    const uint32_t digit_base = in_a ? 0u : ctl->base[pass][bd];
    uint32_t iter = 0;

    while (tile < tiles_f() || prev_tile != kNone) {
        const bool have_cur = tile < tiles_f();
        const bool have_prev = prev_tile != kNone;
        const uint32_t cb = iter & 1;                            // counters / tensor-memory half of `tile`
        uint32_t *tab_cur = s_table + cb * kRows * kRadixBins;
        uint32_t *tab_prev = s_table + (cb ^ 1) * kRows * kRadixBins;
        const uint32_t dbg_tile = have_cur ? tile : prev_tile;
        B200_STAMP(0);
        auto publish = [&]() {
            uint32_t total = 0;
            if (have_cur) {
                // thread = digit: `tile`'s count of my digit -> its status row (and, for the last tile of a group,
                // the group's row: that tile sums its group at once so that nobody waits an iteration for it)
                uint32_t c[kRows];
#pragma unroll
                for (int w = 0; w < kRows; ++w) {
                    c[w] = tab_cur[w * kRadixBins + tid];
                    total += (c[w] & 0xffffu) + (c[w] >> 16);
                }
                const uint32_t group = tile / kLookGroup, r = tile % kLookGroup;
                const bool last_of_group = (r == kLookGroup - 1) || ((size_t)tile + 1 == tiles_f());
                uint32_t *row = status_cur + (size_t)tile * kRadixBins + tid;
                st_relaxed_gpu(row, (r == 0 ? kFlagIncl : kFlagLocal) | total);
                if (status_next != nullptr) {
                    status_next[(size_t)tile * kRadixBins + tid] = 0;
                    if (last_of_group) status_next[(tiles_f() + group) * kRadixBins + tid] = 0;
                }
                // the counters become positions inside the digit's run (warp 2w's keys first, then warp 2w+1's);
                // group B adds the run's first staged word once the look-back has told where the run goes
                uint32_t run = 0;
#pragma unroll
                for (int w = 0; w < kRows; ++w) {
                    const uint32_t lo = c[w] & 0xffffu;
                    tab_cur[w * kRadixBins + tid] = run | ((run + lo) << 16);
                    run += lo + (c[w] >> 16);
                }
                if (last_of_group) {
                    const uint32_t p_in = (r > 0) ? walk_back<16>(row - kRadixBins, r) : 0u;
                    if (r > 0) st_relaxed_gpu(row, kFlagIncl | (p_in + total));
                    uint32_t *grow = status_cur + (tiles_f() + group) * kRadixBins + tid;
                    st_relaxed_gpu(grow, (group == 0 ? kFlagIncl : kFlagLocal) | (p_in + total));
                    s_pin[((INSTEP || ACOUNT) ? cb : 0u) * kRadixBins + tid] = p_in;
                }
                __syncwarp();                                    // the group walk diverges per digit
            }
            // The next tile's ticket is drawn right after the publication: from ticket to publication every tile takes
            // the same write + count + stage time.  (The atomic is issued here and its result used after the slot scan:
            // its global round trip would otherwise hold the whole group at the scan's barrier.)
            uint32_t t_next = 0;
            if (tid == 0) t_next = atomicAdd(&ctl->ticket[pass], 1u);
            {
                // the staging slots of `tile`: whole 16-byte chunks + four spare words per digit, in digit order
                const uint32_t slot = have_cur ? ((total + 3u) & ~3u) + 4u : 0u;
                uint32_t x = slot;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
                    if (lane >= (uint32_t)o) x += y;
                }
                if (lane == 31) s_misc[warp] = x;
                bar_sync(2, kRadixBins);
                const uint4 m0 = reinterpret_cast<const uint4 *>(s_misc)[0], m1 = reinterpret_cast<const uint4 *>(s_misc)[1];
                const uint32_t ms[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
                uint32_t add = 0;
#pragma unroll
                for (int w = 0; w < 8; ++w) add += (w < (int)warp) ? ms[w] : 0u;
                s_ptot[((INSTEP || ACOUNT) ? cb : 0u) * kRadixBins + tid] = total | ((x - slot + add) << 16);
            }
            if (tid == 0) {
                s_misc[8] = t_next;
                // ... and the tile some CTA will draw half a round of tickets from now is sent for: with two CTAs of
                // this size an SM has 28 KB of L1 left, which is all the loads it can have in flight, so how long a load
                // is in flight (HBM or L2) bounds how fast the keys come in
                const size_t t_far = (size_t)t_next + gridDim.x / 2;
                if (t_far < tiles_f()) {
                    const size_t left = (n_f() - t_far * kTile) * 4;
                    const uintptr_t a0 = reinterpret_cast<uintptr_t>(in + t_far * kTile) & ~(uintptr_t)15;
                    const uint32_t bytes = (uint32_t)((left < (size_t)kTile * 4 ? left : (size_t)kTile * 4) & ~(size_t)15);
                    if (bytes > 0) bulk_prefetch_l2(reinterpret_cast<const void *>(a0), bytes);
                }
            }
        };
        auto resolve = [&]() {
            if (have_prev) {
                // thread = digit; the rows the look-back needs were published most of an iteration ago and the nearest
                // of them fetched into shared memory since the last barrier
                const uint32_t pb = cb ^ 1;
                const uint32_t pw = s_ptot[((INSTEP || ACOUNT) ? pb : 0u) * kRadixBins + bd];
                const uint32_t p_total = pw & 0xffffu;
                const uint32_t group = prev_tile / kLookGroup, r = prev_tile % kLookGroup;
                const bool last_tile = (size_t)prev_tile + 1 == tiles_f();
                const bool last_of_group = (r == kLookGroup - 1) || last_tile;
                uint32_t *row = status_cur + (size_t)prev_tile * kRadixBins + bd;
                uint32_t *grow = status_cur + (tiles_f() + group) * kRadixBins + bd;
                uint32_t have1, have2;
                window_rows(prev_tile, have1, have2);
                if (have1 + have2 > 0) { mbar_wait(mbar, win_parity); win_parity ^= 1; }   // the fetched rows have landed
                B200_STAMP(11);
                uint32_t w1[kT3Win1], w2[kT3Win2];
                load_window<kT3Win1>(s_win1 + bd, have1, w1);
                load_window<kT3Win2>(s_win2 + bd, have2, w2);
                uint32_t inprev;
                if (last_of_group) inprev = s_pin[((INSTEP || ACOUNT) ? pb : 0u) * kRadixBins + bd];          // summed when the tile was published
                else               inprev = (r > 0) ? sum_window<kT3Win1, 8>(w1, have1, row - kRadixBins, r) : 0u;
                const uint32_t gprev = (group > 0) ? sum_window<kT3Win2, 8>(w2, have2, grow - kRadixBins, group) : 0u;
                B200_STAMP(10);                                  // previous tile resolved
                // ... the run's first staged word: the word of its slot that is congruent mod 4 to its first
                // destination word; it is ADDED to the counters (positions inside the run since the publication)
                const uint32_t g = digit_base + inprev + gprev + gmis;       // destination word (from out_al)
                B200_CHECK_AT(12, (size_t)g - gmis + (last_tile ? 0u : p_total) <= n_f());
                const uint32_t start = (pw >> 16) + (g & 3u);
#pragma unroll
                for (int w = 0; w < kRows; ++w) atomicAdd(&tab_prev[w * kRadixBins + bd], start * 0x10001u);
                // slots past n (last tile only) carry INT_MAX (KEYS: key_pad, whose image is 0xFFFFFFFF): digit 255,
                // counted behind every real key; they are staged but never written
                uint32_t cw = p_total;
                if (last_tile && bd == kRadixBins - 1) cw -= (uint32_t)(tiles_f() * (size_t)kTile - n_f());
                s_rg[pb * kRadixBins + bd] = make_uint2(start | (cw << 16), g);
                // later walks stop at this tile's rows
                if (last_of_group) { if (group > 0) st_relaxed_gpu(grow, kFlagIncl | ((gprev + inprev + p_total) & kValueMask)); }
                else if (r > 0)    st_relaxed_gpu(row, kFlagIncl | (inprev + p_total));
                __syncwarp();                                    // the walks diverge per digit
            }
        };
        auto request_rows = [&](uint32_t p) {                    // one thread: the TMA unit fetches tile p's look-back rows
            uint32_t have1, have2;
            window_rows(p, have1, have2);
            if (have1 + have2 > 0) {
                const uint32_t group = p / kLookGroup;
                fence_proxy_async_smem();                        // the reads of the windows' last contents are done (barriers)
                mbar_expect_tx(mbar, (have1 + have2) * kRadixBins * 4);
                if (have1) bulk_load(smem_u32(s_win1), status_cur + ((size_t)p - have1) * kRadixBins, have1 * kRadixBins * 4, mbar);
                if (have2) bulk_load(smem_u32(s_win2), status_cur + (tiles_f() + group - have2) * kRadixBins, have2 * kRadixBins * 4, mbar);
            }
        };
        if (ACOUNT) {
            if (in_a) {
                // ---- R: count my keys of `tile` and my partner warp's; P: publish it ---------------------------
                if (have_cur) count_and_park_both(tile, cb, tab_cur);
                B200_STAMP(1);
                bar_sync(2, kRadixBins);                         // group A: `tile`'s counts are final
                publish();
                B200_STAMP(2);
                bar_sync(11, kT2Threads);                        // L: the previous tile's positions are final
                B200_STAMP(3);
            } else {
                // ---- D: the previous tile's prefix and where its runs are staged ------------------------------
                resolve();
                B200_STAMP(1);
                bulk_wait_read_all();                            // my bulk copy of the tile before has READ the staging area
                __threadfence_block();
                bar_arrive(11, kT2Threads);                      // L: group A may stage
                bar_sync(1, kRadixBins);                         // ... and so may group B
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");   // my keys were parked by warp - 8
                B200_STAMP(3);
            }
            if (have_prev) stage_own(cb, tab_prev);              // ---- S
            B200_STAMP(5);
        } else if (INSTEP) {
            // ---- R: everybody counts its keys of `tile` ---------------------------------------------------------
            if (have_cur) count_and_park(tile, cb, tab_cur);
            B200_STAMP(1);
            if (in_a) {
                bulk_wait_read_all();                            // my bulk copy of the tile before has READ the staging area
                bar_arrive(13, kT2Threads);                      // group A is done with the staging area
                bar_sync(12, kT2Threads);                        // X: `tile`'s counts are final
                B200_STAMP(2);
                publish();                                       // ---- P
                B200_STAMP(3);
                bar_sync(11, kT2Threads);                        // L: the previous tile's positions are final
                B200_STAMP(4);
            } else {
                bar_arrive(12, kT2Threads);                      // X: group A may publish
                // the look-back rows are requested as late as possible: a row fetched before it was published costs a
                // global round trip of its own (requested during W instead: 0.613 -> 0.646 ms per pass)
                if (tid == kRadixBins && have_prev) request_rows(prev_tile);
                B200_STAMP(2);
                resolve();                                       // ---- D
                B200_STAMP(3);
                __threadfence_block();
                bar_arrive(11, kT2Threads);                      // L: group A may stage
                bar_sync(1, kRadixBins);                         // ... and so may group B, once ...
                bar_sync(13, kT2Threads);                        // ... group A's copies have read the staging area
                B200_STAMP(4);
            }
            if (have_prev) stage_own(cb, tab_prev);              // ---- S
            B200_STAMP(5);
        } else if (in_a) {
            // ---- 1: count my keys of `tile` -----------------------------------------------------------------
            if (have_cur) count_and_park(tile, cb, tab_cur);
            B200_STAMP(1);
            bulk_wait_read_all();                                // my bulk copy of the tile before has READ the staging area
            bar_sync(11, kT2Threads);                            // L: the previous tile's positions are final
            B200_STAMP(2);
            // ---- 2: stage my keys of the previous tile ------------------------------------------------------
            if (have_prev) stage_own(cb, tab_prev);
            B200_STAMP(3);
            bar_sync(12, kT2Threads);                            // X: `tile`'s counts are final
            B200_STAMP(4);
            // ---- 3: publish `tile` ----------------------------------------------------------------------------
            publish();
            B200_STAMP(5);
        } else {
            // ---- 1: the previous tile's prefix and where its runs are staged ----------------------------------
            resolve();
            B200_STAMP(1);
            __threadfence_block();
            bar_arrive(11, kT2Threads);                          // L: group A may stage
            B200_STAMP(2);
            // ---- 2: count my keys of `tile` -----------------------------------------------------------------
            if (have_cur) count_and_park(tile, cb, tab_cur);
            B200_STAMP(3);
            bar_sync(12, kT2Threads);                            // X: `tile`'s counts are final (group A publishes)
            B200_STAMP(4);
            // ---- 3: stage my keys of the previous tile ------------------------------------------------------
            if (have_prev) stage_own(cb, tab_prev);
            B200_STAMP(5);
        }
        __syncthreads();                                         // Y: the staged tile is complete, the ticket is drawn
        B200_STAMP(6);
        // ---- 4: batch 0 of the next tile is requested; group A writes the previous tile: per digit run one bulk copy
        // for the 16-byte aligned interior, the <= 3 + 3 edge words by ordinary stores; group B asks for the look-back
        // rows of `tile` and goes on to resolve it ----------------------------------------------------------------
        const uint32_t next = s_misc[8];
        if (ACOUNT) {
            // group A only loads (it counts for everybody); group B, thread = digit, writes the previous tile: one bulk
            // copy for the run's 16-byte aligned interior, the <= 3 + 3 edge words by ordinary stores
            if (in_a) {
                if (next < tiles_f()) load_batch(next, 0, ka);
            } else {
                // t's look-back rows are requested first: they were published ~10 k cycles ago and are consumed after
                // the write-out, so the fetch costs the look-back nothing
                if (tid == kRadixBins && have_cur) request_rows(tile);
                if (have_prev) {
                    const uint2 rg = s_rg[(cb ^ 1) * kRadixBins + bd];
                    const uint32_t start = rg.x & 0xffffu, c = rg.x >> 16, g = rg.y;
                    uint32_t head = (4u - (g & 3u)) & 3u;
                    if (head > c) head = c;
                    const uint32_t body = (c - head) & ~3u;
                    const uint32_t tail = c - head - body;
                    B200_CHECK_AT(13, body == 0 || (((g + head) & 3u) == 0 && ((start + head) & 3u) == 0));
                    B200_CHECK_AT(14, (size_t)g - gmis + c <= n_f() && start + c <= (uint32_t)kT3StageWords);
                    int32_t e[6];        // the edge words are read before the copy is issued (~14 instructions per lane), stored after
#pragma unroll
                    for (int j = 0; j < 3; ++j) {
                        e[j]     = ((uint32_t)j < head) ? s_stage[start + j] : 0;
                        e[3 + j] = ((uint32_t)j < tail) ? s_stage[start + head + body + j] : 0;
                    }
                    if (body > 0) bulk_store(out_al + g + head, stage_s + (start + head) * 4u, body * 4u);
                    bulk_commit();
#pragma unroll
                    for (int j = 0; j < 3; ++j) {
                        if ((uint32_t)j < head) st_stream(out_al + g + j, e[j]);
                        if ((uint32_t)j < tail) st_stream(out_al + g + head + body + j, e[3 + j]);
                    }
                }
            }
        } else {
            if (next < tiles_f()) load_batch(next, 0, ka);
            if (have_prev) {
                // thread = digit in both groups: A sends the interior and the head, B the tail
                const uint2 rg = s_rg[(cb ^ 1) * kRadixBins + (in_a ? tid : bd)];
                const uint32_t start = rg.x & 0xffffu, c = rg.x >> 16, g = rg.y;
                uint32_t head = (4u - (g & 3u)) & 3u;
                if (head > c) head = c;
                const uint32_t body = (c - head) & ~3u;
                if (in_a) {
                    B200_CHECK_AT(13, body == 0 || (((g + head) & 3u) == 0 && ((start + head) & 3u) == 0));
                    B200_CHECK_AT(14, (size_t)g - gmis + c <= n_f() && start + c <= (uint32_t)kT3StageWords);
                    if (body > 0) bulk_store(out_al + g + head, stage_s + (start + head) * 4u, body * 4u);
                    bulk_commit();
                }
                const uint32_t cnt = in_a ? head : c - head - body;  // my edge: words [first, first + cnt) of the run
                const uint32_t first = in_a ? 0u : head + body;
                int32_t e[3];
    #pragma unroll
                for (int j = 0; j < 3; ++j) e[j] = ((uint32_t)j < cnt) ? s_stage[start + first + j] : 0;
    #pragma unroll
                for (int j = 0; j < 3; ++j)
                    if ((uint32_t)j < cnt) st_stream(out_al + g + first + j, e[j]);
            }
            if (!INSTEP && tid == kRadixBins && have_cur) request_rows(tile);
        }
        B200_STAMP(7);                                           // previous tile written (bulk copies in flight)
        if (TIMING && g_phase_dbg != nullptr && lane == 0 && (warp == 0 || warp == 8))
            g_phase_dbg[((size_t)dbg_tile * 2 + (warp >> 3)) * 16 + 9] = dbg_tile;
        prev_tile = have_cur ? tile : kNone;
        tile = next;
        ++iter;
    }
    bulk_wait_all();                                             // every bulk copy has landed
    __syncthreads();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "n"(kT2TmemCols) : "memory");
}

template <int TIMING, int DEVN = 0, int INSTEP = 0, int ACOUNT = 0, int KEYS = 0>
__global__ void __launch_bounds__(kT2Threads, 2)
radix_onesweep_tma3_kernel(const int32_t *in_buf, int32_t *out_buf, int32_t *tmp_buf, size_t n, int pass,
                           RadixControl *ctl, uint32_t *status_cur, uint32_t *status_next, int follow_plan)
{
    radix_onesweep_tma3_body<TIMING, DEVN, INSTEP, ACOUNT, KEYS>(in_buf, out_buf, tmp_buf, n, pass, ctl, status_cur, status_next, follow_plan);
}

}  // namespace b200sort
