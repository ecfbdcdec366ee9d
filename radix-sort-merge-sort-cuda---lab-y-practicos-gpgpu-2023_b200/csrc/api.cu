// api.cu -- the extern "C" surface of libb200sort.so (include/b200sort.h) and the host-array
// operator that stands where the lab's order_array stood (SRM/lab.cu:303-402).
#include "common.cuh"
#include "dist.cuh"
#include "merge.cuh"
#include "radix.cuh"
#include "radix16.cuh"
#include "radix64.cuh"
#include "segmented.cuh"
#include "segmented16.cuh"
#include "segmented64.cuh"

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <thread>
#include <vector>

namespace b200sort {

thread_local cudaError_t g_last_cuda_error = cudaSuccess;
thread_local unsigned long long g_launch_count = 0;

// declared in radix.cu
int radix_num_variants();
const char *radix_variant_name(int v);
int radix_set_variant(int v);
void radix_set_skip(int enabled);
int radix_atomic_order_ok();
int radix_set_phase_debug(long long *d_buf);
const char *radix_effective_variant_name();
unsigned long long radix_check_failures(unsigned long long *per_site);
unsigned long long dist_check_failures(unsigned long long *per_site);

namespace {

int device_check() {
    int dev = -1;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) { g_last_cuda_error = e; cudaGetLastError(); return B200SORT_ERR_NO_DEVICE; }
    int major = 0;
    e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    if (e != cudaSuccess) { g_last_cuda_error = e; cudaGetLastError(); return B200SORT_ERR_NO_DEVICE; }
    return major == 10 ? B200SORT_OK : B200SORT_ERR_NO_DEVICE;
}

int check_sort_args(const void *keys, const void *tmp, size_t n) {
    if (n > B200SORT_MAX_N) return B200SORT_ERR_INVALID;
    if (n > 1 && (keys == nullptr || tmp == nullptr)) return B200SORT_ERR_INVALID;
    return B200SORT_OK;
}

// ---- the per-process arena behind the host-array operator ---------------------------------------
constexpr size_t kStageBytes = 8u << 20;       // pinned staging chunk for pageable callers
constexpr size_t kDirectBytes = 4u << 20;      // below this a plain cudaMemcpy is as good as staging
constexpr int kCopyThreads = 16;               // most host threads ever filling / draining the staging chunks
constexpr int kStageSlots = 2 * kCopyThreads;  // two chunks per thread: one being copied, one in DMA
// How many of them a transfer uses: B200SORT_COPY_THREADS (1..16), else one per host core up to 16.
// Measured on the B200 box (16 cores), pageable array of 2^28 keys through order_array (ms):
// 2 threads 115, 4: 76, 8: 72, 12: 62, 16: 54 (profiles/r01_host_copy_threads.txt); the two
// transfers alone take 40 ms from pinned memory.
int copy_threads() {
    static const int n = [] {
        const char *e = getenv("B200SORT_COPY_THREADS");
        const int v = e ? atoi(e) : 0;
        if (v >= 1 && v <= kCopyThreads) return v;
        const unsigned hw = std::thread::hardware_concurrency();
        return (int)(hw < 1 ? 4 : hw > (unsigned)kCopyThreads ? (unsigned)kCopyThreads : hw);
    }();
    return n;
}
// Streamed host-array path (order_host_streamed): from this many keys on, the array is moved in
// kStreamChunks chunks and the sort overlaps the transfers.
constexpr size_t kStreamMinKeys = (size_t)1 << 25;
constexpr int kStreamChunks = 8;               // a power of two

struct HostArena {
    std::mutex mu;
    int device = -1;
    int32_t *d_keys = nullptr, *d_tmp = nullptr;
    size_t cap_keys = 0;
    void *d_ws = nullptr;
    size_t cap_ws = 0;
    void *h_stage[kStageSlots] = {};
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream[kCopyThreads] = {};
    cudaEvent_t ev[kStageSlots] = {};
    cudaEvent_t ev_main = nullptr;
    cudaEvent_t ev_step[2 * kStreamChunks] = {};   // streamed path: chunk i landed / output piece k merged

    void release() {
        if (d_keys) cudaFree(d_keys);
        if (d_tmp) cudaFree(d_tmp);
        if (d_ws) cudaFree(d_ws);
        for (int i = 0; i < kStageSlots; ++i) {
            if (h_stage[i]) cudaFreeHost(h_stage[i]);
            if (ev[i]) cudaEventDestroy(ev[i]);
            h_stage[i] = nullptr; ev[i] = nullptr;
        }
        for (int i = 0; i < kCopyThreads; ++i) {
            if (copy_stream[i]) cudaStreamDestroy(copy_stream[i]);
            copy_stream[i] = nullptr;
        }
        if (ev_main) cudaEventDestroy(ev_main);
        ev_main = nullptr;
        for (auto &e : ev_step) { if (e) cudaEventDestroy(e); e = nullptr; }
        if (stream) cudaStreamDestroy(stream);
        d_keys = d_tmp = nullptr; d_ws = nullptr; stream = nullptr;
        cap_keys = cap_ws = 0; device = -1;
    }

    int ensure(size_t n, size_t ws_bytes) {
        int dev = 0;
        B200_CUDA_TRY(cudaGetDevice(&dev));
        if (dev != device) { release(); device = dev; }
        if (stream == nullptr) {
            B200_CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
            for (int i = 0; i < kCopyThreads; ++i)
                B200_CUDA_TRY(cudaStreamCreateWithFlags(&copy_stream[i], cudaStreamNonBlocking));
            for (int i = 0; i < kStageSlots; ++i) B200_CUDA_TRY(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming));
            B200_CUDA_TRY(cudaEventCreateWithFlags(&ev_main, cudaEventDisableTiming));
            for (auto &e : ev_step) B200_CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        }
        if (n > cap_keys) {
            if (d_keys) cudaFree(d_keys);
            if (d_tmp) cudaFree(d_tmp);
            d_keys = d_tmp = nullptr; cap_keys = 0;
            size_t cap = 1024;
            while (cap < n) cap *= 2;
            B200_CUDA_TRY(cudaMalloc(&d_keys, cap * sizeof(int32_t)));
            B200_CUDA_TRY(cudaMalloc(&d_tmp, cap * sizeof(int32_t)));
            cap_keys = cap;
        }
        if (ws_bytes > cap_ws) {
            if (d_ws) cudaFree(d_ws);
            d_ws = nullptr; cap_ws = 0;
            B200_CUDA_TRY(cudaMalloc(&d_ws, ws_bytes));
            cap_ws = ws_bytes;
        }
        return B200SORT_OK;
    }

    int ensure_stage() {
        for (int i = 0; i < 2 * copy_threads(); ++i)
            if (h_stage[i] == nullptr) B200_CUDA_TRY(cudaMallocHost(&h_stage[i], kStageBytes));
        return B200SORT_OK;
    }
};

HostArena &arena() {
    static HostArena a;
    return a;
}

bool is_device_accessible_host(const void *p) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return attr.type == cudaMemoryTypeHost || attr.type == cudaMemoryTypeManaged;
}

// Pageable host memory <-> device through pinned staging chunks.  kCopyThreads host threads each
// own two chunks and a copy stream: while the DMA engine drains one chunk the thread fills the
// other, so the transfer runs at PCIe speed instead of at one core's memcpy speed (what the
// reference pays inside cudaMemcpy on a malloc'd array, SRM/lab.cu:321,397).
// `after` (may be null): an event the copy streams wait for before they touch device memory.
int staged_copy(HostArena &a, char *dev, char *host, size_t bytes, bool to_device, cudaEvent_t after) {
    B200_TRY(a.ensure_stage());
    int dev_id = 0;
    B200_CUDA_TRY(cudaGetDevice(&dev_id));
    // Small transfers: fewer threads (starting one costs tens of microseconds) and smaller chunks, so
    // that every thread still has at least two chunks to overlap its memcpy with the DMA engine.
    int nthreads = copy_threads();
    const size_t want = bytes / (4u << 20);                    // one thread per 4 MB
    if ((size_t)nthreads > want) nthreads = want < 1 ? 1 : (int)want;
    size_t chunk_bytes = align_up(div_up(bytes, (size_t)2 * nthreads), 4096);
    if (chunk_bytes > kStageBytes) chunk_bytes = kStageBytes;
    if (chunk_bytes < (256u << 10)) chunk_bytes = 256u << 10;
    const size_t chunks = div_up(bytes, chunk_bytes);
    int status[kCopyThreads] = {};
    cudaError_t cuda_err[kCopyThreads] = {};
    auto worker = [&](int t) {
        auto fail = [&](cudaError_t e) { status[t] = B200SORT_ERR_CUDA; cuda_err[t] = e; };
        cudaError_t e = cudaSetDevice(dev_id);
        if (e != cudaSuccess) return fail(e);
        cudaStream_t cs = a.copy_stream[t];
        if (after != nullptr && (e = cudaStreamWaitEvent(cs, after, 0)) != cudaSuccess) return fail(e);
        size_t k = 0;
        size_t prev_c = (size_t)-1;
        int prev_slot = 0;
        for (size_t c = t; c < chunks; c += nthreads, ++k) {
            const int slot = 2 * t + (int)(k & 1);
            const size_t off = c * chunk_bytes;
            const size_t len = bytes - off < chunk_bytes ? bytes - off : chunk_bytes;
            if (to_device) {
                if ((e = cudaEventSynchronize(a.ev[slot])) != cudaSuccess) return fail(e);   // chunk free again
                std::memcpy(a.h_stage[slot], host + off, len);
                if ((e = cudaMemcpyAsync(dev + off, a.h_stage[slot], len, cudaMemcpyHostToDevice, cs)) != cudaSuccess) return fail(e);
                if ((e = cudaEventRecord(a.ev[slot], cs)) != cudaSuccess) return fail(e);
            } else {
                if ((e = cudaMemcpyAsync(a.h_stage[slot], dev + off, len, cudaMemcpyDeviceToHost, cs)) != cudaSuccess) return fail(e);
                if ((e = cudaEventRecord(a.ev[slot], cs)) != cudaSuccess) return fail(e);
                if (prev_c != (size_t)-1) {       // drain the previous chunk while this one is in flight
                    const size_t poff = prev_c * chunk_bytes;
                    const size_t plen = bytes - poff < chunk_bytes ? bytes - poff : chunk_bytes;
                    if ((e = cudaEventSynchronize(a.ev[prev_slot])) != cudaSuccess) return fail(e);
                    std::memcpy(host + poff, a.h_stage[prev_slot], plen);
                }
                prev_c = c;
                prev_slot = slot;
            }
        }
        if (!to_device && prev_c != (size_t)-1) {
            const size_t poff = prev_c * chunk_bytes;
            const size_t plen = bytes - poff < chunk_bytes ? bytes - poff : chunk_bytes;
            if ((e = cudaEventSynchronize(a.ev[prev_slot])) != cudaSuccess) return fail(e);
            std::memcpy(host + poff, a.h_stage[prev_slot], plen);
        }
        if (to_device && (e = cudaStreamSynchronize(cs)) != cudaSuccess) return fail(e);
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < nthreads; ++t) pool.emplace_back(worker, t);
    worker(0);
    for (auto &th : pool) th.join();
    for (int t = 0; t < nthreads; ++t)
        if (status[t] != B200SORT_OK) return record_cuda(cuda_err[t]);
    return B200SORT_OK;
}

int h2d(HostArena &a, int32_t *d, const int32_t *h, size_t bytes) {
    if (bytes <= kDirectBytes || is_device_accessible_host(h)) {
        B200_CUDA_TRY(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, a.stream));
        return B200SORT_OK;
    }
    // every chunk has landed when this returns, so the main stream needs no further dependency
    return staged_copy(a, reinterpret_cast<char *>(d), reinterpret_cast<char *>(const_cast<int32_t *>(h)), bytes, true,
                       nullptr);
}

int d2h(HostArena &a, int32_t *h, const int32_t *d, size_t bytes) {
    if (bytes <= kDirectBytes || is_device_accessible_host(h)) {
        B200_CUDA_TRY(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, a.stream));
        B200_CUDA_TRY(cudaStreamSynchronize(a.stream));
        return B200SORT_OK;
    }
    // the copy streams start after everything queued on the main stream so far (the sort)
    B200_CUDA_TRY(cudaEventRecord(a.ev_main, a.stream));
    return staged_copy(a, reinterpret_cast<char *>(const_cast<int32_t *>(d)), reinterpret_cast<char *>(h), bytes, false,
                       a.ev_main);
}

int sort_dispatch(int algo, const int32_t *in, int32_t *out, int32_t *t, size_t n, void *ws, size_t wsb,
                  cudaStream_t s, float *ms = nullptr) {
    switch (algo) {
        case B200SORT_ALGO_RADIX: return ms ? radix_sort_timed(in, out, t, n, ws, wsb, s, ms)
                                            : radix_sort(in, out, t, n, ws, wsb, s);
        case B200SORT_ALGO_MERGE: return merge_sort(in, out, t, n, ws, wsb, s, ms, false);
        case B200SORT_ALGO_LAB: return merge_sort(in, out, t, n, ws, wsb, s, ms, true);
        default: return B200SORT_ERR_INVALID;
    }
}

size_t workspace_bytes(size_t n, int algo) {
    switch (algo) {
        case B200SORT_ALGO_RADIX: return radix_workspace_bytes(n);
        case B200SORT_ALGO_MERGE:
        case B200SORT_ALGO_LAB: return merge_workspace_bytes(n);
        default: return 0;
    }
}

// Streamed host-array path for large device-accessible (pinned / managed) arrays.  The transfers bound this operator (1 GiB each way over
// PCIe against ~3 ms of sorting at n = 2^28), so the sort is arranged to hide behind them:
//   * the array arrives in kStreamChunks chunks; chunk i is sorted (with the requested algorithm)
//     while chunk i+1 is still on the wire;
//   * sorted neighbours are merged as soon as both exist (merge-path passes, k4/k5'), level by
//     level, ping-ponging between the two device buffers -- when the last chunk lands only its own
//     sort and one merge per level are left;
//   * the last merge is launched as kStreamChunks ranges of output tiles, and every range starts
//     its way back to the host as soon as it is merged.
// Level l reads runs of (chunk << l) keys from d_keys (l even) or d_tmp (l odd) and writes the other;
// any operation on a range of keys only touches that range of the two buffers.
std::atomic<int> g_host_streaming{1};

int order_host_streamed(HostArena &a, int32_t *h_keys, size_t n, int algo) {
    constexpr int C = kStreamChunks;
    int levels = 0;
    while ((1 << levels) < C) ++levels;
    const size_t chunk = align_up(div_up(n, (size_t)C), 2 * merge_tile());
    const size_t sort_ws = align_up(workspace_bytes(chunk, algo), 256);
    const size_t merge_ws = merge_workspace_bytes(n);
    B200_TRY(a.ensure(n, sort_ws + merge_ws));
    auto *splits = reinterpret_cast<uint32_t *>(static_cast<unsigned char *>(a.d_ws) + sort_ws);
    cudaStream_t up = a.copy_stream[0], down = a.copy_stream[1];
    auto buffer_of = [&](int level) { return (level & 1) ? a.d_tmp : a.d_keys; };

    for (int i = 0; i < C; ++i) {
        const size_t off = (size_t)i * chunk;
        const size_t len = n - off < chunk ? n - off : chunk;
        B200_CUDA_TRY(cudaMemcpyAsync(a.d_keys + off, h_keys + off, len * sizeof(int32_t), cudaMemcpyHostToDevice, up));
        B200_CUDA_TRY(cudaEventRecord(a.ev_step[i], up));
        B200_CUDA_TRY(cudaStreamWaitEvent(a.stream, a.ev_step[i], 0));
        B200_TRY(sort_dispatch(algo, a.d_keys + off, a.d_keys + off, a.d_tmp + off, len, a.d_ws, sort_ws, a.stream));
        // every level whose pair of runs is complete now, except the last one
        for (int l = 0; l + 1 < levels && ((i + 1) & ((2 << l) - 1)) == 0; ++l) {
            const size_t run = chunk << l;
            const size_t start = (size_t)(i + 1 - (2 << l)) * chunk;
            const size_t sub = n - start < 2 * run ? n - start : 2 * run;
            B200_TRY(merge_partition(buffer_of(l) + start, sub, run, splits, a.stream));
            B200_TRY(merge_pass(buffer_of(l) + start, buffer_of(l + 1) + start, sub, run, splits, a.stream));
        }
    }
    // last level, range by range, each range followed by its copy back
    const int32_t *src = buffer_of(levels - 1);
    int32_t *dst = buffer_of(levels);
    const size_t run = chunk << (levels - 1);
    const size_t tiles = div_up(n, merge_tile());
    const size_t per = div_up(tiles, (size_t)C);
    B200_TRY(merge_partition(src, n, run, splits, a.stream));
    for (int k = 0; k < C; ++k) {
        B200_TRY(merge_pass_range(src, dst, n, run, splits, (size_t)k * per, (size_t)(k + 1) * per, a.stream));
        B200_CUDA_TRY(cudaEventRecord(a.ev_step[C + k], a.stream));
    }
    for (int k = 0; k < C; ++k) {
        const size_t e0 = (size_t)k * per * merge_tile();
        if (e0 >= n) break;
        const size_t e1 = (size_t)(k + 1) * per * merge_tile() < n ? (size_t)(k + 1) * per * merge_tile() : n;
        B200_CUDA_TRY(cudaStreamWaitEvent(down, a.ev_step[C + k], 0));
        B200_CUDA_TRY(cudaMemcpyAsync(h_keys + e0, dst + e0, (e1 - e0) * sizeof(int32_t), cudaMemcpyDeviceToHost, down));
    }
    B200_CUDA_TRY(cudaStreamSynchronize(down));
    B200_CUDA_TRY(cudaStreamSynchronize(a.stream));
    return B200SORT_OK;
}

int order_host(int32_t *h_keys, size_t n, int algo) {
    if (n > B200SORT_MAX_N) return B200SORT_ERR_INVALID;
    if (algo != B200SORT_ALGO_RADIX && algo != B200SORT_ALGO_MERGE && algo != B200SORT_ALGO_LAB)
        return B200SORT_ERR_INVALID;
    if (n <= 1) return B200SORT_OK;
    if (h_keys == nullptr) return B200SORT_ERR_INVALID;
    B200_TRY(device_check());
    HostArena &a = arena();
    std::lock_guard<std::mutex> lock(a.mu);
    // Pageable arrays move through the staging chunks at the host's memcpy speed; cutting that
    // pipeline into eight short ones costs more than the hidden sort saves (measured: 20.2 ms
    // streamed against 12.9 ms in one go at n = 2^25), so only device-accessible arrays stream.
    if (n >= kStreamMinKeys && g_host_streaming.load() != 0 && is_device_accessible_host(h_keys))
        return order_host_streamed(a, h_keys, n, algo);
    const size_t wsb = workspace_bytes(n, algo);
    B200_TRY(a.ensure(n, wsb));
    const size_t bytes = n * sizeof(int32_t);
    B200_TRY(h2d(a, a.d_keys, h_keys, bytes));
    B200_TRY(sort_dispatch(algo, a.d_keys, a.d_keys, a.d_tmp, n, a.d_ws, a.cap_ws, a.stream));
    B200_TRY(d2h(a, h_keys, a.d_keys, bytes));
    B200_CUDA_TRY(cudaStreamSynchronize(a.stream));
    return B200SORT_OK;
}

}  // namespace
}  // namespace b200sort

using namespace b200sort;

extern "C" {

const char *b200sort_version(void) { return "b200sort 0.1 (sm_100a)"; }

const char *b200sort_status_string(int status) {
    switch (status) {
        case B200SORT_OK: return "ok";
        case B200SORT_ERR_INVALID: return "invalid argument";
        case B200SORT_ERR_WORKSPACE: return "workspace missing, misaligned or too small";
        case B200SORT_ERR_CUDA: return "CUDA runtime error";
        case B200SORT_ERR_NO_DEVICE: return "no sm_100 device (this library has no CPU fallback)";
        case B200SORT_ERR_ALLOC: return "allocation failed";
        default: return "unknown status";
    }
}

int b200sort_last_cuda_error(void) { return (int)g_last_cuda_error; }
const char *b200sort_last_cuda_error_string(void) { return cudaGetErrorString(g_last_cuda_error); }
int b200sort_device_check(void) {
    B200_TRY(device_check());
    (void)radix_atomic_order_ok();      // explicit per-device initialisation: the lane-order self-test (blocks once)
    return B200SORT_OK;
}

size_t b200sort_workspace_bytes(size_t n, int algo) { return workspace_bytes(n, algo); }

int b200sort_radix_i32(int32_t *d_keys, int32_t *d_tmp, size_t n, void *d_ws, size_t ws_bytes, void *stream) {
    B200_TRY(check_sort_args(d_keys, d_tmp, n));
    return radix_sort(d_keys, d_keys, d_tmp, n, d_ws, ws_bytes, static_cast<cudaStream_t>(stream));
}

int b200sort_radix_pairs_i32(int32_t *d_keys, int32_t *d_vals, int32_t *d_tmp_keys, int32_t *d_tmp_vals, size_t n,
                             void *d_ws, size_t ws_bytes, void *stream) {
    B200_TRY(check_sort_args(d_keys, d_tmp_keys, n));
    B200_TRY(check_sort_args(d_vals, d_tmp_vals, n));
    return radix_sort_pairs(d_keys, d_keys, d_tmp_keys, d_vals, d_vals, d_tmp_vals, n, d_ws, ws_bytes,
                            static_cast<cudaStream_t>(stream));
}

int b200sort_radix_pairs_copy_i32(const int32_t *d_keys_in, const int32_t *d_vals_in, int32_t *d_keys_out,
                                  int32_t *d_vals_out, int32_t *d_tmp_keys, int32_t *d_tmp_vals, size_t n,
                                  void *d_ws, size_t ws_bytes, void *stream) {
    B200_TRY(check_sort_args(d_keys_out, d_tmp_keys, n));
    B200_TRY(check_sort_args(d_vals_out, d_tmp_vals, n));
    if (n > 0 && (d_keys_in == nullptr || d_vals_in == nullptr)) return B200SORT_ERR_INVALID;
    return radix_sort_pairs(d_keys_in, d_keys_out, d_tmp_keys, d_vals_in, d_vals_out, d_tmp_vals, n, d_ws, ws_bytes,
                            static_cast<cudaStream_t>(stream));
}

int b200sort_merge_i32(int32_t *d_keys, int32_t *d_tmp, size_t n, void *d_ws, size_t ws_bytes, void *stream) {
    B200_TRY(check_sort_args(d_keys, d_tmp, n));
    return merge_sort(d_keys, d_keys, d_tmp, n, d_ws, ws_bytes, static_cast<cudaStream_t>(stream), nullptr);
}

int b200sort_lab_i32(int32_t *d_keys, int32_t *d_tmp, size_t n, void *d_ws, size_t ws_bytes, void *stream) {
    B200_TRY(check_sort_args(d_keys, d_tmp, n));
    return merge_sort(d_keys, d_keys, d_tmp, n, d_ws, ws_bytes, static_cast<cudaStream_t>(stream), nullptr, true);
}

int b200sort_sort_i32(int algo, int32_t *d_keys, int32_t *d_tmp, size_t n, void *d_ws, size_t ws_bytes,
                      void *stream) {
    B200_TRY(check_sort_args(d_keys, d_tmp, n));
    return sort_dispatch(algo, d_keys, d_keys, d_tmp, n, d_ws, ws_bytes, static_cast<cudaStream_t>(stream));
}

int b200sort_sort_copy_i32(int algo, const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, size_t n,
                           void *d_ws, size_t ws_bytes, void *stream) {
    B200_TRY(check_sort_args(d_out, d_tmp, n));
    if (n > 0 && d_in == nullptr) return B200SORT_ERR_INVALID;
    return sort_dispatch(algo, d_in, d_out, d_tmp, n, d_ws, ws_bytes, static_cast<cudaStream_t>(stream));
}

int b200sort_sort_timed_i32(int algo, const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, size_t n,
                            void *d_ws, size_t ws_bytes, void *stream, float *ms) {
    B200_TRY(check_sort_args(d_out, d_tmp, n));
    if ((n > 0 && d_in == nullptr) || ms == nullptr) return B200SORT_ERR_INVALID;
    return sort_dispatch(algo, d_in, d_out, d_tmp, n, d_ws, ws_bytes, static_cast<cudaStream_t>(stream), ms);
}

int b200sort_sort_keys(int algo, int key_type, int descending, const void *d_in, void *d_out, void *d_tmp, size_t n,
                       void *d_ws, size_t ws_bytes, void *stream) {
    SignXor order;
    if (!key_order(key_type, descending, &order)) return B200SORT_ERR_INVALID;
    B200_TRY(check_sort_args(d_out, d_tmp, n));
    if (n > 0 && d_in == nullptr) return B200SORT_ERR_INVALID;
    const auto *in = static_cast<const int32_t *>(d_in);
    auto *out = static_cast<int32_t *>(d_out), *tmp = static_cast<int32_t *>(d_tmp);
    const auto s = static_cast<cudaStream_t>(stream);
    if (key_type == B200SORT_KEY_I32 && descending == 0) return sort_dispatch(algo, in, out, tmp, n, d_ws, ws_bytes, s);
    switch (algo) {
        case B200SORT_ALGO_RADIX: return radix_sort(in, out, tmp, n, d_ws, ws_bytes, s, &order);
        case B200SORT_ALGO_MERGE: return merge_sort_keys(in, out, tmp, n, d_ws, ws_bytes, s, order);
        default: return B200SORT_ERR_INVALID;      // the lab pipeline sorts int32 ascending only
    }
}

int b200sort_radix_pairs_keys(int key_type, int descending, const void *d_keys_in, const int32_t *d_vals_in,
                              void *d_keys_out, int32_t *d_vals_out, void *d_tmp_keys, int32_t *d_tmp_vals, size_t n,
                              void *d_ws, size_t ws_bytes, void *stream) {
    SignXor order;
    if (!key_order(key_type, descending, &order)) return B200SORT_ERR_INVALID;
    B200_TRY(check_sort_args(d_keys_out, d_tmp_keys, n));
    B200_TRY(check_sort_args(d_vals_out, d_tmp_vals, n));
    if (n > 0 && (d_keys_in == nullptr || d_vals_in == nullptr)) return B200SORT_ERR_INVALID;
    const bool i32_asc = key_type == B200SORT_KEY_I32 && descending == 0;
    return radix_sort_pairs(static_cast<const int32_t *>(d_keys_in), static_cast<int32_t *>(d_keys_out),
                            static_cast<int32_t *>(d_tmp_keys), d_vals_in, d_vals_out, d_tmp_vals, n, d_ws, ws_bytes,
                            static_cast<cudaStream_t>(stream), i32_asc ? nullptr : &order);
}

// Argument checks of the 64-bit entry points that come before the workspace, in the order and with the statuses of
// b200sort_sort_keys, plus the 8-byte alignment of the key pointers.
static int check_keys64_args(int key_type, int descending, SignXor64 *order, size_t n, const void *in, const void *out,
                             const void *tmp) {
    if (!key_order64(key_type, descending, order)) return B200SORT_ERR_INVALID;
    if (n > B200SORT_MAX_N) return B200SORT_ERR_INVALID;
    if (n > 0 && (in == nullptr || out == nullptr || tmp == nullptr)) return B200SORT_ERR_INVALID;
    if (((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(tmp)) & 7) != 0)
        return B200SORT_ERR_INVALID;
    return B200SORT_OK;
}

size_t b200sort_keys64_workspace_bytes(size_t n) { return radix64_workspace_bytes(n); }

int b200sort_sort_keys64(int key_type, int descending, const void *d_in, void *d_out, void *d_tmp, size_t n,
                         void *d_ws, size_t ws_bytes, void *stream) {
    SignXor64 order;
    B200_TRY(check_keys64_args(key_type, descending, &order, n, d_in, d_out, d_tmp));
    return radix64_sort(static_cast<const uint64_t *>(d_in), static_cast<uint64_t *>(d_out),
                        static_cast<uint64_t *>(d_tmp), nullptr, nullptr, nullptr, n, d_ws, ws_bytes,
                        static_cast<cudaStream_t>(stream), order);
}

int b200sort_radix_pairs_keys64(int key_type, int descending, const void *d_keys_in, const int32_t *d_vals_in,
                                void *d_keys_out, int32_t *d_vals_out, void *d_tmp_keys, int32_t *d_tmp_vals, size_t n,
                                void *d_ws, size_t ws_bytes, void *stream) {
    SignXor64 order;
    B200_TRY(check_keys64_args(key_type, descending, &order, n, d_keys_in, d_keys_out, d_tmp_keys));
    if (n > 0 && (d_vals_in == nullptr || d_vals_out == nullptr || d_tmp_vals == nullptr)) return B200SORT_ERR_INVALID;
    if ((d_keys_in == d_keys_out) != (d_vals_in == d_vals_out)) return B200SORT_ERR_INVALID;   // one plan for both
    return radix64_sort(static_cast<const uint64_t *>(d_keys_in), static_cast<uint64_t *>(d_keys_out),
                        static_cast<uint64_t *>(d_tmp_keys), d_vals_in, d_vals_out, d_tmp_vals, n, d_ws, ws_bytes,
                        static_cast<cudaStream_t>(stream), order);
}

// Argument checks of the 16-bit entry points that come before the workspace, in the order and with the statuses of
// the 64-bit ones; key pointers need 2-byte alignment.  d_tmp (pairs only) may be NULL for keys only.
static int check_keys16_args(int key_type, int descending, SignXor16 *order, size_t n, const void *in, const void *out,
                             const void *tmp, bool need_tmp) {
    if (!key_order16(key_type, descending, order)) return B200SORT_ERR_INVALID;
    if (n > B200SORT_MAX_N) return B200SORT_ERR_INVALID;
    if (n > 0 && (in == nullptr || out == nullptr || (need_tmp && tmp == nullptr))) return B200SORT_ERR_INVALID;
    if (((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(tmp)) & 1) != 0)
        return B200SORT_ERR_INVALID;
    return B200SORT_OK;
}

size_t b200sort_keys16_workspace_bytes(size_t n) { return radix16_workspace_bytes(n); }

int b200sort_sort_keys16(int key_type, int descending, const void *d_in, void *d_out, size_t n, void *d_ws,
                         size_t ws_bytes, void *stream) {
    SignXor16 order;
    B200_TRY(check_keys16_args(key_type, descending, &order, n, d_in, d_out, nullptr, false));
    return radix16_sort(static_cast<const uint16_t *>(d_in), static_cast<uint16_t *>(d_out), nullptr, nullptr, nullptr,
                        nullptr, n, d_ws, ws_bytes, static_cast<cudaStream_t>(stream), order);
}

int b200sort_radix_pairs_keys16(int key_type, int descending, const void *d_keys_in, const int32_t *d_vals_in,
                                void *d_keys_out, int32_t *d_vals_out, void *d_tmp_keys, int32_t *d_tmp_vals, size_t n,
                                void *d_ws, size_t ws_bytes, void *stream) {
    SignXor16 order;
    B200_TRY(check_keys16_args(key_type, descending, &order, n, d_keys_in, d_keys_out, d_tmp_keys, true));
    if (n > 0 && (d_vals_in == nullptr || d_vals_out == nullptr || d_tmp_vals == nullptr)) return B200SORT_ERR_INVALID;
    if ((d_keys_in == d_keys_out) != (d_vals_in == d_vals_out)) return B200SORT_ERR_INVALID;   // one plan for both
    return radix16_sort(static_cast<const uint16_t *>(d_keys_in), static_cast<uint16_t *>(d_keys_out),
                        static_cast<uint16_t *>(d_tmp_keys), d_vals_in, d_vals_out, d_tmp_vals, n, d_ws, ws_bytes,
                        static_cast<cudaStream_t>(stream), order);
}

// Argument checks of the segmented entry points, in the order and with the statuses of b200sort_sort_keys.
static int check_segmented_args(size_t n, const int32_t *d_offsets, size_t num_segments, void *d_ws, size_t ws_bytes) {
    if (num_segments > B200SORT_MAX_N || (num_segments > 0 && d_offsets == nullptr)) return B200SORT_ERR_INVALID;
    if (n == 0) return B200SORT_OK;
    if (d_ws == nullptr || (reinterpret_cast<uintptr_t>(d_ws) & 255) != 0 ||
        ws_bytes < segmented_workspace_bytes(n, num_segments))
        return B200SORT_ERR_WORKSPACE;
    return B200SORT_OK;
}

size_t b200sort_segmented_workspace_bytes(size_t n, size_t num_segments) {
    return segmented_workspace_bytes(n, num_segments);
}
size_t b200sort_segmented_class_max(int c) { return segmented_class_max(c); }

int b200sort_segmented_sort_keys(int key_type, int descending, const void *d_in, void *d_out, void *d_tmp, size_t n,
                                 const int32_t *d_offsets, size_t num_segments, void *d_ws, size_t ws_bytes,
                                 void *stream) {
    SignXor order;
    if (!key_order(key_type, descending, &order)) return B200SORT_ERR_INVALID;
    B200_TRY(check_sort_args(d_out, d_tmp, n));
    if (n > 0 && (d_in == nullptr || d_out == nullptr)) return B200SORT_ERR_INVALID;   // n == 1 writes d_out too
    B200_TRY(check_segmented_args(n, d_offsets, num_segments, d_ws, ws_bytes));
    if (n == 0) return B200SORT_OK;
    return segmented_sort(static_cast<const int32_t *>(d_in), static_cast<int32_t *>(d_out), static_cast<int32_t *>(d_tmp),
                          nullptr, nullptr, nullptr, n, d_offsets, num_segments, d_ws, static_cast<cudaStream_t>(stream),
                          order);
}

int b200sort_segmented_pairs_keys(int key_type, int descending, const void *d_keys_in, const int32_t *d_vals_in,
                                  void *d_keys_out, int32_t *d_vals_out, void *d_tmp_keys, int32_t *d_tmp_vals, size_t n,
                                  const int32_t *d_offsets, size_t num_segments, void *d_ws, size_t ws_bytes,
                                  void *stream) {
    SignXor order;
    if (!key_order(key_type, descending, &order)) return B200SORT_ERR_INVALID;
    B200_TRY(check_sort_args(d_keys_out, d_tmp_keys, n));
    B200_TRY(check_sort_args(d_vals_out, d_tmp_vals, n));
    if (n > 0 && (d_keys_in == nullptr || d_vals_in == nullptr || d_keys_out == nullptr || d_vals_out == nullptr))
        return B200SORT_ERR_INVALID;                                                     // n == 1 writes the outputs too
    if ((d_keys_in == d_keys_out) != (d_vals_in == d_vals_out)) return B200SORT_ERR_INVALID;
    B200_TRY(check_segmented_args(n, d_offsets, num_segments, d_ws, ws_bytes));
    if (n == 0) return B200SORT_OK;
    return segmented_sort(static_cast<const int32_t *>(d_keys_in), static_cast<int32_t *>(d_keys_out),
                          static_cast<int32_t *>(d_tmp_keys), d_vals_in, d_vals_out, d_tmp_vals, n, d_offsets,
                          num_segments, d_ws, static_cast<cudaStream_t>(stream), order);
}

// Argument checks of the 16-bit segmented entry points before the workspace: those of b200sort_segmented_sort_keys in
// its order and with its statuses, on the 16-bit key types, plus the 2-byte alignment of the key pointers.
static int check_segmented16_keys(int key_type, int descending, SignXor16 *order, size_t n, const void *in,
                                  const void *out, const void *tmp) {
    if (!key_order16(key_type, descending, order)) return B200SORT_ERR_INVALID;
    B200_TRY(check_sort_args(out, tmp, n));
    if (n > 0 && (in == nullptr || out == nullptr)) return B200SORT_ERR_INVALID;        // n == 1 writes d_out too
    if (((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(tmp)) & 1) != 0)
        return B200SORT_ERR_INVALID;
    return B200SORT_OK;
}

static int check_segmented16_args(size_t n, const int32_t *d_offsets, size_t num_segments, void *d_ws, size_t ws_bytes) {
    if (num_segments > B200SORT_MAX_N || (num_segments > 0 && d_offsets == nullptr)) return B200SORT_ERR_INVALID;
    if (n == 0) return B200SORT_OK;
    if (d_ws == nullptr || (reinterpret_cast<uintptr_t>(d_ws) & 255) != 0 ||
        ws_bytes < segmented16_workspace_bytes(n, num_segments))
        return B200SORT_ERR_WORKSPACE;
    return B200SORT_OK;
}

size_t b200sort_segmented16_workspace_bytes(size_t n, size_t num_segments) {
    return segmented16_workspace_bytes(n, num_segments);
}
size_t b200sort_segmented16_class_max(int c) { return segmented16_class_max(c); }

int b200sort_segmented_sort_keys16(int key_type, int descending, const void *d_in, void *d_out, void *d_tmp, size_t n,
                                   const int32_t *d_offsets, size_t num_segments, void *d_ws, size_t ws_bytes,
                                   void *stream) {
    SignXor16 order;
    B200_TRY(check_segmented16_keys(key_type, descending, &order, n, d_in, d_out, d_tmp));
    B200_TRY(check_segmented16_args(n, d_offsets, num_segments, d_ws, ws_bytes));
    if (n == 0) return B200SORT_OK;
    return segmented16_sort(static_cast<const uint16_t *>(d_in), static_cast<uint16_t *>(d_out),
                            static_cast<uint16_t *>(d_tmp), nullptr, nullptr, nullptr, n, d_offsets, num_segments, d_ws,
                            static_cast<cudaStream_t>(stream), order);
}

int b200sort_segmented_pairs_keys16(int key_type, int descending, const void *d_keys_in, const int32_t *d_vals_in,
                                    void *d_keys_out, int32_t *d_vals_out, void *d_tmp_keys, int32_t *d_tmp_vals,
                                    size_t n, const int32_t *d_offsets, size_t num_segments, void *d_ws,
                                    size_t ws_bytes, void *stream) {
    SignXor16 order;
    B200_TRY(check_segmented16_keys(key_type, descending, &order, n, d_keys_in, d_keys_out, d_tmp_keys));
    B200_TRY(check_sort_args(d_vals_out, d_tmp_vals, n));
    if (n > 0 && (d_vals_in == nullptr || d_vals_out == nullptr)) return B200SORT_ERR_INVALID;
    if ((d_keys_in == d_keys_out) != (d_vals_in == d_vals_out)) return B200SORT_ERR_INVALID;
    B200_TRY(check_segmented16_args(n, d_offsets, num_segments, d_ws, ws_bytes));
    if (n == 0) return B200SORT_OK;
    return segmented16_sort(static_cast<const uint16_t *>(d_keys_in), static_cast<uint16_t *>(d_keys_out),
                            static_cast<uint16_t *>(d_tmp_keys), d_vals_in, d_vals_out, d_tmp_vals, n, d_offsets,
                            num_segments, d_ws, static_cast<cudaStream_t>(stream), order);
}

// Argument checks of the 64-bit segmented entry points before the workspace: those of b200sort_segmented_sort_keys in
// its order and with its statuses, on the 64-bit key types, plus the 8-byte alignment of the key pointers.
static int check_segmented64_keys(int key_type, int descending, SignXor64 *order, size_t n, const void *in,
                                  const void *out, const void *tmp) {
    if (!key_order64(key_type, descending, order)) return B200SORT_ERR_INVALID;
    B200_TRY(check_sort_args(out, tmp, n));
    if (n > 0 && (in == nullptr || out == nullptr)) return B200SORT_ERR_INVALID;        // n == 1 writes d_out too
    if (((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(tmp)) & 7) != 0)
        return B200SORT_ERR_INVALID;
    return B200SORT_OK;
}

static int check_segmented64_args(size_t n, const int32_t *d_offsets, size_t num_segments, void *d_ws, size_t ws_bytes) {
    if (num_segments > B200SORT_MAX_N || (num_segments > 0 && d_offsets == nullptr)) return B200SORT_ERR_INVALID;
    if (n == 0) return B200SORT_OK;
    if (d_ws == nullptr || (reinterpret_cast<uintptr_t>(d_ws) & 255) != 0 ||
        ws_bytes < segmented64_workspace_bytes(n, num_segments))
        return B200SORT_ERR_WORKSPACE;
    return B200SORT_OK;
}

size_t b200sort_segmented64_workspace_bytes(size_t n, size_t num_segments) {
    return segmented64_workspace_bytes(n, num_segments);
}
size_t b200sort_segmented64_class_max(int c) { return segmented64_class_max(c); }

int b200sort_segmented_sort_keys64(int key_type, int descending, const void *d_in, void *d_out, void *d_tmp, size_t n,
                                   const int32_t *d_offsets, size_t num_segments, void *d_ws, size_t ws_bytes,
                                   void *stream) {
    SignXor64 order;
    B200_TRY(check_segmented64_keys(key_type, descending, &order, n, d_in, d_out, d_tmp));
    B200_TRY(check_segmented64_args(n, d_offsets, num_segments, d_ws, ws_bytes));
    if (n == 0) return B200SORT_OK;
    return segmented64_sort(static_cast<const uint64_t *>(d_in), static_cast<uint64_t *>(d_out),
                            static_cast<uint64_t *>(d_tmp), nullptr, nullptr, nullptr, n, d_offsets, num_segments, d_ws,
                            static_cast<cudaStream_t>(stream), order);
}

int b200sort_segmented_pairs_keys64(int key_type, int descending, const void *d_keys_in, const int32_t *d_vals_in,
                                    void *d_keys_out, int32_t *d_vals_out, void *d_tmp_keys, int32_t *d_tmp_vals,
                                    size_t n, const int32_t *d_offsets, size_t num_segments, void *d_ws,
                                    size_t ws_bytes, void *stream) {
    SignXor64 order;
    B200_TRY(check_segmented64_keys(key_type, descending, &order, n, d_keys_in, d_keys_out, d_tmp_keys));
    B200_TRY(check_sort_args(d_vals_out, d_tmp_vals, n));
    if (n > 0 && (d_vals_in == nullptr || d_vals_out == nullptr)) return B200SORT_ERR_INVALID;
    if ((d_keys_in == d_keys_out) != (d_vals_in == d_vals_out)) return B200SORT_ERR_INVALID;
    B200_TRY(check_segmented64_args(n, d_offsets, num_segments, d_ws, ws_bytes));
    if (n == 0) return B200SORT_OK;
    return segmented64_sort(static_cast<const uint64_t *>(d_keys_in), static_cast<uint64_t *>(d_keys_out),
                            static_cast<uint64_t *>(d_tmp_keys), d_vals_in, d_vals_out, d_tmp_vals, n, d_offsets,
                            num_segments, d_ws, static_cast<cudaStream_t>(stream), order);
}

int b200sort_radix_histogram_i32(const int32_t *d_keys, size_t n, uint32_t *d_hist, void *stream) {
    if (d_hist == nullptr || (n > 0 && d_keys == nullptr) || n > B200SORT_MAX_N) return B200SORT_ERR_INVALID;
    return radix_histogram(d_keys, n, d_hist, static_cast<cudaStream_t>(stream));
}

int b200sort_radix_pass_i32(const int32_t *d_in, int32_t *d_out, size_t n, int pass, void *d_ws,
                            size_t ws_bytes, void *stream) {
    if (n > B200SORT_MAX_N || (n > 0 && (d_in == nullptr || d_out == nullptr))) return B200SORT_ERR_INVALID;
    return radix_single_pass(d_in, d_out, n, pass, d_ws, ws_bytes, static_cast<cudaStream_t>(stream));
}

size_t b200sort_block_sort_tile(void) { return merge_block_tile(); }
int b200sort_block_sort_i32(const int32_t *d_in, int32_t *d_out, size_t n, void *stream) {
    if (n > B200SORT_MAX_N || (n > 0 && (d_in == nullptr || d_out == nullptr))) return B200SORT_ERR_INVALID;
    return merge_block_sort(d_in, d_out, n, static_cast<cudaStream_t>(stream), false);
}
int b200sort_lab_tile_sort_i32(const int32_t *d_in, int32_t *d_out, size_t n, void *stream) {
    if (n > B200SORT_MAX_N || (n > 0 && (d_in == nullptr || d_out == nullptr))) return B200SORT_ERR_INVALID;
    return merge_block_sort(d_in, d_out, n, static_cast<cudaStream_t>(stream), true);
}
size_t b200sort_merge_tile(void) { return merge_tile(); }
int b200sort_merge_partition_i32(const int32_t *d_in, size_t n, size_t run, uint32_t *d_splits, void *stream) {
    if (n > B200SORT_MAX_N || (n > 0 && (d_in == nullptr || d_splits == nullptr))) return B200SORT_ERR_INVALID;
    return merge_partition(d_in, n, run, d_splits, static_cast<cudaStream_t>(stream));
}
int b200sort_merge_pass_i32(const int32_t *d_in, int32_t *d_out, size_t n, size_t run,
                            const uint32_t *d_splits, void *stream) {
    if (n > B200SORT_MAX_N || (n > 0 && (d_in == nullptr || d_out == nullptr || d_splits == nullptr)))
        return B200SORT_ERR_INVALID;
    return merge_pass(d_in, d_out, n, run, d_splits, static_cast<cudaStream_t>(stream));
}

int b200sort_merge_set_variant(int variant) { return merge_set_variant(variant); }
int b200sort_merge_num_variants(void) { return merge_num_variants(); }
const char *b200sort_merge_variant_name(int variant) { return merge_variant_name(variant); }
int b200sort_radix_set_variant(int variant) { return radix_set_variant(variant); }
int b200sort_radix_num_variants(void) { return radix_num_variants(); }
const char *b200sort_radix_variant_name(int variant) { return radix_variant_name(variant); }
size_t b200sort_radix_tile(void) { return radix_current_tile(); }
int b200sort_debug_set_phase_buffer(void *d_buf) { return radix_set_phase_debug(static_cast<long long *>(d_buf)); }
int b200sort_radix_atomic_order_ok(void) { return radix_atomic_order_ok(); }
int b200sort_debug_checked_build(void) {
#ifdef B200SORT_CHECKED
    return 1;
#else
    return 0;
#endif
}
unsigned long long b200sort_debug_check_failures(void) {
    return radix_check_failures(nullptr) + dist_check_failures(nullptr) + segmented_check_failures(nullptr) +
           radix64_check_failures(nullptr) + radix16_check_failures(nullptr) + segmented16_check_failures(nullptr) +
           segmented64_check_failures(nullptr);
}
unsigned long long b200sort_debug_check_failures_by_site(unsigned long long *per_site /* [16], overwritten */) {
    if (per_site == nullptr) return 0;
    for (int i = 0; i < 16; ++i) per_site[i] = 0;
    return radix_check_failures(per_site) + dist_check_failures(per_site) + segmented_check_failures(per_site) +
           radix64_check_failures(per_site) + radix16_check_failures(per_site) + segmented16_check_failures(per_site) +
           segmented64_check_failures(per_site);
}
const char *b200sort_radix_effective_variant_name(void) { return radix_effective_variant_name(); }
int b200sort_radix_set_skip(int enabled) { radix_set_skip(enabled); return B200SORT_OK; }
unsigned long long b200sort_launch_count(void) { return g_launch_count; }
void b200sort_launch_count_reset(void) { g_launch_count = 0; }

int b200sort_order_array_host(int32_t *h_keys, size_t n, int algo) { return order_host(h_keys, n, algo); }
int b200sort_host_set_streaming(int enabled) { g_host_streaming.store(enabled ? 1 : 0); return B200SORT_OK; }
int b200sort_order_with_trust_host(int32_t *h_keys, size_t n) {
    return order_host(h_keys, n, B200SORT_ALGO_MERGE);
}
void b200sort_host_release(void) {
    HostArena &a = arena();
    std::lock_guard<std::mutex> lock(a.mu);
    a.release();
}
int b200sort_host_alloc_pinned(void **h_ptr, size_t bytes) {
    if (h_ptr == nullptr) return B200SORT_ERR_INVALID;
    B200_CUDA_TRY(cudaMallocHost(h_ptr, bytes));
    return B200SORT_OK;
}
int b200sort_host_free_pinned(void *h_ptr) {
    B200_CUDA_TRY(cudaFreeHost(h_ptr));
    return B200SORT_OK;
}


// ---- one-box multi-GPU path -------------------------------------------------------------------------
int b200sort_dist_histogram_i32(const int32_t *d_keys, size_t n, int bits, unsigned long long *d_hist,
                                void *stream) {
    if (d_hist == nullptr || (n > 0 && d_keys == nullptr) || n > B200SORT_MAX_N) return B200SORT_ERR_INVALID;
    if (bits < B200SORT_DIST_BITS_MIN) return B200SORT_ERR_INVALID;
    return dist_histogram(d_keys, n, bits, d_hist, static_cast<cudaStream_t>(stream));
}
int b200sort_dist_plan(const unsigned long long *all_hist, int world, int rank, int bits, int *bin_owner,
                       unsigned long long *recv_count, unsigned long long *send_count,
                       unsigned long long *dst_offset) {
    if (bits < B200SORT_DIST_BITS_MIN) return B200SORT_ERR_INVALID;
    return dist_plan(all_hist, world, rank, bits, bin_owner, recv_count, send_count, dst_offset);
}
size_t b200sort_dist_workspace_bytes(size_t n, int bits) { return dist_workspace_bytes(n, bits); }
int b200sort_dist_plan_device(const unsigned long long *d_all_hist, int world, int rank, int bits, unsigned long long cap,
                              int *d_bin_owner, void *d_plan, void *d_ws, size_t ws_bytes, void *stream) {
    B200_TRY(device_check());
    return dist_plan_device(d_all_hist, world, rank, bits, cap, d_bin_owner, d_plan, d_ws, ws_bytes, static_cast<cudaStream_t>(stream));
}
int b200sort_dist_partition_planned_i32(const int32_t *d_keys, size_t n, int bits, int world, int32_t *const *h_dst_base,
                                        const int *d_bin_owner, const void *d_plan, unsigned int *d_src_hist,
                                        void *d_ws, size_t ws_bytes, void *stream) {
    B200_TRY(device_check());
    if (n > B200SORT_MAX_N || (n > 0 && d_keys == nullptr)) return B200SORT_ERR_INVALID;
    return dist_partition_planned(d_keys, n, bits, world, h_dst_base, d_bin_owner, d_plan, d_src_hist, d_ws, ws_bytes,
                                  static_cast<cudaStream_t>(stream));
}
int b200sort_radix_copy_devn_i32(const int32_t *d_in, int32_t *d_out, int32_t *d_tmp, size_t n_max, const uint32_t *d_n,
                                 const uint32_t *d_hist, void *d_ws, size_t ws_bytes, void *stream) {
    B200_TRY(device_check());
    if (n_max > B200SORT_MAX_N || (n_max > 0 && (d_in == nullptr || d_out == nullptr || d_tmp == nullptr)) || d_n == nullptr)
        return B200SORT_ERR_INVALID;
    return radix_sort_devn(d_in, d_out, d_tmp, n_max, d_n, d_hist, d_ws, ws_bytes, static_cast<cudaStream_t>(stream));
}
int b200sort_dist_partition_i32(const int32_t *d_keys, size_t n, int bits, int world,
                                int32_t *const *h_dst_base, const int *d_bin_owner,
                                const unsigned long long *h_dst_offset, void *d_ws, size_t ws_bytes,
                                void *stream) {
    if ((n > 0 && d_keys == nullptr) || n > B200SORT_MAX_N || bits < B200SORT_DIST_BITS_MIN)
        return B200SORT_ERR_INVALID;
    return dist_partition(d_keys, n, bits, world, h_dst_base, d_bin_owner, h_dst_offset, d_ws, ws_bytes,
                          static_cast<cudaStream_t>(stream));
}
int b200sort_device_malloc(void **d_ptr, size_t bytes) {
    if (d_ptr == nullptr) return B200SORT_ERR_INVALID;
    B200_CUDA_TRY(cudaMalloc(d_ptr, bytes));
    return B200SORT_OK;
}
int b200sort_device_free(void *d_ptr) {
    B200_CUDA_TRY(cudaFree(d_ptr));
    return B200SORT_OK;
}
int b200sort_ipc_export(void *d_ptr, unsigned char *handle) {
    static_assert(sizeof(cudaIpcMemHandle_t) == B200SORT_IPC_HANDLE_BYTES, "handle size");
    if (d_ptr == nullptr || handle == nullptr) return B200SORT_ERR_INVALID;
    cudaIpcMemHandle_t h;
    B200_CUDA_TRY(cudaIpcGetMemHandle(&h, d_ptr));
    std::memcpy(handle, &h, sizeof h);
    return B200SORT_OK;
}
int b200sort_ipc_open(const unsigned char *handle, void **d_ptr) {
    if (d_ptr == nullptr || handle == nullptr) return B200SORT_ERR_INVALID;
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof h);
    B200_CUDA_TRY(cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return B200SORT_OK;
}
int b200sort_ipc_close(void *d_ptr) {
    B200_CUDA_TRY(cudaIpcCloseMemHandle(d_ptr));
    return B200SORT_OK;
}

}  // extern "C"
