// cabi.cu -- the extern "C" boundary of include/gbwt_b200.h: index construction (parse + K0 layout + upload),
// kernel launches, and the chunked host<->device pipeline of the host entry points.
//
// There is no CPU implementation of any query behind this boundary: every entry point launches the kernels
// of kernels.cuh on the index's device, and index construction fails with GBWT_B200_E_NO_DEVICE without one.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <functional>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/gbwt_b200.h"
#include "../../include/gbwt_b200_build.h"
#include "../../include/gbwt_b200_insert.h"
#include "../../include/gbwt_b200_ranges.h"
#include "build.h"
#include "find_mixed.h"
#include "find_window.h"
#include "insert.h"
#include "kernels.cuh"
#include "layout_builder.h"
#include "layout_writer.h"
#include "locate.h"
#include "ranges.h"
#include "sds_loader.h"

using namespace gbwt_b200;

struct gbwt_b200_index {
    int device = 0;
    int sm_count = 0;
    uint64_t sequences = 0, size = 0, offset = 0, alphabet_size = 0, flags = 0;
    IndexView view{};
    void* d_desc = nullptr;
    void* d_bodies = nullptr;
    void* d_edges = nullptr;
    void* d_endmarker = nullptr;
    void* d_skips = nullptr;
    uint64_t skip_bytes = 0;
    void* d_stage_body = nullptr;   // IndexView::stage_body (window kernels)
    uint64_t edges_total = 0, edges_local = 0;
    bool window_ok = false;         // the record-window search kernel can run on this index (validated edges, a plan)
    bool window_suits = false;      // ... and is expected to pay: mostly single-edge / dense records, mostly local edges
    WindowPlan window{};
    // GBWT_B200_WINDOW_STATS=1 (tests, tools): queries that went through the window kernel and how many it deferred
    // and the device time of the window kernel alone, in nanoseconds (CUDA events around the launch)
    mutable std::atomic<uint64_t> window_queries{0}, window_deferred{0}, window_kernel_ns{0}, window_launches{0};
    // Path checkpoints (kernels.cuh, k_build_checkpoints): built once when the index is created, immutable afterwards.
    void* d_ckpt_table = nullptr;
    void* d_ckpt_first = nullptr;
    CheckpointView ckpt{};
    bool ckpt_ok = false;
    uint32_t ckpt_shift = 0;
    uint64_t ckpt_entries = 0, ckpt_bytes = 0, ckpt_build_us = 0;
    // DNA bytes of every sequence before each of its checkpoints (k_extract_dna_checkpointed), made when checkpoints and
    // node labels are both there; follows the checkpoint table entry by entry.
    void* d_ckpt_dna = nullptr;
    bool dna_ckpt_ok = false;
    void* d_seq_len = nullptr;  // length of every sequence once some walk has measured it (SEQ_LEN_UNKNOWN before)
    void* d_dna_len = nullptr;  // the same for the DNA of every sequence (valid for the attached graph)
    void* d_label_starts = nullptr;  // node labels of a GBZ file (Graph::sequences), absent for a plain GBWT
    void* d_label_bytes = nullptr;
    bool has_graph = false;
    GraphView graph{};
    uint64_t graph_bytes = 0;
    uint64_t bytes[4] = {0, 0, 0, 0};
    uint64_t format_counts[FMT_COUNT] = {0, 0, 0, 0, 0, 0, 0};
    uint64_t checkpointed_records = 0;
    // Locate samples (GBWT_B200_LAYOUT_LOCATE; kernels.cuh k_build_locate, locate.cu): built once at creation.
    void* d_locate_first = nullptr;    // u32 [records + 1]
    void* d_locate_samples = nullptr;  // LocateSample [locate_samples]
    bool locate_ok = false;
    uint32_t locate_shift = 0;
    uint64_t locate_samples = 0, locate_bytes = 0, locate_build_us = 0;
    mutable std::atomic<uint64_t> locate_steps{0};  // GBWT_B200_LOCATE_STATS=1: LF steps of the locate walks
    Carried carried;  // tags, DA samples, metadata, Graph section: host-side, written back by serialize
};

namespace {

thread_local std::string g_last_error;
std::atomic<uint64_t> g_launches{0};

int fail(int code, const std::string& msg) {
    g_last_error = msg;
    return code;
}

int cuda_fail(cudaError_t e, const char* what) {
    g_last_error = std::string(what) + ": " + cudaGetErrorString(e);
    return GBWT_B200_E_CUDA;
}

#define CUDA_TRY(expr)                                        \
    do {                                                      \
        cudaError_t _e = (expr);                              \
        if (_e != cudaSuccess) return cuda_fail(_e, #expr);   \
    } while (0)

// Selects the index's device for the calling thread and restores the previous one.
struct DeviceScope {
    int previous = -1;
    bool ok = true;
    explicit DeviceScope(int device) {
        if (cudaGetDevice(&previous) != cudaSuccess) previous = -1;
        ok = cudaSetDevice(device) == cudaSuccess;
    }
    ~DeviceScope() { if (previous >= 0) cudaSetDevice(previous); }
};

// Persistent grid: at most one resident wave (8 CTAs of 256 threads per SM), fewer when the batch is small.
unsigned grid_for(const gbwt_b200_index* ix, size_t n, int block = BLOCK_THREADS) {
    size_t blocks = (n + block - 1) / block;
    size_t wave = static_cast<size_t>(ix->sm_count) * (2048 / block);
    return static_cast<unsigned>(std::max<size_t>(1, std::min(blocks, wave)));
}

int launch_done(const char* what) {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, what);
    return GBWT_B200_OK;
}

// ---- kernel launchers (device pointers) ------------------------------------------------------------

int launch_find(const gbwt_b200_index* ix, const uint64_t* nodes, size_t n, gbwt_b200_state* out, cudaStream_t s) {
    if (n == 0) return GBWT_B200_OK;
    k_find<<<grid_for(ix, n), BLOCK_THREADS, 0, s>>>(ix->view, nodes, n, out);
    return launch_done("k_find");
}
int launch_extend(const gbwt_b200_index* ix, const gbwt_b200_state* st, const uint64_t* nodes, size_t n,
                  gbwt_b200_state* out, cudaStream_t s) {
    if (n == 0) return GBWT_B200_OK;
    k_extend<<<grid_for(ix, n), BLOCK_THREADS, 0, s>>>(ix->view, st, nodes, n, out);
    return launch_done("k_extend");
}
// Development / test knob: GBWT_B200_LOCALITY = 0 never bucket the batch, 1 always (lets the tests drive the
// permuted path on tiny indexes); unset = decided by batch and index size.
int env_int(const char* name, int fallback) {
    const char* e = std::getenv(name);
    return e ? std::atoi(e) : fallback;
}

constexpr size_t LOCALITY_MIN_QUERIES = size_t(1) << 16;  // below this the sort costs more than it saves
constexpr uint64_t LOCALITY_MIN_INDEX_BYTES = uint64_t(48) << 20;  // an index that lives in L2 gains nothing

bool has_run_records(const gbwt_b200_index* ix) {
    // (DENSE4 bodies go through the same out-of-line step as the run-length formats)
    return ix->format_counts[FMT_RUN8] + ix->format_counts[FMT_RUN32] + ix->format_counts[FMT_RUN64] + ix->format_counts[FMT_DENSE4] != 0;
}

// The lean find/extend loop handles single-edge and dense records itself and calls out of line for the rest: it is
// the kernel of choice when the rest is a minority (a pangenome index under the dense policy), not for a run-length
// layout. Needs validated edge targets. GBWT_B200_FIND_LEAN=0 forces the general kernels.
bool wants_lean_find(const gbwt_b200_index* ix) {
    const uint64_t runs = ix->format_counts[FMT_RUN8] + ix->format_counts[FMT_RUN32] + ix->format_counts[FMT_RUN64];
    return ix->view.edges_valid && runs <= ix->format_counts[FMT_DENSE2] + ix->format_counts[FMT_SINGLE] / 4 &&
           env_int("GBWT_B200_FIND_LEAN", 1) != 0;
}

// Whether a batch of n queries gets the locality schedule (GBWT_B200_LOCALITY overrides).
bool wants_locality(const gbwt_b200_index* ix, size_t n) {
    const uint64_t index_bytes = ix->bytes[0] + ix->bytes[1] + ix->bytes[2];
    const int locality = env_int("GBWT_B200_LOCALITY", -1);
    if (ix->view.records == 0 || n > 0xFFFFFFFFull) return false;
    return locality == 1 || (locality != 0 && n >= LOCALITY_MIN_QUERIES && index_bytes >= LOCALITY_MIN_INDEX_BYTES);
}

// Locality schedule: counting sort of the batch by the record of each query's first node. `write_keys(shift, keys, counts)`
// launches the kernel that fills keys[q] = bucket of query q and counts the buckets; on success *perm holds the sorted order and the
// caller frees it with cudaFreeAsync on the same stream once the search kernel is enqueued.
// About 256 queries per bucket and at most 2^18 buckets (GBWT_B200_BUCKETS overrides): measured on config 4,
// a full sort (one bucket per record) makes the search kernel 11% faster but the sort itself twice as
// expensive (20 M counters and fully scattered slot writes), a net loss.
// `fixed_shift` >= 0: buckets of exactly 2^fixed_shift records (the record windows of find_window.cu). `bucket_end`, when
// asked for, receives the array whose entry b is the end of bucket b's slots in perm (the caller frees it).
struct DefaultScatter {};
template <class WriteKeys, class Scatter = DefaultScatter>
int build_locality_perm(const gbwt_b200_index* ix, size_t n, cudaStream_t s, WriteKeys write_keys, uint32_t** perm,
                        int fixed_shift = -1, uint32_t** bucket_end = nullptr, uint32_t** keys_out = nullptr, Scatter* scatter = nullptr) {
    const uint64_t max_buckets = static_cast<uint64_t>(std::max(1, env_int("GBWT_B200_BUCKETS", 1 << 18)));
    const uint64_t want_buckets = std::min<uint64_t>(max_buckets, std::max<uint64_t>(256, n / 256));
    uint32_t shift = 0;
    if (fixed_shift >= 0) shift = static_cast<uint32_t>(fixed_shift);
    else while (bucket_count(ix->view.records, shift) > want_buckets) shift++;
    const uint32_t buckets = static_cast<uint32_t>(bucket_count(ix->view.records, shift));
    const uint32_t m = buckets + 1, tiles = (m + SCAN_TILE - 1) / SCAN_TILE;
    uint32_t *counts = nullptr, *tile_sums = nullptr, *keys = nullptr;
    *perm = nullptr;
    CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&counts), m * sizeof(uint32_t), s));
    CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&tile_sums), tiles * sizeof(uint32_t), s));
    CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&keys), n * sizeof(uint32_t), s));
    CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(perm), n * sizeof(uint32_t), s));
    CUDA_TRY(cudaMemsetAsync(counts, 0, m * sizeof(uint32_t), s));
    write_keys(shift, keys, counts);  // keys[q] = bucket of query q, counts[bucket + 1] += 1
    launch_done("k_keys");
    k_scan_tiles<<<tiles, 1024, 0, s>>>(counts, m, tile_sums);
    launch_done("k_scan_tiles");
    if (tiles > 1) {
        k_scan_single<<<1, 1024, 0, s>>>(tile_sums, tiles);
        launch_done("k_scan_single");
        k_scan_add<<<tiles, 1024, 0, s>>>(counts, m, tile_sums);
        launch_done("k_scan_add");
    }
    // (`scatter`: the caller's own placement kernel, which writes more than the permutation)
    if constexpr (std::is_same<Scatter, DefaultScatter>::value) k_bucket_scatter<<<grid_for(ix, n), BLOCK_THREADS, 0, s>>>(keys, n, counts, *perm);
    else (*scatter)(keys, counts, *perm);
    int rc = launch_done("k_bucket_scatter");
    if (bucket_end != nullptr) *bucket_end = counts;  // after the scatter, counts[b] = end of bucket b
    else cudaFreeAsync(counts, s);
    cudaFreeAsync(tile_sums, s);
    if (keys_out != nullptr) *keys_out = keys;  // n words the caller may reuse (the keys are no longer needed)
    else cudaFreeAsync(keys, s);
    return rc;
}

// keys[q] = bucket of query q for either pattern width (the 64-bit kernel of kernels.cuh, or find_window.cu's for 32 bits).
void write_keys_fixed(const gbwt_b200_index* ix, const uint64_t* part, size_t count, size_t k, uint32_t shift, uint32_t* keys,
                      uint32_t* counts, cudaStream_t s) {
    k_keys_fixed<<<grid_for(ix, count), BLOCK_THREADS, 0, s>>>(ix->view, part, count, k, shift, keys, counts);
}
void write_keys_fixed(const gbwt_b200_index* ix, const uint32_t* part, size_t count, size_t k, uint32_t shift, uint32_t* keys,
                      uint32_t* counts, cudaStream_t s) {
    WindowPlan plan{};
    plan.wshift = shift;
    launch_window_keys<uint32_t>(ix->view, plan, part, count, k, keys, counts, grid_for(ix, count), s);
}

// The search kernel for a batch without record windows (small batches, indexes the windows do not suit).
void launch_find_extend_plain(const gbwt_b200_index* ix, const uint64_t* part, const uint32_t* perm, size_t count, size_t k,
                              gbwt_b200_state* out, cudaStream_t s) {
    // development: GBWT_B200_FIND_LEAN = 0 general, 2 general with runs, 3 lean mixed (only with validated edges)
    const int force = env_int("GBWT_B200_FIND_LEAN", 1);
    if (force == 2) k_find_extend<true><<<grid_for(ix, count), BLOCK_THREADS, 0, s>>>(ix->view, part, perm, count, k, out);
    else if (force == 3 && ix->view.edges_valid) launch_find_extend_lean_mixed(ix->view, part, perm, count, k, out, grid_for(ix, count), s);
    else if (wants_lean_find(ix)) {
        // 5 resident CTAs per SM (48 registers): measured 3.06 G queries/s per step on config 4 against 2.85 with 4
        // (53 registers, no spills), 2.69 with 6 and 1.66 with 8 (spills), 2.81 for the general loop
        if (has_run_records(ix)) launch_find_extend_lean_mixed(ix->view, part, perm, count, k, out, grid_for(ix, count), s);
        else k_find_extend_lean<5><<<grid_for(ix, count), BLOCK_THREADS, 0, s>>>(ix->view, part, perm, count, k, out);
    }
    else if (has_run_records(ix)) k_find_extend<true><<<grid_for(ix, count), BLOCK_THREADS, 0, s>>>(ix->view, part, perm, count, k, out);
    else k_find_extend<false><<<grid_for(ix, count), BLOCK_THREADS, 0, s>>>(ix->view, part, perm, count, k, out);
}
void launch_find_extend_plain(const gbwt_b200_index* ix, const uint32_t* part, const uint32_t* perm, size_t count, size_t k,
                              gbwt_b200_state* out, cudaStream_t s) {
    launch_find_extend_u32(ix->view, has_run_records(ix), part, perm, count, k, out, grid_for(ix, count), s);
}

// Whether a sorted batch goes through the record windows of find_window.cu (GBWT_B200_FIND_WINDOW=0 disables them).
// GBWT_B200_FIND_WINDOW=2 forces them onto any index they can run on (tests).
bool wants_windows(const gbwt_b200_index* ix) {
    const int knob = env_int("GBWT_B200_FIND_WINDOW", 1);
    if (!ix->window_ok || knob == 0 || env_int("GBWT_B200_FIND_LEAN", 1) != 1) return false;
    return knob == 2 || ix->window_suits;
}

// T = uint64_t (the crate's usize nodes) or uint32_t (callers that hold 32-bit node identifiers).
template <class T>
int launch_find_extend(const gbwt_b200_index* ix, const T* patterns, size_t n, size_t k, gbwt_b200_state* out, cudaStream_t s) {
    if (n == 0) return GBWT_B200_OK;
    if (k > 0xFFFFFFFFull) return fail(GBWT_B200_E_ARGUMENT, "pattern length must be below 2^32");
    const size_t max_part = 0xFFFFFFFFull;  // the permutation is 32-bit
    for (size_t begin = 0; begin < n; begin += max_part) {
        const size_t count = std::min(max_part, n - begin);
        const T* part = patterns + begin * k;
        const bool sorted = k >= 2 && wants_locality(ix, count);
        // (a window is decoded into shared memory once per batch: it has to be shared by enough queries to pay)
        if (sorted && wants_windows(ix) && (count >= 8 * static_cast<size_t>(ix->window.windows) || env_int("GBWT_B200_FIND_WINDOW", 1) == 2)) {
            // Record windows: one bucket of the sort = one window; the window kernel answers from shared memory and
            // lists what it could not decide, the general kernel finishes the list.
            uint32_t *perm = nullptr, *bucket_end = nullptr, *scratch = nullptr, *counters = nullptr;
            // margins for this batch's pattern length (the windows themselves, and with them the sort, stay the same)
            WindowPlan plan = ix->window;
            if (k != 32 && !plan_windows(ix->view, plan.body_units, plan.edge_span, plan.wide != 0, static_cast<uint32_t>(std::min<size_t>(k, 4096)), plan))
                plan = ix->window;
            CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&counters), 2 * sizeof(uint32_t), s));
            CUDA_TRY(cudaMemsetAsync(counters, 0, 2 * sizeof(uint32_t), s));
            int rc = GBWT_B200_OK;
            const uint64_t cap = std::max<uint64_t>(64, 2 * ((count + plan.windows - 1) / plan.windows));
            if (env_int("GBWT_B200_WINDOW_DIRECT", 1) != 0 && cap * plan.windows <= 0xFFFFFFFFull) {
                // one pass: every window owns `cap` slots, a query takes the next free one of its window (or is deferred)
                plan.direct_cap = static_cast<uint32_t>(cap);
                CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&bucket_end), plan.windows * sizeof(uint32_t), s));
                CUDA_TRY(cudaMemsetAsync(bucket_end, 0, plan.windows * sizeof(uint32_t), s));
                CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&perm), cap * plan.windows * sizeof(uint32_t), s));
                CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&scratch), count * sizeof(uint32_t), s));
                launch_window_place_direct<T>(ix->view, plan, part, count, k, bucket_end, perm, scratch, counters, grid_for(ix, count), s);
                rc = launch_done("k_window_place_direct");
            } else {
                plan.direct_cap = 0;
                rc = build_locality_perm(ix, count, s, [&](uint32_t, uint32_t* keys, uint32_t* counts) {
                    launch_window_keys<T>(ix->view, ix->window, part, count, k, keys, counts, grid_for(ix, count), s);
                }, &perm, static_cast<int>(ix->window.wshift - ix->window.fine), &bucket_end, &scratch);
            }
            if (rc != GBWT_B200_OK) return rc;
            const bool stats = env_int("GBWT_B200_WINDOW_STATS", 0) != 0;
            cudaEvent_t t0 = nullptr, t1 = nullptr;
            if (stats && (cudaEventCreate(&t0) != cudaSuccess || cudaEventCreate(&t1) != cudaSuccess)) { cudaGetLastError(); t0 = t1 = nullptr; }
            if (t0 != nullptr && t1 != nullptr) cudaEventRecord(t0, s);
            const int e = launch_find_window<T>(ix->view, plan, part, perm, bucket_end, count, k, out + begin, scratch, counters, ix->sm_count, s);
            if (t0 != nullptr && t1 != nullptr) cudaEventRecord(t1, s);
            if (e != 0) rc = cuda_fail(static_cast<cudaError_t>(e), "k_find_window");
            g_launches.fetch_add(1, std::memory_order_relaxed);
            if (rc == GBWT_B200_OK) {
                launch_find_deferred<T>(ix->view, part, scratch, counters, k, out + begin, static_cast<unsigned>(ix->sm_count) * 4, s);
                rc = launch_done("k_find_deferred");
            }
            if (rc == GBWT_B200_OK && stats) {
                uint32_t host[2] = {0, 0};
                if (cudaMemcpyAsync(host, counters, sizeof(host), cudaMemcpyDeviceToHost, s) == cudaSuccess && cudaStreamSynchronize(s) == cudaSuccess) {
                    ix->window_queries.fetch_add(count);
                    ix->window_deferred.fetch_add(host[1]);
                    float ms = 0;
                    if (t0 != nullptr && t1 != nullptr && cudaEventElapsedTime(&ms, t0, t1) == cudaSuccess) {
                        ix->window_kernel_ns.fetch_add(static_cast<uint64_t>(ms * 1e6));
                        ix->window_launches.fetch_add(1);
                    }
                }
            }
            if (t0 != nullptr) cudaEventDestroy(t0);
            if (t1 != nullptr) cudaEventDestroy(t1);
            cudaFreeAsync(perm, s); cudaFreeAsync(bucket_end, s); cudaFreeAsync(scratch, s); cudaFreeAsync(counters, s);
            if (rc != GBWT_B200_OK) return rc;
            continue;
        }
        uint32_t* perm = nullptr;
        if (sorted) {
            int rc = build_locality_perm(ix, count, s, [&](uint32_t shift, uint32_t* keys, uint32_t* counts) {
                write_keys_fixed(ix, part, count, k, shift, keys, counts, s);
            }, &perm);
            if (rc != GBWT_B200_OK) return rc;
        }
        launch_find_extend_plain(ix, part, perm, count, k, out + begin, s);
        int rc = launch_done("k_find_extend");
        if (perm != nullptr) cudaFreeAsync(perm, s);
        if (rc != GBWT_B200_OK) return rc;
    }
    return GBWT_B200_OK;
}

int launch_find_extend_ragged(const gbwt_b200_index* ix, const uint64_t* nodes, const uint64_t* offsets, uint64_t base,
                              size_t n, gbwt_b200_state* out, cudaStream_t s) {
    if (n == 0) return GBWT_B200_OK;
    uint32_t* perm = nullptr;
    if (wants_locality(ix, n)) {
        int rc = build_locality_perm(ix, n, s, [&](uint32_t shift, uint32_t* keys, uint32_t* counts) {
            k_keys_ragged<<<grid_for(ix, n), BLOCK_THREADS, 0, s>>>(ix->view, nodes, offsets, base, nullptr, n, shift, keys, counts);
        }, &perm);
        if (rc != GBWT_B200_OK) return rc;
    }
    if (wants_lean_find(ix) && has_run_records(ix))
        launch_find_extend_ragged_lean_mixed(ix->view, nodes, offsets, base, perm, n, out, grid_for(ix, n), s);
    else if (wants_lean_find(ix))
        k_find_extend_ragged<true><<<grid_for(ix, n), BLOCK_THREADS, 0, s>>>(ix->view, nodes, offsets, base, perm, n, out);
    else
        k_find_extend_ragged<false><<<grid_for(ix, n), BLOCK_THREADS, 0, s>>>(ix->view, nodes, offsets, base, perm, n, out);
    int rc = launch_done("k_find_extend_ragged");
    if (perm != nullptr) cudaFreeAsync(perm, s);
    return rc;
}
int launch_bd_find(const gbwt_b200_index* ix, const uint64_t* nodes, size_t n, gbwt_b200_bdstate* out, cudaStream_t s) {
    if (n == 0) return GBWT_B200_OK;
    k_bd_find<<<grid_for(ix, n), BLOCK_THREADS, 0, s>>>(ix->view, nodes, n, out);
    return launch_done("k_bd_find");
}
int launch_bd_extend(const gbwt_b200_index* ix, const gbwt_b200_bdstate* st, const uint64_t* nodes, size_t n, int backward,
                     gbwt_b200_bdstate* out, cudaStream_t s) {
    if (n == 0) return GBWT_B200_OK;
    k_bd_extend<<<grid_for(ix, n), BLOCK_THREADS, 0, s>>>(ix->view, st, nodes, n, backward, out);
    return launch_done("k_bd_extend");
}
int launch_bd_search(const gbwt_b200_index* ix, const uint64_t* nodes, const uint64_t* offsets, uint64_t base,
                     const uint64_t* first, const uint64_t* start, const uint64_t* end, size_t n, gbwt_b200_bdstate* out,
                     cudaStream_t s) {
    if (n == 0) return GBWT_B200_OK;
    uint32_t* perm = nullptr;
    // Record windows (find_window.cu: k_bd_window): the batch sorted by the window of path[first], the searches answered from
    // shared memory, what a window cannot decide finished by the general loop.
    WindowPlan plan;
    if (wants_locality(ix, n) && wants_windows(ix) && (n >= 8 * static_cast<size_t>(ix->window.windows) || env_int("GBWT_B200_FIND_WINDOW", 1) == 2) &&
        env_int("GBWT_B200_BD_WINDOW", 1) != 0 && plan_bd_windows(ix->window, plan)) {
        uint32_t *bucket_end = nullptr, *scratch = nullptr, *counters = nullptr;
        uint4* packed = nullptr;  // per search, in sorted order: where its subpath starts, its length, the position of `first` in it
        CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&counters), 2 * sizeof(uint32_t), s));
        CUDA_TRY(cudaMemsetAsync(counters, 0, 2 * sizeof(uint32_t), s));
        const uint64_t cap = std::max<uint64_t>(64, 2 * ((n + plan.windows - 1) / plan.windows));
        int rc = GBWT_B200_OK;
        if (env_int("GBWT_B200_WINDOW_DIRECT", 1) != 0 && cap * plan.windows <= 0xFFFFFFFFull) {
            // one pass: every window owns `cap` slots, a search takes the next free one of its window (or is deferred)
            plan.direct_cap = static_cast<uint32_t>(cap);
            CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&bucket_end), plan.windows * sizeof(uint32_t), s));
            CUDA_TRY(cudaMemsetAsync(bucket_end, 0, plan.windows * sizeof(uint32_t), s));
            CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&perm), cap * plan.windows * sizeof(uint32_t), s));
            CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&packed), cap * plan.windows * sizeof(uint4), s));
            CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&scratch), n * sizeof(uint32_t), s));
            launch_bd_place_direct(ix->view, plan, nodes, n, bucket_end, perm, offsets, base, first, start, end, packed, scratch, counters, grid_for(ix, n), s);
            rc = launch_done("k_bd_place_direct");
        } else {
            plan.direct_cap = 0;
            CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&packed), n * sizeof(uint4), s));
            auto place = [&](const uint32_t* keys, uint32_t* cursor, uint32_t* perm_out) {
                launch_bd_place(keys, n, cursor, perm_out, offsets, base, first, start, end, packed, grid_for(ix, n), s);
            };
            rc = build_locality_perm(ix, n, s, [&](uint32_t shift, uint32_t* keys, uint32_t* counts) {
                k_keys_ragged<<<grid_for(ix, n), BLOCK_THREADS, 0, s>>>(ix->view, nodes, offsets, base, first, n, shift, keys, counts);
            }, &perm, static_cast<int>(plan.wshift), &bucket_end, &scratch, &place);
        }
        if (rc != GBWT_B200_OK) { cudaFreeAsync(packed, s); cudaFreeAsync(counters, s); return rc; }
        const int e = launch_bd_window(ix->view, plan, nodes, offsets, base, first, start, end, perm, packed, bucket_end, out, scratch, counters,
                                       ix->sm_count, s);
        g_launches.fetch_add(2, std::memory_order_relaxed);
        cudaFreeAsync(perm, s); cudaFreeAsync(bucket_end, s); cudaFreeAsync(scratch, s); cudaFreeAsync(counters, s); cudaFreeAsync(packed, s);
        if (e != 0) return cuda_fail(static_cast<cudaError_t>(e), "k_bd_window");
        return GBWT_B200_OK;
    }
    if (wants_locality(ix, n)) {
        int rc = build_locality_perm(ix, n, s, [&](uint32_t shift, uint32_t* keys, uint32_t* counts) {
            k_keys_ragged<<<grid_for(ix, n), BLOCK_THREADS, 0, s>>>(ix->view, nodes, offsets, base, first, n, shift, keys, counts);
        }, &perm);
        if (rc != GBWT_B200_OK) return rc;
    }
    if (has_run_records(ix)) k_bd_search<true><<<grid_for(ix, n), BLOCK_THREADS, 0, s>>>(ix->view, nodes, offsets, base, first, start, end, perm, n, out);
    else k_bd_search<false><<<grid_for(ix, n), BLOCK_THREADS, 0, s>>>(ix->view, nodes, offsets, base, first, start, end, perm, n, out);
    int rc = launch_done("k_bd_search");
    if (perm != nullptr) cudaFreeAsync(perm, s);
    return rc;
}
int launch_follow(const gbwt_b200_index* ix, const gbwt_b200_bdstate* st, size_t n, int backward, const uint64_t* out_offsets,
                  uint64_t base, gbwt_b200_bdstate* out, uint64_t* counts, cudaStream_t s) {
    if (n == 0) return GBWT_B200_OK;
    k_follow<<<grid_for(ix, n), BLOCK_THREADS, 0, s>>>(ix->view, st, n, backward, out_offsets, base, out, counts);
    return launch_done("k_follow");
}
int launch_start(const gbwt_b200_index* ix, const uint64_t* ids, size_t n, gbwt_b200_pos* out, cudaStream_t s) {
    if (n == 0) return GBWT_B200_OK;
    k_start<<<grid_for(ix, n), BLOCK_THREADS, 0, s>>>(ix->view, ids, n, out);
    return launch_done("k_start");
}
int launch_forward(const gbwt_b200_index* ix, const gbwt_b200_pos* pos, size_t n, gbwt_b200_pos* out, cudaStream_t s) {
    if (n == 0) return GBWT_B200_OK;
    k_forward<<<grid_for(ix, n), BLOCK_THREADS, 0, s>>>(ix->view, pos, n, out);
    return launch_done("k_forward");
}
int launch_backward(const gbwt_b200_index* ix, const gbwt_b200_pos* pos, size_t n, gbwt_b200_pos* out, cudaStream_t s) {
    if (n == 0) return GBWT_B200_OK;
    k_backward<<<grid_for(ix, n), BLOCK_THREADS, 0, s>>>(ix->view, pos, n, out);
    return launch_done("k_backward");
}
int launch_extract(const gbwt_b200_index* ix, const uint64_t* ids, size_t m, const uint64_t* out_offsets, uint64_t base,
                   uint64_t* nodes, uint64_t* lengths, cudaStream_t s) {
    if (m == 0) return GBWT_B200_OK;
    // With checkpoints every sequence is a set of independent segments (GBWT_B200_EXTRACT_CHECKPOINTS=0: the chain walks below).
    if (ix->ckpt_ok && env_int("GBWT_B200_EXTRACT_CHECKPOINTS", 1) != 0 && std::getenv("GBWT_B200_EXTRACT_STRIDE") == nullptr) {
        if (nodes == nullptr) {
            if (lengths != nullptr) k_lengths_from_table<<<grid_for(ix, m), BLOCK_THREADS, 0, s>>>(ix->view.sequences, ix->ckpt.seq_len, ids, m, lengths);
            return launch_done("k_lengths_from_table");
        }
        const uint64_t items = ((m + 31) / 32) * static_cast<uint64_t>(std::max<uint32_t>(1, ix->ckpt.max_segments));
        CheckpointView cv = ix->ckpt;
        cv.max_segments = std::max<uint32_t>(1, cv.max_segments);
        cv.discard = env_int("GBWT_B200_EXTRACT_DISCARD", 0) != 0 ? 1u : 0u;
        // Enough sequences to fill CTAs of 128 to 512 lanes on an index that suits record windows: the lanes of a CTA walk the same
        // records, so the CTA stages them in shared memory (find_window.cu: k_extract_window; GBWT_B200_EXTRACT_WINDOW=0
        // keeps the one-lane walks from global memory, =2 forces the windows).
        {
            const int knob = env_int("GBWT_B200_EXTRACT_WINDOW", 1);
            WindowPlan plan;
            if (knob != 0 && ix->window_ok && (knob == 2 || (ix->window_suits && m >= 96)) && plan_extract_windows(ix->window, m, plan)) {
                uint32_t* counters = nullptr;
                CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&counters), sizeof(uint32_t), s));
                CUDA_TRY(cudaMemsetAsync(counters, 0, sizeof(uint32_t), s));
                const int e = launch_extract_window(ix->view, cv, plan, ids, m, out_offsets, base, nodes, lengths, counters, ix->sm_count, s);
                g_launches.fetch_add(1, std::memory_order_relaxed);
                cudaFreeAsync(counters, s);
                if (e != 0) return cuda_fail(static_cast<cudaError_t>(e), "k_extract_window");
                return GBWT_B200_OK;
            }
        }
        cv.lookahead = static_cast<uint32_t>(std::max(0, env_int("GBWT_B200_EXTRACT_LOOKAHEAD", 256)));  // measured: +4 % over none
        // (the warps of a CTA take consecutive items, i.e. the same segment of neighbouring sequences; a 1024-thread CTA that
        // holds one segment of 1024 sequences was measured 8 % slower than 256-thread CTAs)
        constexpr int threads = BLOCK_THREADS;
        const size_t tile_bytes = static_cast<size_t>(threads / 32) * 32 * TILE_STRIDE * sizeof(uint32_t);
        const uint64_t ctas_wanted = (items * 32 + threads - 1) / threads;
        const unsigned grid = static_cast<unsigned>(std::max<uint64_t>(1, std::min<uint64_t>(ctas_wanted, static_cast<uint64_t>(ix->sm_count) * 8)));
        auto kernel = ix->view.edges_valid ? k_extract_checkpointed<false, threads> : k_extract_checkpointed<true, threads>;
        CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(tile_bytes)));
        kernel<<<grid, threads, tile_bytes, s>>>(ix->view, cv, ids, m, out_offsets, base, nodes, lengths);
        return launch_done("k_extract_checkpointed");
    }
    // Up to 64 Ki sequences: one warp each (GBWT_B200_EXTRACT_STRIDE overrides: threads per sequence, 32 = warp mode).
    uint32_t stride = static_cast<uint32_t>(env_int("GBWT_B200_EXTRACT_STRIDE", m <= (size_t(1) << 16) ? 32 : 1));
    if (stride != 1 && stride != 2 && stride != 4 && stride != 8 && stride != 16 && stride != 32) stride = 1;
    if (stride == 32) {
        // One-warp CTAs spread few chains over all SMs; beyond 32 CTAs per SM, four warps per CTA.
        const int block = m > static_cast<size_t>(ix->sm_count) * 32 ? 128 : 32;
        const unsigned ctas = static_cast<unsigned>((m * 32 + block - 1) / block);
        // How far ahead (in records) the walks ask L2 for the records they are heading to; 0 disables it.
        const uint32_t ahead = static_cast<uint32_t>(std::max(0, env_int("GBWT_B200_EXTRACT_AHEAD", 48)));
        uint64_t* seq_len = static_cast<uint64_t*>(ix->d_seq_len);
        // With an output to fill and a bidirectional index, sequences whose length is already known are walked from
        // both ends by two warps (GBWT_B200_EXTRACT_SPLIT=0 disables it).
        if (nodes != nullptr && ix->view.bidirectional && seq_len != nullptr && env_int("GBWT_B200_EXTRACT_SPLIT", 1) != 0) {
            const unsigned grid = static_cast<unsigned>(std::min<size_t>(m, size_t(1) << 30));
            if (ix->view.edges_valid) k_extract_split<false><<<grid, 64, 0, s>>>(ix->view, ids, m, out_offsets, base, nodes, lengths, seq_len, ahead);
            else k_extract_split<true><<<grid, 64, 0, s>>>(ix->view, ids, m, out_offsets, base, nodes, lengths, seq_len, ahead);
            return launch_done("k_extract_split");
        }
        if (ix->view.edges_valid) k_extract<false><<<ctas, block, 0, s>>>(ix->view, ids, m, out_offsets, base, nodes, lengths, seq_len, ahead);
        else k_extract<true><<<ctas, block, 0, s>>>(ix->view, ids, m, out_offsets, base, nodes, lengths, seq_len, ahead);
        return launch_done("k_extract");
    }
    const int block = 32;
    const size_t threads = m * stride;
    k_extract_lanes<<<static_cast<unsigned>((threads + block - 1) / block), block, 0, s>>>(ix->view, ids, m, out_offsets, base, nodes, lengths, stride);
    return launch_done("k_extract_lanes");
}
// K4 from checkpoints (kernels.cuh: k_extract_dna_checkpointed). seg_bytes != nullptr: the count pass over all sequences.
int launch_extract_dna_checkpointed(const gbwt_b200_index* ix, const uint64_t* ids, size_t m, const uint64_t* out_offsets, uint64_t base,
                                    uint8_t endmarker, uint8_t* bytes, uint64_t* lengths, uint64_t* seg_bytes, cudaStream_t s) {
    if (m == 0) return GBWT_B200_OK;
    constexpr int threads = BLOCK_THREADS;
    const size_t tile_bytes = static_cast<size_t>(threads / 32) * 32 * DNA_TILE_STRIDE * sizeof(uint32_t);
    const uint64_t items = ((m + 31) / 32) * ix->ckpt.max_segments;
    const uint64_t ctas_wanted = (items * 32 + threads - 1) / threads;
    const unsigned grid = static_cast<unsigned>(std::max<uint64_t>(1, std::min<uint64_t>(ctas_wanted, static_cast<uint64_t>(ix->sm_count) * 8)));
    // CTAs per SM the kernel is compiled for (GBWT_B200_DNA_CTAS: 4 = 64 registers, 3 = 85, anything else = what the compiler takes)
    const int ctas = env_int("GBWT_B200_DNA_CTAS", 4);
    auto kernel = k_extract_dna_checkpointed<false, threads, 1>;
    if (ix->view.edges_valid) kernel = ctas >= 4 ? k_extract_dna_checkpointed<false, threads, 4> : (ctas == 3 ? k_extract_dna_checkpointed<false, threads, 3> : k_extract_dna_checkpointed<false, threads, 1>);
    else kernel = ctas >= 4 ? k_extract_dna_checkpointed<true, threads, 4> : (ctas == 3 ? k_extract_dna_checkpointed<true, threads, 3> : k_extract_dna_checkpointed<true, threads, 1>);
    CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(tile_bytes)));
    kernel<<<grid, threads, tile_bytes, s>>>(ix->view, ix->graph, ix->ckpt, static_cast<const uint64_t*>(ix->d_ckpt_dna), seg_bytes,
                                             static_cast<const uint64_t*>(ix->d_dna_len), ids, m, out_offsets, base, endmarker, bytes, lengths);
    return launch_done("k_extract_dna_checkpointed");
}

// Where the DNA of every sequence stands at each of its checkpoints: one count pass over all segments (every node's label
// length, no bytes moved), then a scan per sequence; leaves the DNA length of every sequence in d_dna_len. Called when an
// index has both checkpoints and node labels (at creation, when labels are attached, after an import). Without it DNA is
// extracted by whole-sequence walks; a failure here only means that.
void build_dna_checkpoints(gbwt_b200_index* ix) {
    cudaFree(ix->d_ckpt_dna);
    ix->d_ckpt_dna = nullptr;
    ix->dna_ckpt_ok = false;
    if (!ix->ckpt_ok || !ix->has_graph || ix->d_dna_len == nullptr || ix->ckpt.max_segments == 0 || env_int("GBWT_B200_DNA_CHECKPOINTS", 1) == 0) return;
    DeviceScope scope(ix->device);
    if (!scope.ok) return;
    uint64_t* seg = nullptr;
    if (cudaMalloc(reinterpret_cast<void**>(&seg), std::max<size_t>(256, ix->ckpt_entries * sizeof(uint64_t))) != cudaSuccess) { cudaGetLastError(); return; }
    cudaStream_t s = nullptr;
    int rc = launch_extract_dna_checkpointed(ix, nullptr, ix->view.sequences, nullptr, 0, 0, nullptr, nullptr, seg, s);
    if (rc == GBWT_B200_OK) {
        k_dna_checkpoint_scan<<<grid_for(ix, ix->view.sequences), BLOCK_THREADS, 0, s>>>(ix->view.sequences, ix->ckpt.first, seg,
                                                                                         static_cast<uint64_t*>(ix->d_dna_len));
        rc = launch_done("k_dna_checkpoint_scan");
    }
    if (rc != GBWT_B200_OK || cudaStreamSynchronize(s) != cudaSuccess) { cudaGetLastError(); cudaFree(seg); return; }
    ix->d_ckpt_dna = seg;
    ix->dna_ckpt_ok = true;
}

int launch_extract_dna(const gbwt_b200_index* ix, const uint64_t* ids, size_t m, const uint64_t* out_offsets, uint64_t base,
                       uint8_t endmarker, uint8_t* bytes, uint64_t* lengths, cudaStream_t s) {
    if (m == 0) return GBWT_B200_OK;
    // One warp per sequence. One-warp CTAs spread few chains over all SMs; with more chains than the SMs hold
    // that way (32 CTAs each), four warps per CTA double the chains in flight.
    const int block = m > static_cast<size_t>(ix->sm_count) * 32 ? 128 : 32;
    const size_t ctas = (m * 32 + block - 1) / block;
    const uint32_t ahead = static_cast<uint32_t>(std::max(0, env_int("GBWT_B200_EXTRACT_AHEAD", 48)));
    const unsigned grid = static_cast<unsigned>(std::min<size_t>(ctas, size_t(1) << 30));
    uint64_t *seq_len = static_cast<uint64_t*>(ix->d_seq_len), *dna_len = static_cast<uint64_t*>(ix->d_dna_len);
    // With path checkpoints and their DNA positions every sequence is spelled as independent segments, one lane each
    // (GBWT_B200_DNA_CHECKPOINTS=0: whole-sequence walks), and the lengths are a table lookup.
    if (ix->dna_ckpt_ok && env_int("GBWT_B200_DNA_CHECKPOINTS", 1) != 0) {
        if (bytes == nullptr) {
            if (lengths != nullptr) k_lengths_from_table<<<grid_for(ix, m), BLOCK_THREADS, 0, s>>>(ix->view.sequences, dna_len, ids, m, lengths);
            return launch_done("k_lengths_from_table");
        }
        return launch_extract_dna_checkpointed(ix, ids, m, out_offsets, base, endmarker, bytes, lengths, nullptr, s);
    }
    // sequences whose lengths are known are spelled from both ends by two warps (see launch_extract)
    if (bytes != nullptr && ix->view.bidirectional && env_int("GBWT_B200_EXTRACT_SPLIT", 1) != 0) {
        const unsigned pairs = static_cast<unsigned>(std::min<size_t>(m, size_t(1) << 30));
        if (env_int("GBWT_B200_DNA_RELAY", 1) != 0) {
            if (ix->view.edges_valid) k_extract_dna_relay<false><<<pairs, 96, 0, s>>>(ix->view, ix->graph, ids, m, out_offsets, base, endmarker, bytes, lengths, seq_len, dna_len, ahead);
            else k_extract_dna_relay<true><<<pairs, 96, 0, s>>>(ix->view, ix->graph, ids, m, out_offsets, base, endmarker, bytes, lengths, seq_len, dna_len, ahead);
            return launch_done("k_extract_dna_relay");
        }
        if (ix->view.edges_valid) k_extract_dna_split<false><<<pairs, 64, 0, s>>>(ix->view, ix->graph, ids, m, out_offsets, base, endmarker, bytes, lengths, seq_len, dna_len, ahead);
        else k_extract_dna_split<true><<<pairs, 64, 0, s>>>(ix->view, ix->graph, ids, m, out_offsets, base, endmarker, bytes, lengths, seq_len, dna_len, ahead);
        return launch_done("k_extract_dna_split");
    }
    if (ix->view.edges_valid) k_extract_dna<false><<<grid, block, 0, s>>>(ix->view, ix->graph, ids, m, out_offsets, base, endmarker, bytes, lengths, seq_len, dna_len, ahead);
    else k_extract_dna<true><<<grid, block, 0, s>>>(ix->view, ix->graph, ids, m, out_offsets, base, endmarker, bytes, lengths, seq_len, dna_len, ahead);
    return launch_done("k_extract_dna");
}
int launch_node_sequences(const gbwt_b200_index* ix, const uint64_t* node_ids, size_t n, const uint64_t* out_offsets, uint64_t base,
                          uint8_t* bytes, uint64_t* lengths, cudaStream_t s) {
    if (n == 0) return GBWT_B200_OK;
    k_node_sequences<<<grid_for(ix, n * 32), BLOCK_THREADS, 0, s>>>(ix->view, ix->graph, node_ids, n, out_offsets, base, bytes, lengths);
    return launch_done("k_node_sequences");
}

// ---- host <-> device pipeline ----------------------------------------------------------------------

// How an array of a batched host call is cut for the chunk of items [q0, q1).
enum class Slice {
    Item,      // `width` bytes per item: items q0 .. q1
    Offsets,   // the chunking offsets themselves: words q0 .. q1, both included
    Elements,  // `width` bytes per element: elements offsets[q0] .. offsets[q1] (pattern nodes, output slots)
};

// An array on the host side of a batched call. One with neither `in` nor `out` is device scratch.
struct HostArray {
    const void* in;     // copied to the device before the kernel (may be null)
    void* out;          // copied back after the kernel (may be null)
    size_t width;
    Slice slice = Slice::Item;
    int fill = -1;      // byte written over the device array before the kernel (-1: none), so that output slots larger
                        // than their results carry it back to the caller, not stale pool memory
};

// Chunk size: about 64 MiB of the widest array per chunk, at least 16 Ki items.
size_t chunk_for(size_t widest_item_bytes, size_t target = size_t(64) << 20) {
    if (const int mb = env_int("GBWT_B200_HOST_CHUNK_MB", 0); mb > 0) target = static_cast<size_t>(mb) << 20;  // tests
    return std::max<size_t>(size_t(1) << 14, target / std::max<size_t>(1, widest_item_bytes));
}

// Budget of one chunk of a ragged batch (items, or the pattern nodes, output elements, extensions or occurrences they
// hold). GBWT_B200_HOST_RAGGED_BUDGET=N caps it at N, so that tests cross chunk boundaries with small batches.
uint64_t ragged_budget(uint64_t budget) {
    if (const int cap = env_int("GBWT_B200_HOST_RAGGED_BUDGET", 0); cap > 0) return std::min<uint64_t>(budget, static_cast<uint64_t>(cap));  // tests
    return budget;
}

// Fixed-size batches: `items` per chunk, and with `taper` the last chunk's worth cut into halves (see run_chunked).
size_t fixed_chunk_end(size_t n, size_t q0, size_t items, bool taper) {
    const size_t left = n - q0;
    if (taper && left <= items && left / 2 >= std::max<size_t>(size_t(1) << 14, items / 16)) return q0 + left / 2;
    return q0 + std::min(items, left);
}

// Ragged batches: items [q0, q1) such that offsets[q1] - offsets[q0] <= node_budget (at least one item).
size_t ragged_chunk_end(const uint64_t* offsets, size_t n, size_t q0, size_t item_budget, uint64_t node_budget) {
    size_t q1 = std::min(n, q0 + item_budget);
    if (q1 > q0 + 1 && offsets[q1] - offsets[q0] > node_budget) {
        size_t lo = q0 + 1, hi = q1;  // largest q1 within the node budget, but never fewer than one item
        while (lo < hi) {
            size_t mid = lo + (hi - lo + 1) / 2;
            if (offsets[mid] - offsets[q0] <= node_budget) lo = mid; else hi = mid - 1;
        }
        q1 = lo;
    }
    return q1;
}

bool offsets_valid(const uint64_t* offsets, size_t n) {
    for (size_t i = 0; i < n; i++) if (offsets[i + 1] < offsets[i]) return false;
    return true;
}

// Where the chunks of a batch end, and how many streams they alternate on.
struct Chunking {
    size_t items;                       // items per chunk (ragged: at most)
    int streams;
    bool taper = false;                 // fixed-size: cut the last chunk's worth into halves
    const uint64_t* offsets = nullptr;  // ragged: item i holds elements offsets[i] .. offsets[i+1]
    uint64_t elems = 0;                 // ragged: elements per chunk, at most (but at least one item)
};

// Fixed-size chunks of `items` items: one stream for a batch of one chunk, two for more, four with the tapered tail.
Chunking fixed_chunks(size_t n, size_t items) {
    if (n <= items) return {items, 1};
    const bool taper = env_int("GBWT_B200_HOST_TAPER", 1) != 0;
    return {items, taper ? 4 : 2, taper};
}

// Ragged chunks of at most `items` items and `elems` elements, each capped by ragged_budget.
Chunking ragged_chunks(const uint64_t* offsets, size_t items, uint64_t elems, int streams) {
    return {ragged_budget(items), streams, false, offsets, ragged_budget(elems)};
}

// Processes items [0, n) in chunks on alternating streams: H2D of the chunk's inputs, the kernel(s), D2H of its outputs.
// With page-locked host memory the copies of one chunk overlap the kernels of the others, and the host-to-device copies
// follow each other without a gap: the call takes the time of its input copies plus whatever is left to do when the last
// byte has arrived. That tail is the last chunk's kernels and output copy, so the last chunk's worth of items is cut into
// halves (1/2, 1/4, ... of a chunk, down to 1/16): the kernels of each piece run under the copy of the next, and what
// follows the last copy is the work of a sixteenth of a chunk. (Four streams: a piece must not wait for the output copy of
// the piece two before it.)
// `launch(q0, count, device_ptrs, stream)` receives one device pointer per HostArray. Empty slices are neither filled nor
// copied, but still get a device array.
template <class Launch>
int run_chunked(const gbwt_b200_index* ix, size_t n, const std::vector<HostArray>& arrays, const Chunking& c, Launch launch) {
    if (n == 0) return GBWT_B200_OK;
    DeviceScope scope(ix->device);
    if (!scope.ok) return fail(GBWT_B200_E_CUDA, "cudaSetDevice failed");
    std::vector<cudaStream_t> streams(c.streams, nullptr);
    for (cudaStream_t& s : streams) CUDA_TRY(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    int rc = GBWT_B200_OK;
    std::vector<void*> dptr(arrays.size(), nullptr);
    std::vector<size_t> at(arrays.size()), bytes(arrays.size());  // the chunk's slice of each array on the host
    for (size_t q0 = 0, chunk_index = 0; q0 < n && rc == GBWT_B200_OK; chunk_index++) {
        const size_t q1 = c.offsets != nullptr ? ragged_chunk_end(c.offsets, n, q0, c.items, c.elems)
                                               : fixed_chunk_end(n, q0, c.items, c.taper);
        cudaStream_t s = streams[chunk_index % streams.size()];
        for (size_t a = 0; a < arrays.size() && rc == GBWT_B200_OK; a++) {
            const HostArray& h = arrays[a];
            const size_t first = h.slice == Slice::Elements ? c.offsets[q0] : q0;
            const size_t end = h.slice == Slice::Elements ? c.offsets[q1] : h.slice == Slice::Offsets ? q1 + 1 : q1;
            at[a] = first * h.width;
            bytes[a] = (end - first) * h.width;
            cudaError_t e = cudaMallocAsync(&dptr[a], std::max<size_t>(16, bytes[a]), s);
            if (e != cudaSuccess) rc = cuda_fail(e, "cudaMallocAsync");
        }
        for (size_t a = 0; a < arrays.size() && rc == GBWT_B200_OK; a++) {
            const HostArray& h = arrays[a];
            if (bytes[a] == 0) continue;
            cudaError_t e = h.fill >= 0 ? cudaMemsetAsync(dptr[a], h.fill, bytes[a], s) : cudaSuccess;
            if (e == cudaSuccess && h.in != nullptr)
                e = cudaMemcpyAsync(dptr[a], static_cast<const char*>(h.in) + at[a], bytes[a], cudaMemcpyHostToDevice, s);
            if (e != cudaSuccess) rc = cuda_fail(e, "cudaMemcpyAsync H2D");
        }
        if (rc == GBWT_B200_OK) rc = launch(q0, q1 - q0, dptr, s);
        for (size_t a = 0; a < arrays.size(); a++) {
            if (dptr[a] == nullptr) continue;
            if (rc == GBWT_B200_OK && arrays[a].out != nullptr && bytes[a] > 0) {
                cudaError_t e = cudaMemcpyAsync(static_cast<char*>(arrays[a].out) + at[a], dptr[a], bytes[a], cudaMemcpyDeviceToHost, s);
                if (e != cudaSuccess) rc = cuda_fail(e, "cudaMemcpyAsync D2H");
            }
            cudaFreeAsync(dptr[a], s);
            dptr[a] = nullptr;
        }
        q0 = q1;
    }
    for (cudaStream_t s : streams) {
        cudaError_t e = cudaStreamSynchronize(s);
        if (e != cudaSuccess && rc == GBWT_B200_OK) rc = cuda_fail(e, "cudaStreamSynchronize");
        cudaStreamDestroy(s);
    }
    return rc;
}

// Checks the arguments of a call that writes the `elem_bytes`-sized elements of item i into out[out_offsets[i] ..
// out_offsets[i+1]), and sets `budget` to the elements of one chunk: 60% of the free HBM of the index's device, at least
// 1 Mi. (Such a call puts all its items in one chunk: a path walk is latency-bound, so concurrency is everything.)
int slot_budget(const gbwt_b200_index* ix, const uint64_t* ids, size_t m, const uint64_t* out_offsets, const void* out,
                size_t elem_bytes, uint64_t* budget) {
    if (m == 0) return GBWT_B200_OK;
    if (ids == nullptr || out_offsets == nullptr) return fail(GBWT_B200_E_ARGUMENT, "null array");
    if (!offsets_valid(out_offsets, m)) return fail(GBWT_B200_E_ARGUMENT, "out_offsets must be non-decreasing");
    if (out_offsets[m] > out_offsets[0] && out == nullptr) return fail(GBWT_B200_E_ARGUMENT, "null output");
    DeviceScope scope(ix->device);
    if (!scope.ok) return fail(GBWT_B200_E_CUDA, "cudaSetDevice failed");
    size_t free_bytes = 0, total_bytes = 0;
    CUDA_TRY(cudaMemGetInfo(&free_bytes, &total_bytes));
    *budget = std::max<uint64_t>(uint64_t(1) << 20, (free_bytes / elem_bytes) * 6 / 10);
    return GBWT_B200_OK;
}

int check_index(const gbwt_b200_index* ix) {
    if (ix == nullptr) return fail(GBWT_B200_E_ARGUMENT, "null index handle");
    return GBWT_B200_OK;
}

int check_bidirectional(const gbwt_b200_index* ix) {
    // assert!(self.is_bidirectional(), ...) at src/gbwt.rs:237, 312, 340
    if (!(ix->flags & GBWT_FLAG_BIDIRECTIONAL)) return fail(GBWT_B200_E_NOT_BIDIRECTIONAL, "Bidirectional search requires a bidirectional GBWT");
    return GBWT_B200_OK;
}

int upload(void** d, const void* h, size_t bytes, uint64_t& accounted) {
    *d = nullptr;
    accounted = bytes;
    CUDA_TRY(cudaMalloc(d, std::max<size_t>(bytes, 256)));
    if (bytes > 0) CUDA_TRY(cudaMemcpy(*d, h, bytes, cudaMemcpyHostToDevice));
    return GBWT_B200_OK;
}

// Node labels into HBM: starts[0 .. sequences] and the concatenated bytes (the caller has validated them).
int attach_graph(gbwt_b200_index* ix, const uint64_t* starts, uint64_t sequences, const uint8_t* label_bytes) {
    DeviceScope scope(ix->device);
    if (!scope.ok) return fail(GBWT_B200_E_CUDA, "cudaSetDevice failed");
    cudaFree(ix->d_label_starts); cudaFree(ix->d_label_bytes);
    ix->d_label_starts = ix->d_label_bytes = nullptr;
    ix->has_graph = false;
    ix->dna_ckpt_ok = false;
    ix->carried.graph_section.clear();  // (create_index restores the loaded one after attaching the loaded labels)
    // DNA lengths measured with another graph are void
    if (ix->d_dna_len != nullptr) CUDA_TRY(cudaMemset(ix->d_dna_len, 0xFE, std::max<size_t>(256, ix->sequences * sizeof(uint64_t))));
    uint64_t a = 0, b = 0;
    int rc = upload(&ix->d_label_starts, starts, (sequences + 1) * 8, a);
    if (rc == GBWT_B200_OK) rc = upload(&ix->d_label_bytes, label_bytes, starts[sequences], b);
    if (rc != GBWT_B200_OK) return rc;
    ix->graph.starts = static_cast<const uint64_t*>(ix->d_label_starts);
    ix->graph.bytes = static_cast<const uint8_t*>(ix->d_label_bytes);
    ix->graph.sequences = sequences;
    ix->graph_bytes = a + b;
    ix->has_graph = true;
    build_dna_checkpoints(ix);
    return GBWT_B200_OK;
}

int check_samples(const gbwt_b200_index* ix) {
    if (!ix->locate_ok) return fail(GBWT_B200_E_NO_SAMPLES, "the index was created without locate samples (GBWT_B200_LAYOUT_LOCATE)");
    return GBWT_B200_OK;
}

LocateView locate_view(const gbwt_b200_index* ix) {
    LocateView lv;
    lv.first = static_cast<const uint32_t*>(ix->d_locate_first);
    lv.samples = static_cast<const LocateSample*>(ix->d_locate_samples);
    // a walk meets a sample within 2^shift + 32 steps on a consistent index; the slack and walk_limit end it on a damaged one
    lv.max_steps = std::min<uint64_t>((uint64_t(1) << ix->locate_shift) + 64, ix->view.walk_limit);
    return lv;
}

// Runs `launch(steps)` on stream s; with GBWT_B200_LOCATE_STATS=1 it hands a device counter to the kernels, waits for the
// stream and adds the LF steps they counted to the index's total.
template <class Launch>
int with_locate_stats(const gbwt_b200_index* ix, cudaStream_t s, Launch launch) {
    if (env_int("GBWT_B200_LOCATE_STATS", 0) == 0) return launch(static_cast<unsigned long long*>(nullptr));
    unsigned long long* steps = nullptr;
    CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&steps), sizeof(unsigned long long), s));
    CUDA_TRY(cudaMemsetAsync(steps, 0, sizeof(unsigned long long), s));
    int rc = launch(steps);
    unsigned long long host = 0;
    if (rc == GBWT_B200_OK) {
        cudaError_t e = cudaMemcpyAsync(&host, steps, sizeof(host), cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) rc = cuda_fail(e, "locate step counter");
        else ix->locate_steps.fetch_add(host);
    }
    cudaFreeAsync(steps, s);
    return rc;
}

int launch_locate_positions(const gbwt_b200_index* ix, const gbwt_b200_pos* pos, size_t n, gbwt_b200_occurrence* out, cudaStream_t s) {
    if (n == 0) return GBWT_B200_OK;
    return with_locate_stats(ix, s, [&](unsigned long long* steps) {
        cudaError_t e = launch_locate(ix->view, locate_view(ix), pos, n, out, steps, ix->sm_count, s);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        return e == cudaSuccess ? GBWT_B200_OK : cuda_fail(e, "k_locate");
    });
}

int launch_locate_state_batch(const gbwt_b200_index* ix, const gbwt_b200_state* states, size_t n, const uint64_t* out_offsets, uint64_t base,
                              gbwt_b200_occurrence* out, uint64_t* counts, cudaStream_t s) {
    if (n == 0) return GBWT_B200_OK;
    return with_locate_stats(ix, s, [&](unsigned long long* steps) {
        cudaError_t e = launch_locate_states(ix->view, locate_view(ix), states, n, out_offsets, base, out, counts, steps, ix->sm_count, s);
        g_launches.fetch_add(out != nullptr ? 4 : 1, std::memory_order_relaxed);
        return e == cudaSuccess ? GBWT_B200_OK : cuda_fail(e, "k_locate_states");
    });
}

int check_graph(const gbwt_b200_index* ix) {
    if (!ix->has_graph) return fail(GBWT_B200_E_NO_GRAPH, "the index was not loaded from a GBZ file: no node sequences");
    return GBWT_B200_OK;
}

// The path checkpoints the range walks start from (ranges.h): table == nullptr where the index has none, and for DNA where it
// has no DNA checkpoints (or GBWT_B200_DNA_CHECKPOINTS=0, as in launch_extract_dna).
CheckpointView range_view(const gbwt_b200_index* ix, bool dna) {
    CheckpointView cv = ix->ckpt;
    if (!ix->ckpt_ok || (dna && !(ix->dna_ckpt_ok && env_int("GBWT_B200_DNA_CHECKPOINTS", 1) != 0))) cv.table = nullptr;
    return cv;
}

int launch_seek_batch(const gbwt_b200_index* ix, const uint64_t* ids, const uint64_t* indexes, size_t n, gbwt_b200_pos* out, cudaStream_t s) {
    if (n == 0) return GBWT_B200_OK;
    const cudaError_t e = launch_seek(ix->view, range_view(ix, false), ix->ckpt_shift, ids, indexes, n, out, ix->sm_count, s);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return e == cudaSuccess ? GBWT_B200_OK : cuda_fail(e, "k_seek");
}

int launch_range_batch(const gbwt_b200_index* ix, bool dna, const uint64_t* ids, const uint64_t* starts, const uint64_t* ends, size_t m,
                       const uint64_t* out_offsets, uint64_t base, void* out, uint64_t* lengths, cudaStream_t s) {
    if (m == 0) return GBWT_B200_OK;
    const CheckpointView cv = range_view(ix, dna);
    const cudaError_t e = dna ? launch_range_dna(ix->view, ix->graph, cv, static_cast<const uint64_t*>(ix->d_ckpt_dna),
                                                 static_cast<const uint64_t*>(ix->d_dna_len), ids, starts, ends, m, out_offsets, base,
                                                 static_cast<uint8_t*>(out), lengths, ix->sm_count, s)
                              : launch_range_nodes(ix->view, cv, ix->ckpt_shift, ids, starts, ends, m, out_offsets, base,
                                                   static_cast<uint64_t*>(out), lengths, ix->sm_count, s);
    g_launches.fetch_add(4, std::memory_order_relaxed);  // (the plan, CUB's two scan kernels, the pieces)
    return e == cudaSuccess ? GBWT_B200_OK : cuda_fail(e, dna ? "k_range_pieces<true>" : "k_range_pieces<false>");
}

// Host twin of the range calls: the arguments checked like extract's, then the chunk loop over the output slots.
int ranges_host(const gbwt_b200_index* ix, bool dna, const uint64_t* ids, const uint64_t* starts, const uint64_t* ends, size_t m,
                const uint64_t* out_offsets, void* out, uint64_t* lengths) {
    if (int rc = check_index(ix)) return rc;
    if (dna) { if (int rc = check_graph(ix)) return rc; }
    const size_t width = dna ? 1 : sizeof(uint64_t);
    uint64_t elems = 0;
    if (int rc = slot_budget(ix, ids, m, out_offsets, out, width, &elems)) return rc;
    if (m > 0 && (starts == nullptr || ends == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null array");
    std::vector<HostArray> arrays = {{ids, nullptr, 8}, {starts, nullptr, 8}, {ends, nullptr, 8}, {nullptr, out, width, Slice::Elements, 0x00},
                                     {out_offsets, nullptr, 8, Slice::Offsets}, {nullptr, lengths, 8}};
    return run_chunked(ix, m, arrays, ragged_chunks(out_offsets, m, elems, 1), [&](size_t q0, size_t count, std::vector<void*>& d, cudaStream_t s) {
        auto u = [&](int a) { return static_cast<const uint64_t*>(d[a]); };
        return launch_range_batch(ix, dna, u(0), u(1), u(2), count, u(4), out_offsets[q0], d[3], static_cast<uint64_t*>(d[5]), s);
    });
}

// Device twin: the batch in slices of 2^30 ranges (the scan of a slice is indexed with 64-bit CUB offsets; slices keep each
// launch's temporary arrays bounded).
int ranges_device(const gbwt_b200_index* ix, bool dna, const uint64_t* ids, const uint64_t* starts, const uint64_t* ends, size_t m,
                  const uint64_t* out_offsets, void* out, uint64_t* lengths, cudaStream_t s) {
    if (m > 0 && (ids == nullptr || starts == nullptr || ends == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null array");
    if (m > 0 && (out == nullptr || out_offsets == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null output");
    const size_t chunk = size_t(1) << 30;
    for (size_t begin = 0; begin < m; begin += chunk) {
        const size_t count = std::min(chunk, m - begin);
        int rc = launch_range_batch(ix, dna, ids + begin, starts + begin, ends + begin, count, out_offsets + begin, 0, out,
                                    lengths != nullptr ? lengths + begin : nullptr, s);
        if (rc != GBWT_B200_OK) return rc;
    }
    return GBWT_B200_OK;
}

// In-place inclusive scan of counts[0 .. m) on stream s (the three launches of kernels.cuh).
int scan_counts(uint32_t* counts, uint32_t m, cudaStream_t s) {
    const uint32_t tiles = (m + SCAN_TILE - 1) / SCAN_TILE;
    uint32_t* tile_sums = nullptr;
    CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&tile_sums), tiles * sizeof(uint32_t), s));
    k_scan_tiles<<<tiles, 1024, 0, s>>>(counts, m, tile_sums);
    launch_done("k_scan_tiles");
    if (tiles > 1) {
        k_scan_single<<<1, 1024, 0, s>>>(tile_sums, tiles);
        launch_done("k_scan_single");
        k_scan_add<<<tiles, 1024, 0, s>>>(counts, m, tile_sums);
        launch_done("k_scan_add");
    }
    cudaFreeAsync(tile_sums, s);
    return GBWT_B200_OK;
}

// Path checkpoints: one warp-mode walk over every sequence records its length and its position at about every
// 2^shift-th node; afterwards a sequence can be extracted as independent segments (k_extract_checkpointed). The
// interval is chosen so that the table holds at most ~16 M entries (GBWT_B200_CHECKPOINT_SHIFT overrides).
int build_checkpoints(gbwt_b200_index* ix) {
    const IndexView& v = ix->view;
    if (v.sequences == 0 || v.sequences >= 0xFFFFFFFFull) return GBWT_B200_OK;
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
    uint32_t shift = 6;
    while (shift < 30 && (v.walk_limit >> shift) > (uint64_t(16) << 20)) shift++;
    shift = static_cast<uint32_t>(std::min(30, std::max(6, env_int("GBWT_B200_CHECKPOINT_SHIFT", static_cast<int>(shift)))));
    const uint64_t pool_cap = (v.walk_limit >> shift) + v.sequences + 1024;
    PoolEntry* pool = nullptr;
    unsigned long long* used_dev = nullptr;
    uint32_t* first = nullptr;
    cudaStream_t s = nullptr;
    CUDA_TRY(cudaEventRecord(e0, s));
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&pool), pool_cap * sizeof(PoolEntry)));
    int rc = GBWT_B200_OK;
    auto cleanup = [&]() { cudaFree(pool); cudaFree(used_dev); cudaEventDestroy(e0); cudaEventDestroy(e1); };
    if (cudaMalloc(reinterpret_cast<void**>(&used_dev), sizeof(unsigned long long)) != cudaSuccess ||
        cudaMemset(used_dev, 0, sizeof(unsigned long long)) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void**>(&first), (v.sequences + 1) * sizeof(uint32_t)) != cudaSuccess ||
        cudaMemset(first, 0, (v.sequences + 1) * sizeof(uint32_t)) != cudaSuccess) {
        rc = cuda_fail(cudaGetLastError(), "cudaMalloc(checkpoints)");
        cleanup(); cudaFree(first);
        return rc;
    }
    const int block = 128;
    const unsigned ctas = static_cast<unsigned>(std::min<uint64_t>((v.sequences * 32 + block - 1) / block, uint64_t(1) << 20));
    const uint32_t ahead = static_cast<uint32_t>(std::max(0, env_int("GBWT_B200_EXTRACT_AHEAD", 48)));
    uint64_t* seq_len = static_cast<uint64_t*>(ix->d_seq_len);
    if (v.edges_valid) k_build_checkpoints<false><<<ctas, block, 0, s>>>(v, shift, pool, used_dev, pool_cap, seq_len, ahead);
    else k_build_checkpoints<true><<<ctas, block, 0, s>>>(v, shift, pool, used_dev, pool_cap, seq_len, ahead);
    rc = launch_done("k_build_checkpoints");
    unsigned long long used = 0;
    if (rc == GBWT_B200_OK && cudaMemcpy(&used, used_dev, sizeof(used), cudaMemcpyDeviceToHost) != cudaSuccess)
        rc = cuda_fail(cudaGetLastError(), "k_build_checkpoints");
    if (rc != GBWT_B200_OK || used > pool_cap || used > 0xFFFFFFF0ull) {  // (an overflowing pool: leave the index without checkpoints)
        cleanup(); cudaFree(first);
        return rc;
    }
    Checkpoint* table = nullptr;
    if (cudaMalloc(reinterpret_cast<void**>(&table), std::max<size_t>(256, used * sizeof(Checkpoint))) != cudaSuccess) {
        rc = cuda_fail(cudaGetLastError(), "cudaMalloc(checkpoint table)");
        cleanup(); cudaFree(first);
        return rc;
    }
    if (used > 0) {
        k_checkpoint_count<<<grid_for(ix, used), BLOCK_THREADS, 0, s>>>(pool, used, first);
        launch_done("k_checkpoint_count");
        rc = scan_counts(first, static_cast<uint32_t>(v.sequences + 1), s);
        if (rc == GBWT_B200_OK) {
            k_checkpoint_scatter<<<grid_for(ix, used), BLOCK_THREADS, 0, s>>>(pool, used, shift, first, table);
            rc = launch_done("k_checkpoint_scatter");
        }
    }
    std::vector<uint32_t> host_first(v.sequences + 1, 0);
    if (rc == GBWT_B200_OK && cudaMemcpy(host_first.data(), first, host_first.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost) != cudaSuccess)
        rc = cuda_fail(cudaGetLastError(), "checkpoint table");
    CUDA_TRY(cudaEventRecord(e1, s));
    CUDA_TRY(cudaEventSynchronize(e1));
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    cleanup();
    if (rc != GBWT_B200_OK) { cudaFree(first); cudaFree(table); return rc; }
    uint32_t max_segments = 0;
    for (uint64_t i = 0; i < v.sequences; i++) max_segments = std::max(max_segments, host_first[i + 1] - host_first[i]);
    ix->d_ckpt_table = table; ix->d_ckpt_first = first;
    ix->ckpt.table = table; ix->ckpt.first = first; ix->ckpt.seq_len = seq_len; ix->ckpt.max_segments = max_segments; ix->ckpt.discard = 0; ix->ckpt.lookahead = 0;
    ix->ckpt_shift = shift; ix->ckpt_entries = used;
    ix->ckpt_bytes = used * sizeof(Checkpoint) + (v.sequences + 1) * sizeof(uint32_t);
    ix->ckpt_build_us = static_cast<uint64_t>(ms * 1000.0f);
    ix->ckpt_ok = true;
    return GBWT_B200_OK;
}

// Locate samples: one walk over every sequence emits a sample at every 2^shift-th node (the first flush at or after it) and
// at its last node (LocateSink), and locate.cu sorts them by BWT position. Default interval 2^10 (the C++ GBWT's sample
// interval); GBWT_B200_LOCATE_SHIFT (0 .. 20) overrides it. The flag was asked for, so anything that keeps the table from
// being built fails the creation.
int build_locate(gbwt_b200_index* ix) {
    const IndexView& v = ix->view;
    if (v.sequences > 0xFFFFFFFFull) return fail(GBWT_B200_E_RANGE, "locate samples hold 32-bit sequence ids");
    const uint32_t shift = static_cast<uint32_t>(std::min(20, std::max(0, env_int("GBWT_B200_LOCATE_SHIFT", 10))));
    // at most one sample per multiple of the interval and one at the last node of every sequence (+ slack for the flushes)
    const uint64_t cap = (v.walk_limit >> shift) + 2 * v.sequences + 1024;
    cudaStream_t s = nullptr;
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
    uint64_t* keys = nullptr;
    LocateSample* pool = nullptr;
    unsigned long long* used_dev = nullptr;
    uint32_t* first = nullptr;
    LocateSample* table = nullptr;
    auto cleanup = [&]() { cudaFree(keys); cudaFree(pool); cudaFree(used_dev); cudaEventDestroy(e0); cudaEventDestroy(e1); };
    auto give_up = [&](int rc) { cleanup(); cudaFree(first); cudaFree(table); return rc; };
    CUDA_TRY(cudaEventRecord(e0, s));
    if (cudaMalloc(reinterpret_cast<void**>(&keys), cap * sizeof(uint64_t)) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void**>(&pool), cap * sizeof(LocateSample)) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void**>(&used_dev), sizeof(unsigned long long)) != cudaSuccess ||
        cudaMemset(used_dev, 0, sizeof(unsigned long long)) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void**>(&first), (v.records + 1) * sizeof(uint32_t)) != cudaSuccess)
        return give_up(cuda_fail(cudaGetLastError(), "cudaMalloc(locate samples)"));
    int rc = GBWT_B200_OK;
    if (shift >= 5) {
        const int block = 128;
        const unsigned ctas = static_cast<unsigned>(std::min<uint64_t>((v.sequences * 32 + block - 1) / block, uint64_t(1) << 20));
        const uint32_t ahead = static_cast<uint32_t>(std::max(0, env_int("GBWT_B200_EXTRACT_AHEAD", 48)));
        if (v.sequences > 0) {
            if (v.edges_valid) k_build_locate<false><<<ctas, block, 0, s>>>(v, shift, keys, pool, used_dev, cap, ahead);
            else k_build_locate<true><<<ctas, block, 0, s>>>(v, shift, keys, pool, used_dev, cap, ahead);
        }
    } else if (v.sequences > 0) {
        k_build_locate_lanes<<<grid_for(ix, v.sequences), BLOCK_THREADS, 0, s>>>(v, shift, keys, pool, used_dev, cap);
    }
    rc = launch_done("k_build_locate");
    unsigned long long used = 0;
    if (rc == GBWT_B200_OK && cudaMemcpy(&used, used_dev, sizeof(used), cudaMemcpyDeviceToHost) != cudaSuccess)
        rc = cuda_fail(cudaGetLastError(), "k_build_locate");
    if (rc != GBWT_B200_OK) return give_up(rc);
    if (used > 0xFFFFFFFFull) return give_up(fail(GBWT_B200_E_RANGE, "more than 2^32 - 1 locate samples (raise GBWT_B200_LOCATE_SHIFT)"));
    // (only a damaged index, whose walks run to walk_limit, can emit more samples than the pool holds)
    if (used > cap) return give_up(fail(GBWT_B200_E_INVALID_DATA, "locate samples: the sequences are longer than the index"));
    if (cudaMalloc(reinterpret_cast<void**>(&table), std::max<size_t>(256, used * sizeof(LocateSample))) != cudaSuccess)
        return give_up(cuda_fail(cudaGetLastError(), "cudaMalloc(locate table)"));
    cudaError_t e = locate_sort_samples(keys, pool, used, v.records, table, first, ix->sm_count, s);
    g_launches.fetch_add(2, std::memory_order_relaxed);
    if (e == cudaSuccess) e = cudaEventRecord(e1, s);
    if (e == cudaSuccess) e = cudaEventSynchronize(e1);
    if (e != cudaSuccess) return give_up(cuda_fail(e, "locate sample sort"));
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    cleanup();
    ix->d_locate_first = first; ix->d_locate_samples = table;
    ix->locate_ok = true; ix->locate_shift = shift; ix->locate_samples = used;
    ix->locate_bytes = used * sizeof(LocateSample) + (v.records + 1) * sizeof(uint32_t);
    ix->locate_build_us = static_cast<uint64_t>(ms * 1000.0f);
    return GBWT_B200_OK;
}

int create_index(const ParsedGBWT& parsed, int device, int policy, gbwt_b200_index** out) {
    if (out == nullptr) return fail(GBWT_B200_E_ARGUMENT, "null output handle");
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(GBWT_B200_E_NO_DEVICE, "no CUDA device available (this library has no CPU fallback)");
    }
    if (device < 0 || device >= count) return fail(GBWT_B200_E_ARGUMENT, "invalid device ordinal");
    const int checkpoint_policy = policy & (GBWT_B200_LAYOUT_CHECKPOINTS | GBWT_B200_LAYOUT_NO_CHECKPOINTS);
    const bool want_locate = (policy & GBWT_B200_LAYOUT_LOCATE) != 0;
    policy &= ~(GBWT_B200_LAYOUT_CHECKPOINTS | GBWT_B200_LAYOUT_NO_CHECKPOINTS | GBWT_B200_LAYOUT_LOCATE);
    HostLayout layout;
    std::string err;
    int rc = build_layout(parsed, policy, layout, err);
    if (rc != GBWT_B200_OK) return fail(rc, err);

    DeviceScope scope(device);
    if (!scope.ok) return fail(GBWT_B200_E_CUDA, "cudaSetDevice failed");
    gbwt_b200_index* ix = new gbwt_b200_index();
    ix->device = device;
    cudaDeviceGetAttribute(&ix->sm_count, cudaDevAttrMultiProcessorCount, device);
    ix->sequences = parsed.sequences; ix->size = parsed.size; ix->offset = parsed.offset;
    ix->alphabet_size = parsed.alphabet_size; ix->flags = parsed.flags;
    std::memcpy(ix->format_counts, layout.format_counts, sizeof(layout.format_counts));
    ix->checkpointed_records = layout.checkpointed_records;
    ix->carried.tags = parsed.tags; ix->carried.gbz_tags = parsed.gbz_tags;
    ix->carried.da_samples = parsed.da_samples; ix->carried.metadata = parsed.metadata; ix->carried.graph_section = parsed.graph_section;
    rc = upload(&ix->d_desc, layout.desc.data(), layout.desc.size() * sizeof(RecordDesc), ix->bytes[0]);
    if (rc == GBWT_B200_OK) rc = upload(&ix->d_bodies, layout.bodies.data(), layout.bodies.size() * 8, ix->bytes[1]);
    if (rc == GBWT_B200_OK) rc = upload(&ix->d_edges, layout.edges.data(), layout.edges.size() * sizeof(Edge), ix->bytes[2]);
    if (rc == GBWT_B200_OK) rc = upload(&ix->d_endmarker, layout.endmarker.data(), layout.endmarker.size() * sizeof(Edge), ix->bytes[3]);
    if (rc == GBWT_B200_OK) rc = upload(&ix->d_skips, layout.skips.data(), layout.skips.size() * 8, ix->skip_bytes);
    if (rc == GBWT_B200_OK) {
        uint64_t stage_bytes = 0;
        rc = upload(&ix->d_stage_body, layout.stage_body.data(), layout.stage_body.size() * sizeof(uint32_t), stage_bytes);
        ix->skip_bytes += stage_bytes;
    }
    ix->edges_total = layout.edges_total; ix->edges_local = layout.edges_local;
    if (rc == GBWT_B200_OK) {
        // per sequence: its length, then (behind all lengths) the three words of its signature (kernels.cuh, SigAcc)
        const size_t bytes = std::max<size_t>(256, parsed.sequences * sizeof(uint64_t));
        if (cudaMalloc(&ix->d_seq_len, 4 * bytes) != cudaSuccess || cudaMemset(ix->d_seq_len, 0xFE, 4 * bytes) != cudaSuccess ||
            cudaMalloc(&ix->d_dna_len, bytes) != cudaSuccess || cudaMemset(ix->d_dna_len, 0xFE, bytes) != cudaSuccess) {
            rc = cuda_fail(cudaGetLastError(), "cudaMalloc(sequence lengths)");
        }
    }
    if (rc != GBWT_B200_OK) { gbwt_b200_index_destroy(ix); return rc; }
    // Records are fetched as isolated 32-byte sectors; ask L2 not to widen the DRAM fetches (a hint).
    {
        const char* e = std::getenv("GBWT_B200_L2_FETCH");
        size_t granularity = e ? static_cast<size_t>(std::atoi(e)) : 32;
        if (granularity > 0 && cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, granularity) != cudaSuccess) cudaGetLastError();
    }
    // Keep the stream-ordered pool's memory between calls: the host entry points allocate their staging
    // buffers from it on every call.
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        uint64_t threshold = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold);
    }
    IndexView& v = ix->view;
    v.desc = static_cast<const RecordDesc*>(ix->d_desc);
    v.bodies = static_cast<const Unit16*>(ix->d_bodies);
    v.edges = static_cast<const Edge*>(ix->d_edges);
    v.endmarker = static_cast<const Edge*>(ix->d_endmarker);
    v.records = layout.desc.size();
    v.offset = parsed.offset;
    v.alphabet_size = parsed.alphabet_size;
    v.sequences = parsed.sequences;
    v.endmarker_len = layout.endmarker.size();
    v.bidirectional = (parsed.flags & GBWT_FLAG_BIDIRECTIONAL) != 0;
    v.skips = static_cast<const Unit16*>(ix->d_skips);
    v.edges_valid = layout.edges_valid ? 1 : 0;
    v.walk_limit = layout.total_length;
    v.stage_body = static_cast<const uint32_t*>(ix->d_stage_body);
    // Record windows (find_window.cu) suit an index whose records are mostly single-edge or dense and whose edges
    // mostly lead to nearby records; everything else keeps the scattered-load kernels.
    {
        const uint64_t runs = layout.format_counts[FMT_RUN8] + layout.format_counts[FMT_RUN32] + layout.format_counts[FMT_RUN64];
        const bool mostly_plain = runs * 8 <= layout.format_counts[FMT_DENSE2] + layout.format_counts[FMT_SINGLE];
        const bool local = layout.edges_local * 10 >= layout.edges_total * 9;
        const double edge_span = layout.edges_local != 0 ? static_cast<double>(layout.edges_local_span) / static_cast<double>(layout.edges_local) : 3.0;
        const bool wide = layout.format_counts[FMT_DENSE4] + layout.format_counts[FMT_RUN8] != 0;
        ix->window_ok = plan_windows(v, layout.bodies.size() / 2, edge_span, wide, 32, ix->window);
        ix->window_suits = mostly_plain && local;
    }
    if (parsed.has_graph) {
        rc = attach_graph(ix, parsed.label_starts.data(), parsed.label_starts.size() - 1, parsed.label_bytes.data());
        if (rc != GBWT_B200_OK) { gbwt_b200_index_destroy(ix); return rc; }
        ix->carried.graph_section = parsed.graph_section;
    }
    // Path checkpoints by default for indexes whose sequences are long enough to be worth cutting up
    // (GBWT_B200_LAYOUT_CHECKPOINTS / _NO_CHECKPOINTS decide explicitly; GBWT_B200_CHECKPOINTS=0/1 overrides both).
    {
        bool want = layout.total_length >= (uint64_t(1) << 22);
        if (checkpoint_policy & GBWT_B200_LAYOUT_CHECKPOINTS) want = true;
        if (checkpoint_policy & GBWT_B200_LAYOUT_NO_CHECKPOINTS) want = false;
        const int knob = env_int("GBWT_B200_CHECKPOINTS", -1);
        if (knob >= 0) want = knob != 0;
        if (want) {
            rc = build_checkpoints(ix);
            if (rc != GBWT_B200_OK) { gbwt_b200_index_destroy(ix); return rc; }
            build_dna_checkpoints(ix);
        }
    }
    if (want_locate) {
        rc = build_locate(ix);
        if (rc != GBWT_B200_OK) { gbwt_b200_index_destroy(ix); return rc; }
    }
    *out = ix;
    return GBWT_B200_OK;
}

}  // namespace

// ---- construction ------------------------------------------------------------------------------------

extern "C" {

// No exception crosses the C ABI: the sizes declared in a damaged image can make an allocation fail.
#define GBWT_B200_GUARDED(...)                                                                         \
    try { __VA_ARGS__ } catch (const std::bad_alloc&) {                                                       \
        return fail(GBWT_B200_E_INVALID_DATA, "invalid data (an allocation of the declared size failed)"); \
    } catch (const std::exception& e) {                                                                \
        return fail(GBWT_B200_E_INVALID_DATA, std::string("invalid data (") + e.what() + ")");        \
    }

int gbwt_b200_index_from_bytes(const void* bytes, size_t len, int device, int layout_policy, gbwt_b200_index** out) {
    GBWT_B200_GUARDED(
        ParsedGBWT parsed;
        std::string err;
        int rc = parse_gbwt_image(static_cast<const uint8_t*>(bytes), len, parsed, err);
        if (rc != GBWT_B200_OK) return fail(rc, err);
        return create_index(parsed, device, layout_policy, out);
    )
}

int gbwt_b200_index_load_file(const char* path, int device, int layout_policy, gbwt_b200_index** out) {
    if (path == nullptr) return fail(GBWT_B200_E_ARGUMENT, "null path");
    std::ifstream f(path, std::ios::binary | std::ios::ate);
    if (!f) return fail(GBWT_B200_E_IO, std::string("cannot open ") + path);
    std::streamsize n = f.tellg();
    f.seekg(0);
    GBWT_B200_GUARDED(
        std::vector<uint8_t> buf(static_cast<size_t>(n));
        if (n > 0 && !f.read(reinterpret_cast<char*>(buf.data()), n)) return fail(GBWT_B200_E_IO, std::string("cannot read ") + path);
        return gbwt_b200_index_from_bytes(buf.data(), buf.size(), device, layout_policy, out);
    )
}

int gbwt_b200_index_from_parts(uint64_t sequences, uint64_t size, uint64_t offset, uint64_t alphabet_size, uint64_t flags,
                               const uint8_t* bwt_bytes, uint64_t bwt_len, const uint64_t* record_starts, uint64_t records,
                               int device, int layout_policy, gbwt_b200_index** out) {
    if ((bwt_len > 0 && bwt_bytes == nullptr) || (records > 0 && record_starts == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null input");
    GBWT_B200_GUARDED(
        ParsedGBWT parsed;
        parsed.sequences = sequences; parsed.size = size; parsed.offset = offset; parsed.alphabet_size = alphabet_size;
        parsed.flags = flags | GBWT_FLAG_SIMPLE_SDS;
        parsed.bwt = bwt_bytes; parsed.bwt_len = bwt_len;
        parsed.record_starts.assign(record_starts, record_starts + records);
        for (uint64_t i = 0; i < records; i++) {
            if (record_starts[i] >= bwt_len || (i > 0 && record_starts[i] <= record_starts[i - 1]))
                return fail(GBWT_B200_E_INVALID_DATA, "BWT: invalid index");
        }
        return create_index(parsed, device, layout_policy, out);
    )
}

// The layout comes back from HBM as it is; the encoder runs on the host. `gbz`: a GBZ image (needs node labels).
static int serialize_index(const gbwt_b200_index* ix, bool gbz, void** image, size_t* len) {
    if (int rc = check_index(ix)) return rc;
    if (image == nullptr || len == nullptr) return fail(GBWT_B200_E_ARGUMENT, "null output");
    *image = nullptr; *len = 0;
    if (gbz) { if (int rc = check_graph(ix)) return rc; }
    DeviceScope scope(ix->device);
    if (!scope.ok) return fail(GBWT_B200_E_CUDA, "cudaSetDevice failed");
    GBWT_B200_GUARDED(
        std::vector<RecordDesc> desc(ix->view.records);
        std::vector<uint64_t> bodies(ix->bytes[1] / 8 + 2, 0);
        std::vector<Edge> edges(ix->bytes[2] / sizeof(Edge) + 1, Edge{0, 0});
        if (!desc.empty()) CUDA_TRY(cudaMemcpy(desc.data(), ix->d_desc, desc.size() * sizeof(RecordDesc), cudaMemcpyDeviceToHost));
        if (ix->bytes[1] > 0) CUDA_TRY(cudaMemcpy(bodies.data(), ix->d_bodies, ix->bytes[1], cudaMemcpyDeviceToHost));
        if (ix->bytes[2] > 0) CUDA_TRY(cudaMemcpy(edges.data(), ix->d_edges, ix->bytes[2], cudaMemcpyDeviceToHost));
        LayoutArrays in;
        in.desc = desc.data(); in.records = desc.size(); in.bodies = bodies.data(); in.edges = edges.data();
        GBWTHeaderFields header;
        header.sequences = ix->sequences; header.size = ix->size; header.offset = ix->offset;
        header.alphabet_size = ix->alphabet_size; header.flags = ix->flags;
        std::vector<uint8_t> bytes;
        std::string err;
        int rc;
        if (!gbz) {
            rc = write_gbwt_image(header, in, ix->carried, bytes, err);
        } else {
            // labels attached by hand have no Graph section to pass through: they come back from HBM and are written as one
            std::vector<uint64_t> starts;
            std::vector<uint8_t> labels;
            if (ix->carried.graph_section.empty()) {
                starts.assign(ix->graph.sequences + 1, 0);
                CUDA_TRY(cudaMemcpy(starts.data(), ix->d_label_starts, starts.size() * 8, cudaMemcpyDeviceToHost));
                labels.assign(starts.back(), 0);
                if (!labels.empty()) CUDA_TRY(cudaMemcpy(labels.data(), ix->d_label_bytes, labels.size(), cudaMemcpyDeviceToHost));
            }
            rc = write_gbz_image(header, in, ix->carried, starts.empty() ? nullptr : starts.data(), ix->graph.sequences,
                                 labels.data(), bytes, err);
        }
        if (rc != GBWT_B200_OK) return fail(rc, err);
        void* out = std::malloc(std::max<size_t>(bytes.size(), 1));
        if (out == nullptr) return fail(GBWT_B200_E_IO, "out of memory");
        std::memcpy(out, bytes.data(), bytes.size());
        *image = out; *len = bytes.size();
        return GBWT_B200_OK;
    )
}

static int save_index(const gbwt_b200_index* ix, bool gbz, const char* path) {
    if (path == nullptr) return fail(GBWT_B200_E_ARGUMENT, "null path");
    void* image = nullptr;
    size_t len = 0;
    if (int rc = serialize_index(ix, gbz, &image, &len)) return rc;
    std::ofstream f(path, std::ios::binary | std::ios::trunc);
    bool ok = static_cast<bool>(f);
    if (ok) { f.write(static_cast<const char*>(image), static_cast<std::streamsize>(len)); ok = static_cast<bool>(f); }
    std::free(image);
    return ok ? GBWT_B200_OK : fail(GBWT_B200_E_IO, std::string("cannot write ") + path);
}

// ---- build once, replicate over NVLink -----------------------------------------------------------------------------
// The index of a multi-GPU job is the same on every GPU. Instead of every rank parsing the image and running K0 and the
// checkpoint walk, one rank builds it and exports a small blob: the scalars of the handle, what the loader carried, and
// a CUDA IPC handle per device array. The other ranks (one process per GPU) open the handles and copy the arrays
// device to device -- peer copies over NVLink / NVSwitch -- into allocations of their own.

namespace {

constexpr uint64_t IPC_MAGIC = 0x4350493030324247ull;  // "GB200IPC"
constexpr int IPC_ARRAYS = 14;

struct IpcArray { uint64_t bytes; cudaIpcMemHandle_t handle; };

struct IpcHeader {
    uint64_t magic, version;
    uint64_t sequences, size, offset, alphabet_size, flags;
    uint64_t records, endmarker_len, bidirectional, edges_valid, walk_limit;
    uint64_t bytes[4], skip_bytes, format_counts[FMT_COUNT], checkpointed_records, edges_total, edges_local;
    uint64_t window_ok, window_suits;
    WindowPlan window;
    uint64_t ckpt_ok, ckpt_shift, ckpt_entries, ckpt_bytes, ckpt_build_us, ckpt_max_segments;
    uint64_t has_graph, graph_sequences, graph_bytes;
    uint64_t locate_ok, locate_shift, locate_samples, locate_bytes, locate_build_us;
    uint64_t source_device;
    IpcArray arrays[IPC_ARRAYS];
};

void put_u64(std::vector<uint8_t>& out, uint64_t v) { const uint8_t* p = reinterpret_cast<const uint8_t*>(&v); out.insert(out.end(), p, p + 8); }
void put_blob(std::vector<uint8_t>& out, const void* p, size_t n) {
    put_u64(out, n);
    const uint8_t* b = static_cast<const uint8_t*>(p);
    out.insert(out.end(), b, b + n);
}
void put_tags_blob(std::vector<uint8_t>& out, const std::vector<std::pair<std::string, std::string>>& tags) {
    put_u64(out, tags.size());
    for (const auto& kv : tags) { put_blob(out, kv.first.data(), kv.first.size()); put_blob(out, kv.second.data(), kv.second.size()); }
}

struct BlobReader {
    const uint8_t* p;
    size_t n, at = 0;
    bool ok = true;
    uint64_t u64() {
        if (!ok || n - at < 8) { ok = false; return 0; }
        uint64_t v;
        std::memcpy(&v, p + at, 8);
        at += 8;
        return v;
    }
    std::string str() {
        const uint64_t len = u64();
        if (!ok || len > n - at) { ok = false; return std::string(); }
        std::string s(reinterpret_cast<const char*>(p + at), len);
        at += len;
        return s;
    }
    std::vector<uint8_t> bytes() { const std::string s = str(); return std::vector<uint8_t>(s.begin(), s.end()); }
    void tags(std::vector<std::pair<std::string, std::string>>& out) {
        const uint64_t count = u64();
        out.clear();
        for (uint64_t i = 0; i < count && ok; i++) { std::string k = str(); std::string v = str(); out.emplace_back(k, v); }
    }
};

// The device arrays of a handle in export order, with their sizes in bytes.
void ipc_arrays(const gbwt_b200_index* ix, void* ptrs[IPC_ARRAYS], uint64_t sizes[IPC_ARRAYS]) {
    const uint64_t seq_bytes = std::max<uint64_t>(256, ix->sequences * sizeof(uint64_t));
    void* p[IPC_ARRAYS] = {ix->d_desc, ix->d_bodies, ix->d_edges, ix->d_endmarker, ix->d_skips, ix->d_stage_body, ix->d_seq_len,
                           ix->d_dna_len, ix->d_ckpt_table, ix->d_ckpt_first, ix->d_label_starts, ix->d_label_bytes,
                           ix->d_locate_first, ix->d_locate_samples};
    const uint64_t b[IPC_ARRAYS] = {ix->bytes[0], ix->bytes[1], ix->bytes[2], ix->bytes[3],
                                    (ix->view.records + 1) * 16, (ix->view.records / STAGE_GRANULE + 2) * sizeof(uint32_t), 4 * seq_bytes, seq_bytes,
                                    ix->ckpt_ok ? ix->ckpt_entries * sizeof(Checkpoint) : 0,
                                    ix->ckpt_ok ? (ix->view.sequences + 1) * sizeof(uint32_t) : 0,
                                    ix->has_graph ? (ix->graph.sequences + 1) * 8 : 0,
                                    ix->has_graph ? ix->graph_bytes - (ix->graph.sequences + 1) * 8 : 0,
                                    ix->locate_ok ? (ix->view.records + 1) * sizeof(uint32_t) : 0,
                                    ix->locate_ok ? ix->locate_samples * sizeof(LocateSample) : 0};
    for (int i = 0; i < IPC_ARRAYS; i++) { ptrs[i] = p[i]; sizes[i] = p[i] != nullptr ? b[i] : 0; }
}

}  // namespace

int gbwt_b200_index_export_ipc(const gbwt_b200_index* ix, void** blob, size_t* len) {
    if (int rc = check_index(ix)) return rc;
    if (blob == nullptr || len == nullptr) return fail(GBWT_B200_E_ARGUMENT, "null output");
    *blob = nullptr; *len = 0;
    DeviceScope scope(ix->device);
    if (!scope.ok) return fail(GBWT_B200_E_CUDA, "cudaSetDevice failed");
    CUDA_TRY(cudaDeviceSynchronize());  // everything the build enqueued has landed
    IpcHeader h;
    std::memset(&h, 0, sizeof(h));
    h.magic = IPC_MAGIC; h.version = 2;
    h.sequences = ix->sequences; h.size = ix->size; h.offset = ix->offset; h.alphabet_size = ix->alphabet_size; h.flags = ix->flags;
    h.records = ix->view.records; h.endmarker_len = ix->view.endmarker_len; h.bidirectional = ix->view.bidirectional;
    h.edges_valid = ix->view.edges_valid; h.walk_limit = ix->view.walk_limit;
    for (int i = 0; i < 4; i++) h.bytes[i] = ix->bytes[i];
    h.skip_bytes = ix->skip_bytes;
    for (int i = 0; i < FMT_COUNT; i++) h.format_counts[i] = ix->format_counts[i];
    h.checkpointed_records = ix->checkpointed_records;
    h.edges_total = ix->edges_total; h.edges_local = ix->edges_local;
    h.window_ok = ix->window_ok; h.window_suits = ix->window_suits; h.window = ix->window;
    h.ckpt_ok = ix->ckpt_ok; h.ckpt_shift = ix->ckpt_shift; h.ckpt_entries = ix->ckpt_entries; h.ckpt_bytes = ix->ckpt_bytes;
    h.ckpt_build_us = ix->ckpt_build_us; h.ckpt_max_segments = ix->ckpt.max_segments;
    h.has_graph = ix->has_graph; h.graph_sequences = ix->graph.sequences; h.graph_bytes = ix->graph_bytes;
    h.locate_ok = ix->locate_ok; h.locate_shift = ix->locate_shift; h.locate_samples = ix->locate_samples;
    h.locate_bytes = ix->locate_bytes; h.locate_build_us = ix->locate_build_us;
    h.source_device = static_cast<uint64_t>(ix->device);
    void* ptrs[IPC_ARRAYS];
    uint64_t sizes[IPC_ARRAYS];
    ipc_arrays(ix, ptrs, sizes);
    for (int i = 0; i < IPC_ARRAYS; i++) {
        h.arrays[i].bytes = sizes[i];
        if (sizes[i] > 0) CUDA_TRY(cudaIpcGetMemHandle(&h.arrays[i].handle, ptrs[i]));
    }
    GBWT_B200_GUARDED(
        std::vector<uint8_t> out(reinterpret_cast<const uint8_t*>(&h), reinterpret_cast<const uint8_t*>(&h) + sizeof(h));
        put_tags_blob(out, ix->carried.tags); put_tags_blob(out, ix->carried.gbz_tags);
        put_blob(out, ix->carried.da_samples.data(), ix->carried.da_samples.size());
        put_blob(out, ix->carried.metadata.data(), ix->carried.metadata.size());
        put_blob(out, ix->carried.graph_section.data(), ix->carried.graph_section.size());
        void* mem = std::malloc(out.size());
        if (mem == nullptr) return fail(GBWT_B200_E_IO, "out of memory");
        std::memcpy(mem, out.data(), out.size());
        *blob = mem; *len = out.size();
        return GBWT_B200_OK;
    )
}

int gbwt_b200_index_import_ipc(const void* blob, size_t len, int device, gbwt_b200_index** out) {
    if (out == nullptr || blob == nullptr) return fail(GBWT_B200_E_ARGUMENT, "null argument");
    *out = nullptr;
    if (len < sizeof(IpcHeader)) return fail(GBWT_B200_E_INVALID_DATA, "not an exported index");
    IpcHeader h;
    std::memcpy(&h, blob, sizeof(h));
    if (h.magic != IPC_MAGIC || h.version != 2) return fail(GBWT_B200_E_INVALID_DATA, "not an exported index");
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(GBWT_B200_E_NO_DEVICE, "no CUDA device available (this library has no CPU fallback)");
    }
    if (device < 0 || device >= count) return fail(GBWT_B200_E_ARGUMENT, "invalid device ordinal");
    DeviceScope scope(device);
    if (!scope.ok) return fail(GBWT_B200_E_CUDA, "cudaSetDevice failed");
    GBWT_B200_GUARDED(
        gbwt_b200_index* ix = new gbwt_b200_index();
        ix->device = device;
        cudaDeviceGetAttribute(&ix->sm_count, cudaDevAttrMultiProcessorCount, device);
        ix->sequences = h.sequences; ix->size = h.size; ix->offset = h.offset; ix->alphabet_size = h.alphabet_size; ix->flags = h.flags;
        for (int i = 0; i < 4; i++) ix->bytes[i] = h.bytes[i];
        ix->skip_bytes = h.skip_bytes;
        for (int i = 0; i < FMT_COUNT; i++) ix->format_counts[i] = h.format_counts[i];
        ix->checkpointed_records = h.checkpointed_records;
        ix->edges_total = h.edges_total; ix->edges_local = h.edges_local;
        ix->window_ok = h.window_ok != 0; ix->window_suits = h.window_suits != 0; ix->window = h.window;
        BlobReader rd{static_cast<const uint8_t*>(blob), len, sizeof(IpcHeader)};
        rd.tags(ix->carried.tags); rd.tags(ix->carried.gbz_tags);
        ix->carried.da_samples = rd.bytes(); ix->carried.metadata = rd.bytes(); ix->carried.graph_section = rd.bytes();
        if (!rd.ok) { delete ix; return fail(GBWT_B200_E_INVALID_DATA, "truncated exported index"); }
        // the arrays: open the exporter's allocation, copy it device to device, close it
        void** slots[IPC_ARRAYS] = {&ix->d_desc, &ix->d_bodies, &ix->d_edges, &ix->d_endmarker, &ix->d_skips, &ix->d_stage_body, &ix->d_seq_len,
                                    &ix->d_dna_len, &ix->d_ckpt_table, &ix->d_ckpt_first, &ix->d_label_starts, &ix->d_label_bytes,
                                    &ix->d_locate_first, &ix->d_locate_samples};
        int rc = GBWT_B200_OK;
        for (int i = 0; i < IPC_ARRAYS && rc == GBWT_B200_OK; i++) {
            if (h.arrays[i].bytes == 0) continue;
            void* remote = nullptr;
            cudaError_t e = cudaIpcOpenMemHandle(&remote, h.arrays[i].handle, cudaIpcMemLazyEnablePeerAccess);
            if (e != cudaSuccess) { rc = cuda_fail(e, "cudaIpcOpenMemHandle"); break; }
            e = cudaMalloc(slots[i], std::max<size_t>(h.arrays[i].bytes, 256));
            if (e == cudaSuccess) e = cudaMemcpy(*slots[i], remote, h.arrays[i].bytes, cudaMemcpyDefault);
            cudaIpcCloseMemHandle(remote);
            if (e != cudaSuccess) rc = cuda_fail(e, "copy of an exported array");
        }
        if (rc != GBWT_B200_OK) { gbwt_b200_index_destroy(ix); return rc; }
        // buffers that an exporter may lack (no checkpoints, no graph) but every handle owns
        const size_t seq_bytes = std::max<size_t>(256, h.sequences * sizeof(uint64_t));
        if (ix->d_seq_len == nullptr && (cudaMalloc(&ix->d_seq_len, 4 * seq_bytes) != cudaSuccess || cudaMemset(ix->d_seq_len, 0xFE, 4 * seq_bytes) != cudaSuccess))
            rc = cuda_fail(cudaGetLastError(), "cudaMalloc(sequence lengths)");
        if (rc == GBWT_B200_OK && ix->d_dna_len == nullptr &&
            (cudaMalloc(&ix->d_dna_len, seq_bytes) != cudaSuccess || cudaMemset(ix->d_dna_len, 0xFE, seq_bytes) != cudaSuccess))
            rc = cuda_fail(cudaGetLastError(), "cudaMalloc(sequence lengths)");
        if (rc != GBWT_B200_OK) { gbwt_b200_index_destroy(ix); return rc; }
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            uint64_t threshold = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold);
        }
        IndexView& v = ix->view;
        v.desc = static_cast<const RecordDesc*>(ix->d_desc);
        v.bodies = static_cast<const Unit16*>(ix->d_bodies);
        v.edges = static_cast<const Edge*>(ix->d_edges);
        v.endmarker = static_cast<const Edge*>(ix->d_endmarker);
        v.records = h.records; v.offset = h.offset; v.alphabet_size = h.alphabet_size; v.sequences = h.sequences;
        v.endmarker_len = h.endmarker_len; v.bidirectional = static_cast<uint32_t>(h.bidirectional);
        v.skips = static_cast<const Unit16*>(ix->d_skips);
        v.edges_valid = static_cast<uint32_t>(h.edges_valid);
        v.walk_limit = h.walk_limit;
        v.stage_body = static_cast<const uint32_t*>(ix->d_stage_body);
        if (h.ckpt_ok) {
            ix->ckpt.table = static_cast<const Checkpoint*>(ix->d_ckpt_table);
            ix->ckpt.first = static_cast<const uint32_t*>(ix->d_ckpt_first);
            ix->ckpt.seq_len = static_cast<const uint64_t*>(ix->d_seq_len);
            ix->ckpt.max_segments = static_cast<uint32_t>(h.ckpt_max_segments);
            ix->ckpt_shift = static_cast<uint32_t>(h.ckpt_shift); ix->ckpt_entries = h.ckpt_entries; ix->ckpt_bytes = h.ckpt_bytes;
            ix->ckpt_build_us = h.ckpt_build_us;
            ix->ckpt_ok = true;
        }
        if (h.has_graph) {
            ix->graph.starts = static_cast<const uint64_t*>(ix->d_label_starts);
            ix->graph.bytes = static_cast<const uint8_t*>(ix->d_label_bytes);
            ix->graph.sequences = h.graph_sequences;
            ix->graph_bytes = h.graph_bytes;
            ix->has_graph = true;
        }
        if (h.locate_ok) {
            // (an index without samples has a zero-sized sample array: the table comes over only with its `first`)
            ix->locate_ok = ix->d_locate_first != nullptr;
            if (ix->locate_ok && ix->d_locate_samples == nullptr && cudaMalloc(&ix->d_locate_samples, 256) != cudaSuccess) {
                gbwt_b200_index_destroy(ix);
                return cuda_fail(cudaGetLastError(), "cudaMalloc(locate table)");
            }
            ix->locate_shift = static_cast<uint32_t>(h.locate_shift); ix->locate_samples = h.locate_samples;
            ix->locate_bytes = h.locate_bytes; ix->locate_build_us = h.locate_build_us;
        }
        build_dna_checkpoints(ix);  // (a table of the importer's own: a short count pass, not worth a handle in the blob)
        *out = ix;
        return GBWT_B200_OK;
    )
}

int gbwt_b200_index_serialize(const gbwt_b200_index* ix, void** image, size_t* len) { return serialize_index(ix, false, image, len); }
int gbwt_b200_index_serialize_gbz(const gbwt_b200_index* ix, void** image, size_t* len) { return serialize_index(ix, true, image, len); }
int gbwt_b200_index_save_gbz_file(const gbwt_b200_index* ix, const char* path) { return save_index(ix, true, path); }

int gbwt_b200_index_save_file(const gbwt_b200_index* ix, const char* path) { return save_index(ix, false, path); }

void gbwt_b200_free(void* p) { std::free(p); }

void gbwt_b200_index_destroy(gbwt_b200_index* ix) {
    if (ix == nullptr) return;
    {
        DeviceScope scope(ix->device);
        cudaFree(ix->d_desc); cudaFree(ix->d_bodies); cudaFree(ix->d_edges); cudaFree(ix->d_endmarker); cudaFree(ix->d_skips); cudaFree(ix->d_stage_body); cudaFree(ix->d_ckpt_table); cudaFree(ix->d_ckpt_first); cudaFree(ix->d_seq_len); cudaFree(ix->d_dna_len); cudaFree(ix->d_ckpt_dna);
        cudaFree(ix->d_label_starts); cudaFree(ix->d_label_bytes); cudaFree(ix->d_locate_first); cudaFree(ix->d_locate_samples);
    }
    delete ix;
}

int gbwt_b200_index_attach_graph(gbwt_b200_index* ix, uint64_t sequences, const uint64_t* label_starts, const uint8_t* label_bytes) {
    if (int rc = check_index(ix)) return rc;
    if (label_starts == nullptr || (label_starts[sequences] > 0 && label_bytes == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null input");
    if (label_starts[0] != 0) return fail(GBWT_B200_E_INVALID_DATA, "StringArray: First string does not start at offset 0");
    if (!offsets_valid(label_starts, sequences)) return fail(GBWT_B200_E_INVALID_DATA, "StringArray: invalid index");
    // GBZ::load, src/gbz.rs:686-694
    if (!(ix->flags & GBWT_FLAG_BIDIRECTIONAL)) return fail(GBWT_B200_E_INVALID_DATA, "GBZ: The GBWT index is not bidirectional");
    if (sequences != (ix->alphabet_size - (ix->offset + 1)) / 2)
        return fail(GBWT_B200_E_INVALID_DATA, "GBZ: Mismatch between GBWT alphabet size and Graph sequence count");
    return attach_graph(ix, label_starts, sequences, label_bytes);
}

int gbwt_b200_has_graph(const gbwt_b200_index* ix) { return ix && ix->has_graph; }
uint64_t gbwt_b200_graph_sequences(const gbwt_b200_index* ix) { return ix && ix->has_graph ? ix->graph.sequences : 0; }
uint64_t gbwt_b200_graph_bytes(const gbwt_b200_index* ix) { return ix ? ix->graph_bytes : 0; }
uint64_t gbwt_b200_skip_bytes(const gbwt_b200_index* ix) { return ix ? ix->skip_bytes : 0; }
uint64_t gbwt_b200_run_checkpoint_records(const gbwt_b200_index* ix) { return ix ? ix->checkpointed_records : 0; }
uint64_t gbwt_b200_dense4_records(const gbwt_b200_index* ix) { return ix ? ix->format_counts[FMT_DENSE4] : 0; }

void gbwt_b200_checkpoint_info(const gbwt_b200_index* ix, uint64_t info[6]) {
    if (ix == nullptr || info == nullptr) return;
    const uint64_t values[6] = {ix->ckpt_ok, uint64_t(1) << ix->ckpt_shift, ix->ckpt_entries, ix->ckpt_bytes, ix->ckpt_build_us, ix->ckpt.max_segments};
    for (int i = 0; i < 6; i++) info[i] = values[i];
}

void gbwt_b200_locate_info(const gbwt_b200_index* ix, uint64_t info[6]) {
    if (ix == nullptr || info == nullptr) return;
    const uint64_t values[6] = {ix->locate_ok, ix->locate_ok ? uint64_t(1) << ix->locate_shift : 0, ix->locate_samples, ix->locate_bytes,
                                ix->locate_build_us, ix->locate_steps.load()};
    for (int i = 0; i < 6; i++) info[i] = values[i];
}

void gbwt_b200_window_info(const gbwt_b200_index* ix, uint64_t info[14]) {
    if (ix == nullptr || info == nullptr) return;
    const WindowPlan& w = ix->window;
    const uint64_t values[14] = {ix->window_ok, ix->window_suits, uint64_t(1) << w.wshift, w.margin, w.body_cap, w.threads, w.smem_bytes,
                                 w.windows, ix->edges_total, ix->edges_local, ix->window_queries.load(), ix->window_deferred.load(),
                                 ix->window_kernel_ns.load(), ix->window_launches.load()};
    for (int i = 0; i < 14; i++) info[i] = values[i];
}

const char* gbwt_b200_last_error(void) { return g_last_error.c_str(); }

// ---- statistics (src/gbwt.rs:105-175) ----------------------------------------------------------------

uint64_t gbwt_b200_len(const gbwt_b200_index* ix) { return ix ? ix->size : 0; }
uint64_t gbwt_b200_sequences(const gbwt_b200_index* ix) { return ix ? ix->sequences : 0; }
uint64_t gbwt_b200_alphabet_size(const gbwt_b200_index* ix) { return ix ? ix->alphabet_size : 0; }
uint64_t gbwt_b200_alphabet_offset(const gbwt_b200_index* ix) { return ix ? ix->offset : 0; }
uint64_t gbwt_b200_effective_size(const gbwt_b200_index* ix) { return ix ? ix->alphabet_size - ix->offset : 0; }
uint64_t gbwt_b200_first_node(const gbwt_b200_index* ix) { return ix ? ix->offset + 1 : 0; }
int gbwt_b200_has_node(const gbwt_b200_index* ix, uint64_t id) { return ix && id > ix->offset && id < ix->alphabet_size; }
int gbwt_b200_is_bidirectional(const gbwt_b200_index* ix) { return ix && (ix->flags & GBWT_FLAG_BIDIRECTIONAL) != 0; }
int gbwt_b200_device(const gbwt_b200_index* ix) { return ix ? ix->device : -1; }

uint64_t gbwt_b200_device_bytes(const gbwt_b200_index* ix, uint64_t breakdown[10]) {
    if (ix == nullptr) return 0;
    if (breakdown != nullptr) {
        for (int i = 0; i < 4; i++) breakdown[i] = ix->bytes[i];
        for (int i = 0; i < 6; i++) breakdown[4 + i] = ix->format_counts[i];
        breakdown[4 + FMT_DENSE2] += ix->format_counts[FMT_DENSE4];  // both dense formats in one slot (gbwt_b200_dense4_records tells them apart)
    }
    return ix->bytes[0] + ix->bytes[1] + ix->bytes[2] + ix->bytes[3] + ix->skip_bytes + ix->graph_bytes + ix->ckpt_bytes +
           (ix->locate_ok ? ix->locate_bytes : 0);
}

// ---- device-pointer entry points ---------------------------------------------------------------------

#define DEVICE_ENTRY_PROLOGUE(ix)                                              \
    if (int _rc = check_index(ix)) return _rc;                                 \
    DeviceScope _scope((ix)->device);                                          \
    if (!_scope.ok) return fail(GBWT_B200_E_CUDA, "cudaSetDevice failed");

int gbwt_b200_find_device(const gbwt_b200_index* ix, const uint64_t* d_nodes, size_t n, gbwt_b200_state* d_out, void* stream) {
    DEVICE_ENTRY_PROLOGUE(ix);
    return launch_find(ix, d_nodes, n, d_out, static_cast<cudaStream_t>(stream));
}
int gbwt_b200_extend_device(const gbwt_b200_index* ix, const gbwt_b200_state* d_states, const uint64_t* d_nodes, size_t n,
                            gbwt_b200_state* d_out, void* stream) {
    DEVICE_ENTRY_PROLOGUE(ix);
    return launch_extend(ix, d_states, d_nodes, n, d_out, static_cast<cudaStream_t>(stream));
}
int gbwt_b200_find_extend_device(const gbwt_b200_index* ix, const uint64_t* d_patterns, size_t n, size_t k,
                                 gbwt_b200_state* d_out, void* stream) {
    DEVICE_ENTRY_PROLOGUE(ix);
    return launch_find_extend(ix, d_patterns, n, k, d_out, static_cast<cudaStream_t>(stream));
}
int gbwt_b200_find_extend_u32_device(const gbwt_b200_index* ix, const uint32_t* d_patterns, size_t n, size_t k,
                                     gbwt_b200_state* d_out, void* stream) {
    DEVICE_ENTRY_PROLOGUE(ix);
    return launch_find_extend(ix, d_patterns, n, k, d_out, static_cast<cudaStream_t>(stream));
}
int gbwt_b200_find_extend_ragged_device(const gbwt_b200_index* ix, const uint64_t* d_nodes, const uint64_t* d_offsets, size_t n,
                                        gbwt_b200_state* d_out, void* stream) {
    DEVICE_ENTRY_PROLOGUE(ix);
    return launch_find_extend_ragged(ix, d_nodes, d_offsets, 0, n, d_out, static_cast<cudaStream_t>(stream));
}
int gbwt_b200_bd_find_device(const gbwt_b200_index* ix, const uint64_t* d_nodes, size_t n, gbwt_b200_bdstate* d_out, void* stream) {
    DEVICE_ENTRY_PROLOGUE(ix);
    if (int rc = check_bidirectional(ix)) return rc;
    return launch_bd_find(ix, d_nodes, n, d_out, static_cast<cudaStream_t>(stream));
}
int gbwt_b200_bd_extend_device(const gbwt_b200_index* ix, const gbwt_b200_bdstate* d_states, const uint64_t* d_nodes, size_t n,
                               int backward, gbwt_b200_bdstate* d_out, void* stream) {
    DEVICE_ENTRY_PROLOGUE(ix);
    if (int rc = check_bidirectional(ix)) return rc;
    return launch_bd_extend(ix, d_states, d_nodes, n, backward, d_out, static_cast<cudaStream_t>(stream));
}
int gbwt_b200_bd_search_device(const gbwt_b200_index* ix, const uint64_t* d_nodes, const uint64_t* d_offsets,
                               const uint64_t* d_first, const uint64_t* d_start, const uint64_t* d_end, size_t n,
                               gbwt_b200_bdstate* d_out, void* stream) {
    DEVICE_ENTRY_PROLOGUE(ix);
    if (int rc = check_bidirectional(ix)) return rc;
    return launch_bd_search(ix, d_nodes, d_offsets, 0, d_first, d_start, d_end, n, d_out, static_cast<cudaStream_t>(stream));
}
int gbwt_b200_follow_device(const gbwt_b200_index* ix, const gbwt_b200_bdstate* d_states, size_t n, int backward,
                            const uint64_t* d_out_offsets, gbwt_b200_bdstate* d_out, uint64_t* d_counts, void* stream) {
    DEVICE_ENTRY_PROLOGUE(ix);
    if (int rc = check_bidirectional(ix)) return rc;
    if (d_out != nullptr && d_out_offsets == nullptr) return fail(GBWT_B200_E_ARGUMENT, "null out_offsets");
    return launch_follow(ix, d_states, n, backward, d_out_offsets, 0, d_out, d_counts, static_cast<cudaStream_t>(stream));
}
int gbwt_b200_forward_device(const gbwt_b200_index* ix, const gbwt_b200_pos* d_positions, size_t n, gbwt_b200_pos* d_out, void* stream) {
    DEVICE_ENTRY_PROLOGUE(ix);
    return launch_forward(ix, d_positions, n, d_out, static_cast<cudaStream_t>(stream));
}
int gbwt_b200_sequence_lengths_device(const gbwt_b200_index* ix, const uint64_t* d_seq_ids, size_t m, uint64_t* d_lengths, void* stream) {
    DEVICE_ENTRY_PROLOGUE(ix);
    return launch_extract(ix, d_seq_ids, m, nullptr, 0, nullptr, d_lengths, static_cast<cudaStream_t>(stream));
}
int gbwt_b200_extract_device(const gbwt_b200_index* ix, const uint64_t* d_seq_ids, size_t m, const uint64_t* d_out_offsets,
                             uint64_t* d_nodes, uint64_t* d_lengths, void* stream) {
    DEVICE_ENTRY_PROLOGUE(ix);
    if (m > 0 && (d_nodes == nullptr || d_out_offsets == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null output");
    return launch_extract(ix, d_seq_ids, m, d_out_offsets, 0, d_nodes, d_lengths, static_cast<cudaStream_t>(stream));
}

int gbwt_b200_locate_device(const gbwt_b200_index* ix, const gbwt_b200_pos* d_positions, size_t n, gbwt_b200_occurrence* d_out, void* stream) {
    DEVICE_ENTRY_PROLOGUE(ix);
    if (int rc = check_samples(ix)) return rc;
    if (n > 0 && (d_positions == nullptr || d_out == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null array");
    return launch_locate_positions(ix, d_positions, n, d_out, static_cast<cudaStream_t>(stream));
}
int gbwt_b200_locate_states_device(const gbwt_b200_index* ix, const gbwt_b200_state* d_states, size_t n, const uint64_t* d_out_offsets,
                                   gbwt_b200_occurrence* d_out, uint64_t* d_counts, void* stream) {
    DEVICE_ENTRY_PROLOGUE(ix);
    if (int rc = check_samples(ix)) return rc;
    if (n > 0 && (d_states == nullptr || (d_out != nullptr && d_out_offsets == nullptr) || (d_out == nullptr && d_counts == nullptr)))
        return fail(GBWT_B200_E_ARGUMENT, "null array");
    // (the scan of a chunk is indexed with 64-bit CUB offsets; chunks keep each launch's temporary arrays bounded)
    const size_t chunk = size_t(1) << 30;
    for (size_t begin = 0; begin < n; begin += chunk) {
        const size_t count = std::min(chunk, n - begin);
        int rc = launch_locate_state_batch(ix, d_states + begin, count, d_out_offsets != nullptr ? d_out_offsets + begin : nullptr, 0, d_out,
                                           d_counts != nullptr ? d_counts + begin : nullptr, static_cast<cudaStream_t>(stream));
        if (rc != GBWT_B200_OK) return rc;
    }
    return GBWT_B200_OK;
}

int gbwt_b200_seek_device(const gbwt_b200_index* ix, const uint64_t* d_seq_ids, const uint64_t* d_indexes, size_t n, gbwt_b200_pos* d_out,
                          void* stream) {
    DEVICE_ENTRY_PROLOGUE(ix);
    if (n > 0 && (d_seq_ids == nullptr || d_indexes == nullptr || d_out == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null array");
    return launch_seek_batch(ix, d_seq_ids, d_indexes, n, d_out, static_cast<cudaStream_t>(stream));
}
int gbwt_b200_extract_ranges_device(const gbwt_b200_index* ix, const uint64_t* d_seq_ids, const uint64_t* d_starts, const uint64_t* d_ends,
                                    size_t m, const uint64_t* d_out_offsets, uint64_t* d_nodes, uint64_t* d_lengths, void* stream) {
    DEVICE_ENTRY_PROLOGUE(ix);
    return ranges_device(ix, false, d_seq_ids, d_starts, d_ends, m, d_out_offsets, d_nodes, d_lengths, static_cast<cudaStream_t>(stream));
}
int gbwt_b200_extract_dna_ranges_device(const gbwt_b200_index* ix, const uint64_t* d_seq_ids, const uint64_t* d_starts, const uint64_t* d_ends,
                                        size_t m, const uint64_t* d_out_offsets, uint8_t* d_bytes, uint64_t* d_lengths, void* stream) {
    DEVICE_ENTRY_PROLOGUE(ix);
    if (int rc = check_graph(ix)) return rc;
    return ranges_device(ix, true, d_seq_ids, d_starts, d_ends, m, d_out_offsets, d_bytes, d_lengths, static_cast<cudaStream_t>(stream));
}

int gbwt_b200_dna_lengths_device(const gbwt_b200_index* ix, const uint64_t* d_seq_ids, size_t m, uint64_t* d_lengths, void* stream) {
    DEVICE_ENTRY_PROLOGUE(ix);
    if (int rc = check_graph(ix)) return rc;
    return launch_extract_dna(ix, d_seq_ids, m, nullptr, 0, 0, nullptr, d_lengths, static_cast<cudaStream_t>(stream));
}
int gbwt_b200_extract_dna_device(const gbwt_b200_index* ix, const uint64_t* d_seq_ids, size_t m, uint8_t endmarker,
                                 const uint64_t* d_out_offsets, uint8_t* d_bytes, uint64_t* d_lengths, void* stream) {
    DEVICE_ENTRY_PROLOGUE(ix);
    if (int rc = check_graph(ix)) return rc;
    if (m > 0 && (d_bytes == nullptr || d_out_offsets == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null output");
    return launch_extract_dna(ix, d_seq_ids, m, d_out_offsets, 0, endmarker, d_bytes, d_lengths, static_cast<cudaStream_t>(stream));
}

// ---- host entry points -------------------------------------------------------------------------------

int gbwt_b200_find(const gbwt_b200_index* ix, const uint64_t* nodes, size_t n, gbwt_b200_state* out) {
    if (int rc = check_index(ix)) return rc;
    if (n > 0 && (nodes == nullptr || out == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null array");
    std::vector<HostArray> arrays = {{nodes, nullptr, 8}, {nullptr, out, sizeof(gbwt_b200_state)}};
    return run_chunked(ix, n, arrays, fixed_chunks(n, chunk_for(sizeof(gbwt_b200_state))), [&](size_t, size_t count, std::vector<void*>& d, cudaStream_t s) {
        return launch_find(ix, static_cast<uint64_t*>(d[0]), count, static_cast<gbwt_b200_state*>(d[1]), s);
    });
}

int gbwt_b200_extend(const gbwt_b200_index* ix, const gbwt_b200_state* states, const uint64_t* nodes, size_t n, gbwt_b200_state* out) {
    if (int rc = check_index(ix)) return rc;
    if (n > 0 && (states == nullptr || nodes == nullptr || out == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null array");
    std::vector<HostArray> arrays = {{states, out, sizeof(gbwt_b200_state)}, {nodes, nullptr, 8}};
    return run_chunked(ix, n, arrays, fixed_chunks(n, chunk_for(sizeof(gbwt_b200_state))), [&](size_t, size_t count, std::vector<void*>& d, cudaStream_t s) {
        gbwt_b200_state* st = static_cast<gbwt_b200_state*>(d[0]);
        return launch_extend(ix, st, static_cast<uint64_t*>(d[1]), count, st, s);
    });
}

int gbwt_b200_find_extend(const gbwt_b200_index* ix, const uint64_t* patterns, size_t n, size_t k, gbwt_b200_state* out) {
    if (int rc = check_index(ix)) return rc;
    if (n > 0 && ((k > 0 && patterns == nullptr) || out == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null array");
    std::vector<HostArray> arrays = {{k > 0 ? patterns : nullptr, nullptr, 8 * k}, {nullptr, out, sizeof(gbwt_b200_state)}};
    // (pattern batches take larger chunks: a chunk is sorted and searched on its own, and the record windows of the
    // search kernel want many queries each)
    return run_chunked(ix, n, arrays, fixed_chunks(n, chunk_for(std::max<size_t>(8 * k, sizeof(gbwt_b200_state)), size_t(512) << 20)),
                       [&](size_t, size_t count, std::vector<void*>& d, cudaStream_t s) {
        return launch_find_extend(ix, static_cast<uint64_t*>(d[0]), count, k, static_cast<gbwt_b200_state*>(d[1]), s);
    });
}

int gbwt_b200_find_extend_u32(const gbwt_b200_index* ix, const uint32_t* patterns, size_t n, size_t k, gbwt_b200_state* out) {
    if (int rc = check_index(ix)) return rc;
    if (n > 0 && ((k > 0 && patterns == nullptr) || out == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null array");
    std::vector<HostArray> arrays = {{k > 0 ? patterns : nullptr, nullptr, 4 * k}, {nullptr, out, sizeof(gbwt_b200_state)}};
    return run_chunked(ix, n, arrays, fixed_chunks(n, chunk_for(std::max<size_t>(4 * k, sizeof(gbwt_b200_state)), size_t(256) << 20)),
                       [&](size_t, size_t count, std::vector<void*>& d, cudaStream_t s) {
        return launch_find_extend(ix, static_cast<uint32_t*>(d[0]), count, k, static_cast<gbwt_b200_state*>(d[1]), s);
    });
}

int gbwt_b200_find_extend_ragged(const gbwt_b200_index* ix, const uint64_t* nodes, const uint64_t* offsets, size_t n, gbwt_b200_state* out) {
    if (int rc = check_index(ix)) return rc;
    if (n > 0 && (offsets == nullptr || out == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null array");
    if (!offsets_valid(offsets, n)) return fail(GBWT_B200_E_ARGUMENT, "offsets must be non-decreasing");
    if (n > 0 && nodes == nullptr && offsets[n] > offsets[0]) return fail(GBWT_B200_E_ARGUMENT, "null array");
    std::vector<HostArray> arrays = {{nodes, nullptr, 8, Slice::Elements}, {offsets, nullptr, 8, Slice::Offsets},
                                     {nullptr, out, sizeof(gbwt_b200_state)}};
    return run_chunked(ix, n, arrays, ragged_chunks(offsets, size_t(1) << 20, uint64_t(8) << 20, 2),
                       [&](size_t q0, size_t count, std::vector<void*>& d, cudaStream_t s) {
        return launch_find_extend_ragged(ix, static_cast<uint64_t*>(d[0]), static_cast<uint64_t*>(d[1]), offsets[q0], count,
                                         static_cast<gbwt_b200_state*>(d[2]), s);
    });
}

int gbwt_b200_bd_find(const gbwt_b200_index* ix, const uint64_t* nodes, size_t n, gbwt_b200_bdstate* out) {
    if (int rc = check_index(ix)) return rc;
    if (int rc = check_bidirectional(ix)) return rc;
    if (n > 0 && (nodes == nullptr || out == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null array");
    std::vector<HostArray> arrays = {{nodes, nullptr, 8}, {nullptr, out, sizeof(gbwt_b200_bdstate)}};
    return run_chunked(ix, n, arrays, fixed_chunks(n, chunk_for(sizeof(gbwt_b200_bdstate))), [&](size_t, size_t count, std::vector<void*>& d, cudaStream_t s) {
        return launch_bd_find(ix, static_cast<uint64_t*>(d[0]), count, static_cast<gbwt_b200_bdstate*>(d[1]), s);
    });
}

static int bd_extend_host(const gbwt_b200_index* ix, const gbwt_b200_bdstate* states, const uint64_t* nodes, size_t n, int backward,
                          gbwt_b200_bdstate* out) {
    if (int rc = check_index(ix)) return rc;
    if (int rc = check_bidirectional(ix)) return rc;
    if (n > 0 && (states == nullptr || nodes == nullptr || out == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null array");
    std::vector<HostArray> arrays = {{states, out, sizeof(gbwt_b200_bdstate)}, {nodes, nullptr, 8}};
    return run_chunked(ix, n, arrays, fixed_chunks(n, chunk_for(sizeof(gbwt_b200_bdstate))), [&](size_t, size_t count, std::vector<void*>& d, cudaStream_t s) {
        gbwt_b200_bdstate* st = static_cast<gbwt_b200_bdstate*>(d[0]);
        return launch_bd_extend(ix, st, static_cast<uint64_t*>(d[1]), count, backward, st, s);
    });
}

int gbwt_b200_extend_forward(const gbwt_b200_index* ix, const gbwt_b200_bdstate* states, const uint64_t* nodes, size_t n, gbwt_b200_bdstate* out) {
    return bd_extend_host(ix, states, nodes, n, 0, out);
}
int gbwt_b200_extend_backward(const gbwt_b200_index* ix, const gbwt_b200_bdstate* states, const uint64_t* nodes, size_t n, gbwt_b200_bdstate* out) {
    return bd_extend_host(ix, states, nodes, n, 1, out);
}

int gbwt_b200_bd_search(const gbwt_b200_index* ix, const uint64_t* nodes, const uint64_t* offsets, const uint64_t* first,
                        const uint64_t* start, const uint64_t* end, size_t n, gbwt_b200_bdstate* out) {
    if (int rc = check_index(ix)) return rc;
    if (int rc = check_bidirectional(ix)) return rc;
    if (n > 0 && (offsets == nullptr || first == nullptr || start == nullptr || end == nullptr || out == nullptr))
        return fail(GBWT_B200_E_ARGUMENT, "null array");
    if (!offsets_valid(offsets, n)) return fail(GBWT_B200_E_ARGUMENT, "offsets must be non-decreasing");
    if (n > 0 && nodes == nullptr && offsets[n] > offsets[0]) return fail(GBWT_B200_E_ARGUMENT, "null array");
    std::vector<HostArray> arrays = {{nodes, nullptr, 8, Slice::Elements}, {offsets, nullptr, 8, Slice::Offsets},
                                     {first, nullptr, 8}, {start, nullptr, 8}, {end, nullptr, 8}, {nullptr, out, sizeof(gbwt_b200_bdstate)}};
    return run_chunked(ix, n, arrays, ragged_chunks(offsets, size_t(1) << 20, uint64_t(8) << 20, 2),
                       [&](size_t q0, size_t count, std::vector<void*>& d, cudaStream_t s) {
        auto u = [&](int a) { return static_cast<const uint64_t*>(d[a]); };
        return launch_bd_search(ix, u(0), u(1), offsets[q0], u(2), u(3), u(4), count, static_cast<gbwt_b200_bdstate*>(d[5]), s);
    });
}

int gbwt_b200_follow(const gbwt_b200_index* ix, const gbwt_b200_bdstate* states, size_t n, int backward, const uint64_t* out_offsets,
                     gbwt_b200_bdstate* out, uint64_t* counts) {
    if (int rc = check_index(ix)) return rc;
    if (int rc = check_bidirectional(ix)) return rc;
    if (n == 0) return GBWT_B200_OK;
    if (states == nullptr || (out != nullptr && out_offsets == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null array");
    if (out == nullptr) {
        if (counts == nullptr) return fail(GBWT_B200_E_ARGUMENT, "null array");
        std::vector<HostArray> arrays = {{states, nullptr, sizeof(gbwt_b200_bdstate)}, {nullptr, counts, 8}};
        return run_chunked(ix, n, arrays, fixed_chunks(n, chunk_for(sizeof(gbwt_b200_bdstate))), [&](size_t, size_t count, std::vector<void*>& d, cudaStream_t s) {
            return launch_follow(ix, static_cast<gbwt_b200_bdstate*>(d[0]), count, backward, nullptr, 0, nullptr, static_cast<uint64_t*>(d[1]), s);
        });
    }
    if (!offsets_valid(out_offsets, n)) return fail(GBWT_B200_E_ARGUMENT, "out_offsets must be non-decreasing");
    // (no fill: what a slot holds beyond its result is unspecified, and clearing it would cost a memset per call)
    std::vector<HostArray> arrays = {{states, nullptr, sizeof(gbwt_b200_bdstate)}, {nullptr, out, sizeof(gbwt_b200_bdstate), Slice::Elements},
                                     {out_offsets, nullptr, 8, Slice::Offsets}, {nullptr, counts, 8}};
    return run_chunked(ix, n, arrays, ragged_chunks(out_offsets, size_t(1) << 20, uint64_t(4) << 20, 1),
                       [&](size_t q0, size_t count, std::vector<void*>& d, cudaStream_t s) {
        return launch_follow(ix, static_cast<gbwt_b200_bdstate*>(d[0]), count, backward, static_cast<uint64_t*>(d[2]), out_offsets[q0],
                             static_cast<gbwt_b200_bdstate*>(d[1]), static_cast<uint64_t*>(d[3]), s);
    });
}

int gbwt_b200_start(const gbwt_b200_index* ix, const uint64_t* seq_ids, size_t n, gbwt_b200_pos* out) {
    if (int rc = check_index(ix)) return rc;
    if (n > 0 && (seq_ids == nullptr || out == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null array");
    std::vector<HostArray> arrays = {{seq_ids, nullptr, 8}, {nullptr, out, sizeof(gbwt_b200_pos)}};
    return run_chunked(ix, n, arrays, fixed_chunks(n, chunk_for(sizeof(gbwt_b200_pos))), [&](size_t, size_t count, std::vector<void*>& d, cudaStream_t s) {
        return launch_start(ix, static_cast<uint64_t*>(d[0]), count, static_cast<gbwt_b200_pos*>(d[1]), s);
    });
}

static int step_host(const gbwt_b200_index* ix, const gbwt_b200_pos* positions, size_t n, gbwt_b200_pos* out, bool backward) {
    if (int rc = check_index(ix)) return rc;
    if (backward) {
        // assert!(self.is_bidirectional(), ...) at src/gbwt.rs:237
        if (!(ix->flags & GBWT_FLAG_BIDIRECTIONAL)) return fail(GBWT_B200_E_NOT_BIDIRECTIONAL, "Following sequences backward requires a bidirectional GBWT");
    }
    if (n > 0 && (positions == nullptr || out == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null array");
    std::vector<HostArray> arrays = {{positions, out, sizeof(gbwt_b200_pos)}};
    return run_chunked(ix, n, arrays, fixed_chunks(n, chunk_for(sizeof(gbwt_b200_pos))), [&](size_t, size_t count, std::vector<void*>& d, cudaStream_t s) {
        gbwt_b200_pos* p = static_cast<gbwt_b200_pos*>(d[0]);
        return backward ? launch_backward(ix, p, count, p, s) : launch_forward(ix, p, count, p, s);
    });
}

int gbwt_b200_forward(const gbwt_b200_index* ix, const gbwt_b200_pos* positions, size_t n, gbwt_b200_pos* out) {
    return step_host(ix, positions, n, out, false);
}
int gbwt_b200_backward(const gbwt_b200_index* ix, const gbwt_b200_pos* positions, size_t n, gbwt_b200_pos* out) {
    return step_host(ix, positions, n, out, true);
}

int gbwt_b200_sequence_lengths(const gbwt_b200_index* ix, const uint64_t* seq_ids, size_t m, uint64_t* lengths) {
    if (int rc = check_index(ix)) return rc;
    if (m > 0 && (seq_ids == nullptr || lengths == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null array");
    std::vector<HostArray> arrays = {{seq_ids, nullptr, 8}, {nullptr, lengths, 8}};
    // all chains of the batch in one launch: a path walk is latency-bound, so concurrency is everything
    return run_chunked(ix, m, arrays, fixed_chunks(m, std::max<size_t>(m, 1)), [&](size_t, size_t count, std::vector<void*>& d, cudaStream_t s) {
        return launch_extract(ix, static_cast<uint64_t*>(d[0]), count, nullptr, 0, nullptr, static_cast<uint64_t*>(d[1]), s);
    });
}

int gbwt_b200_extract(const gbwt_b200_index* ix, const uint64_t* seq_ids, size_t m, const uint64_t* out_offsets, uint64_t* nodes,
                      uint64_t* lengths) {
    if (int rc = check_index(ix)) return rc;
    uint64_t elems = 0;
    if (int rc = slot_budget(ix, seq_ids, m, out_offsets, nodes, sizeof(uint64_t), &elems)) return rc;
    std::vector<HostArray> arrays = {{seq_ids, nullptr, 8}, {nullptr, nodes, sizeof(uint64_t), Slice::Elements, 0x00},
                                     {out_offsets, nullptr, 8, Slice::Offsets}, {nullptr, lengths, 8}};
    return run_chunked(ix, m, arrays, ragged_chunks(out_offsets, m, elems, 1), [&](size_t q0, size_t count, std::vector<void*>& d, cudaStream_t s) {
        return launch_extract(ix, static_cast<uint64_t*>(d[0]), count, static_cast<uint64_t*>(d[2]), out_offsets[q0],
                              static_cast<uint64_t*>(d[1]), static_cast<uint64_t*>(d[3]), s);
    });
}

int gbwt_b200_dna_lengths(const gbwt_b200_index* ix, const uint64_t* seq_ids, size_t m, uint64_t* lengths) {
    if (int rc = check_index(ix)) return rc;
    if (int rc = check_graph(ix)) return rc;
    if (m > 0 && (seq_ids == nullptr || lengths == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null array");
    std::vector<HostArray> arrays = {{seq_ids, nullptr, 8}, {nullptr, lengths, 8}};
    return run_chunked(ix, m, arrays, fixed_chunks(m, std::max<size_t>(m, 1)), [&](size_t, size_t count, std::vector<void*>& d, cudaStream_t s) {
        return launch_extract_dna(ix, static_cast<uint64_t*>(d[0]), count, nullptr, 0, 0, nullptr, static_cast<uint64_t*>(d[1]), s);
    });
}

int gbwt_b200_extract_dna(const gbwt_b200_index* ix, const uint64_t* seq_ids, size_t m, uint8_t endmarker, const uint64_t* out_offsets,
                          uint8_t* bytes, uint64_t* lengths) {
    if (int rc = check_index(ix)) return rc;
    if (int rc = check_graph(ix)) return rc;
    uint64_t elems = 0;
    if (int rc = slot_budget(ix, seq_ids, m, out_offsets, bytes, 1, &elems)) return rc;
    std::vector<HostArray> arrays = {{seq_ids, nullptr, 8}, {nullptr, bytes, 1, Slice::Elements, 0x00},
                                     {out_offsets, nullptr, 8, Slice::Offsets}, {nullptr, lengths, 8}};
    return run_chunked(ix, m, arrays, ragged_chunks(out_offsets, m, elems, 1), [&](size_t q0, size_t count, std::vector<void*>& d, cudaStream_t s) {
        return launch_extract_dna(ix, static_cast<uint64_t*>(d[0]), count, static_cast<uint64_t*>(d[2]), out_offsets[q0], endmarker,
                                  static_cast<uint8_t*>(d[1]), static_cast<uint64_t*>(d[3]), s);
    });
}

int gbwt_b200_locate(const gbwt_b200_index* ix, const gbwt_b200_pos* positions, size_t n, gbwt_b200_occurrence* out) {
    if (int rc = check_index(ix)) return rc;
    if (int rc = check_samples(ix)) return rc;
    if (n > 0 && (positions == nullptr || out == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null array");
    std::vector<HostArray> arrays = {{positions, nullptr, sizeof(gbwt_b200_pos)}, {nullptr, out, sizeof(gbwt_b200_occurrence)}};
    return run_chunked(ix, n, arrays, fixed_chunks(n, chunk_for(sizeof(gbwt_b200_pos))), [&](size_t, size_t count, std::vector<void*>& d, cudaStream_t s) {
        return launch_locate_positions(ix, static_cast<gbwt_b200_pos*>(d[0]), count, static_cast<gbwt_b200_occurrence*>(d[1]), s);
    });
}

int gbwt_b200_locate_states(const gbwt_b200_index* ix, const gbwt_b200_state* states, size_t n, const uint64_t* out_offsets,
                            gbwt_b200_occurrence* out, uint64_t* counts) {
    if (int rc = check_index(ix)) return rc;
    if (int rc = check_samples(ix)) return rc;
    if (n == 0) return GBWT_B200_OK;
    if (states == nullptr || (out != nullptr && out_offsets == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null array");
    if (out == nullptr) {
        if (counts == nullptr) return fail(GBWT_B200_E_ARGUMENT, "null array");
        std::vector<HostArray> arrays = {{states, nullptr, sizeof(gbwt_b200_state)}, {nullptr, counts, 8}};
        return run_chunked(ix, n, arrays, fixed_chunks(n, chunk_for(sizeof(gbwt_b200_state))), [&](size_t, size_t count, std::vector<void*>& d, cudaStream_t s) {
            return launch_locate_state_batch(ix, static_cast<gbwt_b200_state*>(d[0]), count, nullptr, 0, nullptr, static_cast<uint64_t*>(d[1]), s);
        });
    }
    if (!offsets_valid(out_offsets, n)) return fail(GBWT_B200_E_ARGUMENT, "out_offsets must be non-decreasing");
    std::vector<HostArray> arrays = {{states, nullptr, sizeof(gbwt_b200_state)}, {nullptr, out, sizeof(gbwt_b200_occurrence), Slice::Elements, 0xFF},
                                     {out_offsets, nullptr, 8, Slice::Offsets}, {nullptr, counts, 8}};
    return run_chunked(ix, n, arrays, ragged_chunks(out_offsets, size_t(1) << 22, uint64_t(16) << 20, 1),
                       [&](size_t q0, size_t count, std::vector<void*>& d, cudaStream_t s) {
        return launch_locate_state_batch(ix, static_cast<gbwt_b200_state*>(d[0]), count, static_cast<uint64_t*>(d[2]), out_offsets[q0],
                                         static_cast<gbwt_b200_occurrence*>(d[1]), static_cast<uint64_t*>(d[3]), s);
    });
}

int gbwt_b200_seek(const gbwt_b200_index* ix, const uint64_t* seq_ids, const uint64_t* indexes, size_t n, gbwt_b200_pos* out) {
    if (int rc = check_index(ix)) return rc;
    if (n > 0 && (seq_ids == nullptr || indexes == nullptr || out == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null array");
    std::vector<HostArray> arrays = {{seq_ids, nullptr, 8}, {indexes, nullptr, 8}, {nullptr, out, sizeof(gbwt_b200_pos)}};
    return run_chunked(ix, n, arrays, fixed_chunks(n, chunk_for(sizeof(gbwt_b200_pos))), [&](size_t, size_t count, std::vector<void*>& d, cudaStream_t s) {
        return launch_seek_batch(ix, static_cast<uint64_t*>(d[0]), static_cast<uint64_t*>(d[1]), count, static_cast<gbwt_b200_pos*>(d[2]), s);
    });
}

int gbwt_b200_extract_ranges(const gbwt_b200_index* ix, const uint64_t* seq_ids, const uint64_t* starts, const uint64_t* ends, size_t m,
                             const uint64_t* out_offsets, uint64_t* nodes, uint64_t* lengths) {
    return ranges_host(ix, false, seq_ids, starts, ends, m, out_offsets, nodes, lengths);
}

int gbwt_b200_extract_dna_ranges(const gbwt_b200_index* ix, const uint64_t* seq_ids, const uint64_t* starts, const uint64_t* ends, size_t m,
                                 const uint64_t* out_offsets, uint8_t* bytes, uint64_t* lengths) {
    return ranges_host(ix, true, seq_ids, starts, ends, m, out_offsets, bytes, lengths);
}

int gbwt_b200_node_sequence_lengths(const gbwt_b200_index* ix, const uint64_t* node_ids, size_t n, uint64_t* lengths) {
    if (int rc = check_index(ix)) return rc;
    if (int rc = check_graph(ix)) return rc;
    if (n > 0 && (node_ids == nullptr || lengths == nullptr)) return fail(GBWT_B200_E_ARGUMENT, "null array");
    std::vector<HostArray> arrays = {{node_ids, nullptr, 8}, {nullptr, lengths, 8}};
    return run_chunked(ix, n, arrays, fixed_chunks(n, chunk_for(16)), [&](size_t, size_t count, std::vector<void*>& d, cudaStream_t s) {
        return launch_node_sequences(ix, static_cast<uint64_t*>(d[0]), count, nullptr, 0, nullptr, static_cast<uint64_t*>(d[1]), s);
    });
}

int gbwt_b200_node_sequences(const gbwt_b200_index* ix, const uint64_t* node_ids, size_t n, const uint64_t* out_offsets, uint8_t* bytes,
                             uint64_t* lengths) {
    if (int rc = check_index(ix)) return rc;
    if (int rc = check_graph(ix)) return rc;
    uint64_t elems = 0;
    if (int rc = slot_budget(ix, node_ids, n, out_offsets, bytes, 1, &elems)) return rc;
    std::vector<HostArray> arrays = {{node_ids, nullptr, 8}, {nullptr, bytes, 1, Slice::Elements, 0x00},
                                     {out_offsets, nullptr, 8, Slice::Offsets}, {nullptr, lengths, 8}};
    return run_chunked(ix, n, arrays, ragged_chunks(out_offsets, n, elems, 1), [&](size_t q0, size_t count, std::vector<void*>& d, cudaStream_t s) {
        return launch_node_sequences(ix, static_cast<uint64_t*>(d[0]), count, static_cast<uint64_t*>(d[2]), out_offsets[q0],
                                     static_cast<uint8_t*>(d[1]), static_cast<uint64_t*>(d[3]), s);
    });
}

// ---- building a GBWT from paths (gbwt_b200_build.h) ---------------------------------------------------------

static int build_to_image(const uint64_t* d_nodes, const uint64_t* d_offsets, size_t n, int bidirectional, uint64_t extra_bytes,
                          cudaStream_t s, void** image, size_t* len, uint64_t info[4]) {
    std::vector<uint8_t> bytes;
    std::string err;
    const int rc = build_gbwt_image(d_nodes, d_offsets, n, bidirectional != 0, extra_bytes, s, bytes, info, err);
    if (rc != GBWT_B200_OK) return fail(rc, err);
    void* out = std::malloc(std::max<size_t>(bytes.size(), 1));
    if (out == nullptr) return fail(GBWT_B200_E_IO, "out of memory");
    std::memcpy(out, bytes.data(), bytes.size());
    *image = out; *len = bytes.size();
    return GBWT_B200_OK;
}

static int check_build_call(int device, void** image, size_t* len, size_t n) {
    if (image == nullptr || len == nullptr) return fail(GBWT_B200_E_ARGUMENT, "null output");
    *image = nullptr; *len = 0;
    if (n == 0) return fail(GBWT_B200_E_ARGUMENT, "no paths");
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(GBWT_B200_E_NO_DEVICE, "no CUDA device available (this library has no CPU fallback)");
    }
    if (device < 0 || device >= count) return fail(GBWT_B200_E_ARGUMENT, "invalid device ordinal");
    return GBWT_B200_OK;
}

// Host paths on the current device for a build or an insertion: the checks of build_check_paths, the memory check (`need`
// from the records and the bytes of the copies), then the copies on a new stream, freed on every path.
struct PathUpload {
    void* nodes = nullptr;
    void* offsets = nullptr;
    cudaStream_t s = nullptr;
    uint64_t bytes = 0;
    PathUpload() = default;
    PathUpload(const PathUpload&) = delete;
    PathUpload& operator=(const PathUpload&) = delete;
    ~PathUpload() { cudaFree(nodes); cudaFree(offsets); if (s) cudaStreamDestroy(s); }
};

static int upload_paths(const uint64_t* nodes, const uint64_t* offsets, size_t n, bool bidirectional, const char* what,
                        const std::function<uint64_t(uint64_t, uint64_t)>& need_of, PathUpload& in) {
    std::string err;
    uint64_t records = 0;
    if (int rc = build_check_paths(nodes, offsets, n, bidirectional, records, err)) return fail(rc, err);
    const uint64_t path_nodes = offsets[n] - offsets[0];
    std::vector<uint64_t> rebased(offsets, offsets + n + 1);
    for (uint64_t& o : rebased) o -= offsets[0];
    in.bytes = 8 * (path_nodes + n + 1);
    size_t free_bytes = 0, total_bytes = 0;
    CUDA_TRY(cudaMemGetInfo(&free_bytes, &total_bytes));
    const uint64_t need = need_of(path_nodes, records) + in.bytes;
    if (need > free_bytes)
        return fail(GBWT_B200_E_CUDA, std::string("the ") + what + " needs about " + std::to_string(need) + " bytes of device memory; " +
                                      std::to_string(free_bytes) + " are free");
    CUDA_TRY(cudaStreamCreateWithFlags(&in.s, cudaStreamNonBlocking));
    CUDA_TRY(cudaMalloc(&in.nodes, std::max<uint64_t>(8 * path_nodes, 8)));
    CUDA_TRY(cudaMalloc(&in.offsets, 8 * (n + 1)));
    if (path_nodes > 0) CUDA_TRY(cudaMemcpyAsync(in.nodes, nodes + offsets[0], 8 * path_nodes, cudaMemcpyHostToDevice, in.s));
    CUDA_TRY(cudaMemcpyAsync(in.offsets, rebased.data(), 8 * (n + 1), cudaMemcpyHostToDevice, in.s));
    return GBWT_B200_OK;
}

// A null d_nodes is refused once the offsets show the paths are not all empty.
static int check_device_nodes(const uint64_t* d_nodes, const uint64_t* d_offsets, size_t n, cudaStream_t s) {
    if (d_nodes != nullptr) return GBWT_B200_OK;
    uint64_t ends[2] = {0, 0};
    CUDA_TRY(cudaMemcpyAsync(&ends[0], d_offsets, 8, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(&ends[1], d_offsets + n, 8, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    if (ends[1] != ends[0]) return fail(GBWT_B200_E_ARGUMENT, "null nodes");
    return GBWT_B200_OK;
}

int gbwt_b200_build_image(const uint64_t* nodes, const uint64_t* offsets, size_t n, int bidirectional, int device, void** image,
                          size_t* len, uint64_t info[4]) {
    if (int rc = check_build_call(device, image, len, n)) return rc;
    if (offsets == nullptr) return fail(GBWT_B200_E_ARGUMENT, "null offsets");
    GBWT_B200_GUARDED(
        DeviceScope scope(device);
        if (!scope.ok) return fail(GBWT_B200_E_CUDA, "cudaSetDevice failed");
        PathUpload in;
        if (int rc = upload_paths(nodes, offsets, n, bidirectional != 0, "build", [&](uint64_t path_nodes, uint64_t records) {
                return build_device_bytes(n, path_nodes, bidirectional != 0, records);
            }, in)) return rc;
        return build_to_image(static_cast<const uint64_t*>(in.nodes), static_cast<const uint64_t*>(in.offsets), n, bidirectional,
                              in.bytes, in.s, image, len, info);
    )
}

int gbwt_b200_build_image_device(const uint64_t* d_nodes, const uint64_t* d_offsets, size_t n, int bidirectional, int device,
                                 void* stream, void** image, size_t* len, uint64_t info[4]) {
    if (int rc = check_build_call(device, image, len, n)) return rc;
    if (d_offsets == nullptr) return fail(GBWT_B200_E_ARGUMENT, "null offsets");
    GBWT_B200_GUARDED(
        DeviceScope scope(device);
        if (!scope.ok) return fail(GBWT_B200_E_CUDA, "cudaSetDevice failed");
        if (int rc = check_device_nodes(d_nodes, d_offsets, n, static_cast<cudaStream_t>(stream))) return rc;
        return build_to_image(d_nodes, d_offsets, n, bidirectional, 0, static_cast<cudaStream_t>(stream), image, len, info);
    )
}

// ---- inserting paths into an index (gbwt_b200_insert.h) ----------------------------------------------------------

static InsertTarget insert_target(const gbwt_b200_index* ix) {
    InsertTarget a;
    a.view = ix->view;
    a.size = ix->size;
    a.edges_total = ix->edges_total;
    a.body_bytes = ix->bytes[1];
    return a;
}

static int insert_to_image(const gbwt_b200_index* ix, const uint64_t* d_nodes, const uint64_t* d_offsets, size_t n, uint64_t extra_bytes,
                           cudaStream_t s, void** image, size_t* len, uint64_t info[6]) {
    std::vector<uint8_t> bytes;
    std::string err;
    const int rc = insert_gbwt_image(insert_target(ix), d_nodes, d_offsets, n, extra_bytes, s, bytes, info, err);
    if (rc != GBWT_B200_OK) return fail(rc, err);
    void* out = std::malloc(std::max<size_t>(bytes.size(), 1));
    if (out == nullptr) return fail(GBWT_B200_E_IO, "out of memory");
    std::memcpy(out, bytes.data(), bytes.size());
    *image = out; *len = bytes.size();
    return GBWT_B200_OK;
}

static int check_insert_call(const gbwt_b200_index* ix, void** image, size_t* len, size_t n) {
    if (int rc = check_index(ix)) return rc;
    return check_build_call(ix->device, image, len, n);
}

int gbwt_b200_insert_image(const gbwt_b200_index* ix, const uint64_t* nodes, const uint64_t* offsets, size_t n, void** image, size_t* len,
                           uint64_t info[6]) {
    if (int rc = check_insert_call(ix, image, len, n)) return rc;
    if (offsets == nullptr) return fail(GBWT_B200_E_ARGUMENT, "null offsets");
    GBWT_B200_GUARDED(
        DeviceScope scope(ix->device);
        if (!scope.ok) return fail(GBWT_B200_E_CUDA, "cudaSetDevice failed");
        const bool bidirectional = (ix->flags & GBWT_FLAG_BIDIRECTIONAL) != 0;
        PathUpload in;
        if (int rc = upload_paths(nodes, offsets, n, bidirectional, "insertion", [&](uint64_t path_nodes, uint64_t) {
                return build_device_bytes(n, path_nodes, bidirectional, 1);
            }, in)) return rc;
        return insert_to_image(ix, static_cast<const uint64_t*>(in.nodes), static_cast<const uint64_t*>(in.offsets), n, in.bytes, in.s,
                               image, len, info);
    )
}

int gbwt_b200_insert_image_device(const gbwt_b200_index* ix, const uint64_t* d_nodes, const uint64_t* d_offsets, size_t n, void* stream,
                                  void** image, size_t* len, uint64_t info[6]) {
    if (int rc = check_insert_call(ix, image, len, n)) return rc;
    if (d_offsets == nullptr) return fail(GBWT_B200_E_ARGUMENT, "null offsets");
    GBWT_B200_GUARDED(
        DeviceScope scope(ix->device);
        if (!scope.ok) return fail(GBWT_B200_E_CUDA, "cudaSetDevice failed");
        if (int rc = check_device_nodes(d_nodes, d_offsets, n, static_cast<cudaStream_t>(stream))) return rc;
        return insert_to_image(ix, d_nodes, d_offsets, n, 0, static_cast<cudaStream_t>(stream), image, len, info);
    )
}

// ---- utilities ---------------------------------------------------------------------------------------

void* gbwt_b200_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, std::max<size_t>(bytes, 1), cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
void gbwt_b200_host_free(void* p) { if (p) cudaFreeHost(p); }
uint64_t gbwt_b200_kernel_launches(void) { return g_launches.load(); }
const char* gbwt_b200_version(void) { return "gbwt-rs_b200 0.1.0 (sm_100a)"; }

}  // extern "C"
