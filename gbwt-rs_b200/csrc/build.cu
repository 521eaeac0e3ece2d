// build.cu -- the GBWT of a set of paths, built on the device (gbwt_b200_build_image, include/gbwt_b200_build.h).
//
// The visits to a node are sorted by their reversed prefixes, ties at the start of a sequence broken by sequence id
// (the definition of tests/gbwt_builder.py, which the C++ GBWT's construction follows). With T nodes in n sequences,
// position p gets a rank: terminators rank 0 .. n-1 (the sequence id), nodes rank in [n, n + T), so every terminator
// sorts below every node. Prefix doubling orders all positions:
//   1. sort by symbol; R_1(p) = n + the dense group number of p;
//   2. round h: key(p) = (R_h(p), R_h(p - h) if p - h is in the same sequence, else the sequence id); sort; R_2h from the
//      group numbers. Stop when all T keys differ. A key that reaches its terminator is unique, so this happens once 2h
//      exceeds the longest sequence at the latest.
// The final order is the BWT order of every record but record 0, which is the n sequences in id order. From it:
// the successor of each entry, the edges (an entry starts an edge block where its predecessor differs from the previous
// entry's in the same record), the edge rank of each entry, maximal runs, and the record bytes (record_encode.h), each
// run written by one thread at an offset from exclusive scans. The host then writes the file (layout_writer.h).
#include "build.h"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>

#include <algorithm>
#include <chrono>
#include <utility>

#include "../../include/gbwt_b200.h"
#include "layout_writer.h"
#include "record_encode.h"

namespace gbwt_b200 {

namespace {

constexpr int BUILD_THREADS = 256;
constexpr uint32_t BAD_OFFSETS = 1, BAD_NODE = 2, NODE_RANGE = 4;

struct BuildStats {
    uint32_t flags;
    uint32_t min_node, max_node;  // over both orientations when bidirectional
    uint32_t pad;
    unsigned long long count;     // edges emitted, groups after a sort
};

unsigned grid_of(uint64_t n, int sm_count) {
    const uint64_t blocks = (n + BUILD_THREADS - 1) / BUILD_THREADS;
    const uint64_t wave = static_cast<uint64_t>(std::max(1, sm_count)) * (2048 / BUILD_THREADS);
    return static_cast<unsigned>(std::max<uint64_t>(1, std::min(blocks, wave)));
}

__device__ __forceinline__ uint64_t stride() { return static_cast<uint64_t>(gridDim.x) * blockDim.x; }
__device__ __forceinline__ uint64_t first_index() { return blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; }

// First i in [lo, hi) with a[i] >= key.
template <class T>
__device__ __forceinline__ uint64_t lower_bound(const T* __restrict__ a, uint64_t lo, uint64_t hi, uint64_t key) {
    while (lo < hi) {
        const uint64_t mid = lo + (hi - lo) / 2;
        if (static_cast<uint64_t>(a[mid]) < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// Sequence s: its first position in the expanded array and its length.
struct SeqSpan { uint64_t start, len; };
__device__ __forceinline__ SeqSpan seq_span(const uint64_t* __restrict__ offsets, uint64_t s, bool bidirectional) {
    const uint64_t q = bidirectional ? s >> 1 : s, base = offsets[0];
    const uint64_t lo = offsets[q] - base, len = offsets[q + 1] - offsets[q];
    if (!bidirectional) return {lo, len};
    return {2 * lo + (s & 1) * len, len};
}

__global__ void __launch_bounds__(BUILD_THREADS) k_build_check_offsets(const uint64_t* __restrict__ offsets, uint64_t n,
                                                                       BuildStats* __restrict__ stats) {
    for (uint64_t q = first_index(); q < n; q += stride())
        if (offsets[q + 1] < offsets[q]) atomicOr(&stats->flags, BAD_OFFSETS);
}

// Flags node 0 (and node 1 when bidirectional: its flip is the endmarker) and nodes >= 2^32; min / max node.
__global__ void __launch_bounds__(BUILD_THREADS) k_build_check_nodes(const uint64_t* __restrict__ nodes, uint64_t count, bool bidirectional,
                                                                     BuildStats* __restrict__ stats) {
    uint32_t flags = 0, lo = 0xFFFFFFFFu, hi = 0;
    for (uint64_t base = blockIdx.x * static_cast<uint64_t>(blockDim.x); base < count; base += stride()) {
        const uint64_t i = base + threadIdx.x;
        if (i < count) {
            const uint64_t v = nodes[i];
            if (v == 0 || (bidirectional && v == 1)) flags |= BAD_NODE;
            if (v >> 32) { flags |= NODE_RANGE; continue; }
            const uint32_t a = bidirectional ? static_cast<uint32_t>(v & ~1ull) : static_cast<uint32_t>(v);
            const uint32_t b = bidirectional ? static_cast<uint32_t>(v | 1ull) : static_cast<uint32_t>(v);
            lo = min(lo, a); hi = max(hi, b);
        }
    }
    flags = __reduce_or_sync(0xFFFFFFFFu, flags);
    lo = __reduce_min_sync(0xFFFFFFFFu, lo);
    hi = __reduce_max_sync(0xFFFFFFFFu, hi);
    if ((threadIdx.x & 31u) == 0) {
        if (flags) atomicOr(&stats->flags, flags);
        atomicMin(&stats->min_node, lo);
        atomicMax(&stats->max_node, hi);
    }
}

// Expanded sequences: symbol and sequence id of every position (the reverse strand written after the forward one).
__global__ void __launch_bounds__(BUILD_THREADS) k_build_expand(const uint64_t* __restrict__ nodes, const uint64_t* __restrict__ offsets,
                                                                uint64_t n, uint64_t path_nodes, bool bidirectional,
                                                                uint32_t* __restrict__ sym, uint32_t* __restrict__ seq) {
    const uint64_t base = offsets[0];
    for (uint64_t i = first_index(); i < path_nodes; i += stride()) {
        const uint64_t g = base + i;
        uint64_t lo = 0, hi = n;  // last path q with offsets[q] <= g
        while (hi - lo > 1) {
            const uint64_t mid = lo + (hi - lo) / 2;
            if (offsets[mid] <= g) lo = mid; else hi = mid;
        }
        const uint64_t v = nodes[g], j = g - offsets[lo];
        if (!bidirectional) { sym[i] = static_cast<uint32_t>(v); seq[i] = static_cast<uint32_t>(lo); continue; }
        const uint64_t start = 2 * (offsets[lo] - base), len = offsets[lo + 1] - offsets[lo];
        sym[start + j] = static_cast<uint32_t>(v);
        seq[start + j] = static_cast<uint32_t>(2 * lo);
        sym[start + 2 * len - 1 - j] = static_cast<uint32_t>(v ^ 1);
        seq[start + 2 * len - 1 - j] = static_cast<uint32_t>(2 * lo + 1);
    }
}

__global__ void __launch_bounds__(BUILD_THREADS) k_build_symbol_keys(const uint32_t* __restrict__ sym, uint64_t count,
                                                                     uint64_t* __restrict__ keys, uint32_t* __restrict__ pos) {
    for (uint64_t p = first_index(); p < count; p += stride()) { keys[p] = sym[p]; pos[p] = static_cast<uint32_t>(p); }
}

// key(p) = R_h(p) << bits | (R_h(p - h) within the sequence, else the sequence id).
__global__ void __launch_bounds__(BUILD_THREADS) k_build_keys(const uint32_t* __restrict__ rank, const uint32_t* __restrict__ seq,
                                                              uint64_t count, uint64_t h, int bits, uint64_t* __restrict__ keys,
                                                              uint32_t* __restrict__ pos) {
    for (uint64_t p = first_index(); p < count; p += stride()) {
        const uint32_t s = seq[p];
        const uint32_t next = (p >= h && seq[p - h] == s) ? rank[p - h] : s;
        keys[p] = (static_cast<uint64_t>(rank[p]) << bits) | next;
        pos[p] = static_cast<uint32_t>(p);
    }
}

// 1 where a sorted key differs from its predecessor (the scan of these numbers the groups).
__global__ void __launch_bounds__(BUILD_THREADS) k_build_group_heads(const uint64_t* __restrict__ keys, uint64_t count,
                                                                     uint32_t* __restrict__ heads) {
    for (uint64_t i = first_index(); i < count; i += stride()) heads[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1u : 0u;
}

__global__ void __launch_bounds__(BUILD_THREADS) k_build_ranks(const uint32_t* __restrict__ order, const uint32_t* __restrict__ group,
                                                               uint64_t count, uint64_t sequences, uint32_t* __restrict__ rank) {
    for (uint64_t i = first_index(); i < count; i += stride())
        rank[order[i]] = static_cast<uint32_t>(sequences + group[i] - 1);
}

// Entry e of the BWT: e < n is sequence e in record 0, e >= n the position order[e - n]. Its record, successor and
// predecessor (0 = the endmarker).
__global__ void __launch_bounds__(BUILD_THREADS) k_build_entries(const uint32_t* __restrict__ order, const uint32_t* __restrict__ sym,
                                                                 const uint32_t* __restrict__ seq, const uint64_t* __restrict__ offsets,
                                                                 uint64_t sequences, uint64_t count, bool bidirectional, uint64_t offset,
                                                                 uint32_t* __restrict__ rec, uint32_t* __restrict__ succ,
                                                                 uint32_t* __restrict__ pred) {
    const uint64_t entries = sequences + count;
    for (uint64_t e = first_index(); e < entries; e += stride()) {
        if (e < sequences) {
            const SeqSpan sp = seq_span(offsets, e, bidirectional);
            rec[e] = 0;
            succ[e] = sp.len > 0 ? sym[sp.start] : 0;
            pred[e] = 0;
            continue;
        }
        const uint64_t p = order[e - sequences];
        const uint32_t s = seq[p];
        rec[e] = static_cast<uint32_t>(sym[p] - offset);
        succ[e] = (p + 1 < count && seq[p + 1] == s) ? sym[p + 1] : 0;
        pred[e] = (p >= 1 && seq[p - 1] == s) ? sym[p - 1] : 0;
    }
}

// out[r] = first i with a[i] >= r, r < count - 1; out[count - 1] = len.
template <class T>
__global__ void __launch_bounds__(BUILD_THREADS) k_build_record_firsts(const T* __restrict__ a, uint64_t len, int shift, uint64_t count,
                                                                       uint32_t* __restrict__ out) {
    for (uint64_t r = first_index(); r < count; r += stride())
        out[r] = static_cast<uint32_t>(r + 1 == count ? len : lower_bound(a, 0, len, r << shift));
}

// Edges (from record << 32 | to node, offset in the record of `to`): one where an entry of record w starts a block of one
// predecessor, and (v -> 0, 0) for every entry whose successor is the endmarker (duplicates removed after the sort).
// keys == nullptr: count only. One atomic per warp.
__global__ void __launch_bounds__(BUILD_THREADS) k_build_edges(const uint32_t* __restrict__ rec, const uint32_t* __restrict__ succ,
                                                               const uint32_t* __restrict__ pred, const uint32_t* __restrict__ rec_first,
                                                               uint64_t sequences, uint64_t entries, uint64_t offset,
                                                               BuildStats* __restrict__ stats, uint64_t* __restrict__ keys,
                                                               uint32_t* __restrict__ offs) {
    const unsigned lane = threadIdx.x & 31u;
    for (uint64_t base = blockIdx.x * static_cast<uint64_t>(blockDim.x); base < entries; base += stride()) {
        const uint64_t e = base + threadIdx.x;
        uint64_t k0 = 0, k1 = 0;  // the block edge first, then the edge to the endmarker
        uint32_t o0 = 0, emit = 0;
        if (e < entries) {
            const uint32_t r = rec[e];
            if (e >= sequences) {
                const uint64_t first = rec_first[r];
                const uint32_t v = pred[e];
                if (e == first || v != pred[e - 1]) {
                    k0 = (static_cast<uint64_t>(v == 0 ? 0 : v - offset) << 32) | (r + offset);
                    o0 = static_cast<uint32_t>(e - first);
                    emit = 1;
                }
            }
            if (succ[e] == 0) {
                const uint64_t k = static_cast<uint64_t>(r) << 32;
                if (emit == 1) k1 = k; else k0 = k;
                emit++;
            }
        }
        uint32_t before = emit;  // inclusive scan over the warp
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t x = __shfl_up_sync(0xFFFFFFFFu, before, d);
            if (lane >= static_cast<unsigned>(d)) before += x;
        }
        const uint32_t total = __shfl_sync(0xFFFFFFFFu, before, 31);
        unsigned long long at = 0;
        if (lane == 31 && total) at = atomicAdd(&stats->count, static_cast<unsigned long long>(total));
        at = __shfl_sync(0xFFFFFFFFu, at, 31) + before - emit;
        if (keys != nullptr && emit) {
            keys[at] = k0; offs[at] = o0;
            if (emit == 2) { keys[at + 1] = k1; offs[at + 1] = 0; }
        }
    }
}

// Entry e's value: the rank of its successor in its record's edge list (written over the successor).
__global__ void __launch_bounds__(BUILD_THREADS) k_build_values(const uint32_t* __restrict__ rec, uint32_t* __restrict__ succ, uint64_t entries,
                                                                const uint32_t* __restrict__ edge_first, const uint64_t* __restrict__ edge_keys) {
    for (uint64_t e = first_index(); e < entries; e += stride()) {
        const uint32_t r = rec[e];
        const uint64_t lo = edge_first[r], hi = edge_first[r + 1];
        succ[e] = static_cast<uint32_t>(lower_bound(edge_keys, lo, hi, (static_cast<uint64_t>(r) << 32) | succ[e]) - lo);
    }
}

__device__ __forceinline__ bool run_head(const uint32_t* __restrict__ rec, const uint32_t* __restrict__ value, uint64_t e) {
    return e == 0 || rec[e] != rec[e - 1] || value[e] != value[e - 1];
}

__global__ void __launch_bounds__(BUILD_THREADS) k_build_run_heads(const uint32_t* __restrict__ rec, const uint32_t* __restrict__ value,
                                                                   uint64_t entries, uint32_t* __restrict__ heads) {
    for (uint64_t e = first_index(); e < entries; e += stride()) heads[e] = run_head(rec, value, e) ? 1u : 0u;
}

// run_start[i] = first entry of run i (from the inclusive scan of the heads); run_start[runs] = entries.
__global__ void __launch_bounds__(BUILD_THREADS) k_build_run_starts(const uint32_t* __restrict__ rec, const uint32_t* __restrict__ value,
                                                                    const uint32_t* __restrict__ scan, uint64_t entries,
                                                                    uint32_t* __restrict__ run_start) {
    for (uint64_t e = first_index(); e < entries; e += stride())
        if (run_head(rec, value, e)) run_start[scan[e] - 1] = static_cast<uint32_t>(e);
    if (first_index() == 0) run_start[scan[entries - 1]] = static_cast<uint32_t>(entries);
}

__device__ __forceinline__ uint64_t edge_count(const uint32_t* __restrict__ edge_first, uint64_t r) {
    return edge_first[r + 1] - edge_first[r];
}

__global__ void __launch_bounds__(BUILD_THREADS) k_build_run_bytes(const uint32_t* __restrict__ run_start, uint64_t runs,
                                                                   const uint32_t* __restrict__ rec, const uint32_t* __restrict__ value,
                                                                   const uint32_t* __restrict__ edge_first, uint64_t* __restrict__ bytes) {
    for (uint64_t i = first_index(); i <= runs; i += stride()) {
        if (i == runs) { bytes[i] = 0; continue; }
        const uint64_t e = run_start[i];
        ByteSink count;
        put_run(count, edge_count(edge_first, rec[e]), value[e], run_start[i + 1] - e);
        bytes[i] = count.n;
    }
}

__device__ __forceinline__ void put_header(ByteSink& out, const uint32_t* __restrict__ edge_first, const uint64_t* __restrict__ edge_keys,
                                           const uint32_t* __restrict__ edge_offs, uint64_t r) {
    const uint64_t lo = edge_first[r];
    put_edges(out, edge_first[r + 1] - lo, [&](uint64_t e) { return EdgeValue{edge_keys[lo + e] & 0xFFFFFFFFull, edge_offs[lo + e]}; });
}

// First run of record r (its first entry starts a run; an empty record gets the first run of the next one).
__device__ __forceinline__ uint64_t first_run(const uint32_t* __restrict__ run_start, uint64_t runs, const uint32_t* __restrict__ rec_first, uint64_t r) {
    return lower_bound(run_start, 0, runs, rec_first[r]);
}

__global__ void __launch_bounds__(BUILD_THREADS) k_build_record_bytes(uint64_t records, const uint32_t* __restrict__ rec_first,
                                                                      const uint32_t* __restrict__ run_start, uint64_t runs,
                                                                      const uint64_t* __restrict__ run_off, const uint32_t* __restrict__ edge_first,
                                                                      const uint64_t* __restrict__ edge_keys, const uint32_t* __restrict__ edge_offs,
                                                                      uint64_t* __restrict__ bytes) {
    for (uint64_t r = first_index(); r <= records; r += stride()) {
        if (r == records) { bytes[r] = 0; continue; }
        ByteSink count;
        put_header(count, edge_first, edge_keys, edge_offs, r);
        bytes[r] = count.n + run_off[first_run(run_start, runs, rec_first, r + 1)] - run_off[first_run(run_start, runs, rec_first, r)];
    }
}

// Writes the header of every record; run_base[r] = where the runs of r go, minus the scan offset of its first run.
__global__ void __launch_bounds__(BUILD_THREADS) k_build_write_records(uint64_t records, const uint64_t* __restrict__ rec_start,
                                                                       const uint32_t* __restrict__ rec_first, const uint32_t* __restrict__ run_start,
                                                                       uint64_t runs, const uint64_t* __restrict__ run_off,
                                                                       const uint32_t* __restrict__ edge_first, const uint64_t* __restrict__ edge_keys,
                                                                       const uint32_t* __restrict__ edge_offs, uint8_t* __restrict__ data,
                                                                       uint64_t* __restrict__ run_base) {
    for (uint64_t r = first_index(); r < records; r += stride()) {
        ByteSink out;
        out.at = data + rec_start[r];
        put_header(out, edge_first, edge_keys, edge_offs, r);
        run_base[r] = rec_start[r] + out.n - run_off[first_run(run_start, runs, rec_first, r)];
    }
}

__global__ void __launch_bounds__(BUILD_THREADS) k_build_write_runs(const uint32_t* __restrict__ run_start, uint64_t runs,
                                                                    const uint32_t* __restrict__ rec, const uint32_t* __restrict__ value,
                                                                    const uint32_t* __restrict__ edge_first, const uint64_t* __restrict__ run_off,
                                                                    const uint64_t* __restrict__ run_base, uint8_t* __restrict__ data) {
    for (uint64_t i = first_index(); i < runs; i += stride()) {
        const uint64_t e = run_start[i];
        const uint32_t r = rec[e];
        ByteSink out;
        out.at = data + run_base[r] + run_off[i];
        put_run(out, edge_count(edge_first, r), value[e], run_start[i + 1] - e);
    }
}

// Device scratch with a byte count: every block is freed when the scratch goes out of scope.
struct Scratch {
    std::vector<std::pair<void*, uint64_t>> blocks;
    uint64_t live = 0, peak = 0;
    ~Scratch() { for (auto& b : blocks) cudaFree(b.first); }
    template <class T>
    cudaError_t get(T*& p, uint64_t count) {
        const uint64_t bytes = std::max<uint64_t>(count * sizeof(T), 16);
        void* raw = nullptr;
        const cudaError_t e = cudaMalloc(&raw, bytes);
        p = static_cast<T*>(raw);
        if (e != cudaSuccess) return e;
        blocks.emplace_back(raw, bytes);
        live += bytes;
        peak = std::max(peak, live);
        return cudaSuccess;
    }
    void drop(const void* p) {
        if (p == nullptr) return;
        for (size_t i = 0; i < blocks.size(); i++) {
            if (blocks[i].first != p) continue;
            cudaFree(blocks[i].first);
            live -= blocks[i].second;
            blocks.erase(blocks.begin() + static_cast<std::ptrdiff_t>(i));
            return;
        }
    }
};

int bits_for(uint64_t v) {  // bits needed for every value below v
    int b = 0;
    while (b < 64 && (v - 1) >> b) b++;
    return std::max(b, 1);
}

int status_of(uint32_t flags, std::string& err) {
    if (flags & BAD_OFFSETS) { err = "offsets decrease"; return GBWT_B200_E_ARGUMENT; }
    if (flags & BAD_NODE) { err = "node 0, or node 1 in a bidirectional build (its flip is the endmarker)"; return GBWT_B200_E_ARGUMENT; }
    if (flags & NODE_RANGE) { err = "a node does not fit 32 bits"; return GBWT_B200_E_RANGE; }
    return GBWT_B200_OK;
}

}  // namespace

int build_check_sizes(uint64_t paths, uint64_t path_nodes, bool bidirectional, std::string& err) {
    const uint64_t limit = uint64_t(1) << 32;
    if (paths >= limit || path_nodes >= limit || (paths + path_nodes) * (bidirectional ? 2 : 1) >= limit) {
        err = "nodes + sequences must be below 2^32";
        return GBWT_B200_E_RANGE;
    }
    return GBWT_B200_OK;
}

int build_check_paths(const uint64_t* nodes, const uint64_t* offsets, uint64_t n, bool bidirectional, uint64_t& records, std::string& err) {
    uint32_t flags = 0;
    for (uint64_t q = 0; q < n; q++) if (offsets[q + 1] < offsets[q]) flags |= BAD_OFFSETS;
    if (int rc = status_of(flags, err)) return rc;
    if (int rc = build_check_sizes(n, offsets[n] - offsets[0], bidirectional, err)) return rc;
    if (offsets[n] > offsets[0] && nodes == nullptr) { err = "null nodes"; return GBWT_B200_E_ARGUMENT; }
    uint64_t lo = ~0ull, hi = 0;
    for (uint64_t i = offsets[0]; i < offsets[n]; i++) {
        const uint64_t v = nodes[i];
        if (v == 0 || (bidirectional && v == 1)) flags |= BAD_NODE;
        if (v >> 32) flags |= NODE_RANGE;
        lo = std::min(lo, bidirectional ? v & ~uint64_t(1) : v);
        hi = std::max(hi, bidirectional ? v | uint64_t(1) : v);
    }
    records = offsets[n] > offsets[0] ? hi - lo + 2 : 1;
    return status_of(flags, err);
}

uint64_t build_device_bytes(uint64_t paths, uint64_t path_nodes, bool bidirectional, uint64_t records) {
    const uint64_t scale = bidirectional ? 2 : 1, positions = scale * path_nodes, entries = scale * paths + positions;
    return 36 * entries + 28 * (records + 1) + (uint64_t(64) << 20);
}

int build_gbwt_image(const uint64_t* d_nodes, const uint64_t* d_offsets, uint64_t n, bool bidirectional, uint64_t extra_bytes,
                     cudaStream_t s, std::vector<uint8_t>& image, uint64_t* info, std::string& err) {
    cudaError_t ce = cudaSuccess;
#define BUILD_TRY(expr)                                                                              \
    do {                                                                                             \
        ce = (expr);                                                                                 \
        if (ce != cudaSuccess) { err = std::string(#expr) + ": " + cudaGetErrorString(ce); return GBWT_B200_E_CUDA; } \
    } while (0)
    int device = 0, sm_count = 0;
    BUILD_TRY(cudaGetDevice(&device));
    BUILD_TRY(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, device));
    Scratch scratch;
    const auto t0 = std::chrono::steady_clock::now();

    // ---- checks, read back before any working memory is taken ----
    BuildStats* d_stats = nullptr;
    BUILD_TRY(scratch.get(d_stats, 1));
    BuildStats h_stats{0, 0xFFFFFFFFu, 0, 0, 0};
    uint64_t ends[2] = {0, 0};
    BUILD_TRY(cudaMemcpyAsync(d_stats, &h_stats, sizeof(BuildStats), cudaMemcpyHostToDevice, s));
    k_build_check_offsets<<<grid_of(n, sm_count), BUILD_THREADS, 0, s>>>(d_offsets, n, d_stats);
    BUILD_TRY(cudaGetLastError());
    BUILD_TRY(cudaMemcpyAsync(&h_stats, d_stats, sizeof(BuildStats), cudaMemcpyDeviceToHost, s));
    BUILD_TRY(cudaMemcpyAsync(&ends[0], d_offsets, 8, cudaMemcpyDeviceToHost, s));
    BUILD_TRY(cudaMemcpyAsync(&ends[1], d_offsets + n, 8, cudaMemcpyDeviceToHost, s));
    BUILD_TRY(cudaStreamSynchronize(s));
    if (int rc = status_of(h_stats.flags, err)) return rc;
    const uint64_t path_nodes = ends[1] - ends[0];
    if (int rc = build_check_sizes(n, path_nodes, bidirectional, err)) return rc;
    if (path_nodes > 0) {
        k_build_check_nodes<<<grid_of(path_nodes, sm_count), BUILD_THREADS, 0, s>>>(d_nodes + ends[0], path_nodes, bidirectional, d_stats);
        BUILD_TRY(cudaGetLastError());
        BUILD_TRY(cudaMemcpyAsync(&h_stats, d_stats, sizeof(BuildStats), cudaMemcpyDeviceToHost, s));
        BUILD_TRY(cudaStreamSynchronize(s));
        if (int rc = status_of(h_stats.flags, err)) return rc;
    }
    const uint64_t N = bidirectional ? 2 * n : n, T = bidirectional ? 2 * path_nodes : path_nodes, M = N + T;
    const uint64_t offset = T > 0 ? h_stats.min_node - 1 : 0, alphabet_size = T > 0 ? uint64_t(h_stats.max_node) + 1 : 1;
    const uint64_t records = alphabet_size - offset;
    const int bits = bits_for(M);
    size_t sort_bytes = 0, scan_bytes = 0;
    if (T > 0) {
        cub::DoubleBuffer<uint64_t> kb(nullptr, nullptr);
        cub::DoubleBuffer<uint32_t> pb(nullptr, nullptr);
        BUILD_TRY(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, kb, pb, static_cast<uint32_t>(T), 0, 2 * bits, s));
        BUILD_TRY(cub::DeviceScan::InclusiveSum(nullptr, scan_bytes, pb.Current(), pb.Current(), static_cast<int64_t>(T), s));
    }
    const size_t temp_bytes = std::max(sort_bytes, scan_bytes);
    {
        size_t free_bytes = 0, total_bytes = 0;
        BUILD_TRY(cudaMemGetInfo(&free_bytes, &total_bytes));
        const uint64_t need = build_device_bytes(n, path_nodes, bidirectional, records) + temp_bytes;
        if (need > free_bytes) {
            err = "the build needs about " + std::to_string(need) + " bytes of device memory; " + std::to_string(free_bytes) + " are free";
            return GBWT_B200_E_CUDA;
        }
    }

    // ---- prefix doubling over the T positions ----
    uint32_t* order = nullptr;  // the final order of the positions
    uint32_t *sym = nullptr, *seq = nullptr;
    uint64_t rounds = 0;
    if (T > 0) {
        uint32_t *rank = nullptr, *pos[2] = {nullptr, nullptr};
        uint64_t* keys[2] = {nullptr, nullptr};
        BUILD_TRY(scratch.get(sym, T));
        BUILD_TRY(scratch.get(seq, T));
        BUILD_TRY(scratch.get(rank, T));
        for (int b = 0; b < 2; b++) { BUILD_TRY(scratch.get(keys[b], T)); BUILD_TRY(scratch.get(pos[b], T)); }
        cub::DoubleBuffer<uint64_t> kb(keys[0], keys[1]);
        cub::DoubleBuffer<uint32_t> pb(pos[0], pos[1]);
        uint8_t* temp = nullptr;
        BUILD_TRY(scratch.get(temp, temp_bytes));
        k_build_expand<<<grid_of(path_nodes, sm_count), BUILD_THREADS, 0, s>>>(d_nodes, d_offsets, n, path_nodes, bidirectional, sym, seq);
        BUILD_TRY(cudaGetLastError());
        const unsigned grid = grid_of(T, sm_count);
        for (uint64_t h = 0;; h = h == 0 ? 1 : 2 * h) {
            if (h == 0) k_build_symbol_keys<<<grid, BUILD_THREADS, 0, s>>>(sym, T, kb.Current(), pb.Current());
            else k_build_keys<<<grid, BUILD_THREADS, 0, s>>>(rank, seq, T, h, bits, kb.Current(), pb.Current());
            BUILD_TRY(cudaGetLastError());
            size_t tb = temp_bytes;
            BUILD_TRY(cub::DeviceRadixSort::SortPairs(temp, tb, kb, pb, static_cast<uint32_t>(T), 0,
                                                      h == 0 ? bits_for(uint64_t(h_stats.max_node) + 1) : 2 * bits, s));
            uint32_t* group = pb.Alternate();
            k_build_group_heads<<<grid, BUILD_THREADS, 0, s>>>(kb.Current(), T, group);
            BUILD_TRY(cudaGetLastError());
            tb = temp_bytes;
            BUILD_TRY(cub::DeviceScan::InclusiveSum(temp, tb, group, group, static_cast<int64_t>(T), s));
            k_build_ranks<<<grid, BUILD_THREADS, 0, s>>>(pb.Current(), group, T, N, rank);
            BUILD_TRY(cudaGetLastError());
            uint32_t groups = 0;
            BUILD_TRY(cudaMemcpyAsync(&groups, group + T - 1, 4, cudaMemcpyDeviceToHost, s));
            BUILD_TRY(cudaStreamSynchronize(s));
            if (h > 0) rounds++;
            if (groups == T) break;
        }
        order = pb.Current();
        scratch.drop(temp); scratch.drop(rank); scratch.drop(pb.Alternate());
        scratch.drop(keys[0]); scratch.drop(keys[1]);
    }

    // ---- entries, records, edges ----
    uint32_t *rec = nullptr, *value = nullptr, *pred = nullptr, *rec_first = nullptr;
    BUILD_TRY(scratch.get(rec, M));
    BUILD_TRY(scratch.get(value, M));
    BUILD_TRY(scratch.get(pred, M));
    BUILD_TRY(scratch.get(rec_first, records + 1));
    const unsigned grid = grid_of(M, sm_count);
    k_build_entries<<<grid, BUILD_THREADS, 0, s>>>(order, sym, seq, d_offsets, N, T, bidirectional, offset, rec, value, pred);
    BUILD_TRY(cudaGetLastError());
    scratch.drop(order); scratch.drop(sym); scratch.drop(seq);
    k_build_record_firsts<<<grid_of(records + 1, sm_count), BUILD_THREADS, 0, s>>>(rec, M, 0, records + 1, rec_first);
    BUILD_TRY(cudaGetLastError());
    BUILD_TRY(cudaMemsetAsync(&d_stats->count, 0, 8, s));
    k_build_edges<<<grid, BUILD_THREADS, 0, s>>>(rec, value, pred, rec_first, N, M, offset, d_stats, nullptr, nullptr);
    BUILD_TRY(cudaGetLastError());
    unsigned long long raw_edges = 0;
    BUILD_TRY(cudaMemcpyAsync(&raw_edges, &d_stats->count, 8, cudaMemcpyDeviceToHost, s));
    BUILD_TRY(cudaStreamSynchronize(s));
    uint64_t* ekeys[2] = {nullptr, nullptr};
    uint32_t* eoffs[2] = {nullptr, nullptr};
    for (int b = 0; b < 2; b++) { BUILD_TRY(scratch.get(ekeys[b], raw_edges)); BUILD_TRY(scratch.get(eoffs[b], raw_edges)); }
    BUILD_TRY(cudaMemsetAsync(&d_stats->count, 0, 8, s));
    k_build_edges<<<grid, BUILD_THREADS, 0, s>>>(rec, value, pred, rec_first, N, M, offset, d_stats, ekeys[0], eoffs[0]);
    BUILD_TRY(cudaGetLastError());
    uint64_t edges = 0;
    uint64_t* edge_keys = nullptr;
    uint32_t* edge_offs = nullptr;
    {
        cub::DoubleBuffer<uint64_t> kb(ekeys[0], ekeys[1]);
        cub::DoubleBuffer<uint32_t> ob(eoffs[0], eoffs[1]);
        unsigned long long* d_selected = &d_stats->count;
        size_t sort_bytes = 0, unique_bytes = 0;
        const int end_bit = 32 + bits_for(records);
        BUILD_TRY(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, kb, ob, static_cast<uint32_t>(raw_edges), 0, end_bit, s));
        BUILD_TRY(cub::DeviceSelect::UniqueByKey(nullptr, unique_bytes, kb.Current(), ob.Current(), kb.Alternate(), ob.Alternate(), d_selected,
                                                 static_cast<int64_t>(raw_edges), s));
        uint8_t* temp = nullptr;
        const size_t temp_bytes = std::max(sort_bytes, unique_bytes);
        BUILD_TRY(scratch.get(temp, temp_bytes));
        size_t tb = temp_bytes;
        BUILD_TRY(cub::DeviceRadixSort::SortPairs(temp, tb, kb, ob, static_cast<uint32_t>(raw_edges), 0, end_bit, s));
        tb = temp_bytes;
        BUILD_TRY(cub::DeviceSelect::UniqueByKey(temp, tb, kb.Current(), ob.Current(), kb.Alternate(), ob.Alternate(), d_selected,
                                                 static_cast<int64_t>(raw_edges), s));
        unsigned long long selected = 0;
        BUILD_TRY(cudaMemcpyAsync(&selected, d_selected, 8, cudaMemcpyDeviceToHost, s));
        BUILD_TRY(cudaStreamSynchronize(s));
        edges = selected;
        edge_keys = kb.Alternate(); edge_offs = ob.Alternate();
        scratch.drop(temp); scratch.drop(kb.Current()); scratch.drop(ob.Current());
    }
    uint32_t* edge_first = nullptr;
    BUILD_TRY(scratch.get(edge_first, records + 1));
    k_build_record_firsts<<<grid_of(records + 1, sm_count), BUILD_THREADS, 0, s>>>(edge_keys, edges, 32, records + 1, edge_first);
    BUILD_TRY(cudaGetLastError());
    k_build_values<<<grid, BUILD_THREADS, 0, s>>>(rec, value, M, edge_first, edge_keys);
    BUILD_TRY(cudaGetLastError());

    // ---- runs and bytes ----
    uint32_t* heads = pred;  // the predecessors are done with
    k_build_run_heads<<<grid, BUILD_THREADS, 0, s>>>(rec, value, M, heads);
    BUILD_TRY(cudaGetLastError());
    uint64_t runs = 0;
    uint32_t* run_start = nullptr;
    uint64_t *run_off = nullptr, *rec_start = nullptr, *run_base = nullptr;
    {
        size_t temp_bytes = 0;
        BUILD_TRY(cub::DeviceScan::InclusiveSum(nullptr, temp_bytes, heads, heads, static_cast<int64_t>(M), s));
        uint8_t* temp = nullptr;
        BUILD_TRY(scratch.get(temp, temp_bytes));
        BUILD_TRY(cub::DeviceScan::InclusiveSum(temp, temp_bytes, heads, heads, static_cast<int64_t>(M), s));
        uint32_t h_runs = 0;
        BUILD_TRY(cudaMemcpyAsync(&h_runs, heads + M - 1, 4, cudaMemcpyDeviceToHost, s));
        BUILD_TRY(cudaStreamSynchronize(s));
        scratch.drop(temp);
        runs = h_runs;
        BUILD_TRY(scratch.get(run_start, runs + 1));
        k_build_run_starts<<<grid, BUILD_THREADS, 0, s>>>(rec, value, heads, M, run_start);
        BUILD_TRY(cudaGetLastError());
        scratch.drop(pred);
    }
    BUILD_TRY(scratch.get(run_off, runs + 1));
    BUILD_TRY(scratch.get(rec_start, records + 1));
    k_build_run_bytes<<<grid_of(runs + 1, sm_count), BUILD_THREADS, 0, s>>>(run_start, runs, rec, value, edge_first, run_off);
    BUILD_TRY(cudaGetLastError());
    {
        size_t a = 0, b = 0;
        BUILD_TRY(cub::DeviceScan::ExclusiveSum(nullptr, a, run_off, run_off, static_cast<int64_t>(runs + 1), s));
        BUILD_TRY(cub::DeviceScan::ExclusiveSum(nullptr, b, rec_start, rec_start, static_cast<int64_t>(records + 1), s));
        uint8_t* temp = nullptr;
        const size_t temp_bytes = std::max(a, b);
        BUILD_TRY(scratch.get(temp, temp_bytes));
        size_t tb = temp_bytes;
        BUILD_TRY(cub::DeviceScan::ExclusiveSum(temp, tb, run_off, run_off, static_cast<int64_t>(runs + 1), s));
        k_build_record_bytes<<<grid_of(records + 1, sm_count), BUILD_THREADS, 0, s>>>(records, rec_first, run_start, runs, run_off, edge_first,
                                                                                     edge_keys, edge_offs, rec_start);
        BUILD_TRY(cudaGetLastError());
        tb = temp_bytes;
        BUILD_TRY(cub::DeviceScan::ExclusiveSum(temp, tb, rec_start, rec_start, static_cast<int64_t>(records + 1), s));
        scratch.drop(temp);
    }
    uint64_t data_len = 0;
    BUILD_TRY(cudaMemcpyAsync(&data_len, rec_start + records, 8, cudaMemcpyDeviceToHost, s));
    BUILD_TRY(cudaStreamSynchronize(s));
    uint8_t* data = nullptr;
    BUILD_TRY(scratch.get(data, data_len));
    BUILD_TRY(scratch.get(run_base, records));
    k_build_write_records<<<grid_of(records, sm_count), BUILD_THREADS, 0, s>>>(records, rec_start, rec_first, run_start, runs, run_off, edge_first,
                                                                              edge_keys, edge_offs, data, run_base);
    BUILD_TRY(cudaGetLastError());
    k_build_write_runs<<<grid_of(runs, sm_count), BUILD_THREADS, 0, s>>>(run_start, runs, rec, value, edge_first, run_off, run_base, data);
    BUILD_TRY(cudaGetLastError());
    std::vector<uint8_t> h_data(data_len);
    std::vector<uint64_t> h_starts(records);
    if (data_len > 0) BUILD_TRY(cudaMemcpyAsync(h_data.data(), data, data_len, cudaMemcpyDeviceToHost, s));
    BUILD_TRY(cudaMemcpyAsync(h_starts.data(), rec_start, records * 8, cudaMemcpyDeviceToHost, s));
    BUILD_TRY(cudaStreamSynchronize(s));
    const uint64_t device_us = std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
#undef BUILD_TRY

    GBWTHeaderFields header;
    header.sequences = N; header.size = M; header.offset = offset; header.alphabet_size = alphabet_size;
    header.flags = bidirectional ? 1 : 0;
    write_gbwt_image(header, h_data.data(), data_len, h_starts, Carried{}, image);
    if (info != nullptr) { info[0] = M; info[1] = rounds; info[2] = device_us; info[3] = scratch.peak + extra_bytes; }
    return GBWT_B200_OK;
}

}  // namespace gbwt_b200
