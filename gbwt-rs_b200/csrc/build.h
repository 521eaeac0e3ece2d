// build.h -- the GBWT of a set of paths, built on the device (build.cu; gbwt_b200_build_image in gbwt_b200_build.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <functional>
#include <string>
#include <utility>
#include <vector>

namespace gbwt_b200 {

// The statuses of build_gbwt_image from host arrays (offsets absolute, n >= 1), before anything is copied; on success
// `records` = the number of records of the GBWT.
int build_check_paths(const uint64_t* nodes, const uint64_t* offsets, uint64_t n, bool bidirectional, uint64_t& records, std::string& err);
// Device memory a build of `paths` paths with `path_nodes` nodes in all takes, without the sort's temporary storage:
// about 36 bytes per position (nodes + sequences) and 28 per record.
uint64_t build_device_bytes(uint64_t paths, uint64_t path_nodes, bool bidirectional, uint64_t records);

// Path q = d_nodes[d_offsets[q] .. d_offsets[q+1]), q < n, read on stream s of the current device. With `bidirectional`,
// sequence 2q = path q and 2q+1 = its reverse with every node flipped; otherwise sequence q = path q. On success `image`
// is the Simple-SDS GBWT file of the sequences. `extra_bytes`: device memory the caller already holds for the inputs,
// counted into info[3]. info (may be null): positions sorted, doubling rounds, device microseconds, peak device bytes.
// Returns a GBWT_B200_* status; `err` says why when it is not OK. Everything allocated here is freed before it returns.
int build_gbwt_image(const uint64_t* d_nodes, const uint64_t* d_offsets, uint64_t n, bool bidirectional, uint64_t extra_bytes,
                     cudaStream_t s, std::vector<uint8_t>& image, uint64_t* info, std::string& err);

// ---- the phases of build_gbwt_image, shared with the insertion (insert.cu) ----------------------------------------

// Device scratch with a byte count: every block is freed when the scratch goes out of scope.
struct Scratch {
    std::vector<std::pair<void*, uint64_t>> blocks;
    uint64_t live = 0, peak = 0;
    Scratch() = default;
    Scratch(const Scratch&) = delete;
    Scratch& operator=(const Scratch&) = delete;
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

// Sequence s: its first position in the expanded array (sym / seq of SortedPaths) and its length.
struct SeqSpan { uint64_t start, len; };
__device__ __forceinline__ SeqSpan seq_span(const uint64_t* __restrict__ offsets, uint64_t s, bool bidirectional) {
    const uint64_t q = bidirectional ? s >> 1 : s, base = offsets[0];
    const uint64_t lo = offsets[q] - base, len = offsets[q + 1] - offsets[q];
    if (!bidirectional) return {lo, len};
    return {2 * lo + (s & 1) * len, len};
}

struct SortedPaths;
// Device memory a caller needs beside the build's own, counted into the check against free memory that build_sort makes
// before its first working allocation; `bytes` sees the sizes and header fields of the paths (may be empty).
struct ExtraNeed {
    const char* what = "build";
    std::function<uint64_t(const SortedPaths&)> bytes;
};

// Phase 1: the checks and the prefix doubling. N sequences, T positions, M = N + T entries; the header fields of the
// paths' own GBWT. order[i] = the position of entry N + i; sym / seq = symbol and sequence of every position; with
// keep_rank, rank[p] = the entry of position p (the caller drops it).
struct SortedPaths {
    uint64_t n = 0, path_nodes = 0, N = 0, T = 0, M = 0, offset = 0, alphabet_size = 1, records = 1, rounds = 0;
    bool bidirectional = false;
    uint32_t *order = nullptr, *sym = nullptr, *seq = nullptr, *rank = nullptr;
};
// Phase 2: per entry its record, edge rank (value) and predecessor node (0 = the endmarker); rec_first[r] = first entry of
// record r; the edges (from record << 32 | to node, offset), sorted, edge_first[r] = first edge of record r. Drops order /
// sym / seq.
struct BuiltEdges {
    uint32_t *rec = nullptr, *value = nullptr, *pred = nullptr, *rec_first = nullptr, *edge_first = nullptr, *edge_offs = nullptr;
    uint64_t* edge_keys = nullptr;
    uint64_t edges = 0;
};

int build_check_sizes(uint64_t paths, uint64_t path_nodes, bool bidirectional, std::string& err);
int device_sm_count(int& sm_count, std::string& err);
int build_sort(const uint64_t* d_nodes, const uint64_t* d_offsets, uint64_t n, bool bidirectional, const ExtraNeed& extra, bool keep_rank,
               int sm_count, cudaStream_t s, Scratch& scratch, SortedPaths& sp, std::string& err);
int build_entries_edges(SortedPaths& sp, const uint64_t* d_offsets, int sm_count, cudaStream_t s, Scratch& scratch, BuiltEdges& be,
                        std::string& err);
// Phase 3: maximal runs and record bytes; the records and their starts on the host. Drops pred.
int build_write_records(const SortedPaths& sp, BuiltEdges& be, int sm_count, cudaStream_t s, Scratch& scratch, std::vector<uint8_t>& data,
                        std::vector<uint64_t>& starts, std::string& err);

}  // namespace gbwt_b200
