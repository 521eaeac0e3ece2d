// insert.cu -- new paths inserted into a loaded GBWT on the device (gbwt_b200_insert_image, include/gbwt_b200_insert.h).
//
// The result is the GBWT of (A's sequences, then the new sequences S), written without expanding A's records:
//   1. S alone goes through the build's checks and prefix doubling (build.cu). That gives, for every entry e of S in
//      record w, beta(e) = its index among the S entries of w, and rank[p] = the entry of position p.
//   2. alpha(e) = the A entries of w that sort before e, from a walk along each new sequence with one lane per sequence
//      (insert_step.h). The walk reads A's records in place and a table of A's incoming edges, sorted here.
//   3. Merged record w: S entry e goes to alpha(e) + beta(e), A's entry i to i + #{S entries e of w : alpha(e) <= i}.
//      Edges are the union of A's and S's successors; the offset of w -> v is before_A(v, w) + before_S(v, w) (0 for the
//      endmarker). One thread per merged record merges the entries of S into the runs of A's body, read in place
//      (for_each_run, record_encode.h), and counts or writes the record with maximal runs.
// Device memory beside A's layout: the build's 36 bytes per S position, about 36 bytes per A edge (the incoming-edge table
// with its sort buffers and the map of A's edge ranks), 4 bytes per S entry for alpha, a few words per merged record,
// and the output bytes. Nothing is proportional to A's length or its run count.
#include "insert.h"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <chrono>

#include "../../include/gbwt_b200.h"
#include "build.h"
#include "insert_step.h"
#include "layout_writer.h"
#include "record_encode.h"

namespace gbwt_b200 {

namespace {

constexpr int INSERT_THREADS = 256;
constexpr uint32_t RECORD_RANGE = 1;

unsigned grid_of(uint64_t n, int sm_count) {
    const uint64_t blocks = (n + INSERT_THREADS - 1) / INSERT_THREADS;
    const uint64_t wave = static_cast<uint64_t>(std::max(1, sm_count)) * (2048 / INSERT_THREADS);
    return static_cast<unsigned>(std::max<uint64_t>(1, std::min(blocks, wave)));
}

__device__ __forceinline__ uint64_t stride() { return static_cast<uint64_t>(gridDim.x) * blockDim.x; }
__device__ __forceinline__ uint64_t first_index() { return blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; }

// What the build of S left: per entry its edge rank (value), predecessor node and alpha; records and edges as in
// BuiltEdges (build.h).
struct SView {
    const uint32_t *value, *pred, *alpha, *rec_first, *edge_first, *edge_offs;
    const uint64_t* edge_keys;
    uint64_t offset, records;
};

// Where the records of node w lie in the result, in A and in S.
struct Geometry {
    uint64_t offset, records;  // of the result
};

__device__ __forceinline__ bool s_record(const SView& sv, uint64_t w, uint64_t& r) {
    if (w != 0 && (w <= sv.offset || w - sv.offset >= sv.records)) return false;
    r = w == 0 ? 0 : w - sv.offset;
    return sv.rec_first[r + 1] > sv.rec_first[r];
}

// before_S(v, w): S's entries of record v whose predecessor is below w (entries are sorted by predecessor first).
__device__ __forceinline__ uint64_t before_s(const SView& sv, uint64_t v, uint64_t w) {
    uint64_t r;
    if (!s_record(sv, v, r)) return 0;
    uint64_t lo = sv.rec_first[r], hi = sv.rec_first[r + 1];
    const uint64_t first = lo;
    while (lo < hi) {
        const uint64_t mid = lo + (hi - lo) / 2;
        if (sv.pred[mid] < w) lo = mid + 1; else hi = mid;
    }
    return lo - first;
}

__device__ __forceinline__ uint64_t node_of(const Geometry& g, uint64_t r) { return r == 0 ? 0 : r + g.offset; }

// ---- A's incoming edges ----

__global__ void __launch_bounds__(INSERT_THREADS) k_insert_a_degree(IndexView ix, uint32_t* __restrict__ degree) {
    for (uint64_t r = first_index(); r <= ix.records; r += stride()) {
        if (r == ix.records) { degree[r] = 0; continue; }
        const Desc d = load_desc(ix, r);
        degree[r] = d.fmt() == FMT_EMPTY ? 0 : d.sigma();
    }
}

__global__ void __launch_bounds__(INSERT_THREADS) k_insert_a_edges(IndexView ix, const uint32_t* __restrict__ a_first,
                                                                   uint64_t* __restrict__ keys, uint32_t* __restrict__ offs) {
    for (uint64_t r = first_index(); r < ix.records; r += stride()) {
        const Desc d = load_desc(ix, r);
        if (d.fmt() == FMT_EMPTY) continue;
        const uint64_t u = r == 0 ? 0 : r + ix.offset, base = a_first[r];
        for (uint32_t k = 0; k < d.sigma(); k++) {
            const Edge e = edge_at(ix, d, k);
            keys[base + k] = (static_cast<uint64_t>(e.node) << 32) | u;
            offs[base + k] = e.offset;
        }
    }
}

// ---- the walk: alpha of every S entry, one lane per new sequence ----

__global__ void __launch_bounds__(INSERT_THREADS) k_insert_walk(IndexView ix, InEdges in, const uint64_t* __restrict__ offsets,
                                                                uint64_t sequences, bool bidirectional, const uint32_t* __restrict__ sym,
                                                                const uint32_t* __restrict__ rank, uint32_t* __restrict__ alpha,
                                                                unsigned long long* __restrict__ longest) {
    for (uint64_t s = first_index(); s < sequences; s += stride()) {
        alpha[s] = static_cast<uint32_t>(ix.sequences);
        const SeqSpan sp = seq_span(offsets, s, bidirectional);
        uint64_t w = 0, a = ix.sequences;
        for (uint64_t k = 0; k < sp.len; k++) {
            const uint64_t p = sp.start + k, v = sym[p];
            a = insert_step(ix, in, w, a, v);
            alpha[rank[p]] = static_cast<uint32_t>(a);
            w = v;
        }
        atomicMax(longest, static_cast<unsigned long long>(sp.len));
    }
}

// ---- merged edges ----

// The edges of merged record r (node w) in node order: counts them, or writes them with their offsets and the merged
// rank of every edge of A (amap, at A's edge index) and of S (smap, at S's edge index).
template <bool WRITE>
__device__ uint32_t merge_edges(const IndexView& ix, const InEdges& in, const uint32_t* __restrict__ a_first, const SView& sv, uint64_t w,
                                Edge* __restrict__ out, uint32_t* __restrict__ amap, uint32_t* __restrict__ smap) {
    Desc da;
    const bool has_a = insert_record(ix, w, da);
    uint64_t rs = 0;
    const bool has_s = s_record(sv, w, rs);
    const uint32_t na = has_a ? da.sigma() : 0;
    const uint64_t sb = has_s ? sv.edge_first[rs] : 0, ns = has_s ? sv.edge_first[rs + 1] - sb : 0;
    const uint64_t ab = has_a ? a_first[w == 0 ? 0 : w - ix.offset] : 0;
    uint32_t i = 0, k = 0;
    uint64_t j = 0;
    while (i < na || j < ns) {
        Edge ea{0xFFFFFFFFu, 0};
        if (i < na) ea = edge_at(ix, da, i);
        const uint64_t vs = j < ns ? (sv.edge_keys[sb + j] & 0xFFFFFFFFull) : ~0ull;
        const uint64_t v = i < na && ea.node < vs ? static_cast<uint64_t>(ea.node) : vs;
        const bool in_a = i < na && ea.node == v, in_s = j < ns && vs == v;
        if (WRITE) {
            uint64_t off = 0;
            if (v != 0) off = (in_a ? ea.offset : insert_before(ix, in, v, w)) + (in_s ? sv.edge_offs[sb + j] : before_s(sv, v, w));
            out[k] = Edge{static_cast<uint32_t>(v), static_cast<uint32_t>(off)};
            if (in_a) amap[ab + i] = k;
            if (in_s) smap[sb + j] = k;
        }
        i += in_a; j += in_s; k++;
    }
    return k;
}

// Outdegree of every merged record (degree[records] = 0); flags a record of 2^32 positions or more.
__global__ void __launch_bounds__(INSERT_THREADS) k_insert_edge_count(IndexView ix, InEdges in, const uint32_t* __restrict__ a_first, SView sv,
                                                                      Geometry g, uint32_t* __restrict__ degree, uint32_t* __restrict__ flags) {
    for (uint64_t r = first_index(); r <= g.records; r += stride()) {
        if (r == g.records) { degree[r] = 0; continue; }
        const uint64_t w = node_of(g, r);
        degree[r] = merge_edges<false>(ix, in, a_first, sv, w, nullptr, nullptr, nullptr);
        Desc da;
        uint64_t rs = 0, len = 0;
        if (insert_record(ix, w, da)) len += da.total_len();
        if (s_record(sv, w, rs)) len += sv.rec_first[rs + 1] - sv.rec_first[rs];
        if (len >> 32) atomicOr(flags, RECORD_RANGE);
    }
}

__global__ void __launch_bounds__(INSERT_THREADS) k_insert_edge_write(IndexView ix, InEdges in, const uint32_t* __restrict__ a_first, SView sv,
                                                                      Geometry g, const uint32_t* __restrict__ m_first, Edge* __restrict__ edges,
                                                                      uint32_t* __restrict__ amap, uint32_t* __restrict__ smap) {
    for (uint64_t r = first_index(); r < g.records; r += stride())
        merge_edges<true>(ix, in, a_first, sv, node_of(g, r), edges + m_first[r], amap, smap);
}

// ---- merged records ----

// Merged record r in the encoding of BWTBuilder::append: the merged edges, then maximal runs of A's body (read in place)
// with the S entries placed among them.
__device__ void put_merged_record(ByteSink& out, const IndexView& ix, const uint32_t* __restrict__ a_first, const SView& sv, const Geometry& g,
                                  const uint32_t* __restrict__ m_first, const Edge* __restrict__ edges, const uint32_t* __restrict__ amap,
                                  const uint32_t* __restrict__ smap, uint64_t r) {
    const uint64_t lo = m_first[r], sigma = m_first[r + 1] - lo;
    put_edges(out, sigma, [&](uint64_t e) { return EdgeValue{edges[lo + e].node, edges[lo + e].offset}; });
    if (sigma == 0) return;
    const uint64_t w = node_of(g, r);
    uint64_t rs = 0, j = 0, s_end = 0;
    if (s_record(sv, w, rs)) { j = sv.rec_first[rs]; s_end = sv.rec_first[rs + 1]; }
    const uint64_t sb = s_end > j ? sv.edge_first[rs] : 0;
    uint64_t run_value = 0, run_len = 0, i = 0;
    auto emit = [&](uint64_t value, uint64_t len) {
        if (run_len > 0 && value != run_value) { put_run(out, sigma, run_value, run_len); run_len = 0; }
        run_value = value; run_len += len;
    };
    Desc da;
    if (insert_record(ix, w, da)) {
        const uint64_t ra = w == 0 ? 0 : w - ix.offset, ab = a_first[ra];
        const RecordDesc d = ix.desc[ra];
        for_each_run(d, ix.bodies, [&](uint64_t value, uint64_t len) {
            const uint64_t mv = amap[ab + value];
            while (len > 0) {
                while (j < s_end && sv.alpha[j] <= i) { emit(smap[sb + sv.value[j]], 1); j++; }
                const uint64_t gap = j < s_end ? sv.alpha[j] - i : len, take = gap < len ? gap : len;
                emit(mv, take);
                i += take; len -= take;
            }
        });
    }
    for (; j < s_end; j++) emit(smap[sb + sv.value[j]], 1);
    if (run_len > 0) put_run(out, sigma, run_value, run_len);
}

__global__ void __launch_bounds__(INSERT_THREADS) k_insert_record_bytes(IndexView ix, const uint32_t* __restrict__ a_first, SView sv, Geometry g,
                                                                        const uint32_t* __restrict__ m_first, const Edge* __restrict__ edges,
                                                                        const uint32_t* __restrict__ amap, const uint32_t* __restrict__ smap,
                                                                        uint64_t* __restrict__ bytes) {
    for (uint64_t r = first_index(); r <= g.records; r += stride()) {
        if (r == g.records) { bytes[r] = 0; continue; }
        ByteSink count;
        put_merged_record(count, ix, a_first, sv, g, m_first, edges, amap, smap, r);
        bytes[r] = count.n;
    }
}

__global__ void __launch_bounds__(INSERT_THREADS) k_insert_write_records(IndexView ix, const uint32_t* __restrict__ a_first, SView sv, Geometry g,
                                                                         const uint32_t* __restrict__ m_first, const Edge* __restrict__ edges,
                                                                         const uint32_t* __restrict__ amap, const uint32_t* __restrict__ smap,
                                                                         const uint64_t* __restrict__ rec_start, uint8_t* __restrict__ data) {
    for (uint64_t r = first_index(); r < g.records; r += stride()) {
        ByteSink out;
        out.at = data + rec_start[r];
        put_merged_record(out, ix, a_first, sv, g, m_first, edges, amap, smap, r);
    }
}

uint64_t elapsed_us(std::chrono::steady_clock::time_point t0) {
    return std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
}

}  // namespace

int insert_gbwt_image(const InsertTarget& a, const uint64_t* d_nodes, const uint64_t* d_offsets, uint64_t n, uint64_t extra_bytes,
                      cudaStream_t s, std::vector<uint8_t>& image, uint64_t* info, std::string& err) {
#define INSERT_TRY(expr)                                                                             \
    do {                                                                                             \
        const cudaError_t ce_ = (expr);                                                              \
        if (ce_ != cudaSuccess) { err = std::string(#expr) + ": " + cudaGetErrorString(ce_); return GBWT_B200_E_CUDA; } \
    } while (0)
    int sm_count = 0;
    if (int rc = device_sm_count(sm_count, err)) return rc;
    const IndexView& ix = a.view;
    const bool bidirectional = ix.bidirectional != 0;
    const bool a_nodes = ix.records > 1;
    const uint64_t a_edges_bound = a.edges_total + 2 * ix.records;
    Scratch scratch;
    const auto t0 = std::chrono::steady_clock::now();

    // The header of the result from S's own one; A without nodes (all its sequences empty) has no say in it.
    uint64_t offset = 0, alphabet_size = 1;
    auto geometry = [&](const SortedPaths& sp) {
        if (sp.T == 0) { offset = ix.offset; alphabet_size = ix.alphabet_size; }
        else if (!a_nodes) { offset = sp.offset; alphabet_size = sp.alphabet_size; }
        else { offset = std::min(ix.offset, sp.offset); alphabet_size = std::max(ix.alphabet_size, sp.alphabet_size); }
    };
    ExtraNeed extra;
    extra.what = "insertion";
    extra.bytes = [&](const SortedPaths& sp) {
        geometry(sp);
        const uint64_t records = alphabet_size - offset;
        // A's edges: table keys and offsets with their sort buffers, the merged-rank map, the merged edges; alpha per S
        // entry; per merged record its degree and byte offset; the output: A's bodies and a few bytes per S entry.
        return 36 * a_edges_bound + 8 * (ix.records + 1) + 4 * sp.M + 12 * (records + 1) + a.body_bytes + 12 * sp.M + (uint64_t(16) << 20);
    };

    // ---- 1. S alone: checks and prefix doubling ----
    SortedPaths sp;
    if (int rc = build_sort(d_nodes, d_offsets, n, bidirectional, extra, true, sm_count, s, scratch, sp, err)) return rc;
    geometry(sp);
    const uint64_t records = alphabet_size - offset;

    // ---- 2. A's incoming edges, then the walk ----
    uint32_t *a_first = nullptr, *flags = nullptr, *alpha = nullptr;
    unsigned long long* longest = nullptr;
    INSERT_TRY(scratch.get(a_first, ix.records + 1));
    INSERT_TRY(scratch.get(flags, 4));
    INSERT_TRY(scratch.get(longest, 1));
    INSERT_TRY(cudaMemsetAsync(flags, 0, 16, s));
    INSERT_TRY(cudaMemsetAsync(longest, 0, 8, s));
    k_insert_a_degree<<<grid_of(ix.records + 1, sm_count), INSERT_THREADS, 0, s>>>(ix, a_first);
    INSERT_TRY(cudaGetLastError());
    {
        size_t tb = 0;
        INSERT_TRY(cub::DeviceScan::ExclusiveSum(nullptr, tb, a_first, a_first, static_cast<int64_t>(ix.records + 1), s));
        uint8_t* temp = nullptr;
        INSERT_TRY(scratch.get(temp, tb));
        INSERT_TRY(cub::DeviceScan::ExclusiveSum(temp, tb, a_first, a_first, static_cast<int64_t>(ix.records + 1), s));
        scratch.drop(temp);
    }
    uint32_t h_a_edges = 0;
    INSERT_TRY(cudaMemcpyAsync(&h_a_edges, a_first + ix.records, 4, cudaMemcpyDeviceToHost, s));
    INSERT_TRY(cudaStreamSynchronize(s));
    const uint64_t a_edges = h_a_edges;
    InEdges in{nullptr, nullptr, a_edges};
    {
        uint64_t* keys[2] = {nullptr, nullptr};
        uint32_t* offs[2] = {nullptr, nullptr};
        for (int b = 0; b < 2; b++) { INSERT_TRY(scratch.get(keys[b], a_edges)); INSERT_TRY(scratch.get(offs[b], a_edges)); }
        k_insert_a_edges<<<grid_of(ix.records, sm_count), INSERT_THREADS, 0, s>>>(ix, a_first, keys[0], offs[0]);
        INSERT_TRY(cudaGetLastError());
        cub::DoubleBuffer<uint64_t> kb(keys[0], keys[1]);
        cub::DoubleBuffer<uint32_t> ob(offs[0], offs[1]);
        size_t tb = 0;
        INSERT_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tb, kb, ob, static_cast<uint32_t>(a_edges), 0, 64, s));
        uint8_t* temp = nullptr;
        INSERT_TRY(scratch.get(temp, tb));
        INSERT_TRY(cub::DeviceRadixSort::SortPairs(temp, tb, kb, ob, static_cast<uint32_t>(a_edges), 0, 64, s));
        scratch.drop(temp); scratch.drop(kb.Alternate()); scratch.drop(ob.Alternate());
        in.keys = kb.Current(); in.offs = ob.Current();
    }
    INSERT_TRY(scratch.get(alpha, sp.M));
    INSERT_TRY(cudaStreamSynchronize(s));
    const auto t_walk = std::chrono::steady_clock::now();
    k_insert_walk<<<grid_of(sp.N, sm_count), INSERT_THREADS, 0, s>>>(ix, in, d_offsets, sp.N, bidirectional, sp.sym, sp.rank, alpha, longest);
    INSERT_TRY(cudaGetLastError());
    unsigned long long h_longest = 0;
    INSERT_TRY(cudaMemcpyAsync(&h_longest, longest, 8, cudaMemcpyDeviceToHost, s));
    INSERT_TRY(cudaStreamSynchronize(s));
    const uint64_t walk_us = elapsed_us(t_walk);
    scratch.drop(sp.rank);
    sp.rank = nullptr;

    // ---- 3. S's entries and edges, then the merged edges ----
    BuiltEdges be;
    if (int rc = build_entries_edges(sp, d_offsets, sm_count, s, scratch, be, err)) return rc;
    const SView sv{be.value, be.pred, alpha, be.rec_first, be.edge_first, be.edge_offs, be.edge_keys, sp.offset, sp.records};
    const Geometry g{offset, records};
    uint32_t* m_first = nullptr;
    INSERT_TRY(scratch.get(m_first, records + 1));
    k_insert_edge_count<<<grid_of(records + 1, sm_count), INSERT_THREADS, 0, s>>>(ix, in, a_first, sv, g, m_first, flags);
    INSERT_TRY(cudaGetLastError());
    uint32_t h_flags = 0;
    INSERT_TRY(cudaMemcpyAsync(&h_flags, flags, 4, cudaMemcpyDeviceToHost, s));
    INSERT_TRY(cudaStreamSynchronize(s));
    if (h_flags & RECORD_RANGE) { err = "a record of the result would hold 2^32 positions or more"; return GBWT_B200_E_RANGE; }
    {
        size_t tb = 0;
        INSERT_TRY(cub::DeviceScan::ExclusiveSum(nullptr, tb, m_first, m_first, static_cast<int64_t>(records + 1), s));
        uint8_t* temp = nullptr;
        INSERT_TRY(scratch.get(temp, tb));
        INSERT_TRY(cub::DeviceScan::ExclusiveSum(temp, tb, m_first, m_first, static_cast<int64_t>(records + 1), s));
        scratch.drop(temp);
    }
    uint32_t h_m_edges = 0;
    INSERT_TRY(cudaMemcpyAsync(&h_m_edges, m_first + records, 4, cudaMemcpyDeviceToHost, s));
    INSERT_TRY(cudaStreamSynchronize(s));
    Edge* edges = nullptr;
    uint32_t *amap = nullptr, *smap = nullptr;
    INSERT_TRY(scratch.get(edges, h_m_edges));
    INSERT_TRY(scratch.get(amap, a_edges));
    INSERT_TRY(scratch.get(smap, be.edges));
    k_insert_edge_write<<<grid_of(records, sm_count), INSERT_THREADS, 0, s>>>(ix, in, a_first, sv, g, m_first, edges, amap, smap);
    INSERT_TRY(cudaGetLastError());

    // ---- 4. merged records: bytes, offsets, bytes written ----
    uint64_t* rec_start = nullptr;
    INSERT_TRY(scratch.get(rec_start, records + 1));
    k_insert_record_bytes<<<grid_of(records + 1, sm_count), INSERT_THREADS, 0, s>>>(ix, a_first, sv, g, m_first, edges, amap, smap, rec_start);
    INSERT_TRY(cudaGetLastError());
    {
        size_t tb = 0;
        INSERT_TRY(cub::DeviceScan::ExclusiveSum(nullptr, tb, rec_start, rec_start, static_cast<int64_t>(records + 1), s));
        uint8_t* temp = nullptr;
        INSERT_TRY(scratch.get(temp, tb));
        INSERT_TRY(cub::DeviceScan::ExclusiveSum(temp, tb, rec_start, rec_start, static_cast<int64_t>(records + 1), s));
        scratch.drop(temp);
    }
    uint64_t data_len = 0;
    INSERT_TRY(cudaMemcpyAsync(&data_len, rec_start + records, 8, cudaMemcpyDeviceToHost, s));
    INSERT_TRY(cudaStreamSynchronize(s));
    uint8_t* data = nullptr;
    INSERT_TRY(scratch.get(data, data_len));
    k_insert_write_records<<<grid_of(records, sm_count), INSERT_THREADS, 0, s>>>(ix, a_first, sv, g, m_first, edges, amap, smap, rec_start, data);
    INSERT_TRY(cudaGetLastError());
    std::vector<uint8_t> h_data(data_len);
    std::vector<uint64_t> h_starts(records);
    if (data_len > 0) INSERT_TRY(cudaMemcpyAsync(h_data.data(), data, data_len, cudaMemcpyDeviceToHost, s));
    INSERT_TRY(cudaMemcpyAsync(h_starts.data(), rec_start, records * 8, cudaMemcpyDeviceToHost, s));
    INSERT_TRY(cudaStreamSynchronize(s));
    const uint64_t device_us = elapsed_us(t0);
#undef INSERT_TRY

    GBWTHeaderFields header;
    header.sequences = ix.sequences + sp.N; header.size = a.size + sp.M; header.offset = offset; header.alphabet_size = alphabet_size;
    header.flags = bidirectional ? 1 : 0;
    write_gbwt_image(header, h_data.data(), data_len, h_starts, Carried{}, image);
    if (info != nullptr) {
        info[0] = sp.M; info[1] = sp.rounds; info[2] = device_us; info[3] = scratch.peak + extra_bytes;
        info[4] = h_longest; info[5] = walk_us;
    }
    return GBWT_B200_OK;
}

}  // namespace gbwt_b200
