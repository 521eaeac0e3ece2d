// ranges.cu -- gbwt_b200_seek / gbwt_b200_extract_ranges / gbwt_b200_extract_dna_ranges (gbwt_b200_ranges.h): walks that
// start from the path checkpoint (kernels.cuh: k_build_checkpoints) nearest to the node or byte they need, instead of from
// the start of the sequence.
//
// A range is cut at the checkpoints it crosses into pieces, and every piece is one lane's walk: from its checkpoint to
// the next one, storing what falls in the range and in the caller's slot. A per-range piece count and its exclusive scan
// (CUB) give the lanes their work, as in k_locate_states. So no lane walks more than about one interval plus the skip
// from the first piece's checkpoint to the range start, however long the range is.
#include "ranges.h"

#include <cub/device/device_scan.cuh>

#include <algorithm>

#include "record_scan.cuh"

namespace gbwt_b200 {

namespace {

constexpr int RANGE_THREADS = 256;

unsigned grid_of(uint64_t n, int sm_count) {
    const uint64_t blocks = (n + RANGE_THREADS - 1) / RANGE_THREADS;
    const uint64_t wave = static_cast<uint64_t>(std::max(1, sm_count)) * (2048 / RANGE_THREADS);
    return static_cast<unsigned>(std::max<uint64_t>(1, std::min(blocks, wave)));
}

__global__ void __launch_bounds__(RANGE_THREADS) k_seek(IndexView ix, CheckpointView cv, uint32_t shift, const uint64_t* __restrict__ ids,
                                                        const uint64_t* __restrict__ indexes, uint64_t n, gbwt_b200_pos* __restrict__ out) {
    for (uint64_t q = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; q < n; q += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        gbwt_b200_pos p;
        uint64_t steps;
        gbwt_seek(ix, cv, shift, __ldg(ids + q), __ldg(indexes + q), p, steps);
        out[q] = p;
    }
}

// What range i writes: elements [start, last) of its sequence (last - start = the full clipped size, cut to the slot),
// walked from checkpoint slots slot .. slot + pieces - 1.
struct Plan {
    uint64_t start, last;
    uint32_t slot, pieces;
};

// min(end, len) - start clipped at 0: the size of range [start, end) of something `len` long.
__device__ __forceinline__ uint64_t clipped(uint64_t start, uint64_t end, uint64_t len) {
    const uint64_t e = end < len ? end : len;
    return e > start ? e - start : 0;
}

// Nodes, with checkpoints. Returns lengths[i].
__device__ __forceinline__ uint64_t plan_nodes(const IndexView& ix, const CheckpointView& cv, uint32_t shift, uint64_t id, uint64_t start,
                                               uint64_t end, uint64_t cap, Plan& p) {
    p.start = p.last = start; p.slot = 0; p.pieces = 0;
    if (id >= ix.sequences) return ~0ull;
    const uint64_t want = clipped(start, end, cv.seq_len[id]);
    p.last = start + (want < cap ? want : cap);
    if (p.last > start) {
        p.slot = checkpoint_slot(cv, shift, id, start);
        p.pieces = checkpoint_slot(cv, shift, id, p.last - 1) - p.slot + 1;
    }
    return want;
}

// Last slot of [lo, hi) whose DNA position is at or below x (dna_at[lo] = 0 <= x).
__device__ __forceinline__ uint32_t dna_slot(const uint64_t* dna_at, uint32_t lo, uint32_t hi, uint64_t x) {
    while (hi - lo > 1) {
        const uint32_t mid = lo + (hi - lo) / 2;
        if (__ldg(dna_at + mid) <= x) lo = mid; else hi = mid;
    }
    return lo;
}

// DNA bytes, with DNA checkpoints. Returns lengths[i].
__device__ __forceinline__ uint64_t plan_dna(const IndexView& ix, const CheckpointView& cv, const uint64_t* dna_at, const uint64_t* dna_len,
                                             uint64_t id, uint64_t start, uint64_t end, uint64_t cap, Plan& p) {
    p.start = p.last = start; p.slot = 0; p.pieces = 0;
    if (id >= ix.sequences) return ~0ull;
    const uint64_t want = clipped(start, end, __ldg(dna_len + id) - 1);
    p.last = start + (want < cap ? want : cap);
    if (p.last > start) {
        const uint32_t lo = __ldg(cv.first + id), hi = __ldg(cv.first + id + 1);
        p.slot = dna_slot(dna_at, lo, hi, start);
        p.pieces = dna_slot(dna_at, p.slot, hi, p.last - 1) - p.slot + 1;
    }
    return want;
}

__device__ __forceinline__ uint64_t slot_of(const uint64_t* out_offsets, uint64_t i) {
    const uint64_t lo = __ldg(out_offsets + i), hi = __ldg(out_offsets + i + 1);
    return hi > lo ? hi - lo : 0;
}

// Without checkpoints a range is one walk from the start of its sequence, and that walk also finds its length.
__device__ __forceinline__ uint64_t plan_chain(const IndexView& ix, uint64_t id, uint64_t start, uint64_t end, Plan& p) {
    p.start = p.last = start; p.slot = 0; p.pieces = 0;
    if (id >= ix.sequences) return ~0ull;
    if (start >= end) return 0;
    p.pieces = 1;
    return ~0ull;  // (written by the walk)
}

// take[i] = pieces of range i; lengths[i] where the plan knows it.
template <bool DNA>
__global__ void __launch_bounds__(RANGE_THREADS) k_range_plan(IndexView ix, CheckpointView cv, uint32_t shift, const uint64_t* __restrict__ dna_at,
                                                              const uint64_t* __restrict__ dna_len, const uint64_t* __restrict__ ids,
                                                              const uint64_t* __restrict__ starts, const uint64_t* __restrict__ ends, uint64_t m,
                                                              const uint64_t* __restrict__ out_offsets, uint64_t* __restrict__ take,
                                                              uint64_t* __restrict__ lengths) {
    for (uint64_t i = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; i < m; i += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        const uint64_t id = __ldg(ids + i), start = __ldg(starts + i), end = __ldg(ends + i);
        Plan p;
        uint64_t len;
        if (cv.table == nullptr) len = plan_chain(ix, id, start, end, p);
        else if (DNA) len = plan_dna(ix, cv, dna_at, dna_len, id, start, end, slot_of(out_offsets, i), p);
        else len = plan_nodes(ix, cv, shift, id, start, end, slot_of(out_offsets, i), p);
        take[i] = p.pieces;
        if (lengths != nullptr && !(cv.table == nullptr && p.pieces != 0)) lengths[i] = len;
    }
}

// Walks from node number `at` (at `pos`) through node number stop - 1 or to the end of the sequence, whichever comes first,
// and stores node x of [a, b) at out[x] (`out` is the slot's address minus the range start). Returns the number of the node
// after the last one reached; `ended` = the sequence ended there (or the walk reached walk_limit).
__device__ __forceinline__ uint64_t walk_nodes(const IndexView& ix, gbwt_b200_pos pos, uint64_t at, uint64_t stop, uint64_t a, uint64_t b,
                                               uint64_t* out, bool& ended) {
    ended = false;
    for (;;) {
        if (at >= a && at < b) out[at] = pos.node;
        if (at + 1 >= stop) return at + 1;
        gbwt_b200_pos next;
        if (at >= ix.walk_limit || !gbwt_forward(ix, pos, next)) { ended = true; return at + 1; }
        pos = next;
        at++;
    }
}

// The same in DNA: `cursor` = bytes of the sequence before the node at `pos`; byte x of [a, b) is stored at out[x]; stops
// once the cursor reaches `stop`. Returns the cursor. Labels as in spell_group (kernels.cuh).
__device__ __forceinline__ uint64_t walk_dna(const IndexView& ix, const GraphView& graph, gbwt_b200_pos pos, uint64_t cursor, uint64_t stop,
                                             uint64_t a, uint64_t b, uint8_t* out, bool& ended) {
    ended = false;
    const uint64_t node_base = ix.offset + 1;
    for (uint64_t steps = 0;; steps++) {
        const uint64_t sid = ((pos.node & ~1ull) - node_base) >> 1;  // GBZ::gbwt_node_to_sequence, src/gbz.rs:253-255
        uint64_t lo = 0, len = 0;
        if (sid < graph.sequences) { lo = __ldg(graph.starts + sid); len = __ldg(graph.starts + sid + 1) - lo; }
        const uint64_t from = cursor > a ? cursor : a, to = cursor + len < b ? cursor + len : b;
        const bool rev = (pos.node & 1) != 0;
        for (uint64_t x = from; x < to; x++) {
            const uint64_t k = x - cursor;
            const uint32_t c = __ldg(graph.bytes + (rev ? lo + len - 1 - k : lo + k));
            out[x] = static_cast<uint8_t>(rev ? complement_base(c) : c);
        }
        cursor += len;
        if (cursor >= stop) return cursor;
        gbwt_b200_pos next;
        if (steps >= ix.walk_limit || !gbwt_forward(ix, pos, next)) { ended = true; return cursor; }
        pos = next;
    }
}

// Piece p of all ranges: lane p finds its range in the exclusive scan of take[] and walks its piece.
template <bool DNA>
// (At most 64 registers: with fewer, ptxas spills around the out-of-line rank_runs call of the LF step.)
__global__ void __launch_bounds__(RANGE_THREADS, 4) k_range_pieces(IndexView ix, GraphView graph, CheckpointView cv, uint32_t shift,
                                                                const uint64_t* __restrict__ dna_at, const uint64_t* __restrict__ dna_len,
                                                                const uint64_t* __restrict__ ids, const uint64_t* __restrict__ starts,
                                                                const uint64_t* __restrict__ ends, uint64_t m, const uint64_t* __restrict__ scan,
                                                                const uint64_t* __restrict__ take, const uint64_t* __restrict__ out_offsets,
                                                                uint64_t base, void* __restrict__ out, uint64_t* __restrict__ lengths) {
    const uint64_t total = scan[m - 1] + take[m - 1];
    for (uint64_t p = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; p < total; p += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        uint64_t lo = 0, hi = m;  // last i with scan[i] <= p (ranges without pieces share their scan value)
        while (hi - lo > 1) {
            const uint64_t mid = lo + (hi - lo) / 2;
            if (__ldg(scan + mid) <= p) lo = mid; else hi = mid;
        }
        const uint64_t i = lo, piece = p - __ldg(scan + i);
        const uint64_t id = __ldg(ids + i), start = __ldg(starts + i), end = __ldg(ends + i), cap = slot_of(out_offsets, i);
        // element x of the sequence goes to out[out_offsets[i] - base + x - start] (the address arithmetic wraps like the index's)
        const uint64_t shift_by = __ldg(out_offsets + i) - base - start;
        uint64_t* const nodes = reinterpret_cast<uint64_t*>(reinterpret_cast<uintptr_t>(out) + shift_by * sizeof(uint64_t));
        uint8_t* const bytes = reinterpret_cast<uint8_t*>(reinterpret_cast<uintptr_t>(out) + shift_by);
        // where the walk starts (`at`: node number, `cursor`: DNA bytes before it), where it stops, what it stores
        gbwt_b200_pos pos;
        uint64_t at = 0, cursor = 0, stop, a = start, b;
        const bool chain = cv.table == nullptr;
        if (chain) {
            // one walk from GBWT::start: it stores [start, start + cap) and runs on to `end` for the length
            stop = end;
            b = cap < end - start ? start + cap : end;
            if (!gbwt_start(ix, id, pos)) {
                if (lengths != nullptr) lengths[i] = 0;
                continue;
            }
        } else {
            Plan plan;
            if (DNA) plan_dna(ix, cv, dna_at, dna_len, id, start, end, cap, plan);
            else plan_nodes(ix, cv, shift, id, start, end, cap, plan);
            const uint32_t slot = plan.slot + static_cast<uint32_t>(piece);
            const bool next = slot + 1 < __ldg(cv.first + id + 1);
            pos = checkpoint_pos(cv, slot, at);
            b = plan.last;
            if (DNA) {
                cursor = __ldg(dna_at + slot);
                if (next && __ldg(dna_at + slot + 1) < b) b = __ldg(dna_at + slot + 1);
                if (cursor > a) a = cursor;
            } else {
                if (next && GBWT_LDG(&cv.table[slot + 1].index) < b) b = GBWT_LDG(&cv.table[slot + 1].index);
                if (at > a) a = at;
            }
            stop = b;
        }
        bool ended;
        uint64_t len = DNA ? walk_dna(ix, graph, pos, cursor, stop, a, b, bytes, ended) : walk_nodes(ix, pos, at, stop, a, b, nodes, ended);
        if (chain && lengths != nullptr) {
            if (!ended) len = end;  // reached `end`: the sequence is at least that long
            lengths[i] = clipped(start, end, len);
        }
    }
}

// take / scan over the m ranges, then one lane per piece (the total is read on the device: a full wave loops over it).
template <bool DNA>
cudaError_t launch_ranges(const IndexView& ix, const GraphView& graph, const CheckpointView& cv, uint32_t shift, const uint64_t* dna_at,
                          const uint64_t* dna_len, const uint64_t* ids, const uint64_t* starts, const uint64_t* ends, uint64_t m,
                          const uint64_t* out_offsets, uint64_t base, void* out, uint64_t* lengths, int sm_count, cudaStream_t s) {
    if (m == 0) return cudaSuccess;
    uint64_t *take = nullptr, *scan = nullptr;
    void* temp = nullptr;
    size_t temp_bytes = 0;
    cudaError_t e = cudaMallocAsync(reinterpret_cast<void**>(&take), m * sizeof(uint64_t), s);
    if (e == cudaSuccess) e = cudaMallocAsync(reinterpret_cast<void**>(&scan), m * sizeof(uint64_t), s);
    if (e == cudaSuccess) {
        k_range_plan<DNA><<<grid_of(m, sm_count), RANGE_THREADS, 0, s>>>(ix, cv, shift, dna_at, dna_len, ids, starts, ends, m, out_offsets, take, lengths);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(nullptr, temp_bytes, take, scan, static_cast<int64_t>(m), s);
    if (e == cudaSuccess) e = cudaMallocAsync(&temp, std::max<size_t>(temp_bytes, 16), s);
    if (e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(temp, temp_bytes, take, scan, static_cast<int64_t>(m), s);
    if (e == cudaSuccess) {
        k_range_pieces<DNA><<<grid_of(uint64_t(1) << 40, sm_count), RANGE_THREADS, 0, s>>>(ix, graph, cv, shift, dna_at, dna_len, ids, starts, ends, m,
                                                                                            scan, take, out_offsets, base, out, lengths);
        e = cudaGetLastError();
    }
    if (temp != nullptr) cudaFreeAsync(temp, s);
    if (take != nullptr) cudaFreeAsync(take, s);
    if (scan != nullptr) cudaFreeAsync(scan, s);
    return e;
}

}  // namespace

cudaError_t launch_seek(const IndexView& ix, const CheckpointView& cv, uint32_t shift, const uint64_t* ids, const uint64_t* indexes,
                        uint64_t n, gbwt_b200_pos* out, int sm_count, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    k_seek<<<grid_of(n, sm_count), RANGE_THREADS, 0, s>>>(ix, cv, shift, ids, indexes, n, out);
    return cudaGetLastError();
}

cudaError_t launch_range_nodes(const IndexView& ix, const CheckpointView& cv, uint32_t shift, const uint64_t* ids, const uint64_t* starts,
                               const uint64_t* ends, uint64_t m, const uint64_t* out_offsets, uint64_t base, uint64_t* nodes,
                               uint64_t* lengths, int sm_count, cudaStream_t s) {
    return launch_ranges<false>(ix, GraphView{}, cv, shift, nullptr, nullptr, ids, starts, ends, m, out_offsets, base, nodes, lengths, sm_count, s);
}

cudaError_t launch_range_dna(const IndexView& ix, const GraphView& graph, const CheckpointView& cv, const uint64_t* dna_at,
                             const uint64_t* dna_len, const uint64_t* ids, const uint64_t* starts, const uint64_t* ends, uint64_t m,
                             const uint64_t* out_offsets, uint64_t base, uint8_t* bytes, uint64_t* lengths, int sm_count,
                             cudaStream_t s) {
    return launch_ranges<true>(ix, graph, cv, 0, dna_at, dna_len, ids, starts, ends, m, out_offsets, base, bytes, lengths, sm_count, s);
}

}  // namespace gbwt_b200
