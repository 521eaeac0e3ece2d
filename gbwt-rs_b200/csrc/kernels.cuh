// kernels.cuh -- the CUDA kernels of the hot path (sm_100a). One thread owns one query (or one path) and
// runs the one-lane code of record_scan.cuh; thousands of independent queries per SM hide the HBM latency
// of the random record fetches. Grids are persistent: gridDim = SMs x resident CTAs, grid-stride loops.
//
//   K1  k_find / k_extend / k_find_extend(_ragged)   GBWT::find, extend          (src/gbwt.rs:269-304)
//   K2  k_bd_find / k_bd_extend / k_bd_search        bd_find, extend_forward/backward (src/gbwt.rs:311-384)
//   K3  k_start / k_forward / k_backward / k_sequence_lengths / k_extract   (src/gbwt.rs:213-261, 557-568)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "find_lean.cuh"
#include "record_scan.cuh"

namespace gbwt_b200 {

#define GBWT_GRID_STRIDE(i, n) \
    for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < (n); i += static_cast<size_t>(gridDim.x) * blockDim.x)

__global__ void __launch_bounds__(BLOCK_THREADS) k_find(IndexView ix, const uint64_t* __restrict__ nodes, size_t n,
                                                         gbwt_b200_state* __restrict__ out) {
    GBWT_GRID_STRIDE(q, n) {
        gbwt_b200_state st;
        gbwt_find(ix, __ldg(nodes + q), st);
        store_state(out + q, st);
    }
}

__global__ void __launch_bounds__(BLOCK_THREADS) k_extend(IndexView ix, const gbwt_b200_state* states,
                                                           const uint64_t* __restrict__ nodes, size_t n,
                                                           gbwt_b200_state* out) {
    GBWT_GRID_STRIDE(q, n) {
        const gbwt_b200_state in = states[q];  // out may alias states
        gbwt_b200_state st;
        gbwt_extend(ix, in, __ldg(nodes + q), st);
        store_state(out + q, st);
    }
}

// K1: find(p[0]) + extends, one thread per pattern. With `perm` the threads take the queries in bucket order
// (locality schedule below; results always go to out[q]). RUNS = false is the instantiation for indexes
// without run-length bodies (record_scan.cuh: rank_pair).
template <bool RUNS>
__global__ void __launch_bounds__(BLOCK_THREADS) k_find_extend(IndexView ix, const uint64_t* __restrict__ patterns,
                                                                const uint32_t* __restrict__ perm, size_t n, size_t k,
                                                                gbwt_b200_state* __restrict__ out) {
    GBWT_FOR_EACH_QUERY(q, n, perm) {
        gbwt_b200_state st;
        ChunkReader rd(patterns + q * k, static_cast<uint32_t>(k));
        query_find_extend_rounds<RUNS>(ix, rd, static_cast<uint32_t>(k), st);
        store_state(out + q, st);
    }
}

// The same for an index that has only EMPTY / SINGLE / DENSE2 records and validated edges (query_find_extend_lean).
// With the lean loop the issue slots are no longer the bound (38 % busy) and the kernel waits for its scattered
// sector loads, so it is compiled for CTAS resident CTAs of 256 threads per SM (more warps to hide the latency).
template <int CTAS>
__global__ void __launch_bounds__(BLOCK_THREADS, CTAS) k_find_extend_lean(IndexView ix, const uint64_t* __restrict__ patterns,
                                                                           const uint32_t* __restrict__ perm, size_t n, size_t k,
                                                                           gbwt_b200_state* __restrict__ out) {
    GBWT_FOR_EACH_QUERY(q, n, perm) {
        gbwt_b200_state st;
        ChunkReader rd(patterns + q * k, static_cast<uint32_t>(k));
        query_find_extend_lean<false>(ix, rd, static_cast<uint32_t>(k), st);
        store_state(out + q, st);
    }
}

// ---- locality schedule ------------------------------------------------------------------------------
// A batch of random queries touches ~65 isolated 32-byte sectors per query; HBM serves such accesses at a
// fraction of its streaming bandwidth (every access opens a new DRAM row). The records a pattern needs lie
// next to the record of its first node (node ids follow the graph's topological order), so the batch is
// bucketed by the record of pattern[0] with a counting sort, and threads take queries in bucket order:
// the queries in flight at any moment then share a few MB of the index, which stays in L1/L2, and HBM
// only streams each part of the index once per batch.

// Sort key of a query: the record of its first node, coarsened by `shift`. (Moving the orientation bit to the
// top, so that walks heading the same way sit together, was measured 16% slower: the two orientations of a node
// share a 64-byte descriptor pair, and a bucket that uses only one of them needs twice the lines.)
__device__ __forceinline__ uint32_t bucket_of(const IndexView& ix, uint64_t node, uint32_t shift) {
    uint64_t rec;
    if (!record_of(ix, node, rec)) return 0;
    return static_cast<uint32_t>(rec >> shift);
}

__host__ __device__ inline uint64_t bucket_count(uint64_t records, uint32_t shift) { return ((records - 1) >> shift) + 1; }

// keys[q] = bucket of query q: its first node is pattern row q, column 0 ...
__global__ void __launch_bounds__(BLOCK_THREADS) k_keys_fixed(IndexView ix, const uint64_t* __restrict__ patterns, size_t n,
                                                               size_t k, uint32_t shift, uint32_t* __restrict__ keys,
                                                               uint32_t* __restrict__ counts) {
    GBWT_GRID_STRIDE(q, n) {
        const uint32_t b = bucket_of(ix, __ldg(patterns + q * k), shift);
        keys[q] = b;
        atomicAdd(counts + 1 + b, 1u);  // counts[0] stays 0 for the exclusive scan
    }
}

// ... or nodes[offsets[q] - base + first[q]] for ragged batches (first == nullptr: the first node of the pattern).
__global__ void __launch_bounds__(BLOCK_THREADS) k_keys_ragged(IndexView ix, const uint64_t* __restrict__ nodes,
                                                                const uint64_t* __restrict__ offsets, uint64_t base,
                                                                const uint64_t* __restrict__ first, size_t n, uint32_t shift,
                                                                uint32_t* __restrict__ keys, uint32_t* __restrict__ counts) {
    GBWT_GRID_STRIDE(q, n) {
        const uint64_t lo = __ldg(offsets + q), hi = __ldg(offsets + q + 1);
        const uint64_t at = first != nullptr ? __ldg(first + q) : 0;
        const uint32_t b = (hi > lo && at < hi - lo) ? bucket_of(ix, __ldg(nodes + (lo - base) + at), shift) : 0;
        keys[q] = b;
        atomicAdd(counts + 1 + b, 1u);
    }
}

// Inclusive scan of counts[0 .. m) in three launches: every CTA scans one tile of SCAN_TILE entries in place and
// records its total, one CTA scans the tile totals, every CTA adds the total of the tiles before it. After the
// scan counts[b] is the first slot of bucket b.
constexpr uint32_t SCAN_TILE = 4096;  // 1024 threads x 4 entries

__device__ __forceinline__ uint32_t block_inclusive_scan(uint32_t x, uint32_t* warp_sums) {
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t d = 1; d < 32; d <<= 1) {
        const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, d);
        if (lane >= d) x += y;
    }
    if (lane == 31) warp_sums[warp] = x;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = warp_sums[lane];
        for (uint32_t d = 1; d < 32; d <<= 1) {
            const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, w, d);
            if (lane >= d) w += y;
        }
        warp_sums[lane] = w;
    }
    __syncthreads();
    const uint32_t result = x + (warp > 0 ? warp_sums[warp - 1] : 0);
    __syncthreads();
    return result;
}

__global__ void __launch_bounds__(1024) k_scan_tiles(uint32_t* __restrict__ counts, uint32_t m, uint32_t* __restrict__ tile_sums) {
    __shared__ uint32_t warp_sums[32];
    const uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * 4;
    uint32_t v[4];
    for (uint32_t j = 0; j < 4; j++) v[j] = base + j < m ? counts[base + j] : 0;
    v[1] += v[0]; v[2] += v[1]; v[3] += v[2];
    const uint32_t before = block_inclusive_scan(v[3], warp_sums) - v[3];
    for (uint32_t j = 0; j < 4; j++) if (base + j < m) counts[base + j] = before + v[j];
    if (threadIdx.x == 1023) tile_sums[blockIdx.x] = before + v[3];
}

// In-place inclusive scan of a short array by one CTA (the tile totals).
__global__ void __launch_bounds__(1024) k_scan_single(uint32_t* __restrict__ a, uint32_t m) {
    __shared__ uint32_t warp_sums[32];
    __shared__ uint32_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < m; base += 1024) {
        const uint32_t i = base + threadIdx.x;
        const uint32_t x = block_inclusive_scan(i < m ? a[i] : 0, warp_sums);
        const uint32_t c = carry;
        if (i < m) a[i] = c + x;
        __syncthreads();
        if (threadIdx.x == 1023) carry = c + x;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(1024) k_scan_add(uint32_t* __restrict__ counts, uint32_t m, const uint32_t* __restrict__ tile_sums) {
    if (blockIdx.x == 0) return;
    const uint32_t add = tile_sums[blockIdx.x - 1];
    const uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * 4;
    for (uint32_t j = 0; j < 4; j++) if (base + j < m) counts[base + j] += add;
}

// perm[slot] = q, slots handed out per bucket by atomics (the order inside a bucket does not matter).
__global__ void __launch_bounds__(BLOCK_THREADS) k_bucket_scatter(const uint32_t* __restrict__ keys, size_t n,
                                                                   uint32_t* __restrict__ cursor, uint32_t* __restrict__ perm) {
    GBWT_GRID_STRIDE(q, n) {
        const uint32_t slot = atomicAdd(cursor + __ldg(keys + q), 1u);
        perm[slot] = static_cast<uint32_t>(q);
    }
}

// `base` = offsets[0] of the chunk that `nodes` starts at (host entry points upload node chunks).
// LEAN: the index qualifies for query_find_extend_lean (see k_find_extend_lean).
template <bool LEAN>
__global__ void __launch_bounds__(BLOCK_THREADS, LEAN ? 5 : 1) k_find_extend_ragged(IndexView ix, const uint64_t* __restrict__ nodes,
                                                                                     const uint64_t* __restrict__ offsets, uint64_t base,
                                                                                     const uint32_t* __restrict__ perm, size_t n,
                                                                                     gbwt_b200_state* __restrict__ out) {
    GBWT_FOR_EACH_QUERY(q, n, perm) {
        const uint64_t lo = __ldg(offsets + q), hi = __ldg(offsets + q + 1);
        const uint64_t len = hi > lo ? hi - lo : 0;
        gbwt_b200_state st;
        if (LEAN && len <= 0xFFFFFFFFull) {
            ChunkReader rd(nodes + (lo - base), static_cast<uint32_t>(len));
            query_find_extend_lean<false>(ix, rd, static_cast<uint32_t>(len), st);
        } else {
            query_find_extend(ix, nodes + (lo - base), len, st);
        }
        store_state(out + q, st);
    }
}

__global__ void __launch_bounds__(BLOCK_THREADS) k_bd_find(IndexView ix, const uint64_t* __restrict__ nodes, size_t n,
                                                            gbwt_b200_bdstate* __restrict__ out) {
    GBWT_GRID_STRIDE(q, n) {
        gbwt_b200_bdstate st;
        gbwt_bd_find(ix, __ldg(nodes + q), st);
        out[q] = st;
    }
}

__global__ void __launch_bounds__(BLOCK_THREADS) k_bd_extend(IndexView ix, const gbwt_b200_bdstate* states,
                                                              const uint64_t* __restrict__ nodes, size_t n, int backward,
                                                              gbwt_b200_bdstate* out) {
    GBWT_GRID_STRIDE(q, n) {
        const gbwt_b200_bdstate in = states[q];
        gbwt_b200_bdstate st;
        if (backward) gbwt_extend_backward(ix, in, __ldg(nodes + q), st);
        else gbwt_extend_forward(ix, in, __ldg(nodes + q), st);
        out[q] = st;
    }
}

template <bool RUNS>
__global__ void __launch_bounds__(BLOCK_THREADS) k_bd_search(IndexView ix, const uint64_t* __restrict__ nodes,
                                                              const uint64_t* __restrict__ offsets, uint64_t base,
                                                              const uint64_t* __restrict__ first,
                                                              const uint64_t* __restrict__ start,
                                                              const uint64_t* __restrict__ end,
                                                              const uint32_t* __restrict__ perm, size_t n,
                                                              gbwt_b200_bdstate* __restrict__ out) {
    GBWT_FOR_EACH_QUERY(q, n, perm) {
        const uint64_t lo = __ldg(offsets + q), hi = __ldg(offsets + q + 1);
        gbwt_b200_bdstate st;
        query_bd_search_fast<RUNS>(ix, nodes + (lo - base), hi > lo ? hi - lo : 0, __ldg(first + q), __ldg(start + q), __ldg(end + q), st);
        out[q] = st;
    }
}

// All extensions of a state (GBZ::follow_forward / follow_backward): one thread per state; `out == nullptr` only counts.
__global__ void __launch_bounds__(BLOCK_THREADS) k_follow(IndexView ix, const gbwt_b200_bdstate* __restrict__ states, size_t n,
                                                           int backward, const uint64_t* __restrict__ out_offsets, uint64_t base,
                                                           gbwt_b200_bdstate* __restrict__ out, uint64_t* __restrict__ counts) {
    GBWT_GRID_STRIDE(q, n) {
        gbwt_b200_bdstate* dst = nullptr;
        uint64_t cap = 0;
        if (out != nullptr) {
            const uint64_t lo = __ldg(out_offsets + q), hi = __ldg(out_offsets + q + 1);
            dst = out + (lo - base);
            cap = hi > lo ? hi - lo : 0;
        }
        const gbwt_b200_bdstate st = states[q];
        const uint64_t c = gbwt_follow_all(ix, st, backward != 0, dst, cap);
        if (counts != nullptr) counts[q] = c;
    }
}

__global__ void __launch_bounds__(BLOCK_THREADS) k_start(IndexView ix, const uint64_t* __restrict__ ids, size_t n,
                                                          gbwt_b200_pos* __restrict__ out) {
    GBWT_GRID_STRIDE(q, n) {
        gbwt_b200_pos p;
        gbwt_start(ix, __ldg(ids + q), p);
        out[q] = p;
    }
}

__global__ void __launch_bounds__(BLOCK_THREADS) k_forward(IndexView ix, const gbwt_b200_pos* positions, size_t n,
                                                            gbwt_b200_pos* out) {
    GBWT_GRID_STRIDE(q, n) {
        const gbwt_b200_pos in = positions[q];
        gbwt_b200_pos p;
        gbwt_forward(ix, in, p);
        out[q] = p;
    }
}

__global__ void __launch_bounds__(BLOCK_THREADS) k_backward(IndexView ix, const gbwt_b200_pos* positions, size_t n,
                                                             gbwt_b200_pos* out) {
    GBWT_GRID_STRIDE(q, n) {
        const gbwt_b200_pos in = positions[q];
        gbwt_b200_pos p;
        gbwt_backward(ix, in, p);
        out[q] = p;
    }
}

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// Descriptor of the record of `node`, or an empty one when BWT::record() would be None.
__device__ __forceinline__ Desc load_desc_of(const IndexView& ix, uint64_t node) {
    Desc d;
    d.a.x = d.a.y = d.a.z = d.a.w = d.b.x = d.b.y = d.b.z = d.b.w = 0;  // fmt() == FMT_EMPTY
    uint64_t rec;
    if (node >= ix.offset + 1 && record_of(ix, node, rec)) d = load_desc(ix, rec);
    return d;
}

// Record::lf (src/bwt.rs:480-496) on a RUN8 body by a whole warp: every lane calls it with the same arguments.
// Each lane takes one 16-byte unit of the body (512 bytes per round, ONE memory round trip for a whole anchor
// record instead of one per unit), decodes its runs, and a shuffle prefix sum over the per-lane run totals plus a
// ballot locate the lane whose unit covers position i; that lane finds the run and its symbol, the lanes before
// it count that symbol, and a warp reduction adds the counts up. Returns symbol == NO_SYMBOL if i is past the end.
__device__ __forceinline__ void warp_lf_runs8(const IndexView& ix, const Desc& d, uint32_t i, uint32_t& symbol, uint32_t& rank_i) {
    constexpr uint32_t FULL = 0xFFFFFFFFu;
    const uint32_t lane = threadIdx.x & 31u;
    const Unit16* body = ix.bodies + d.body();
    const uint32_t n = d.body_len(), sigma = d.sigma();
    const uint32_t magic = d.inline_edges() ? 32769u : d.magic();
    symbol = NO_SYMBOL; rank_i = 0;
    uint32_t off = 0, found_base = 0;
    for (uint32_t base = 0; base < n; base += 512) {
        const uint32_t at = base + 16 * lane;
        Quad q;
        q.x = q.y = q.z = q.w = 0;
        if (at < n) q = load_quad(body + (at >> 4));
        const uint32_t nb = at < n ? (n - at < 16 ? n - at : 16) : 0;
        const uint32_t words[4] = {q.x, q.y, q.z, q.w};
        uint32_t total = 0;
#pragma unroll
        for (uint32_t j = 0; j < 16; j++) {
            if (j < nb) total += (((words[j >> 2] >> (8 * (j & 3))) & 0xFF) * magic >> 16) + 1;
        }
        uint32_t incl = total;
#pragma unroll
        for (uint32_t dlt = 1; dlt < 32; dlt <<= 1) {
            const uint32_t y = __shfl_up_sync(FULL, incl, dlt);
            if (lane >= dlt) incl += y;
        }
        const uint32_t before = off + incl - total;
        const uint32_t hit = __ballot_sync(FULL, total != 0 && i >= before && i - before < total);
        if (hit != 0) {
            const uint32_t owner = __ffs(hit) - 1;
            uint32_t sym = 0, part = 0;
            if (lane == owner) {
                uint32_t o = before;
                bool have = false;
#pragma unroll
                for (uint32_t j = 0; j < 16; j++) {
                    if (j < nb && !have) {
                        const uint32_t b = (words[j >> 2] >> (8 * (j & 3))) & 0xFF;
                        const uint32_t quot = (b * magic) >> 16;
                        if (i - o < quot + 1) { sym = b - quot * sigma; have = true; }
                        else o += quot + 1;
                    }
                }
                o = before;
#pragma unroll
                for (uint32_t j = 0; j < 16; j++) {
                    if (j < nb && o < i) {
                        const uint32_t b = (words[j >> 2] >> (8 * (j & 3))) & 0xFF;
                        const uint32_t quot = (b * magic) >> 16;
                        if (b - quot * sigma == sym) part += (i - o < quot + 1) ? i - o : quot + 1;
                        o += quot + 1;
                    }
                }
            }
            sym = __shfl_sync(FULL, sym, owner);
            part = __shfl_sync(FULL, part, owner);
            uint32_t cnt = 0;
            if (lane < owner) {
#pragma unroll
                for (uint32_t j = 0; j < 16; j++) {
                    if (j < nb) {
                        const uint32_t b = (words[j >> 2] >> (8 * (j & 3))) & 0xFF;
                        const uint32_t quot = (b * magic) >> 16;
                        if (b - quot * sigma == sym) cnt += quot + 1;
                    }
                }
            }
            symbol = sym;
            rank_i = __reduce_add_sync(FULL, cnt) + part;
            found_base = base;
            break;
        }
        off += __shfl_sync(FULL, incl, 31);
    }
    if (symbol == NO_SYMBOL) return;
    // bodies longer than one round: the symbol's runs in the rounds before the one that holds position i
    for (uint32_t base = 0; base < found_base; base += 512) {
        const Quad q = load_quad(body + ((base + 16 * lane) >> 4));
        const uint32_t words[4] = {q.x, q.y, q.z, q.w};
        uint32_t cnt = 0;
#pragma unroll
        for (uint32_t j = 0; j < 16; j++) {
            const uint32_t b = (words[j >> 2] >> (8 * (j & 3))) & 0xFF;
            const uint32_t quot = (b * magic) >> 16;
            if (b - quot * sigma == symbol) cnt += quot + 1;
        }
        rank_i += __reduce_add_sync(FULL, cnt);
    }
}

// ---- what a walk does with the nodes it visits -------------------------------------------------------
// A warp-mode walk parks the nodes it visits one per lane and hands the sink a group of up to 32 of them at a
// time: `count` nodes, the first of which is number `first` of the sequence.

// ---- are the two strands of a path mirror images? -----------------------------------------------------------------------
// The two-ended walks rest on sequence id ^ 1 being sequence id reversed and flipped (support::reverse_path,
// src/support.rs:310-314). That is what "bidirectional" promises, but the flag is only a flag: on an index whose strands
// differ somewhere a two-ended walk would splice two different paths. (Comparing the halves where they meet, as the first
// version did, only proves that they agree THERE.) So every whole-sequence walk also leaves a signature of the sequence,
// three 64-bit sums over its nodes n_j (flipped when the walk is on an odd, i.e. reverse, sequence id):
//     A = sum a(n_j),   B = sum a(n_j) * j,   C = sum b(n_j)          (a, b: two 64-bit mixers)
// If sequence o = id ^ 1 is the mirror image of sequence id, its node j is the flip of node len - 1 - j, hence
//     A_o = A_id,   C_o = C_id,   B_o = (len - 1) * A_id - B_id       (mod 2^64)
// and any difference in a node or in a position breaks one of the three with probability 1 - 2^-64. A sequence is walked
// from both ends only when both strands have signatures and they agree; otherwise it is walked like the reference does.
struct SeqSignature { uint64_t a, b, c; };

__device__ __forceinline__ uint64_t sig_mix(uint64_t x) {
    x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull;
    x ^= x >> 27; x *= 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

struct SigAcc {
    uint64_t a = 0, b = 0, c = 0;  // this lane's share
    // the lane's node of a group: node number first + lane of the walk, if lane < count
    __device__ __forceinline__ void add(uint64_t mine, uint32_t count, uint64_t first, uint64_t flip) {
        const uint32_t lane = threadIdx.x & 31u;
        if (lane >= count) return;
        const uint64_t n = mine ^ flip, wa = sig_mix(n + 0x9E3779B97F4A7C15ull);
        a += wa; b += wa * (first + lane); c += sig_mix(n ^ 0xD6E8FEB86659FD93ull);
    }
    __device__ __forceinline__ SeqSignature total() const {
        SeqSignature s{a, b, c};
#pragma unroll
        for (uint32_t d = 16; d != 0; d >>= 1) {
            s.a += __shfl_xor_sync(0xFFFFFFFFu, s.a, d);
            s.b += __shfl_xor_sync(0xFFFFFFFFu, s.b, d);
            s.c += __shfl_xor_sync(0xFFFFFFFFu, s.c, d);
        }
        return s;
    }
};

// The signatures live behind the lengths in one allocation: seq_len[0 .. sequences), then three words per sequence.
__device__ __forceinline__ uint64_t* signatures_of(uint64_t* seq_len, uint64_t sequences) { return seq_len + sequences; }
__device__ __forceinline__ const uint64_t* signatures_of(const uint64_t* seq_len, uint64_t sequences) { return seq_len + sequences; }

constexpr uint64_t SIG_UNKNOWN = 0xFEFEFEFEFEFEFEFEull;  // what cudaMemset(0xFE) leaves (as for the length cache below)

__device__ __forceinline__ void store_signature(uint64_t* seq_sig, uint64_t id, const SeqSignature& s) {
    seq_sig[3 * id] = s.a; seq_sig[3 * id + 1] = s.b; seq_sig[3 * id + 2] = s.c == SIG_UNKNOWN ? s.c + 1 : s.c;
}

// Both strands of sequence `id` have been walked and they are mirror images of each other.
__device__ __forceinline__ bool strands_mirror(const uint64_t* seq_len, const uint64_t* seq_sig, uint64_t id, uint64_t sequences) {
    const uint64_t other = id ^ 1ull;
    if (id >= sequences || other >= sequences || seq_sig == nullptr) return false;
    const uint64_t len = seq_len[id];
    if (len == SIG_UNKNOWN || seq_len[other] != len) return false;
    const uint64_t a = seq_sig[3 * id], b = seq_sig[3 * id + 1], c = seq_sig[3 * id + 2];
    const uint64_t oa = seq_sig[3 * other], ob = seq_sig[3 * other + 1], oc = seq_sig[3 * other + 2];
    if (c == SIG_UNKNOWN || oc == SIG_UNKNOWN) return false;
    return a == oa && c == oc && ob == (len - 1) * a - b;
}

// GBWT::sequence(id): the node identifiers themselves, up to 256 contiguous bytes per group.
struct NodeSink {
    static constexpr bool CHECKPOINTS = false;
    uint64_t* out;
    uint64_t cap;
    uint64_t flip;  // 1 on a reverse (odd) sequence id: the signature is taken over the flipped nodes
    SigAcc sig;
    __device__ __forceinline__ void group(uint64_t mine, uint32_t count, uint64_t first) {
        const uint32_t lane = threadIdx.x & 31u;
        if (lane < count && first + lane < cap) out[first + lane] = mine;
        sig.add(mine, count, first, flip);
    }
    __device__ __forceinline__ void finish() {}
};

// One half of a sequence walked from either end. Forward: node j of the walk is position j. Reverse: the walk is on
// the other strand of a bidirectional index, where node j of sequence id ^ 1 is the flipped node at position
// len - 1 - j of sequence id (support::reverse_path, src/support.rs:310-314). Positions [lo, hi) are written; the
// node at position `probe` is also kept in `value` (all lanes) so that the two halves can be compared where they meet.
struct HalfSink {
    static constexpr bool CHECKPOINTS = false;
    uint64_t* out;
    uint64_t cap, len, lo, hi, probe, value;
    bool reverse;
    uint64_t flip;  // signature of a whole-sequence walk (see SigAcc): 1 on an odd sequence id
    SigAcc sig;
    __device__ __forceinline__ void group(uint64_t mine, uint32_t count, uint64_t first) {
        const uint32_t lane = threadIdx.x & 31u;
        const uint64_t j = first + lane;
        sig.add(mine, count, first, flip);
        const uint64_t p = reverse ? len - 1 - j : j, node = reverse ? mine ^ 1ull : mine;
        const bool valid = lane < count && (!reverse || j < len);
        if (valid && p >= lo && p < hi && p < cap) out[p] = node;
        const unsigned hit = __ballot_sync(0xFFFFFFFFu, valid && p == probe);
        if (hit != 0) value = __shfl_sync(0xFFFFFFFFu, node, __ffs(static_cast<int>(hit)) - 1);
    }
    __device__ __forceinline__ void finish() {}
};

// (struct GraphView: layout.h; complement_base: record_scan.cuh)

// extract_sequence (src/bin/gbz-extract.rs:173-189): the labels of the visited nodes, reverse-complemented for
// reverse-oriented nodes (support::reverse_complement, src/support.rs:104-110). Per group of 32 nodes every lane
// fetches the label range of its node (32 independent loads instead of one per step of the chain), a warp scan
// turns the lengths into output offsets, and the warp writes the group's bytes as consecutive 32-byte rows, each
// lane finding the node that owns its byte by a 5-step search over the scanned lengths.
// The walk is a latency-bound dependent chain, so the sink must not add round trips to it: the label ranges
// requested for one group are only consumed when the next group arrives (32 steps later, long since landed),
// and label bytes are fetched eight rows (256 bytes, a typical group) at a time before any of them is stored.
struct DnaSink {
    static constexpr bool CHECKPOINTS = false;
    GraphView graph;
    uint64_t node_base;  // alphabet offset + 1: GBZ::gbwt_node_to_sequence, src/gbz.rs:253-255
    uint8_t* out;        // nullptr: count only
    uint64_t cap;
    uint64_t written;
    // the group whose label ranges are in flight
    uint64_t pend_lo, pend_hi;
    uint32_t pend_rev;
    bool pend_valid, pending;
    // Walking one half of a sequence (k_extract_dna split mode): only nodes with index < node_limit are spelled; the
    // node with index `probe` is kept in `value`. mirror: the walk is on the other strand (sequence id ^ 1), whose DNA
    // is the reverse complement of this sequence's, so byte t of the walk is byte end - 1 - t of the result: the same
    // label bytes in the same order within the group, written downwards, and complemented exactly when the node is
    // forward on the walked strand (= reverse on the requested one).
    uint64_t node_limit, probe, value, end;
    bool mirror;
    uint64_t flip = 0;  // signature of a whole-sequence walk (SigAcc): 1 on an odd sequence id
    SigAcc sig;

    __device__ __forceinline__ void copy_pending() {
        constexpr unsigned FULL = 0xFFFFFFFFu;
        constexpr uint32_t ROWS = 8;
        const uint32_t lane = threadIdx.x & 31u;
        const uint32_t len = pend_valid ? static_cast<uint32_t>(pend_hi - pend_lo) : 0u;
        uint32_t incl = len;
#pragma unroll
        for (uint32_t d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(FULL, incl, d);
            if (lane >= d) incl += t;
        }
        const uint32_t total = __shfl_sync(FULL, incl, 31);
        if (out != nullptr) {
            // byte b of the group comes from label byte key + b (forward node) or key - b (reverse node); the keys
            // carry a bias of 2^32 so that they stay positive (bit 63 is the orientation)
            constexpr uint64_t BIAS = 1ull << 32;
            const uint32_t excl = incl - len;
            const uint64_t key = BIAS + (pend_rev ? pend_lo + len - 1 + excl : pend_lo - excl);
            const uint32_t key_lo = static_cast<uint32_t>(key), key_hi = static_cast<uint32_t>(key >> 32) | (pend_rev << 31);
            for (uint32_t row = 0; row < total; row += 32 * ROWS) {
                uint32_t c[ROWS], rev[ROWS];
#pragma unroll
                for (uint32_t j = 0; j < ROWS; j++) {
                    const uint32_t b = row + 32 * j + lane;
                    // owner = number of nodes that end at or before byte b (incl is non-decreasing over the lanes)
                    uint32_t owner = 0;
#pragma unroll
                    for (uint32_t step = 16; step != 0; step >>= 1) {
                        const uint32_t v = __shfl_sync(FULL, incl, (owner + step - 1) & 31u);
                        if (v <= b) owner += step;
                    }
                    const uint32_t k_lo = __shfl_sync(FULL, key_lo, owner & 31u), k_hi = __shfl_sync(FULL, key_hi, owner & 31u);
                    const uint64_t k = (static_cast<uint64_t>(k_hi & 0x7FFFFFFFu) << 32) | k_lo;
                    rev[j] = k_hi >> 31;
                    c[j] = 0;
                    const uint64_t t = written + b;
                    const bool wanted = b < total && (mirror ? t < end && end - 1 - t < cap : t < cap);
                    if (wanted) c[j] = __ldg(graph.bytes + ((rev[j] ? k - b : k + b) - BIAS));
                }
#pragma unroll
                for (uint32_t j = 0; j < ROWS; j++) {
                    const uint32_t b = row + 32 * j + lane;
                    const uint64_t t = written + b;
                    const bool wanted = b < total && (mirror ? t < end && end - 1 - t < cap : t < cap);
                    const bool comp = (rev[j] != 0) != mirror;
                    if (wanted) out[mirror ? end - 1 - t : t] = static_cast<uint8_t>(comp ? complement_base(c[j]) : c[j]);
                }
            }
        }
        written += total;
    }
    __device__ __forceinline__ void group(uint64_t mine, uint32_t count, uint64_t first) {
        const uint32_t lane = threadIdx.x & 31u;
        sig.add(mine, count, first, flip);
        if (pending) copy_pending();
        const unsigned hit = __ballot_sync(0xFFFFFFFFu, lane < count && first + lane == probe);
        if (hit != 0) value = __shfl_sync(0xFFFFFFFFu, mirror ? mine ^ 1ull : mine, __ffs(static_cast<int>(hit)) - 1);
        // the loads are unconditional (clamped index) and nothing here reads their results: a select between the
        // loaded value and zero would make this group wait for them
        const uint64_t sid = ((mine & ~1ull) - node_base) >> 1;
        pend_valid = lane < count && first + lane < node_limit && sid < graph.sequences;
        const uint64_t at = sid < graph.sequences ? sid : 0;
        pend_lo = __ldg(graph.starts + at);
        pend_hi = __ldg(graph.starts + at + 1);
        pend_rev = static_cast<uint32_t>(mine & 1u);
        pending = true;
    }
    __device__ __forceinline__ void finish() {
        if (pending) copy_pending();
        pending = false;
    }
};

// GBWT::sequence(id).collect() (src/gbwt.rs:253-261, 557-568; Record::lf, src/bwt.rs:480-496) by ONE lane: same
// results as walk_sequence(), with the descriptors of both successors of an outdegree-2 record requested together
// with the body block that decides between them. Used when a batch has more sequences than warps worth running
// (one sequence per thread); the warp-mode walk below is the fast path.
__device__ __forceinline__ uint64_t walk_sequence_lane(const IndexView& ix, uint64_t id, uint64_t* out, uint64_t cap) {
    if (id >= ix.sequences) return ~0ull;
    gbwt_b200_pos pos;
    if (!gbwt_start(ix, id, pos)) return 0;
    uint64_t node = pos.node, offset = pos.offset, n = 0;
    Desc d = load_desc_of(ix, node);
    for (;;) {
        if (n < cap) out[n] = node;
        n++;
        const uint32_t fmt = d.fmt();
        if (fmt == FMT_EMPTY || offset >= d.total_len() || n > ix.walk_limit) break;  // GBWT::forward -> None
        const uint32_t i = static_cast<uint32_t>(offset);
        if (fmt == FMT_SINGLE) {
            if (d.node0() == 0) break;
            offset = static_cast<uint64_t>(d.offset0()) + i;
            node = d.node0();
            d = load_desc_of(ix, node);
            continue;
        }
        if (fmt == FMT_DENSE2) {
            const Desc d0 = load_desc_of(ix, d.node0());
            const Desc d1 = load_desc_of(ix, d.node1());
            uint32_t symbol;
            const uint32_t ones = dense_rank1(ix.bodies + d.body(), d.body_len(), i, symbol);
            const uint32_t next = symbol ? d.node1() : d.node0();
            if (next == 0) break;
            offset = static_cast<uint64_t>(symbol ? d.offset1() : d.offset0()) + (symbol ? ones : i - ones);
            node = next;
            d = symbol ? d1 : d0;
            continue;
        }
        gbwt_b200_pos cur, next;
        cur.node = node; cur.offset = offset;
        if (!gbwt_forward(ix, cur, next)) break;
        node = next.node; offset = next.offset;
        d = load_desc_of(ix, node);
    }
    return n;
}

// ---- warp-mode walk: the lean chain ------------------------------------------------------------------
// ncu on the first version of the warp-mode walk showed the chain was not waiting for memory most of the time: a
// step was 186 instructions (64-bit positions, per-step prefetch arithmetic, descriptors spilled to the stack
// around non-inlined calls), and with one warp per chain every dependent instruction costs its full latency.
// This walk keeps a step of the two formats that make up a dense-policy pangenome index (SINGLE and DENSE2) to a
// few dozen 32-bit instructions, moves everything else off the per-step path, and uses the 31 lanes that would
// otherwise repeat lane 0's work: once per 32 steps the warp hands its 32 parked nodes to the sink and issues ONE
// warp-wide round of prefetches for the records it is heading to (one address per lane).

// Record::lf on a run-length body that the warp does not scan cooperatively (RUN32 / RUN64: rare), out of line so
// that it does not weigh on the registers of the walk. The descriptor travels as scalars and the two arrays by
// value: nothing of the caller has its address taken. (No 256-bit inline-asm load in here: inside a non-inlined
// device function that crashes ptxas 12.9.) Returns (offset << 32) | node, 0 = GBWT::forward is None.
__device__ __noinline__ uint64_t forward_other_record(const Unit16* bodies, const Edge* edges, uint32_t d0, uint32_t d1, uint32_t d2,
                                                      uint32_t d3, uint32_t d4, uint32_t d5, uint32_t d6, uint32_t d7, uint32_t i) {
    Desc d;
    d.a.x = d0; d.a.y = d1; d.a.z = d2; d.a.w = d3; d.b.x = d4; d.b.y = d5; d.b.z = d6; d.b.w = d7;
    IndexView view;  // the run scan only looks at the bodies and the edge lists
    view.desc = nullptr; view.bodies = bodies; view.edges = edges; view.endmarker = nullptr;
    view.records = 0; view.offset = 0; view.alphabet_size = 0; view.sequences = 0; view.endmarker_len = 0;
    view.bidirectional = 0; view.skips = nullptr; view.edges_valid = 1;
    const uint32_t symbol = symbol_at_runs(view, d, i);
    if (symbol == NO_SYMBOL) return 0;
    FlipSet fs;
    fs.lt = 0; fs.extra = NO_SYMBOL;
    Ranks r;
    r.at_start = r.at_end = r.flipped = 0;
    rank_runs_inline<false>(view, d, symbol, fs, i, i, r);
    const Edge e = edge_at(view, d, symbol);
    if (e.node == 0) return 0;  // successor is the endmarker: the sequence ends (src/bwt.rs:485-486)
    return (static_cast<uint64_t>(e.offset + r.at_start) << 32) | e.node;
}

// Record index of node v for a load that must be safe but whose result is only used when v has a record: edge
// targets were validated when the layout was built (IndexView::edges_valid), so clamping is enough.
__device__ __forceinline__ uint32_t record_clamped(uint32_t base, uint32_t records, uint32_t v) {
    const uint32_t rec = v - base;
    return rec < records ? rec : records - 1u;
}

// Descriptor and two-hop shortcut of node v. CHECKED: empty (fmt 0, no shortcut) where BWT::record() is None.
template <bool CHECKED>
__device__ __forceinline__ void load_landing(const RecordDesc* descs, const Unit16* skips, uint32_t base, uint32_t records,
                                             uint32_t v, Desc& d, Quad& k) {
    if (CHECKED) {
        d.a.x = d.a.y = d.a.z = d.a.w = d.b.x = d.b.y = d.b.z = d.b.w = 0;
        k.x = k.y = k.z = k.w = 0;
        const uint32_t rec = v - base;
        if (rec - 1u < records - 1u) {
            load_sector(reinterpret_cast<const Unit16*>(descs + rec), d.a, d.b);
            k = load_quad(skips + rec);
        }
    } else {
        const uint32_t rec = record_clamped(base, records, v);
        load_sector(reinterpret_cast<const Unit16*>(descs + rec), d.a, d.b);
        k = load_quad(skips + rec);
    }
}

// The steady state of a walk through a chain of bubbles, as tight as it gets: `cur` is a DENSE2 record whose two
// successors are single-edge records that rejoin at one node L (shortcuts on both edges, same landing). One
// iteration emits cur's node and the allele taken, and lands on L, whose descriptor and shortcut are requested into
// `nxt` before the body block of `cur` is. Returns false (nothing done) when `cur` is anything else, or when the
// lanes are full. The caller alternates (cur, nxt) so that no register is copied.
template <bool CHECKED>
__device__ __forceinline__ bool walk_bubble_step(Desc& cur_d, Quad& cur_k, Desc& nxt_d, Quad& nxt_k, const RecordDesc* descs,
                                                 const Unit16* bodies, const Unit16* skips, uint32_t base, uint32_t records,
                                                 uint32_t lane, uint32_t& node, uint32_t& offset, uint32_t& mine, uint32_t& in_group) {
    const uint32_t land = cur_k.x, i = offset;
    if (cur_d.fmt() != FMT_DENSE2 || land == 0 || land != cur_k.z || i >= cur_d.total_len() || in_group >= 31) return false;
    load_landing<CHECKED>(descs, skips, base, records, land, nxt_d, nxt_k);
    const uint32_t blk = __umulhi(i, 0xAAAAAAABu) >> 7;  // i / 192
    Quad lo, hi;
    load_sector(bodies + cur_d.body() + 2u * blk, lo, hi);
    if (in_group == lane) mine = node;
    uint32_t b;
    const uint32_t ones = dense_block_rank_lean(lo, hi, i - blk * DENSE_BITS, b);
    const uint32_t v = b ? cur_d.node1() : cur_d.node0();
    if (in_group + 1 == lane) mine = v;
    in_group += 2;
    node = land;
    offset = b ? cur_k.w + ones : cur_k.y + (i - ones);
    return true;
}

// GBWT::sequence(id) by one warp (all lanes hold the same state). Per iteration: one record u with inline edges
// (outdegree <= 2), the edge b the sequence takes and the rank r of b before its offset (no body for SINGLE, one
// 32-byte block for DENSE2, a warp scan for RUN8). If the successor v_b is a single-edge record, the shortcut of u
// gives LF(LF(u, i)) directly, so v_b is emitted without its record being read and the walk lands two nodes
// further. The descriptors and shortcuts of both possible landing nodes are requested at the top of the iteration,
// next to the body block that decides between them: ONE memory round trip per iteration.
// CHECKED = false relies on IndexView::edges_valid (no bounds tests on edge targets).
// `limit`: stop once at least that many nodes have been handed to the sink (checked when the lanes are flushed, so
// the walk may run up to 32 nodes further; the sink clips).
// A sink that also wants the position of the sequence's last node defines last_node(node, offset, index) (LocateSink).
template <class Sink, class = void> struct sink_wants_last_node : std::false_type {};
template <class Sink> struct sink_wants_last_node<Sink, std::void_t<decltype(&Sink::last_node)>> : std::true_type {};

template <bool CHECKED, class Sink>
__device__ __forceinline__ uint64_t walk_sequence_warp(const IndexView& ix, uint64_t id, Sink& sink, uint32_t ahead,
                                                       uint64_t limit = ~0ull) {
    uint32_t lane;
    asm volatile("mov.u32 %0, %%laneid;" : "=r"(lane));  // read once: the compiler would re-read the special register per step
    if (id >= ix.sequences) return ~0ull;
    gbwt_b200_pos pos;
    if (!gbwt_start(ix, id, pos)) { sink.finish(); return 0; }
    // the device layout holds node identifiers, offsets and record counts in 32 bits (GBWT_B200_E_RANGE at load)
    const RecordDesc* const descs = ix.desc;
    const Unit16* const bodies = ix.bodies;
    const Unit16* const skips = ix.skips;
    const uint32_t base = static_cast<uint32_t>(ix.offset), records = static_cast<uint32_t>(ix.records);
    uint32_t node = static_cast<uint32_t>(pos.node), offset = static_cast<uint32_t>(pos.offset);
    uint32_t mine = 0, in_group = 0, flush_node = node;
    uint64_t flushed = 0;
    Desc pf;  // this lane's look-ahead descriptor, requested one flush ago
    pf.a.x = pf.a.y = pf.a.z = pf.a.w = pf.b.x = pf.b.y = pf.b.z = pf.b.w = 0;
    Desc d;
    Quad k;
    load_landing<true>(descs, skips, base, records, node, d, k);
    if constexpr (Sink::CHECKPOINTS) sink.checkpoint(node, offset, 0);
    for (;;) {
        if (in_group >= 31) {  // an iteration parks up to two nodes
            sink.group(static_cast<uint64_t>(mine), in_group, flushed);
            flushed += in_group;
            in_group = 0;
            if (flushed >= limit || flushed > ix.walk_limit) break;  // (walk_limit: a damaged index with a cycle)
            // (node, offset) is the position of node number `flushed` of the sequence: what a checkpoint records
            if constexpr (Sink::CHECKPOINTS) sink.checkpoint(node, offset, flushed);
            if (ahead != 0) {
                // Sequences that walk the graph together arrive at a record together and would all wait for the same
                // HBM miss. Node ids follow the graph's topological order, so the records the walk needs next lie a
                // little further in the direction it is moving: lane l asks for the lines of descriptors and
                // shortcuts `ahead + 4 l` records away (the descriptor also as a real load: its body offset is used
                // at the next flush, some 32 nodes later), and for the bodies of the four records it asked for last
                // time.
                // bodies lie in record order: this lane's four records own [its body offset, the next lane's)
                const uint32_t body_at = pf.body(), body_next = __shfl_down_sync(0xFFFFFFFFu, body_at, 1);
                uint32_t span = body_next > body_at ? body_next - body_at : body_at - body_next;
                if (lane == 31 || span > 64u) span = span > 64u ? 64u : 24u;  // at most 1 KiB per lane
                for (uint32_t unit = 0; unit < span; unit += 8) prefetch_l2(bodies + body_at + unit);
                const uint32_t rec = node - base, step = ahead + 4u * lane;
                const bool up = node >= flush_node;
                flush_node = node;
                uint32_t target = up ? rec + step : rec - step;
                if (up ? (target < rec || target >= records) : (target > rec)) target = up ? records - 1u : 0u;
                load_sector(reinterpret_cast<const Unit16*>(descs + target), pf.a, pf.b);
                prefetch_l2(descs + target);  // the whole line: the descriptors of this lane's four records
                prefetch_l2(skips + target);
            }
        }
        // chains of bubbles run here, two register sets alternating; everything else takes the general iteration
        {
            Desc e;
            Quad f;
            bool moved = false;
            for (;;) {
                if (!walk_bubble_step<CHECKED>(d, k, e, f, descs, bodies, skips, base, records, lane, node, offset, mine, in_group)) break;
                if (!walk_bubble_step<CHECKED>(e, f, d, k, descs, bodies, skips, base, records, lane, node, offset, mine, in_group)) { d = e; k = f; break; }
                moved = true;
            }
            (void)moved;
            if (in_group >= 31) continue;
        }
        if (in_group == lane) mine = node;
        in_group++;
        const uint32_t fmt = d.fmt(), i = offset;
        if (i >= d.total_len()) break;  // GBWT::forward -> None (an empty record has length 0)
        if (!d.inline_edges()) {
            // outdegree > 2: the warp scans a byte-per-run body, anything else takes the general one-lane step
            uint32_t next_node, next_offset;
            if (fmt == FMT_RUN8 && d.checkpoints() == 0) {  // (a checkpointed body is a short scan for one lane)
                uint32_t symbol, rank_i;
                warp_lf_runs8(ix, d, i, symbol, rank_i);
                if (symbol == NO_SYMBOL) break;
                const Edge e = edge_at(ix, d, symbol);
                next_node = e.node; next_offset = e.offset + rank_i;
            } else {
                const uint64_t next = forward_other_record(bodies, ix.edges, d.a.x, d.a.y, d.a.z, d.a.w, d.b.x, d.b.y, d.b.z, d.b.w, i);
                next_node = static_cast<uint32_t>(next); next_offset = static_cast<uint32_t>(next >> 32);
            }
            if (next_node == 0) break;
            node = next_node; offset = next_offset;
            load_landing<CHECKED>(descs, skips, base, records, node, d, k);
            continue;
        }
        // where the walk lands over edge 0 / edge 1: two nodes further when the shortcut applies
        const uint32_t land0 = k.x != 0 ? k.x : d.node0(), land1 = k.z != 0 ? k.z : d.node1();
        // A single-edge record, or a bubble whose alleles rejoin at one node (SNPs, indels: most of a pangenome
        // graph): the landing record does not depend on the edge taken, so it is requested once and used as it is.
        const bool same = fmt == FMT_SINGLE || land0 == land1;
        Desc t0, t1;
        Quad s0, s1;
        load_landing<CHECKED>(descs, skips, base, records, land0, t0, s0);
        // (copying t0 into t1 instead of a second request would make the copy wait for the first load before the
        // body block is even requested)
        if (!same) load_landing<CHECKED>(descs, skips, base, records, land1, t1, s1);
        uint32_t b = 0, r = i;  // SINGLE: every position maps to edge 0
        if (fmt != FMT_SINGLE) {
            if (fmt == FMT_DENSE2) {
                const uint32_t blk = __umulhi(i, 0xAAAAAAABu) >> 7;  // i / 192
                Quad lo, hi;
                load_sector(bodies + d.body() + 2u * blk, lo, hi);
                const uint32_t ones = dense_block_rank_lean(lo, hi, i - blk * DENSE_BITS, b);
                r = b ? ones : i - ones;
            } else if (fmt == FMT_RUN8 && d.checkpoints() == 0) {
                warp_lf_runs8(ix, d, i, b, r);
                if (b == NO_SYMBOL) break;
            } else {
                const uint64_t next = forward_other_record(bodies, ix.edges, d.a.x, d.a.y, d.a.z, d.a.w, d.b.x, d.b.y, d.b.z, d.b.w, i);
                if (next == 0) break;
                b = static_cast<uint32_t>(next) == d.node1() && d.node1() != d.node0() ? 1u : 0u;
                r = static_cast<uint32_t>(next >> 32) - (b ? d.offset1() : d.offset0());
            }
        }
        const uint32_t v = b ? d.node1() : d.node0();
        if (v == 0) break;  // successor is the endmarker: the sequence ends (src/bwt.rs:485-486)
        const uint32_t w = b ? k.z : k.x;
        if (w != 0) {
            if (in_group == lane) mine = v;
            in_group++;
            node = w;
            offset = (b ? k.w : k.y) + r;
        } else {
            node = v;
            offset = (b ? d.offset1() : d.offset0()) + r;
        }
        if (same || b == 0) { d = t0; k = s0; }
        else { d = t1; k = s1; }
    }
    if (in_group != 0) sink.group(static_cast<uint64_t>(mine), in_group, flushed);
    // (node, offset) is the position of the last node the walk emitted, unless it stopped at a flush (walk_limit)
    if constexpr (sink_wants_last_node<Sink>::value) { if (in_group != 0) sink.last_node(node, offset, flushed + in_group - 1); }
    sink.finish();
    return flushed + in_group;
}

// K3. GBWT::sequence(id) for a batch (src/gbwt.rs:253-261, 557-568). A path walk is a dependent chain of LF steps,
// so its speed is chains in flight / time per step; paths of a pangenome move through the same records at about
// the same time, so after the first chain has pulled a record into L2 the others hit there.
// k_extract: one warp per sequence (walk_sequence_warp). `nodes == nullptr` only counts.
template <bool CHECKED>
__global__ void __launch_bounds__(128) k_extract(IndexView ix, const uint64_t* __restrict__ ids, size_t m,
                                                  const uint64_t* __restrict__ out_offsets, uint64_t base,
                                                  uint64_t* __restrict__ nodes, uint64_t* __restrict__ lengths,
                                                  uint64_t* __restrict__ seq_len, uint32_t ahead) {
    const size_t warp = (static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x) / 32;
    const size_t warps = (static_cast<size_t>(gridDim.x) * blockDim.x) / 32;
    for (size_t i = warp; i < m; i += warps) {
        const uint64_t id = __ldg(ids + i);
        NodeSink sink{nullptr, 0, id & 1ull, SigAcc{}};
        if (nodes != nullptr) {
            const uint64_t lo = __ldg(out_offsets + i), hi = __ldg(out_offsets + i + 1);
            sink.out = nodes + (lo - base);
            sink.cap = hi > lo ? hi - lo : 0;
        }
        const uint64_t len = walk_sequence_warp<CHECKED>(ix, id, sink, ahead);
        const SeqSignature signature = sink.sig.total();
        if ((threadIdx.x & 31u) == 0) {
            if (lengths != nullptr) lengths[i] = len;
            if (seq_len != nullptr && id < ix.sequences) {  // remembered for k_extract_split
                store_signature(signatures_of(seq_len, ix.sequences), id, signature);
                seq_len[id] = len;
            }
        }
    }
}

constexpr uint64_t SEQ_LEN_UNKNOWN = 0xFEFEFEFEFEFEFEFEull;  // what cudaMemset(0xFE) leaves in the length cache

// k_extract_split: a walk is a dependent chain, and a bidirectional index offers a second way in: sequence id ^ 1 is
// the same path on the other strand, so it starts where sequence id ends. Once the length of a sequence is known
// (any earlier k_extract, e.g. the sequence_lengths call that sized the output, leaves it in `seq_len`), two warps
// of one CTA walk it from both ends and meet in the middle: twice the chains in flight, half the chain length.
// A sequence is only split when both of its strands have been walked whole before and their signatures say that they
// are mirror images (strands_mirror above); the halves are still compared where they meet, and if they disagree the
// first warp redoes the sequence from the front alone, which is what the reference does. One call site of the walk
// serves all three cases, so the kernel stays at the register count of the plain one.
template <bool CHECKED>
__global__ void __launch_bounds__(64) k_extract_split(IndexView ix, const uint64_t* __restrict__ ids, size_t m,
                                                       const uint64_t* __restrict__ out_offsets, uint64_t base,
                                                       uint64_t* __restrict__ nodes, uint64_t* __restrict__ lengths,
                                                       uint64_t* __restrict__ seq_len, uint32_t ahead) {
    __shared__ uint64_t meet[2];
    const uint32_t half = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    for (size_t i = blockIdx.x; i < m; i += gridDim.x) {
        const uint64_t id = __ldg(ids + i);
        const uint64_t lo = __ldg(out_offsets + i), hi = __ldg(out_offsets + i + 1);
        const uint64_t cap = hi > lo ? hi - lo : 0;
        const uint64_t known = id < ix.sequences ? seq_len[id] : SEQ_LEN_UNKNOWN;
        // (a short sequence is not worth two warps)
        bool split = known != SEQ_LEN_UNKNOWN && known >= 128 && strands_mirror(seq_len, signatures_of(seq_len, ix.sequences), id, ix.sequences);
        uint64_t len = known;
        // at most two rounds: the halves, then (only if they disagree where they meet) the whole sequence from the front
        for (;;) {
            const uint64_t mid = known / 2;  // both halves produce position `mid`; the far half writes it
            HalfSink sink;
            sink.out = nodes + (lo - base); sink.cap = cap; sink.value = ~0ull; sink.flip = id & 1ull;
            if (!split) { sink.len = 0; sink.lo = 0; sink.hi = ~0ull; sink.probe = ~0ull; sink.reverse = false; }
            else if (half == 0) { sink.len = known; sink.lo = 0; sink.hi = mid; sink.probe = mid; sink.reverse = false; }
            else { sink.len = known; sink.lo = mid; sink.hi = known; sink.probe = mid; sink.reverse = true; }
            if (split || half == 0) {
                const uint64_t walked = walk_sequence_warp<CHECKED>(ix, split && half == 1 ? id ^ 1ull : id, sink, ahead,
                                                                    !split ? ~0ull : (half == 0 ? mid + 1 : known - mid));
                if (!split) {
                    len = walked;
                    const SeqSignature signature = sink.sig.total();
                    if (lane == 0 && id < ix.sequences) {
                        store_signature(signatures_of(seq_len, ix.sequences), id, signature);
                        seq_len[id] = walked;
                    }
                } else if (lane == 0) {
                    meet[half] = sink.value;
                }
            }
            __syncthreads();
            const bool agree = !split || (meet[0] == meet[1] && meet[0] != ~0ull);
            __syncthreads();
            if (agree) break;
            split = false;
        }
        if (threadIdx.x == 0 && lengths != nullptr) lengths[i] = len;
    }
}

// k_extract_lanes: `stride` threads per sequence, the first of them walks (stride 1 = one sequence per thread, for
// batches with far more sequences than the device has warp slots).
__global__ void __launch_bounds__(64) k_extract_lanes(IndexView ix, const uint64_t* __restrict__ ids, size_t m,
                                                       const uint64_t* __restrict__ out_offsets, uint64_t base,
                                                       uint64_t* __restrict__ nodes, uint64_t* __restrict__ lengths, uint32_t stride) {
    const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (tid % stride != 0) return;
    for (size_t i = tid / stride; i < m; i += (static_cast<size_t>(gridDim.x) * blockDim.x) / stride) {
        uint64_t* out = nullptr;
        uint64_t cap = 0;
        if (nodes != nullptr) {
            const uint64_t lo = __ldg(out_offsets + i), hi = __ldg(out_offsets + i + 1);
            out = nodes + (lo - base);
            cap = hi > lo ? hi - lo : 0;
        }
        const uint64_t len = walk_sequence_lane(ix, __ldg(ids + i), out, cap);
        if (lengths != nullptr) lengths[i] = len;
    }
}

// K4. extract_sequence of src/bin/gbz-extract.rs:173-189 for many GBWT sequences: one warp per sequence walks the
// path (K3) and spells the node labels as it goes, then appends the endmarker byte. lengths[i] = bytes of the
// full result (endmarker included), UINT64_MAX where GBZ::path is None; `bytes == nullptr` only measures.
template <bool CHECKED>
__global__ void __launch_bounds__(128) k_extract_dna(IndexView ix, GraphView graph, const uint64_t* __restrict__ ids, size_t m,
                                                      const uint64_t* __restrict__ out_offsets, uint64_t base, uint32_t endmarker,
                                                      uint8_t* __restrict__ bytes, uint64_t* __restrict__ lengths,
                                                      uint64_t* __restrict__ seq_len, uint64_t* __restrict__ dna_len, uint32_t ahead) {
    const size_t warp = (static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x) / 32;
    const size_t warps = (static_cast<size_t>(gridDim.x) * blockDim.x) / 32;
    for (size_t i = warp; i < m; i += warps) {
        DnaSink sink{graph, ix.offset + 1, nullptr, 0, 0, 0, 0, 0, false, false, ~0ull, ~0ull, ~0ull, 0, false};
        if (bytes != nullptr) {
            const uint64_t lo = __ldg(out_offsets + i), hi = __ldg(out_offsets + i + 1);
            sink.out = bytes + (lo - base);
            sink.cap = hi > lo ? hi - lo : 0;
        }
        const uint64_t id = __ldg(ids + i);
        sink.flip = id & 1ull;
        const uint64_t len = walk_sequence_warp<CHECKED>(ix, id, sink, ahead);
        const SeqSignature signature = sink.sig.total();
        if ((threadIdx.x & 31u) != 0) continue;
        if (len == ~0ull) {
            if (lengths != nullptr) lengths[i] = ~0ull;
            continue;
        }
        if (sink.out != nullptr && sink.written < sink.cap) sink.out[sink.written] = static_cast<uint8_t>(endmarker);
        if (lengths != nullptr) lengths[i] = sink.written + 1;
        store_signature(signatures_of(seq_len, ix.sequences), id, signature);
        seq_len[id] = len;               // remembered for k_extract_dna_split
        dna_len[id] = sink.written + 1;
    }
}

// K4, two-ended: as k_extract_split, for DNA. With the node count and the DNA length of a sequence known, the first
// warp spells nodes [0, mid) from the front and the second walks the other strand and writes the rest downwards from
// the end. Accepted only if the halves meet at the same node and their bytes add up to the known length.
template <bool CHECKED>
__global__ void __launch_bounds__(64) k_extract_dna_split(IndexView ix, GraphView graph, const uint64_t* __restrict__ ids, size_t m,
                                                           const uint64_t* __restrict__ out_offsets, uint64_t base, uint32_t endmarker,
                                                           uint8_t* __restrict__ bytes, uint64_t* __restrict__ lengths,
                                                           uint64_t* __restrict__ seq_len, uint64_t* __restrict__ dna_len, uint32_t ahead) {
    __shared__ uint64_t meet[2], spelled[2];
    const uint32_t half = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    for (size_t i = blockIdx.x; i < m; i += gridDim.x) {
        const uint64_t id = __ldg(ids + i);
        const uint64_t lo = __ldg(out_offsets + i), hi = __ldg(out_offsets + i + 1);
        const uint64_t cap = hi > lo ? hi - lo : 0;
        const bool in_range = id < ix.sequences;
        const uint64_t known = in_range ? seq_len[id] : SEQ_LEN_UNKNOWN, known_dna = in_range ? dna_len[id] : SEQ_LEN_UNKNOWN;
        bool split = known != SEQ_LEN_UNKNOWN && known_dna != SEQ_LEN_UNKNOWN && known >= 128 &&
                     strands_mirror(seq_len, signatures_of(seq_len, ix.sequences), id, ix.sequences);
        uint64_t result = known_dna;
        for (;;) {
            const uint64_t mid = known / 2;
            DnaSink sink{graph, ix.offset + 1, bytes + (lo - base), cap, 0, 0, 0, 0, false, false, ~0ull, ~0ull, ~0ull, 0, false};
            if (split) {
                sink.probe = half == 0 ? mid : known - 1 - mid;
                sink.node_limit = half == 0 ? mid : known - mid;
                sink.mirror = half == 1;
                sink.end = known_dna - 1;
            }
            if (split || half == 0) {
                sink.flip = id & 1ull;
                const uint64_t walked = walk_sequence_warp<CHECKED>(ix, split && half == 1 ? id ^ 1ull : id, sink, ahead,
                                                                    !split ? ~0ull : (half == 0 ? mid + 1 : known - mid));
                const SeqSignature signature = sink.sig.total();
                if (lane == 0) {
                    if (!split) {
                        result = walked == ~0ull ? ~0ull : sink.written + 1;
                        if (walked != ~0ull) {
                            if (sink.written < cap) sink.out[sink.written] = static_cast<uint8_t>(endmarker);
                            store_signature(signatures_of(seq_len, ix.sequences), id, signature);
                            seq_len[id] = walked;
                            dna_len[id] = sink.written + 1;
                        }
                    } else {
                        meet[half] = sink.value;
                        spelled[half] = sink.written;
                        if (half == 0 && known_dna - 1 < cap) sink.out[known_dna - 1] = static_cast<uint8_t>(endmarker);
                    }
                }
            }
            __syncthreads();
            const bool agree = !split || (meet[0] == meet[1] && meet[0] != ~0ull && spelled[0] + spelled[1] == known_dna - 1);
            __syncthreads();
            if (agree) break;
            split = false;
        }
        if (threadIdx.x == 0 && lengths != nullptr) lengths[i] = result;
    }
}

// ---- K4 with a spelling warp ---------------------------------------------------------------------------------------
// The walk is a latency-bound dependent chain; spelling a group of nodes costs a few hundred instructions that have
// nothing to do with it. In this variant the two walking warps of a CTA only park their nodes in a shared-memory ring
// and a third warp does all the spelling (label ranges, scan, byte copy) for both: the walks run at the speed of plain
// node extraction. Ring protocol per slot: the walker waits for full == 0, writes the 32 nodes + count + first index,
// fences and sets full = 1; the speller waits for full == 1, spells, sets full = 0. count == RELAY_DONE ends a walk.
constexpr uint32_t RELAY_SLOTS = 4, RELAY_DONE = 0xFFFFFFFFu;

struct RelayRing {
    uint32_t nodes[RELAY_SLOTS][32];
    uint64_t first[RELAY_SLOTS];
    uint32_t count[RELAY_SLOTS];
    uint32_t full[RELAY_SLOTS];
};

__device__ __forceinline__ uint32_t relay_flag(const uint32_t* flag) { return *reinterpret_cast<const volatile uint32_t*>(flag); }
__device__ __forceinline__ void relay_set(uint32_t* flag, uint32_t v) { *reinterpret_cast<volatile uint32_t*>(flag) = v; }

// The walker's side of the ring (also keeps the node at index `probe`, flipped on the mirrored strand).
struct RelaySink {
    static constexpr bool CHECKPOINTS = false;
    RelayRing* ring;
    uint32_t slot;
    uint64_t probe, value;
    bool mirror;
    uint64_t flip = 0;
    SigAcc sig;
    __device__ __forceinline__ void post(uint32_t node, uint32_t count, uint64_t first) {
        const uint32_t lane = threadIdx.x & 31u;
        while (relay_flag(&ring->full[slot]) != 0) __nanosleep(40);
        ring->nodes[slot][lane] = node;
        if (lane == 0) { ring->count[slot] = count; ring->first[slot] = first; }
        __syncwarp();
        __threadfence_block();
        if (lane == 0) relay_set(&ring->full[slot], 1u);
        slot = (slot + 1u) % RELAY_SLOTS;
    }
    __device__ __forceinline__ void group(uint64_t mine, uint32_t count, uint64_t first) {
        const uint32_t lane = threadIdx.x & 31u;
        const unsigned hit = __ballot_sync(0xFFFFFFFFu, lane < count && first + lane == probe);
        if (hit != 0) value = __shfl_sync(0xFFFFFFFFu, mirror ? mine ^ 1ull : mine, __ffs(static_cast<int>(hit)) - 1);
        sig.add(mine, count, first, flip);
        post(static_cast<uint32_t>(mine), count, first);
    }
    __device__ __forceinline__ void finish() {}
};

// The speller's side: takes whatever is ready on the ring; returns true when the walk has ended.
__device__ __forceinline__ bool relay_take(RelayRing* ring, uint32_t& slot, DnaSink& sink, bool& progressed) {
    const uint32_t lane = threadIdx.x & 31u;
    if (relay_flag(&ring->full[slot]) != 1u) return false;
    __threadfence_block();
    const uint32_t count = ring->count[slot];
    const uint64_t first = ring->first[slot];
    const uint32_t node = ring->nodes[slot][lane];
    __syncwarp();
    if (lane == 0) relay_set(&ring->full[slot], 0u);  // the values are in registers: the walker may reuse the slot
    slot = (slot + 1u) % RELAY_SLOTS;
    progressed = true;
    if (count == RELAY_DONE) { sink.finish(); return true; }
    sink.group(static_cast<uint64_t>(node), count, first);
    return false;
}

template <bool CHECKED>
__global__ void __launch_bounds__(96, 7) k_extract_dna_relay(IndexView ix, GraphView graph, const uint64_t* __restrict__ ids, size_t m,
                                                              const uint64_t* __restrict__ out_offsets, uint64_t base, uint32_t endmarker,
                                                              uint8_t* __restrict__ bytes, uint64_t* __restrict__ lengths,
                                                              uint64_t* __restrict__ seq_len, uint64_t* __restrict__ dna_len, uint32_t ahead) {
    __shared__ RelayRing rings[2];
    __shared__ uint64_t meet[2], spelled[2], walked_nodes;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    for (size_t i = blockIdx.x; i < m; i += gridDim.x) {
        const uint64_t id = __ldg(ids + i);
        const uint64_t lo = __ldg(out_offsets + i), hi = __ldg(out_offsets + i + 1);
        const uint64_t cap = hi > lo ? hi - lo : 0;
        uint8_t* out = bytes + (lo - base);
        const bool in_range = id < ix.sequences;
        const uint64_t known = in_range ? seq_len[id] : SEQ_LEN_UNKNOWN, known_dna = in_range ? dna_len[id] : SEQ_LEN_UNKNOWN;
        bool split = known != SEQ_LEN_UNKNOWN && known_dna != SEQ_LEN_UNKNOWN && known >= 128 &&
                     strands_mirror(seq_len, signatures_of(seq_len, ix.sequences), id, ix.sequences);
        uint64_t result = known_dna;
        for (;;) {
            const uint64_t mid = known / 2;
            if (threadIdx.x < 2 * RELAY_SLOTS) rings[threadIdx.x / RELAY_SLOTS].full[threadIdx.x % RELAY_SLOTS] = 0;
            __syncthreads();
            if (warp < 2) {
                if (split || warp == 0) {
                    RelaySink sink{&rings[warp], 0, ~0ull, ~0ull, split && warp == 1};
                    sink.flip = id & 1ull;
                    if (split) sink.probe = warp == 0 ? mid : known - 1 - mid;
                    const uint64_t walked = walk_sequence_warp<CHECKED>(ix, split && warp == 1 ? id ^ 1ull : id, sink, ahead,
                                                                        !split ? ~0ull : (warp == 0 ? mid + 1 : known - mid));
                    sink.post(0, RELAY_DONE, 0);
                    const SeqSignature signature = sink.sig.total();
                    if (lane == 0) {
                        meet[warp] = sink.value;
                        if (warp == 0) walked_nodes = walked;
                        // (a whole walk; its length is stored below by thread 0 once the speller is done)
                        if (!split && walked != ~0ull) store_signature(signatures_of(seq_len, ix.sequences), id, signature);
                    }
                }
            } else {
                // the spelling warp: one DnaSink per walking warp
                DnaSink front{graph, ix.offset + 1, out, cap, 0, 0, 0, 0, false, false, ~0ull, ~0ull, ~0ull, 0, false};
                DnaSink back{graph, ix.offset + 1, out, cap, 0, 0, 0, 0, false, false, ~0ull, ~0ull, ~0ull, 0, false};
                if (split) {
                    front.node_limit = mid;
                    back.node_limit = known - mid; back.mirror = true; back.end = known_dna - 1;
                }
                bool front_done = false, back_done = !split;
                uint32_t front_slot = 0, back_slot = 0;
                while (!(front_done && back_done)) {
                    bool progressed = false;
                    if (!front_done) front_done = relay_take(&rings[0], front_slot, front, progressed);
                    if (!back_done) back_done = relay_take(&rings[1], back_slot, back, progressed);
                    if (!progressed) __nanosleep(100);
                }
                if (lane == 0) { spelled[0] = front.written; spelled[1] = back.written; }
            }
            __syncthreads();
            const bool ended = walked_nodes != ~0ull;  // (non-split) ~0: GBZ::path is None
            const bool agree = !split || (meet[0] == meet[1] && meet[0] != ~0ull && spelled[0] + spelled[1] == known_dna - 1);
            if (threadIdx.x == 0) {
                if (!split) {
                    result = ended ? spelled[0] + 1 : ~0ull;
                    if (ended) {
                        if (spelled[0] < cap) out[spelled[0]] = static_cast<uint8_t>(endmarker);
                        seq_len[id] = walked_nodes;
                        dna_len[id] = spelled[0] + 1;
                    }
                } else if (agree && known_dna - 1 < cap) {
                    out[known_dna - 1] = static_cast<uint8_t>(endmarker);
                }
            }
            __syncthreads();
            if (agree) break;
            split = false;
        }
        if (threadIdx.x == 0 && lengths != nullptr) lengths[i] = result;
    }
}

// GBZ::sequence(node_id) for a batch of original-graph node identifiers (src/gbz.rs:286-298): lengths[i] = label
// length, UINT64_MAX where the reference returns None (no such node: outside the alphabet or an empty record);
// with `bytes`, label i is copied to bytes[out_offsets[i] - base ..), truncated to its slot. One warp per node.
__global__ void k_node_sequences(IndexView ix, GraphView graph, const uint64_t* __restrict__ node_ids, size_t n,
                                 const uint64_t* __restrict__ out_offsets, uint64_t base, uint8_t* __restrict__ bytes,
                                 uint64_t* __restrict__ lengths) {
    const uint32_t lane = threadIdx.x & 31u;
    const size_t warp = (static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x) / 32;
    const size_t warps = (static_cast<size_t>(gridDim.x) * blockDim.x) / 32;
    for (size_t i = warp; i < n; i += warps) {
        const uint64_t id = __ldg(node_ids + i);
        uint64_t len = ~0ull, lo = 0;
        // GBZ::has_node: inside the alphabet and a non-empty record
        if (id <= (~0ull >> 1) && 2 * id > ix.offset && 2 * id < ix.alphabet_size) {
            const uint64_t sid = (2 * id - (ix.offset + 1)) >> 1;
            const Desc d = load_desc_of(ix, 2 * id);
            if (d.fmt() != FMT_EMPTY && sid < graph.sequences) {
                lo = __ldg(graph.starts + sid);
                len = __ldg(graph.starts + sid + 1) - lo;
            }
        }
        if (lane == 0 && lengths != nullptr) lengths[i] = len;
        if (bytes == nullptr || len == ~0ull) continue;
        const uint64_t o_lo = __ldg(out_offsets + i), o_hi = __ldg(out_offsets + i + 1);
        const uint64_t cap = o_hi > o_lo ? o_hi - o_lo : 0;
        const uint64_t count = len < cap ? len : cap;
        for (uint64_t j = lane; j < count; j += 32) bytes[o_lo - base + j] = __ldg(graph.bytes + lo + j);
    }
}

// ---- K3 with checkpoints: extraction that is parallel ALONG the paths ---------------------------------------------------
// A path walk is a dependent chain (src/gbwt.rs:557-568): however many paths a batch has, nothing can make one chain
// of 6.7 M LF steps take less than 6.7 M round trips. What breaks the chain is knowing positions in its middle. When
// the index is created, one pass of the warp-mode walk over every sequence records the position (node, offset) at
// about every `interval`-th node (k_build_checkpoints; like the DA samples of the reference's GBWT, but indexed by
// sequence and rank instead of by BWT position). A sequence is then extracted as independent segments, each walked
// from its checkpoint to the next by ONE lane: a batch of 1024 paths of 6.7 M nodes is 6.7 M independent walks of
// ~1024 steps instead of 1024 chains, latency is hidden by occupancy like in the search kernels, and the 32 lanes of
// a warp take the same segment number of 32 neighbouring sequences, which in a pangenome walk the same records at the
// same time (their loads coalesce into a handful of sectors). Every node is still produced by an LF step.

// (struct Checkpoint and CheckpointView: layout.h)
struct PoolEntry { uint32_t seq, node, offset, pad; uint64_t index, pad2; };  // as the build walk emits them
static_assert(sizeof(Checkpoint) == 16 && sizeof(PoolEntry) == 32, "checkpoint records are loaded with vector loads");

struct CheckpointSink {
    static constexpr bool CHECKPOINTS = true;
    PoolEntry* pool;
    unsigned long long* pool_used;
    uint64_t pool_cap;
    uint32_t seq, shift;
    uint64_t next;  // first index that wants a checkpoint
    SigAcc sig;
    __device__ __forceinline__ void group(uint64_t mine, uint32_t count, uint64_t first) { sig.add(mine, count, first, seq & 1u); }
    __device__ __forceinline__ void finish() {}
    // called at every flush of the walk (at most 32 nodes apart), so every multiple of the interval gets the first
    // flush at or after it
    __device__ __forceinline__ void checkpoint(uint32_t node, uint32_t offset, uint64_t index) {
        if (index < next) return;
        next = ((index >> shift) + 1) << shift;
        if ((threadIdx.x & 31u) != 0) return;
        const unsigned long long slot = atomicAdd(pool_used, 1ull);
        if (slot >= pool_cap) return;  // cannot happen on a consistent index (the pool holds total length / interval + sequences)
        PoolEntry e;
        e.seq = seq; e.node = node; e.offset = offset; e.pad = 0; e.index = index; e.pad2 = 0;
        pool[slot] = e;
    }
};

// One warp per sequence: walks it once, leaves its length in seq_len[] and its checkpoints in the pool.
template <bool CHECKED>
__global__ void __launch_bounds__(128) k_build_checkpoints(IndexView ix, uint32_t shift, PoolEntry* __restrict__ pool,
                                                            unsigned long long* __restrict__ pool_used, uint64_t pool_cap,
                                                            uint64_t* __restrict__ seq_len, uint32_t ahead) {
    const size_t warp = (static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x) / 32;
    const size_t warps = (static_cast<size_t>(gridDim.x) * blockDim.x) / 32;
    for (size_t id = warp; id < ix.sequences; id += warps) {
        CheckpointSink sink{pool, pool_used, pool_cap, static_cast<uint32_t>(id), shift, 0, SigAcc{}};
        const uint64_t len = walk_sequence_warp<CHECKED>(ix, id, sink, ahead);
        const SeqSignature signature = sink.sig.total();
        if ((threadIdx.x & 31u) == 0) {
            store_signature(signatures_of(seq_len, ix.sequences), id, signature);
            seq_len[id] = len;
        }
    }
}

// counts[1 + seq] = checkpoints of the sequence (the exclusive scan of it gives every sequence's first slot).
__global__ void __launch_bounds__(BLOCK_THREADS) k_checkpoint_count(const PoolEntry* __restrict__ pool, uint64_t used,
                                                                     uint32_t* __restrict__ counts) {
    GBWT_GRID_STRIDE(i, used) atomicAdd(counts + 1 + pool[i].seq, 1u);
}

// table[first[seq] + index / interval] = the checkpoint (slots of a sequence are consecutive, see CheckpointSink).
__global__ void __launch_bounds__(BLOCK_THREADS) k_checkpoint_scatter(const PoolEntry* __restrict__ pool, uint64_t used, uint32_t shift,
                                                                       const uint32_t* __restrict__ first, Checkpoint* __restrict__ table) {
    GBWT_GRID_STRIDE(i, used) {
        const PoolEntry e = pool[i];
        Checkpoint c;
        c.node = e.node; c.offset = e.offset; c.index = e.index;
        table[first[e.seq] + static_cast<uint32_t>(e.index >> shift)] = c;
    }
}


// ---- locate samples (gbwt_b200_locate; DESIGN.md "Locate") ---------------------------------------------------------
// The same walk as the checkpoints, with the table inverted: indexed by BWT position instead of by sequence. Every
// sample is emitted as a sort key (record << 32 | offset) and the sample itself; locate.cu sorts them into the table.
// Rule: a sample at the first flush at or after every multiple of 2^shift (flushes are at most 32 nodes apart), and at
// the sequence's last node. A locate walk therefore meets one within 2^shift + 32 LF steps. The last node is sampled
// because that is where every walk would otherwise leave the sequence: GBWT::forward is None there, and nothing in the
// format ties the endmarker position it would enter to the sequence id.
struct LocateSink {
    static constexpr bool CHECKPOINTS = true;
    uint64_t* keys;
    LocateSample* samples;
    unsigned long long* used;
    uint64_t cap, base, records;  // base = alphabet offset (record = node - base)
    uint32_t seq, shift;
    uint64_t next, last;  // first index that wants a sample; index of the last sample emitted (~0 = none)
    __device__ __forceinline__ void emit(uint32_t node, uint32_t offset, uint64_t index) {
        last = index;
        // (a damaged index can lead a walk to a node without a record: no position there can be located)
        if ((threadIdx.x & 31u) != 0 || node <= base || node - base >= records) return;
        const unsigned long long slot = atomicAdd(used, 1ull);
        if (slot >= cap) return;  // (the caller sees used > cap and fails: cannot happen on a consistent index)
        keys[slot] = (static_cast<uint64_t>(node - base) << 32) | offset;
        LocateSample e;
        e.offset = offset; e.seq = seq; e.index = index;
        samples[slot] = e;
    }
    __device__ __forceinline__ void group(uint64_t, uint32_t, uint64_t) {}
    __device__ __forceinline__ void finish() {}
    __device__ __forceinline__ void checkpoint(uint32_t node, uint32_t offset, uint64_t index) {
        if (index < next) return;
        next = ((index >> shift) + 1) << shift;
        emit(node, offset, index);
    }
    __device__ __forceinline__ void last_node(uint32_t node, uint32_t offset, uint64_t index) {
        if (index != last) emit(node, offset, index);
    }
};

// One warp per sequence (shift >= 5: the flushes are denser than the samples).
template <bool CHECKED>
__global__ void __launch_bounds__(128) k_build_locate(IndexView ix, uint32_t shift, uint64_t* __restrict__ keys,
                                                       LocateSample* __restrict__ samples, unsigned long long* __restrict__ used,
                                                       uint64_t cap, uint32_t ahead) {
    const size_t warp = (static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x) / 32;
    const size_t warps = (static_cast<size_t>(gridDim.x) * blockDim.x) / 32;
    for (size_t id = warp; id < ix.sequences; id += warps) {
        LocateSink sink{keys, samples, used, cap, ix.offset, ix.records, static_cast<uint32_t>(id), shift, 0, ~0ull};
        walk_sequence_warp<CHECKED>(ix, id, sink, ahead);
    }
}

// Intervals shorter than a flush (shift < 5; shift 0 is the whole document array, for tests): one lane per sequence
// walks it with GBWT::forward and samples exactly every multiple of 2^shift and the last node.
__global__ void __launch_bounds__(BLOCK_THREADS) k_build_locate_lanes(IndexView ix, uint32_t shift, uint64_t* __restrict__ keys,
                                                                       LocateSample* __restrict__ samples,
                                                                       unsigned long long* __restrict__ used, uint64_t cap) {
    GBWT_GRID_STRIDE(id, ix.sequences) {
        gbwt_b200_pos pos;
        if (!gbwt_start(ix, id, pos)) continue;
        for (uint64_t j = 0; j <= ix.walk_limit; j++) {
            gbwt_b200_pos next;
            const bool more = gbwt_forward(ix, pos, next);
            const bool located = pos.node > ix.offset && pos.node - ix.offset < ix.records;  // (see LocateSink::emit)
            if (located && (!more || (j & ((uint64_t(1) << shift) - 1)) == 0)) {
                const unsigned long long slot = atomicAdd(used, 1ull);
                if (slot < cap) {
                    keys[slot] = ((pos.node - ix.offset) << 32) | pos.offset;
                    LocateSample e;
                    e.offset = static_cast<uint32_t>(pos.offset); e.seq = static_cast<uint32_t>(id); e.index = j;
                    samples[slot] = e;
                }
            }
            if (!more) break;
            pos = next;
        }
    }
}

// Work item (segment j, block of 32 batch entries): lane l walks segment j of sequence ids[32 * block + l] from its
// checkpoint to the next one (or to the end of the sequence): Record::lf (src/bwt.rs:480-496) per step, two nodes per
// step where the two-hop shortcut applies (layout.h). Items are ordered by segment number first, so the CTAs running at
// any moment are all in the same part of the graph.
//
// Output: a first version stored every node straight from its lane, 8 bytes to 32 different rows per instruction. ncu
// (profiles/r2_extract_checkpointed_v1_ncu.txt): 1.7 G partial-sector writes churn through L2, evict the index (L2 read
// hit rate 18 %) and the walks wait on DRAM for every record -- 39 G LF steps/s. Now every lane parks its nodes in a row
// of a shared-memory tile (as 32-bit values), and when a row is nearly full the warp writes all rows out, up to 512
// contiguous bytes per row with streaming stores: whole sectors that L2 need not keep, in pieces long enough for DRAM
// (with 128-byte pieces the 300 k concurrent output streams ran at 1.4 TB/s, every piece opening a DRAM page of its own).
constexpr uint32_t TILE_NODES = 64, TILE_STRIDE = 65;  // nodes (32-bit) per lane between flushes; row stride in words

// Index loads of the segment walks: the output of an extraction streams tens of GB through L2 and, even written with
// evict-first stores, pushed the index out (L2 read hit rate 9 % in the capture of that version: every record fetch went to DRAM
// behind the writes; the shipped kernel's capture is profiles/r2_extract_checkpointed_v3_ncu.txt). These loads ask L2 to keep what they touch (evict_last).
__device__ __forceinline__ uint64_t keep_policy() {
    uint64_t policy;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(policy));
    return policy;
}
__device__ __forceinline__ void load_sector_keep(const Unit16* p, uint64_t policy, Quad& lo, Quad& hi) {
    asm volatile("ld.global.nc.L2::cache_hint.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8], %9;"
                 : "=r"(lo.x), "=r"(lo.y), "=r"(lo.z), "=r"(lo.w), "=r"(hi.x), "=r"(hi.y), "=r"(hi.z), "=r"(hi.w)
                 : "l"(p), "l"(policy));
}
__device__ __forceinline__ Quad load_quad_keep(const Unit16* p, uint64_t policy) {
    Quad q;
    asm volatile("ld.global.nc.L2::cache_hint.v4.b32 {%0, %1, %2, %3}, [%4], %5;" : "=r"(q.x), "=r"(q.y), "=r"(q.z), "=r"(q.w) : "l"(p), "l"(policy));
    return q;
}

// State of one lane's segment walk. `left` = nodes of the segment still to be emitted (0 = done).
struct SegmentLane {
    uint32_t node, offset, left, parked;
};

// Descriptor + shortcut of node v. A node without a record (only possible on an index with invalid edge targets) gets
// an all-zero descriptor: length 0, so the walk emits the node and ends there, like GBWT::forward returning None.
template <bool CHECKED>
__device__ __forceinline__ void load_segment_record(const RecordDesc* descs, const Unit16* skips, uint32_t base, uint32_t records,
                                                    uint64_t keep, uint32_t v, Desc& d, Quad& k) {
    uint32_t rec = v - base;
    if (CHECKED && rec - 1u >= records - 1u) {
        d.a.x = d.a.y = d.a.z = d.a.w = d.b.x = d.b.y = d.b.z = d.b.w = 0;
        k.x = k.y = k.z = k.w = 0;
        return;
    }
    rec = rec < records ? rec : records - 1u;  // (v == 0, the endmarker as a successor: any valid address will do, the result is unused)
    load_sector_keep(reinterpret_cast<const Unit16*>(descs + rec), keep, d.a, d.b);
    k = load_quad_keep(skips + rec, keep);
}

// One step of a segment walk: emits the current node (whose record is in cur_d / cur_k) and, over a two-hop shortcut, its
// successor; leaves the record of the node it lands on in nxt_d / nxt_k. The caller alternates the two register sets, so
// no descriptor is ever copied. The landing record over edge 0 is requested BEFORE the block that decides the edge is
// looked at: in a bubble both edges land on the same node and a step is one memory round trip; otherwise edge 1 pays a
// second one.
template <bool CHECKED>
__device__ __forceinline__ void segment_step(SegmentLane& st, const Desc& cur_d, const Quad& cur_k, Desc& nxt_d, Quad& nxt_k, uint32_t* row,
                                             const RecordDesc* descs, const Unit16* bodies, const Unit16* skips, const Edge* edges,
                                             uint32_t base, uint32_t records, uint64_t keep) {
    row[st.parked++] = st.node;
    const uint32_t fmt = cur_d.fmt(), at = st.offset;
    if (at >= cur_d.total_len()) { st.left = 0; return; }  // GBWT::forward -> None (an empty record has length 0)
    if (fmt == FMT_SINGLE || fmt == FMT_DENSE2) {
        const uint32_t land0 = cur_k.x != 0 ? cur_k.x : cur_d.node0();
        load_segment_record<CHECKED>(descs, skips, base, records, keep, land0, nxt_d, nxt_k);  // (node 0: the endmarker's record, unused)
        uint32_t b = 0, r = at;
        if (fmt == FMT_DENSE2) {
            const uint32_t blk = __umulhi(at, 0xAAAAAAABu) >> 7;  // at / 192
            Quad lo, hi;
            load_sector_keep(bodies + cur_d.body() + 2u * blk, keep, lo, hi);
            const uint32_t ones = dense_block_rank_lean(lo, hi, at - blk * DENSE_BITS, b);
            r = b ? ones : at - ones;
        }
        const uint32_t v = b ? cur_d.node1() : cur_d.node0();
        const uint32_t w = b ? cur_k.z : cur_k.x;
        if (v == 0) { st.left = 0; return; }  // successor is the endmarker: the sequence ends (src/bwt.rs:485-486)
        uint32_t advance = 1;
        if (w != 0) {
            if (st.left > 1) row[st.parked++] = v;
            st.node = w; st.offset = (b ? cur_k.w : cur_k.y) + r;
            advance = 2;
        } else {
            st.node = v; st.offset = (b ? cur_d.offset1() : cur_d.offset0()) + r;
        }
        st.left = st.left > advance ? st.left - advance : 0;
        if (st.left != 0 && st.node != land0) load_segment_record<CHECKED>(descs, skips, base, records, keep, st.node, nxt_d, nxt_k);
    } else {
        const uint64_t next = forward_other_record(bodies, edges, cur_d.a.x, cur_d.a.y, cur_d.a.z, cur_d.a.w, cur_d.b.x, cur_d.b.y, cur_d.b.z,
                                                   cur_d.b.w, at);
        if (next == 0) { st.left = 0; return; }
        st.node = static_cast<uint32_t>(next); st.offset = static_cast<uint32_t>(next >> 32);
        st.left -= 1;
        if (st.left != 0) load_segment_record<CHECKED>(descs, skips, base, records, keep, st.node, nxt_d, nxt_k);
    }
}

template <bool CHECKED, int THREADS>
__global__ void __launch_bounds__(THREADS) k_extract_checkpointed(IndexView ix, CheckpointView cv, const uint64_t* __restrict__ ids,
                                                                         size_t m, const uint64_t* __restrict__ out_offsets, uint64_t base_offset,
                                                                         uint64_t* __restrict__ nodes, uint64_t* __restrict__ lengths) {
    constexpr unsigned FULL = 0xFFFFFFFFu;
    extern __shared__ __align__(16) unsigned char tile_bytes[];  // [THREADS / 32][32][TILE_STRIDE] words
    uint32_t (*tiles)[32][TILE_STRIDE] = reinterpret_cast<uint32_t (*)[32][TILE_STRIDE]>(tile_bytes);
    const uint32_t lane = threadIdx.x & 31u;
    uint32_t (*tile)[TILE_STRIDE] = tiles[threadIdx.x >> 5];
    uint32_t* const row = tile[lane];
    const uint64_t keep = keep_policy();
    const RecordDesc* const descs = ix.desc;
    const Unit16* const bodies = ix.bodies;
    const Unit16* const skips = ix.skips;
    const Edge* const edges = ix.edges;
    const uint32_t base = static_cast<uint32_t>(ix.offset), records = static_cast<uint32_t>(ix.records);
    const uint64_t blocks = (m + 31) / 32;
    const uint64_t items = blocks * cv.max_segments;
    const uint64_t warp = (static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x) / 32;
    const uint64_t warps = (static_cast<uint64_t>(gridDim.x) * blockDim.x) / 32;
    for (uint64_t item = warp; item < items; item += warps) {
        const uint64_t j = item / blocks, i = (item - j * blocks) * 32 + lane;
        // this lane's segment, if it has one
        SegmentLane st;
        st.node = 0; st.offset = 0; st.left = 0; st.parked = 0;
        uint64_t* dst = nodes;  // where node number `parked` of the tile row goes
        if (i < m) {
            const uint64_t id = __ldg(ids + i);
            if (id >= ix.sequences) {
                if (j == 0 && lengths != nullptr) lengths[i] = ~0ull;  // GBWT::sequence() is None
            } else {
                const uint64_t len = cv.seq_len[id];
                if (j == 0 && lengths != nullptr) lengths[i] = len;
                const uint32_t first = __ldg(cv.first + id), count = __ldg(cv.first + id + 1) - first;
                if (j < count) {
                    const uint64_t lo = __ldg(out_offsets + i), hi = __ldg(out_offsets + i + 1);
                    const uint64_t cap = hi > lo ? hi - lo : 0;
                    const uint4 raw = __ldg(reinterpret_cast<const uint4*>(cv.table + first + j));
                    st.node = raw.x; st.offset = raw.y;
                    const uint64_t index = (static_cast<uint64_t>(raw.w) << 32) | raw.z;
                    uint64_t end = len;
                    if (j + 1 < count) {
                        const uint4 next = __ldg(reinterpret_cast<const uint4*>(cv.table + first + j + 1));
                        end = (static_cast<uint64_t>(next.w) << 32) | next.z;
                    }
                    if (end > cap) end = cap;  // nothing beyond the caller's slot is written
                    const uint64_t todo = end > index ? end - index : 0;
                    st.left = todo < 0xFFFFFFFFull ? static_cast<uint32_t>(todo) : 0xFFFFFFFFu;
                    dst = nodes + (lo - base_offset) + index;
                }
            }
        }
        Desc d0, d1;
        Quad k0, k1;
        if (st.left != 0) load_segment_record<CHECKED>(descs, skips, base, records, keep, st.node, d0, k0);
        // Look-ahead (see the round loop): where the warp was a round ago, the bodies it has yet to touch, and the words
        // its touches returned (folded into `sink` a round later, so that nothing ever waits for them).
        uint32_t prev_rec = 0xFFFFFFFFu, ahead_body = 0, ahead_span = 0;
        uint32_t t0 = 0, t1 = 0, t2 = 0, t3 = 0, t4 = 0, t5 = 0, sink = 0;
        for (;;) {
            // The 32 lanes walk the same stretch of the graph (the same segment of 32 sequences), and so do the other
            // warps of the CTA and the CTAs next to it: whoever gets to a record first waits for DRAM, and everybody
            // else then waits with it. Node identifiers follow the graph's topological order, so once per round the
            // warp touches the records it is heading for -- lane l the descriptors and shortcuts of 8 records
            // `lookahead + 8 l` records further on, and the bodies of the 8 records it touched a round ago (their
            // offset comes from the descriptor that touch returned) -- and the walks find them in L2 / L1.
            if (cv.lookahead != 0) {
                sink ^= t0 ^ t1 ^ t2 ^ t3 ^ t4 ^ t5;
                const unsigned walking = __ballot_sync(FULL, st.left != 0);
                if (walking != 0) {
                    const uint32_t here = __shfl_sync(FULL, st.node, __ffs(static_cast<int>(walking)) - 1) - base;
                    const bool up = prev_rec == 0xFFFFFFFFu ? (here & 1u) == ((base & 1u) ^ 0u) : here >= prev_rec;
                    prev_rec = here;
                    for (uint32_t u = 0; u < ahead_span; u += 8) {  // bodies: 128-byte lines, at most four per lane
                        asm volatile("ld.global.nc.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(t5) : "l"(bodies + ahead_body + u), "l"(keep));
                    }
                    const uint32_t step = cv.lookahead + 8u * lane;
                    uint32_t target = up ? here + step : here - step - 7u;
                    if (up ? (target < here || target + 8u > records) : (target > here)) target = up ? (records > 8u ? records - 8u : 0u) : 0u;
                    if (records >= 8u) {
                        asm volatile("ld.global.nc.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(t0) : "l"(&descs[target].body), "l"(keep));
                        asm volatile("ld.global.nc.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(t1) : "l"(&descs[target + 4u].body), "l"(keep));
                        asm volatile("ld.global.nc.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(t2) : "l"(skips + target), "l"(keep));
                        asm volatile("ld.global.nc.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(t3) : "l"(&descs[target + 7u].body), "l"(keep));
                        t4 = target;
                    }
                }
            }

            // A round: as many steps as fit the tile rows whatever the lanes do (a step parks at most two nodes), two
            // per iteration on alternating register sets. No votes inside: lanes that are done just sit the round out.
#pragma unroll 1
            for (uint32_t step = 0; step < TILE_NODES / 4; step++) {
                if (st.left != 0) segment_step<CHECKED>(st, d0, k0, d1, k1, row, descs, bodies, skips, edges, base, records, keep);
                if (st.left != 0) segment_step<CHECKED>(st, d1, k1, d0, k0, row, descs, bodies, skips, edges, base, records, keep);
            }
            // all rows out, one after the other: up to 512 contiguous bytes per row, 256 per store instruction
            __syncwarp();
            const uint64_t row_addr = reinterpret_cast<uint64_t>(dst);
#pragma unroll 4
            for (uint32_t r = 0; r < 32; r++) {
                const uint32_t n = __shfl_sync(FULL, st.parked, r);
                const uint32_t a_lo = __shfl_sync(FULL, static_cast<uint32_t>(row_addr), r);
                const uint32_t a_hi = __shfl_sync(FULL, static_cast<uint32_t>(row_addr >> 32), r);
                uint64_t* to = reinterpret_cast<uint64_t*>((static_cast<uint64_t>(a_hi) << 32) | a_lo);
                if (cv.discard) continue;
                if (lane < n) __stcs(to + lane, static_cast<uint64_t>(tile[r][lane]));
                if (lane + 32 < n) __stcs(to + lane + 32, static_cast<uint64_t>(tile[r][lane + 32]));
            }
            __syncwarp();
            dst += st.parked;
            st.parked = 0;
            if (cv.lookahead != 0) {
                // by now (a round later) the touched descriptors have arrived: the bodies of this lane's 8 records lie between
                // the body offset of its first record and that of its last (bodies lie in record order)
                // (up to the START of the last one's body: whatever lies in between is inside the array)
                const uint32_t lo = t0 < t3 ? t0 : t3, hi = t0 < t3 ? t3 : t0;
                ahead_body = lo;
                ahead_span = hi - lo < 32u ? hi - lo : 32u;
            }
            if (!__any_sync(FULL, st.left != 0)) break;
        }
        if (sink == 0x9E3779B9u && lengths != nullptr && m == ~size_t(0)) lengths[0] = sink;  // (keeps the touches alive; never true)
    }
}

// ---- K4 with checkpoints: DNA extraction that is parallel ALONG the paths ----------------------------------------------
// One group of up to 32 consecutive nodes of a path (lane l holds node l of the group, l < count) spelled at byte `at` of
// the path's DNA: the stateless form of DnaSink (extract_sequence, src/bin/gbz-extract.rs:173-189; reverse-oriented nodes
// reverse-complemented, support::reverse_complement, src/support.rs:104-110). Every lane fetches the label range of its
// node, a warp scan turns the lengths into offsets, and the warp writes the group's bytes as consecutive 32-byte rows,
// each lane finding the node that owns its byte by a 5-step search over the scanned lengths. out == nullptr only counts.
// Returns the bytes of the group, written or not (nothing beyond out[cap) is written).
__device__ __forceinline__ uint32_t spell_group(const GraphView& graph, uint64_t node_base, uint32_t mine, uint32_t count,
                                                uint8_t* out, uint64_t cap, uint64_t at) {
    constexpr unsigned FULL = 0xFFFFFFFFu;
    constexpr uint32_t ROWS = 8;
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t sid = ((static_cast<uint64_t>(mine) & ~1ull) - node_base) >> 1;  // GBZ::gbwt_node_to_sequence, src/gbz.rs:253-255
    const bool valid = lane < count && sid < graph.sequences;
    const uint64_t idx = valid ? sid : 0;
    const uint64_t lo = __ldg(graph.starts + idx), hi = __ldg(graph.starts + idx + 1);
    const uint32_t rev = mine & 1u;
    const uint32_t len = valid ? static_cast<uint32_t>(hi - lo) : 0u;
    uint32_t incl = len;
#pragma unroll
    for (uint32_t d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(FULL, incl, d);
        if (lane >= d) incl += t;
    }
    const uint32_t total = __shfl_sync(FULL, incl, 31);
    if (out != nullptr) {
        // byte b of the group comes from label byte key + b (forward node) or key - b (reverse node); the keys carry a bias
        // of 2^32 so that they stay positive (bit 63 is the orientation)
        constexpr uint64_t BIAS = 1ull << 32;
        const uint32_t excl = incl - len;
        const uint64_t key = BIAS + (rev ? lo + len - 1 + excl : lo - excl);
        const uint32_t key_lo = static_cast<uint32_t>(key), key_hi = static_cast<uint32_t>(key >> 32) | (rev << 31);
        for (uint32_t row = 0; row < total; row += 32 * ROWS) {
            uint32_t c[ROWS], flip[ROWS];
#pragma unroll
            for (uint32_t j = 0; j < ROWS; j++) {
                const uint32_t b = row + 32 * j + lane;
                uint32_t owner = 0;  // number of nodes that end at or before byte b (incl is non-decreasing over the lanes)
#pragma unroll
                for (uint32_t step = 16; step != 0; step >>= 1) {
                    const uint32_t v = __shfl_sync(FULL, incl, (owner + step - 1) & 31u);
                    if (v <= b) owner += step;
                }
                const uint32_t k_lo = __shfl_sync(FULL, key_lo, owner & 31u), k_hi = __shfl_sync(FULL, key_hi, owner & 31u);
                const uint64_t k = (static_cast<uint64_t>(k_hi & 0x7FFFFFFFu) << 32) | k_lo;
                flip[j] = k_hi >> 31;
                c[j] = 0;
                if (b < total && at + b < cap) c[j] = __ldg(graph.bytes + ((flip[j] ? k - b : k + b) - BIAS));
            }
#pragma unroll
            for (uint32_t j = 0; j < ROWS; j++) {
                const uint32_t b = row + 32 * j + lane;
                if (b < total && at + b < cap) out[at + b] = static_cast<uint8_t>(flip[j] ? complement_base(c[j]) : c[j]);
            }
        }
    }
    return total;
}

// Work item (segment j, block of 32 sequences) as in k_extract_checkpointed: lane l walks segment j of its sequence from
// the checkpoint, parks the nodes in its row of the tile, and once per round the warp spells the rows one after the
// other (spell_group) at each lane's own byte position, which starts at dna_at[checkpoint] = the DNA bytes of the
// sequence before the checkpoint's node.
// Count mode (bytes == nullptr, seg_bytes != nullptr, ids == nullptr: all sequences): seg_bytes[checkpoint] = DNA bytes of
// the segment -- the pass that dna_at[] is made from when a graph and checkpoints are both there.
// (Rounds of 32 nodes per lane: spelling a row is two memory round trips however long it is, so what counts is how many
// warps an SM holds, and the tile is what limits that.)
constexpr uint32_t DNA_TILE_NODES = 32, DNA_TILE_STRIDE = 33;

template <bool CHECKED, int THREADS, int CTAS>
__global__ void __launch_bounds__(THREADS, CTAS) k_extract_dna_checkpointed(IndexView ix, GraphView graph, CheckpointView cv,
                                                                             const uint64_t* __restrict__ dna_at, uint64_t* __restrict__ seg_bytes,
                                                                             const uint64_t* __restrict__ dna_len, const uint64_t* __restrict__ ids,
                                                                             size_t m, const uint64_t* __restrict__ out_offsets, uint64_t base_offset,
                                                                             uint32_t endmarker, uint8_t* __restrict__ bytes,
                                                                             uint64_t* __restrict__ lengths) {
    constexpr unsigned FULL = 0xFFFFFFFFu;
    extern __shared__ __align__(16) unsigned char tile_bytes[];  // [THREADS / 32][32][DNA_TILE_STRIDE] words
    uint32_t (*tiles)[32][DNA_TILE_STRIDE] = reinterpret_cast<uint32_t (*)[32][DNA_TILE_STRIDE]>(tile_bytes);
    const uint32_t lane = threadIdx.x & 31u;
    uint32_t (*tile)[DNA_TILE_STRIDE] = tiles[threadIdx.x >> 5];
    uint32_t* const row = tile[lane];
    const uint64_t keep = keep_policy();
    const RecordDesc* const descs = ix.desc;
    const Unit16* const bodies = ix.bodies;
    const Unit16* const skips = ix.skips;
    const Edge* const edges = ix.edges;
    const uint32_t base = static_cast<uint32_t>(ix.offset), records = static_cast<uint32_t>(ix.records);
    const uint64_t node_base = ix.offset + 1;
    const bool counting = bytes == nullptr;
    const uint64_t blocks = (m + 31) / 32;
    const uint64_t items = blocks * cv.max_segments;
    const uint64_t warp = (static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x) / 32;
    const uint64_t warps = (static_cast<uint64_t>(gridDim.x) * blockDim.x) / 32;
    for (uint64_t item = warp; item < items; item += warps) {
        const uint64_t j = item / blocks, i = (item - j * blocks) * 32 + lane;
        SegmentLane st;
        st.node = 0; st.offset = 0; st.left = 0; st.parked = 0;
        uint8_t* out = nullptr;  // this lane's sequence slot
        uint64_t cap = 0, cursor = 0;
        uint64_t slot = ~0ull;   // the checkpoint this lane walks from
        bool last = false;       // ... is the last one of its sequence: the endmarker byte follows
        if (i < m) {
            const uint64_t id = ids != nullptr ? __ldg(ids + i) : i;
            if (id >= ix.sequences) {
                if (j == 0 && lengths != nullptr) lengths[i] = ~0ull;  // GBZ::path() is None
            } else {
                if (j == 0 && lengths != nullptr) lengths[i] = dna_len[id];
                const uint32_t first = __ldg(cv.first + id), count = __ldg(cv.first + id + 1) - first;
                if (!counting) {
                    const uint64_t lo = __ldg(out_offsets + i), hi = __ldg(out_offsets + i + 1);
                    out = bytes + (lo - base_offset);
                    cap = hi > lo ? hi - lo : 0;
                    if (j == 0 && count == 0 && cap > 0) out[0] = static_cast<uint8_t>(endmarker);  // an empty path: the endmarker alone
                }
                if (j < count) {
                    slot = first + j;
                    const uint4 raw = __ldg(reinterpret_cast<const uint4*>(cv.table + slot));
                    st.node = raw.x; st.offset = raw.y;
                    const uint64_t index = (static_cast<uint64_t>(raw.w) << 32) | raw.z;
                    uint64_t end = cv.seq_len[id];
                    if (j + 1 < count) {
                        const uint4 next = __ldg(reinterpret_cast<const uint4*>(cv.table + slot + 1));
                        end = (static_cast<uint64_t>(next.w) << 32) | next.z;
                    } else {
                        last = true;
                    }
                    const uint64_t todo = end > index ? end - index : 0;
                    st.left = todo < 0xFFFFFFFFull ? static_cast<uint32_t>(todo) : 0xFFFFFFFFu;
                    if (!counting) cursor = __ldg(dna_at + slot);
                }
            }
        }
        Desc d0, d1;
        Quad k0, k1;
        if (st.left != 0) load_segment_record<CHECKED>(descs, skips, base, records, keep, st.node, d0, k0);
        for (;;) {
#pragma unroll 1
            for (uint32_t step = 0; step < DNA_TILE_NODES / 4; step++) {
                if (st.left != 0) segment_step<CHECKED>(st, d0, k0, d1, k1, row, descs, bodies, skips, edges, base, records, keep);
                if (st.left != 0) segment_step<CHECKED>(st, d1, k1, d0, k0, row, descs, bodies, skips, edges, base, records, keep);
            }
            // every lane asks L1 for the label ranges of the nodes it parked (neighbouring lanes walk neighbouring haplotypes:
            // a few lines), so that the warp's loads of them below do not each wait for L2 / DRAM
            for (uint32_t p = 0; p < st.parked; p++) {
                const uint64_t sid = ((static_cast<uint64_t>(row[p]) & ~1ull) - node_base) >> 1;
                if (sid < graph.sequences) asm volatile("prefetch.global.L1 [%0];" ::"l"(graph.starts + sid));
            }
            // the rows one after the other, each at its lane's own position in its own sequence
            __syncwarp();
#pragma unroll 1
            for (uint32_t r = 0; r < 32; r++) {
                const uint32_t n = __shfl_sync(FULL, st.parked, r);
                if (n == 0) continue;
                uint64_t at = __shfl_sync(FULL, cursor, r);
                const uint64_t to = __shfl_sync(FULL, reinterpret_cast<uint64_t>(out), r), limit = __shfl_sync(FULL, cap, r);
                for (uint32_t g = 0; g < n; g += 32) {
                    const uint32_t mine = g + lane < n ? tile[r][g + lane] : 0u;
                    at += spell_group(graph, node_base, mine, n - g < 32u ? n - g : 32u, reinterpret_cast<uint8_t*>(to), limit, at);
                }
                if (lane == r) cursor = at;
            }
            __syncwarp();
            st.parked = 0;
            if (!__any_sync(FULL, st.left != 0)) break;
        }
        if (slot != ~0ull) {
            if (counting) seg_bytes[slot] = cursor;
            else if (last && cursor < cap) out[cursor] = static_cast<uint8_t>(endmarker);
        }
    }
}

// dna_at[checkpoint] = DNA bytes of the sequence before the checkpoint's node (exclusive scan of the segment sizes the
// count pass left there); dna_len[id] = bytes of the whole result, endmarker included (1 for an empty path).
__global__ void __launch_bounds__(BLOCK_THREADS) k_dna_checkpoint_scan(uint64_t sequences, const uint32_t* __restrict__ first,
                                                                        uint64_t* __restrict__ seg, uint64_t* __restrict__ dna_len) {
    GBWT_GRID_STRIDE(id, sequences) {
        uint64_t total = 0;
        for (uint32_t s = first[id]; s < first[id + 1]; s++) {
            const uint64_t t = seg[s];
            seg[s] = total;
            total += t;
        }
        dna_len[id] = total + 1;
    }
}

// GBWT::sequence(id).count() from the table the checkpoint build left.
__global__ void __launch_bounds__(BLOCK_THREADS) k_lengths_from_table(uint64_t sequences, const uint64_t* __restrict__ seq_len,
                                                                       const uint64_t* __restrict__ ids, size_t m, uint64_t* __restrict__ lengths) {
    GBWT_GRID_STRIDE(i, m) {
        const uint64_t id = __ldg(ids + i);
        lengths[i] = id < sequences ? seq_len[id] : ~0ull;
    }
}

}  // namespace gbwt_b200
