// find_window.cu -- the record-window kernels: GBWT::find + extends (src/gbwt.rs:269-304 over Record::follow,
// src/bwt.rs:595-616), bidirectional searches (src/gbwt.rs:311-384) and checkpointed path extraction (Record::lf,
// src/bwt.rs:480-496) with the records in shared memory.
//
// After the locality sort the queries of one bucket all start inside one window of consecutive records, and a
// pattern stays close to its first record (node identifiers follow the graph's topological order). So a CTA takes a
// window, decodes the window plus a margin either side -- descriptors, two-hop shortcuts and the contiguous range of
// bodies -- into tables laid out for the search loop (16-bit window-relative fields, one 4-byte entry per 16 positions
// of a bitvector), and its warps resolve the window's queries from shared memory: a dependent step costs a
// shared-memory round trip (~30 cycles) instead of an L2 / HBM one (300 / 800), the index is read from HBM once per
// batch in large sequential pieces, and the only scattered global accesses left are the pattern rows (read by a warp
// together, whole lines at a time) and the results. (The first version staged the raw records with cp.async.bulk and an
// mbarrier and read them in their global layout; the bank conflicts of that layout are why the window is decoded
// instead: profiles/r2_find_window_v1_tma_raw_layout_ncu.txt.)
//
// Per step: the record u of the current node, the pattern node x1 (which must equal one of u's edge targets), and --
// the two-hop shortcut of layout.h -- if the successor over that edge is a single-edge record whose only target is the
// pattern node after x1, both nodes are consumed at once without looking at the successor's record. A bubble
// (SNP / indel site) is therefore ONE step: one 16-byte record entry and one or two 4-byte rank entries.
//
// Anything the window cannot answer exactly -- a record outside the staged range, a body that did not fit, a record
// format it does not decode -- puts the query on a deferred list, and the general kernel finishes the list
// afterwards. Results are therefore always those of the general kernel; the window only makes the common case fast.
#include "find_window.h"

#include <algorithm>
#include <cstdlib>

#include "find_lean.cuh"

namespace gbwt_b200 {

namespace {

// ---- shared-memory accessors (32-bit shared-space addresses: no generic-pointer arithmetic in the loop) --------------

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ uint4 lds128(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t a) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts128(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ void sts64(uint32_t a, uint32_t x, uint32_t y) {
    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void sts32(uint32_t a, uint32_t x) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(x) : "memory"); }

// ---- pattern rows -----------------------------------------------------------------------------------------------------
// A warp takes 32 queries at a time and reads their pattern rows TOGETHER, one segment of 16 nodes per round: the lanes
// that share a row read consecutive 32-byte sectors of it, so a load instruction moves whole 128-byte lines (64-bit
// nodes: 4 lanes per row, 8 rows per instruction, 4 instructions per segment) instead of 32 isolated sectors. (The
// first versions had every thread read its own row sector by sector: one L1 wavefront per 32 bytes, 3.9 M of the
// 12.2 M data-stage wavefronts per SM, and the consumer waited for DRAM eight times per query -- 21 % of the stall
// samples in profiles/r2_find_window_v2_ncu.txt.) Each node is narrowed on the spot to a 16-bit index into the staged
// window (NODE_OUTSIDE if it is not in there) and stored in the warp's tile, node-major: tile[t][row], so that in the
// search loop a lane reads node t of its own row with one conflict-free 16-bit load however t moves.
constexpr uint32_t SEGMENT = 16;            // pattern nodes per round
constexpr uint32_t TILE_PITCH = 34;         // 16-bit slots per tile line: 32 rows + 2 (the lanes that share a row store 4 lines apart: 16 distinct banks)
constexpr uint32_t TILE_LINE = TILE_PITCH * 2u;  // bytes from node t to node t + 1 of a row
constexpr uint32_t TILE_BYTES = (SEGMENT + 1u) * TILE_LINE;  // one line more than a segment: the line after the last node always reads NODE_OUTSIDE
constexpr uint32_t NODE_OUTSIDE = 0xFFFFu;  // not a record of the staged window (or node 0, the endmarker)

// Window index of an edge target (node 0, the endmarker, is never a record to go on with).
__device__ __forceinline__ uint32_t window_index(uint32_t node, uint32_t origin, uint32_t count) {
    const uint32_t rel = node - origin;
    return node != 0 && rel < count ? rel : NODE_OUTSIDE;
}
// Window index of a pattern node. No test for node 0: if record 0 is staged at all (origin == 0) it is the endmarker's,
// which window_find defers and which no table entry names as a target, so a pattern node 0 never matches anything.
__device__ __forceinline__ uint32_t pattern_index(uint64_t node, uint32_t origin, uint32_t count) {
    const uint64_t rel = node - origin;
    return rel < count ? static_cast<uint32_t>(rel) : NODE_OUTSIDE;
}
__device__ __forceinline__ uint32_t pattern_index(uint32_t node, uint32_t origin, uint32_t count) {
    const uint32_t rel = node - origin;
    return rel < count ? rel : NODE_OUTSIDE;
}

// (16-bit shared accesses on 32-bit registers: the load zero-extends, the store writes the low half)
__device__ __forceinline__ void sts16(uint32_t a, uint32_t x) { asm volatile("st.shared.b16 [%0], %1;" ::"r"(a), "r"(x) : "memory"); }
__device__ __forceinline__ uint32_t lds16(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}

// One 32-byte sector of pattern nodes, bypassing L1 (every byte is used once). The loads ask L2 for the whole row (256
// bytes of 64-bit nodes, 128 of 32-bit nodes: two 16-node segments), so that the second segment's loads find it there
// instead of paying DRAM latency again (6.34 -> 6.84 G queries/s; prefetching the NEXT 32 rows on top of that is slower).
__device__ __forceinline__ void load_nodes(const uint64_t* p, uint64_t (&v)[4]) {
    asm volatile("ld.global.nc.L1::no_allocate.L2::256B.v4.u64 {%0, %1, %2, %3}, [%4];" : "=l"(v[0]), "=l"(v[1]), "=l"(v[2]), "=l"(v[3]) : "l"(p));
}
__device__ __forceinline__ void load_nodes(const uint32_t* p, uint32_t (&v)[8]) {
    asm volatile("ld.global.nc.L1::no_allocate.L2::128B.v8.u32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) : "l"(p));
}

// Fills the warp's tile with nodes [seg, seg + n_seg) of its 32 rows. `q` is this lane's own query (NO_QUERY: none);
// row r is the row of lane r's query. Sector loads when every row segment starts on a 32-byte boundary and n_seg is a
// whole number of sectors, else node by node.
constexpr uint32_t NO_QUERY = 0xFFFFFFFFu;

template <class T>
__device__ __forceinline__ void load_tile(const T* __restrict__ patterns, uint32_t q, uint32_t k, uint32_t seg, uint32_t n_seg, bool sectors,
                                          uint32_t tile, uint32_t origin, uint32_t count, uint32_t lane) {
    constexpr uint32_t PER_SECTOR = 32u / sizeof(T);          // nodes per 32-byte sector: 4 or 8
    constexpr uint32_t MAX_LANES_PER_ROW = SEGMENT / PER_SECTOR;  // 4 or 2
    if (sectors) {
        const uint32_t per_row = n_seg / PER_SECTOR;  // sectors per row segment: 1 .. MAX_LANES_PER_ROW (whole lanes only when a power of two)
        // lanes_per_row = MAX_LANES_PER_ROW always (a shorter segment leaves the extra lanes idle: only the last round of a pattern)
        const uint32_t sub = lane % MAX_LANES_PER_ROW, first = lane / MAX_LANES_PER_ROW;
        constexpr uint32_t ROWS_PER_LOAD = 32u / MAX_LANES_PER_ROW;  // 8 or 16
        constexpr uint32_t LOADS = 32u / ROWS_PER_LOAD;  // 4 or 2 load instructions per segment
        // (64-bit nodes: two loads = 16 registers in flight at a time; all four at once spill under the 64-register budget)
        constexpr uint32_t GROUP = 2;
        const uint32_t at = tile + (sub * PER_SECTOR * TILE_PITCH + first) * 2u;
#pragma unroll
        for (uint32_t g = 0; g < LOADS; g += GROUP) {
            T v[GROUP][PER_SECTOR];
            bool have[GROUP];
#pragma unroll
            for (uint32_t j = 0; j < GROUP; j++) {
                const uint32_t owner = __shfl_sync(0xFFFFFFFFu, q, (g + j) * ROWS_PER_LOAD + first);
                have[j] = owner != NO_QUERY && sub < per_row;
                if (have[j]) load_nodes(patterns + static_cast<size_t>(owner) * k + seg + sub * PER_SECTOR, v[j]);
            }
#pragma unroll
            for (uint32_t j = 0; j < GROUP; j++) {
                if (have[j]) {
#pragma unroll
                    for (uint32_t t = 0; t < PER_SECTOR; t++)
                        sts16(at + (t * TILE_PITCH + (g + j) * ROWS_PER_LOAD) * 2u, pattern_index(v[j][t], origin, count));
                }
            }
        }
    } else {
        for (uint32_t e = lane; e < 32u * n_seg; e += 32u) {
            const uint32_t r = e / n_seg, t = e - r * n_seg;
            const uint32_t owner = __shfl_sync(0xFFFFFFFFu, q, r);
            if (owner != NO_QUERY) sts16(tile + (t * TILE_PITCH + r) * 2u, pattern_index(__ldg(patterns + static_cast<size_t>(owner) * k + seg + t), origin, count));
        }
    }
}

// Asks L2 for a pattern row ahead of its use: its first two 128-byte lines (a length-32 pattern is two lines of 64-bit
// nodes, one of 32-bit nodes).
template <class T>
__device__ __forceinline__ void prefetch_row(const T* row, uint32_t k) {
    asm volatile("prefetch.global.L2 [%0];" ::"l"(row));
    if (k * sizeof(T) > 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(row) + 128));
}

// First node of pattern row q as a 64-bit value (the sort key is computed from it).
__device__ __forceinline__ uint64_t first_node(const uint64_t* patterns, size_t q, size_t k) { return __ldg(patterns + q * k); }
__device__ __forceinline__ uint64_t first_node(const uint32_t* patterns, size_t q, size_t k) { return __ldg(patterns + q * k); }

// ---- the staged window -----------------------------------------------------------------------------------------------
// What a CTA decodes into shared memory for the records [lo, lo + count) -- once per window, used by ~3 queries per
// record times 16 steps. Arranged for the loop, not like the global layout, and in 16-bit fields: the data stage of
// L1 was the busiest unit of the first versions (78 % with 32-bit patterns), half of its shared-memory wavefronts
// being bank conflicts of 8- and 16-byte loads at random records, so every table entry is as narrow as it can be.
// Nodes are indexes into the window (NODE_OUTSIDE when the node is not staged); a record with a field that does not
// fit 16 bits is marked KIND_DEFER.
//   rec[r]   16 B  {target0 | target1 << 16, total_len | kind << 16, shortcut0, shortcut1}: kind = index of the record's
//                  first rank entry for a dense record, or KIND_SINGLE / KIND_EMPTY / KIND_DEFER (run-length body,
//                  outdegree > 2, body not staged); shortcut = the two-hop shortcut of the edge {landing node | offset << 16}
//                  (layout.h, IndexView::skips). One 16-byte load per step.
//   offs[r]   4 B  {offset0 | offset1 << 16}: only read when a step cannot take the shortcut
//   ranks[]   4 B  {ones before | 16 bits << 16}: rank at position p of a record is ONE 4-byte load at kind + p / 16
//   wide records (up to four edges with a DENSE4 or byte-per-run body, or two edges with a byte-per-run body: what a
//   multi-allelic site or a record with few runs looks like) take the slower path of wide_follow():
//   rec[r]         {aux index | sigma << 16, total_len | KIND_WIDE << 16, body slot | body_len << 16, format | checkpoints << 8}
//   aux[a]   32 B  {target0 | target1 << 16, target2 | target3 << 16, shortcut0 .. shortcut3, offset0 | offset1 << 16,
//                  offset2 | offset3 << 16}: handed out from a small pool while the records are decoded
//   body slots: every 32-byte block of the staged body range owns 48 bytes of `ranks`; a DENSE2 block fills them with its
//   twelve rank entries, a DENSE4 block with two 16-byte entries {64 bits of codes, count1 | count2 << 16, count3} of 32
//   positions each, a run-length body (with its checkpoint table) is copied as it is, 32 bytes per slot. kinds[] says
//   which (one byte per block, written by the record's thread before the blocks are decoded).
constexpr uint32_t KIND_SINGLE = 0xFFFFu, KIND_EMPTY = 0xFFFEu, KIND_DEFER = 0xFFFDu, KIND_WIDE = 0xFFFCu;  // anything below: dense
constexpr uint32_t RECORD_BYTES = 20;  // rec + offs
constexpr uint32_t AUX_BYTES = 32;
constexpr uint32_t NO_SHORTCUT = 0xFFFFu;  // (its node half is NODE_OUTSIDE: never equal to a pattern node that passed the x2 test)
enum : uint32_t { BLOCK_UNUSED = 0, BLOCK_DENSE2 = 1, BLOCK_DENSE4 = 2, BLOCK_RAW = 3 };

struct Staged {
    uint32_t rec, offs, ranks;  // shared-space addresses
    uint32_t lo, count;         // staged records [lo, lo + count)
    uint32_t aux, kinds;        // wide records: edge tables, and what each body block holds
};

// Shared address of 16-byte unit u of a body copied as it is into the slots from `slot` on.
__device__ __forceinline__ uint32_t raw_unit(uint32_t ranks, uint32_t slot, uint32_t u) { return ranks + 48u * (slot + (u >> 1)) + 16u * (u & 1u); }

// Occurrences of `symbol` in [0, pos) of a byte-per-run body (layout.h: FMT_RUN8, sigma 2 .. 4) held in the slots from
// `slot` on, starting at the checkpoint before pos when the body has a table (record_scan.cuh: load_checkpoint /
// scan_runs_to, here on the shared-memory copy; a table entry of a record with at most four edges is one 16-byte unit).
__device__ __forceinline__ uint32_t staged_rank_runs8(uint32_t ranks, uint32_t slot, uint32_t n, uint32_t sigma, uint32_t checkpoints,
                                                      uint32_t total, uint32_t symbol, uint32_t pos) {
    uint32_t run = 0, off = 0, count = 0;
    if (checkpoints != 0) {
        const uint32_t shift = checkpoints - 1u, last = (total - 1u) >> shift;
        uint32_t j = pos >> shift;
        if (j > last) j = last;
        if (j != 0) {
            const uint4 e = lds128(raw_unit(ranks, slot, ((((n + 15u) >> 4) + 1u) & ~1u) + j - 1u));
            off = j << shift;
            run = sigma == 2 ? e.y : (sigma == 3 ? e.z : e.w);
            const uint32_t upto = symbol + 1u < sigma ? (symbol == 0 ? e.x : (symbol == 1 ? e.y : e.z)) : off;
            const uint32_t below = symbol == 0 ? 0u : (symbol == 1 ? e.x : (symbol == 2 ? e.y : e.z));
            count = upto - below;
        }
    }
    const uint32_t magic = sigma == 2 ? 32769u : (sigma == 3 ? 21846u : 16385u);  // div_magic(sigma)
    for (uint32_t base = run & ~15u; base < n && off < pos; base += 16) {
        const uint4 q = lds128(raw_unit(ranks, slot, base >> 4));
        const uint32_t words[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (uint32_t j = 0; j < 16; j++) {
            if (base + j >= run && base + j < n && off < pos) {
                const uint32_t byte = (words[j >> 2] >> (8 * (j & 3))) & 0xFFu;
                const uint32_t quot = (byte * magic) >> 16, len = quot + 1u;
                if (byte - quot * sigma == symbol) count += pos - off < len ? pos - off : len;
                off += len;
            }
        }
    }
    return count;
}

// Occurrences of `symbol` in [0, pos) of a DENSE4 body held as 16-byte entries of 32 positions (two per slot).
__device__ __forceinline__ uint32_t staged_rank_dense4(uint32_t ranks, uint32_t slot, uint32_t blocks, uint32_t symbol, uint32_t pos) {
    uint32_t half = pos >> 5;
    if (half >= 2u * blocks) half = 2u * blocks - 1u;  // pos == total_len on a block boundary
    const uint32_t r = pos - 32u * half;               // 0 .. 32 fields of this entry
    const uint4 e = lds128(ranks + 48u * (slot + (half >> 1)) + 16u * (half & 1u));
    const uint32_t c1 = e.z & 0xFFFFu, c2 = e.z >> 16, c3 = e.w;
    const uint32_t before = symbol == 0 ? 32u * half - c1 - c2 - c3 : (symbol == 1 ? c1 : (symbol == 2 ? c2 : c3));
    const unsigned long long codes = (static_cast<unsigned long long>(e.y) << 32) | e.x;
    const unsigned long long y = codes ^ (symbol * 0x5555555555555555ull);
    unsigned long long t = ~(y | (y >> 1)) & 0x5555555555555555ull;
    if (r < 32u) t &= (1ull << (2u * r)) - 1ull;
    return before + static_cast<uint32_t>(__popcll(t));
}

// Record::follow on a wide record (src/bwt.rs:595-616): {rank(s), rank(e), shortcut, shared address of the edge offset}
// for the edge to window index x1; rank(s) == rank(e) == 0 when x1 is not a successor. Out of line: it is the rare case,
// and inlined it would set the register budget of the whole search loop.
__device__ __noinline__ uint4 wide_follow(uint32_t ranks, uint32_t aux, uint32_t h_z, uint32_t h_w, uint32_t sigma, uint32_t total,
                                          uint32_t x1, uint32_t s, uint32_t e) {
    const uint4 a0 = lds128(aux), a1 = lds128(aux + 16u);
    uint32_t b = 4;
    if (x1 == (a0.x & 0xFFFFu)) b = 0;
    else if (x1 == (a0.x >> 16)) b = 1;
    else if (x1 == (a0.y & 0xFFFFu)) b = 2;
    else if (x1 == (a0.y >> 16)) b = 3;
    uint4 out;
    out.x = 0; out.y = 0; out.z = NO_SHORTCUT; out.w = aux + 24u;
    if (b >= sigma) return out;
    const uint32_t slot = h_z & 0xFFFFu, n = h_z >> 16, fmt = h_w & 0xFFu, checkpoints = (h_w >> 8) & 0xFFu;
    if (fmt == FMT_DENSE4) {
        out.x = staged_rank_dense4(ranks, slot, n, b, s);
        out.y = staged_rank_dense4(ranks, slot, n, b, e);
    } else {
        out.x = staged_rank_runs8(ranks, slot, n, sigma, checkpoints, total, b, s);
        out.y = staged_rank_runs8(ranks, slot, n, sigma, checkpoints, total, b, e);
    }
    out.z = b == 0 ? a0.z : (b == 1 ? a0.w : (b == 2 ? a1.x : a1.y));
    out.w = aux + 24u + 2u * b;
    return out;
}

enum : uint32_t { QUERY_ACTIVE = 0, QUERY_FOUND = 1, QUERY_NONE = 2, QUERY_DEFER = 3, QUERY_WIDE = 4 };

// The state of one query between rounds.
struct WindowQuery {
    uint32_t idx;         // window index of the current node
    uint32_t start, end;  // the range in its record
    uint32_t i;           // next pattern position
    uint32_t status;
};

// GBWT::find on the first pattern node (window index x, NODE_OUTSIDE if it is not staged).
__device__ __forceinline__ void window_find(const Staged& st, uint32_t x, uint32_t k, WindowQuery& q) {
    q.idx = x; q.start = 0; q.end = 0; q.i = 1; q.status = QUERY_ACTIVE;
    if (x == NODE_OUTSIDE || x + st.lo == 0) { q.status = QUERY_DEFER; return; }  // (record 0 is the endmarker: find() is None; let the general code say so)
    const uint2 h = lds64(st.rec + 16u * x);
    const uint32_t kind = h.y >> 16;
    q.end = h.y & 0xFFFFu;
    if (kind == KIND_DEFER) q.status = QUERY_DEFER;
    else if (kind == KIND_EMPTY || q.end == 0) q.status = QUERY_NONE;  // GBWT::find: no record
    else if (k == 1) q.status = QUERY_FOUND;
}

// Extends an active query through the pattern nodes [q.i, seg + n_seg) that the warp's tile holds (tile line t = node
// seg + t of every row, the line after the last node reads NODE_OUTSIDE; `slot` = this lane's column). QUERY_FOUND:
// (idx, start, end) is the reference's SearchState; QUERY_NONE: the reference returns None; QUERY_DEFER: the window
// could not decide and the general kernel redoes the query from the start. The inner loop has ONE exit (every failure
// breaks out with its status), so the lanes of a warp reconverge after every step instead of carrying a stack of
// divergent returns. Per step: the two pattern nodes, one 16-byte record entry, one or two rank entries.
// A wide record ends the inner loop as well: the lanes that met one take that step together (wide_follow, out of
// line) once every lane has left the loop, and go back in -- the common records never pay for the rare ones, and the
// rare steps of different lanes run side by side instead of one after the other.
template <bool WIDE>
__device__ __forceinline__ void window_extend(const Staged& st, uint32_t slot, uint32_t seg, uint32_t n_seg, uint32_t k, WindowQuery& q) {
    uint32_t idx = q.idx, start = q.start, end = q.end, status = QUERY_ACTIVE;
    uint32_t pat = slot + (q.i - seg) * TILE_LINE;
    const uint32_t pat_end = slot + n_seg * TILE_LINE;
    uint4 h = lds128(st.rec + 16u * idx);
    for (;;) {
        while (pat < pat_end) {
            const uint32_t x1 = lds16(pat), x2 = lds16(pat + TILE_LINE);
            const uint32_t total = h.y & 0xFFFFu, kind = h.y >> 16;
            const uint32_t s = start < total ? start : total, e = end < total ? end : total;
            if (x1 == NODE_OUTSIDE) { status = QUERY_DEFER; break; }
            // Record::follow on an empty range; a record of 0xFFFF positions or more is staged with total 0 (KIND_DEFER), and
            // its range is only empty here because it was not staged
            if (s >= e) { status = kind == KIND_DEFER ? QUERY_DEFER : QUERY_NONE; break; }
            const uint32_t b = x1 == (h.x >> 16) ? 1u : 0u;
            uint32_t rs = s, re = e;
            if (kind < KIND_WIDE) {
                // dense record: rank1(s), and rank1(e) = ones up to and including position e - 1
                if (x1 != (h.x & 0xFFFFu) && b == 0) { status = QUERY_NONE; break; }
                const uint32_t last = e - 1u;
                const uint32_t ws = lds32(st.ranks + 4u * (kind + (s >> 4))), we = lds32(st.ranks + 4u * (kind + (last >> 4)));
                const uint32_t ones_s = (ws & 0xFFFFu) + static_cast<uint32_t>(__popc((ws >> 16) & ~(0xFFFFFFFFu << (s & 15u))));
                const uint32_t ones_e = (we & 0xFFFFu) + static_cast<uint32_t>(__popc((we >> 16) & ~(0xFFFFFFFEu << (last & 15u))));
                rs = b ? ones_s : s - ones_s;
                re = b ? ones_e : e - ones_e;
                if (rs >= re) { status = QUERY_NONE; break; }
            } else if (kind == KIND_SINGLE) {
                if (x1 != (h.x & 0xFFFFu)) { status = QUERY_NONE; break; }
            } else {
                // a wide record (below), BWT::record() is None, or a record the window does not decode
                status = WIDE && kind == KIND_WIDE ? QUERY_WIDE : (kind == KIND_EMPTY ? QUERY_NONE : QUERY_DEFER);
                break;
            }
            // two hops at once when the successor is a single-edge record leading to the pattern node after x1
            const uint32_t hop = b ? h.w : h.z;
            uint32_t offset;
            if (x2 == (hop & 0xFFFFu) && x2 != NODE_OUTSIDE) {
                offset = hop >> 16; idx = x2; pat += 2u * TILE_LINE;
            } else {
                offset = lds16(st.offs + 4u * idx + 2u * b); idx = x1; pat += TILE_LINE;
            }
            start = offset + rs; end = offset + re;
            if (pat >= pat_end) break;
            h = lds128(st.rec + 16u * idx);
        }
        if (!WIDE || status != QUERY_WIDE) break;
        // the same step on a wide record (the tests on x1 and on the range have passed)
        {
            const uint32_t x1 = lds16(pat), x2 = lds16(pat + TILE_LINE);
            const uint32_t total = h.y & 0xFFFFu;
            const uint32_t s = start < total ? start : total, e = end < total ? end : total;
            const uint4 f = wide_follow(st.ranks, st.aux + AUX_BYTES * (h.x & 0xFFFFu), h.z, h.w, h.x >> 16, total, x1, s, e);
            if (f.x >= f.y) { status = QUERY_NONE; break; }
            uint32_t offset;
            if (x2 == (f.z & 0xFFFFu) && x2 != NODE_OUTSIDE) {
                offset = f.z >> 16; idx = x2; pat += 2u * TILE_LINE;
            } else {
                offset = lds16(f.w); idx = x1; pat += TILE_LINE;
            }
            start = offset + f.x; end = offset + f.y;
            status = QUERY_ACTIVE;
            if (pat >= pat_end) break;
            h = lds128(st.rec + 16u * idx);
        }
    }
    q.idx = idx; q.start = start; q.end = end; q.i = seg + (pat - slot) / TILE_LINE;
    q.status = status == QUERY_ACTIVE && q.i >= k ? QUERY_FOUND : status;
}

__device__ __forceinline__ void sts8(uint32_t a, uint32_t x) { asm volatile("st.shared.b8 [%0], %1;" ::"r"(a), "r"(x) : "memory"); }
__device__ __forceinline__ uint32_t lds8(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}

// One record of the window, from its descriptor and shortcuts to its table entries. `aux_counter` = shared address of
// the pool counter, aux_cap = entries in the pool.
template <bool WIDE>
__device__ __forceinline__ void stage_record(const Staged& st, const IndexView& ix, uint32_t r, const Desc& d, const Quad& skip, uint32_t origin,
                                             uint32_t body_lo, uint32_t body_units, uint32_t* aux_counter, uint32_t aux_cap) {
    const uint32_t fmt = d.fmt();
    uint32_t kind = KIND_DEFER, x = NODE_OUTSIDE | (NODE_OUTSIDE << 16), total = 0, offsets = 0;
    uint32_t z = NO_SHORTCUT, w = NO_SHORTCUT;  // inline records: the two-hop shortcuts of the two edges
    const uint32_t unit0 = d.body() - body_lo;  // bodies are 32-byte aligned and lie in record order
    if (fmt == FMT_EMPTY) kind = KIND_EMPTY;
    else if (d.total_len() < 0xFFFFu) {
        total = d.total_len();
        const uint32_t sigma = d.sigma();
        if (fmt == FMT_SINGLE && d.offset0() <= 0xFFFFu) {
            kind = KIND_SINGLE; x = window_index(d.node0(), origin, st.count) | (NODE_OUTSIDE << 16); offsets = d.offset0();
        } else if (fmt == FMT_DENSE2 && d.offset0() <= 0xFFFFu && d.offset1() <= 0xFFFFu) {
            if (d.body() >= body_lo && unit0 + 2u * d.body_len() <= body_units && (unit0 / 2u) * 12u < KIND_WIDE) {
                kind = (unit0 / 2u) * 12u;
                x = window_index(d.node0(), origin, st.count) | (window_index(d.node1(), origin, st.count) << 16);
                offsets = d.offset0() | (d.offset1() << 16);
                if (WIDE) { for (uint32_t j = 0; j < d.body_len(); j++) sts8(st.kinds + unit0 / 2u + j, BLOCK_DENSE2); }
            }
        } else if (WIDE && (fmt == FMT_DENSE4 || fmt == FMT_RUN8) && sigma >= 2 && sigma <= 4 && d.body_len() <= 0xFFFFu) {
            // a wide record: its whole body (runs and checkpoint table) has to be staged, and the pool must have an entry left
            uint32_t units = 2u * d.body_len();
            if (fmt == FMT_RUN8) {
                units = (((d.body_len() + 15u) >> 4) + 1u) & ~1u;
                if (d.checkpoints() != 0) units += ((((total - 1u) >> (d.checkpoints() - 1u)) + 1u) & ~1u);  // one unit per entry (sigma <= 4)
            }
            uint32_t targets[4] = {0, 0, 0, 0}, edge_offsets[4] = {0, 0, 0, 0};
            bool fits = d.body() >= body_lo && unit0 + units <= body_units;
            if (fits) {
                if (d.inline_edges()) {
                    targets[0] = d.node0(); edge_offsets[0] = d.offset0(); targets[1] = d.node1(); edge_offsets[1] = d.offset1();
                } else {
#pragma unroll
                    for (uint32_t e = 0; e < 4; e++) {
                        if (e < sigma) {
                            targets[e] = __ldg(&ix.edges[d.edge_base() + e].node);
                            edge_offsets[e] = __ldg(&ix.edges[d.edge_base() + e].offset);
                        }
                    }
                }
                fits = fits && (edge_offsets[0] | edge_offsets[1] | edge_offsets[2] | edge_offsets[3]) <= 0xFFFFu;
            }
            uint32_t a = aux_cap;
            if (fits) a = atomicAdd(aux_counter, 1u);
            if (a < aux_cap) {
                uint32_t t[4];
#pragma unroll
                for (uint32_t e = 0; e < 4; e++) t[e] = e < sigma ? window_index(targets[e], origin, st.count) : NODE_OUTSIDE;
                const uint32_t at = st.aux + AUX_BYTES * a;
                sts128(at, t[0] | (t[1] << 16), t[2] | (t[3] << 16), NO_SHORTCUT, NO_SHORTCUT);
                sts128(at + 16u, NO_SHORTCUT, NO_SHORTCUT, edge_offsets[0] | (edge_offsets[1] << 16), edge_offsets[2] | (edge_offsets[3] << 16));
                kind = KIND_WIDE;
                x = a | (sigma << 16); z = (unit0 / 2u) | (d.body_len() << 16); w = fmt | (d.checkpoints() << 8);
                for (uint32_t j = 0; j < units / 2u; j++) sts8(st.kinds + unit0 / 2u + j, fmt == FMT_DENSE4 ? BLOCK_DENSE4 : BLOCK_RAW);
            }
        }
    }
    if (kind != KIND_WIDE) {
        // a shortcut whose landing node is not staged or whose offset does not fit is left out (the step then takes one hop)
        z = skip.y <= 0xFFFFu ? (window_index(skip.x, origin, st.count) | (skip.y << 16)) : NO_SHORTCUT;
        w = skip.w <= 0xFFFFu ? (window_index(skip.z, origin, st.count) | (skip.w << 16)) : NO_SHORTCUT;
    }
    sts128(st.rec + 16u * r, x, total | (kind << 16), z, w);
    sts32(st.offs + 4u * r, offsets);
}

// The two-hop shortcuts of a wide record's edges, from the staged tables (the global shortcut array only covers records
// with inline edges): edge b leads to a single-edge record -> {that record's target, offset_b + its edge offset}.
__device__ __forceinline__ void stage_wide_shortcuts(const Staged& st, uint32_t a) {
    const uint32_t at = st.aux + AUX_BYTES * a;
    const uint2 targets = lds64(at);
    const uint2 offsets = lds64(at + 24u);
    uint32_t hops[4];
#pragma unroll
    for (uint32_t b = 0; b < 4; b++) {
        const uint32_t target = ((b < 2 ? targets.x : targets.y) >> (16u * (b & 1u))) & 0xFFFFu;
        const uint32_t offset = ((b < 2 ? offsets.x : offsets.y) >> (16u * (b & 1u))) & 0xFFFFu;
        hops[b] = NO_SHORTCUT;
        if (target != NODE_OUTSIDE) {
            const uint2 next = lds64(st.rec + 16u * target);
            const uint32_t through = offset + (lds32(st.offs + 4u * target) & 0xFFFFu);
            if ((next.y >> 16) == KIND_SINGLE && (next.x & 0xFFFFu) != NODE_OUTSIDE && through <= 0xFFFFu) hops[b] = (next.x & 0xFFFFu) | (through << 16);
        }
    }
    sts64(at + 8u, hops[0], hops[1]);
    sts64(at + 16u, hops[2], hops[3]);
}

// One 32-byte block of the staged body range, according to what its record said it holds.
__device__ __forceinline__ void stage_block(const Staged& st, uint32_t what, uint32_t blk, const Quad& lo, const Quad& hi) {
    const uint32_t at_block = st.ranks + 48u * blk;
    if (what == BLOCK_DENSE2) {
        // a 192-bit dense block (layout.h) as twelve rank entries
        const uint32_t bits[6] = {lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
        uint32_t ones = lo.x;
#pragma unroll
        for (uint32_t j = 0; j < 6; j += 2) {
            const uint32_t a0 = bits[j] & 0xFFFFu, a1 = bits[j] >> 16, b0 = bits[j + 1] & 0xFFFFu, b1 = bits[j + 1] >> 16;
            const uint32_t o1 = ones + static_cast<uint32_t>(__popc(a0)), o2 = o1 + static_cast<uint32_t>(__popc(a1));
            const uint32_t o3 = o2 + static_cast<uint32_t>(__popc(b0));
            sts128(at_block + 8u * j, (ones & 0xFFFFu) | (a0 << 16), (o1 & 0xFFFFu) | (a1 << 16), (o2 & 0xFFFFu) | (b0 << 16), (o3 & 0xFFFFu) | (b1 << 16));
            ones = o3 + static_cast<uint32_t>(__popc(b1));
        }
    } else if (what == BLOCK_DENSE4) {
        // 64 positions of two bits: two entries of 32 positions, the second with the counts of the first half added
        uint32_t c[3] = {lo.x, lo.y & ~DENSE4_TAG, lo.z};
        sts128(at_block, hi.x, hi.y, c[0] | (c[1] << 16), c[2]);
#pragma unroll
        for (uint32_t v = 1; v <= 3; v++) {
            const uint32_t y0 = hi.x ^ (v * 0x55555555u), y1 = hi.y ^ (v * 0x55555555u);
            c[v - 1] += static_cast<uint32_t>(__popc(~(y0 | (y0 >> 1)) & 0x55555555u) + __popc(~(y1 | (y1 >> 1)) & 0x55555555u));
        }
        sts128(at_block + 16u, hi.z, hi.w, c[0] | (c[1] << 16), c[2]);
    } else if (what == BLOCK_RAW) {
        sts128(at_block, lo.x, lo.y, lo.z, lo.w);
        sts128(at_block + 16u, hi.x, hi.y, hi.z, hi.w);
    }
}

constexpr uint32_t SMEM_HEADER = 128;  // control words, keeps the staged arrays 128-byte aligned

// Bytes of shared memory a plan needs.
__host__ __device__ inline uint32_t window_kinds_bytes(uint32_t body_cap) { return (body_cap / 2u + 15u) & ~15u; }
__host__ __device__ inline uint32_t window_smem_bytes(uint32_t max_records, uint32_t body_cap, uint32_t threads, uint32_t aux_cap) {
    return SMEM_HEADER + max_records * RECORD_BYTES + aux_cap * AUX_BYTES + (aux_cap != 0 ? window_kinds_bytes(body_cap) : 0u) +
           (body_cap / 2u) * 48u + (threads / 32u) * TILE_BYTES;
}

// WIDE = false: the instantiation for an index without DENSE4 / byte-per-run records (every staged body block is a
// DENSE2 block: no block kinds, no pool, one barrier less per window).
template <class T, int THREADS, int CTAS, bool WIDE>
__global__ void __launch_bounds__(THREADS, CTAS) k_find_window(IndexView ix, WindowPlan wp, const T* __restrict__ patterns,
                                                                const uint32_t* __restrict__ perm, const uint32_t* __restrict__ bucket_end,
                                                                uint32_t k, gbwt_b200_state* __restrict__ out,
                                                                uint32_t* __restrict__ deferred, uint32_t* __restrict__ counters) {
    extern __shared__ __align__(128) unsigned char smem[];
    volatile uint32_t* ctrl = reinterpret_cast<volatile uint32_t*>(smem);  // [0] window ticket, [1] next query slot
    const uint32_t tid = threadIdx.x, lane = tid & 31u;
    const uint32_t base = static_cast<uint32_t>(ix.offset), records = static_cast<uint32_t>(ix.records);
    Staged st;
    st.rec = smem_addr(smem) + SMEM_HEADER;
    st.offs = st.rec + 16u * wp.max_records;
    st.aux = st.offs + 4u * wp.max_records;
    st.kinds = st.aux + AUX_BYTES * wp.aux_cap;
    st.ranks = st.kinds + (WIDE ? window_kinds_bytes(wp.body_cap) : 0u);
    uint32_t tile = st.ranks + (wp.body_cap / 2u) * 48u + (tid >> 5) * TILE_BYTES;
    // (opaque to the compiler: it would otherwise recompute the shared-window addresses from special registers in every step)
    if (WIDE) asm volatile("" : "+r"(st.rec), "+r"(st.offs), "+r"(st.ranks), "+r"(st.aux), "+r"(tile));
    else asm volatile("" : "+r"(st.rec), "+r"(st.offs), "+r"(st.ranks), "+r"(tile));
    const uint32_t slot = tile + 2u * lane;
    sts16(slot + SEGMENT * TILE_LINE, NODE_OUTSIDE);  // the line after a full segment
    // sector loads need every row segment on a 32-byte boundary
    const bool aligned = (reinterpret_cast<uintptr_t>(patterns) & 31u) == 0 && (k * sizeof(T)) % 32u == 0;
    for (;;) {
        __syncthreads();  // everybody has left the previous window: its shared memory and ctrl[] may be reused
        if (tid == 0) { ctrl[0] = atomicAdd(&counters[0], 1u); ctrl[1] = 0; ctrl[2] = 0; }
        if (WIDE) { for (uint32_t i = tid; i < window_kinds_bytes(wp.body_cap) / 4u; i += THREADS) sts32(st.kinds + 4u * i, 0u); }  // BLOCK_UNUSED
        __syncthreads();
        const uint32_t w = ctrl[0];
        if (w >= wp.windows) break;
        uint32_t q_begin, q_end;
        if (wp.direct_cap != 0) {
            // one-pass placement (k_window_place_direct): window w owns the slots [w cap, (w + 1) cap) of perm, bucket_end[w] = its count
            const uint32_t filled = __ldg(bucket_end + w);
            q_begin = w * wp.direct_cap;
            q_end = q_begin + (filled < wp.direct_cap ? filled : wp.direct_cap);
        } else {
            // (bucket_end[] has one entry per sort bucket, 2^fine of them per window)
            const uint32_t fine_buckets = ((records - 1u) >> (wp.wshift - wp.fine)) + 1u, after = (w + 1u) << wp.fine;
            q_begin = w == 0 ? 0u : __ldg(bucket_end + (w << wp.fine) - 1u);
            q_end = __ldg(bucket_end + (after < fine_buckets ? after : fine_buckets) - 1u);
        }
        if (q_begin >= q_end) continue;
        // Queries are handed out 32 at a time per warp; with wp.prefetch the pattern rows of a warp's NEXT 32 queries are
        // requested from L2 before it works on the current ones.
        uint32_t at = 0, q_cur = 0;
        if (lane == 0) at = q_begin + atomicAdd(const_cast<uint32_t*>(&ctrl[1]), 32u);
        at = __shfl_sync(0xFFFFFFFFu, at, 0);
        if (at + lane < q_end) {
            q_cur = __ldg(perm + at + lane);
            if (wp.prefetch) prefetch_row(patterns + static_cast<size_t>(q_cur) * k, k);
        }
        const uint32_t r0 = w << wp.wshift;
        st.lo = r0 > wp.margin ? r0 - wp.margin : 0u;
        const uint32_t want_hi = r0 + (1u << wp.wshift) + wp.margin;
        const uint32_t hi = want_hi < records ? want_hi : records;
        st.count = hi - st.lo;
        const uint32_t origin = base + st.lo;
        const uint32_t body_lo = __ldg(ix.stage_body + st.lo / STAGE_GRANULE);
        const uint32_t body_hi = __ldg(ix.stage_body + (hi + STAGE_GRANULE - 1u) / STAGE_GRANULE);
        const uint32_t body_units = body_hi - body_lo < wp.body_cap ? body_hi - body_lo : wp.body_cap;
        // decode the window into shared memory: descriptors + shortcuts first (a record also says what its body blocks
        // hold), then the body blocks and, from the finished record table, the shortcuts of the wide records. (Requesting
        // two records or blocks per thread before decoding either was measured: the extra live registers spill under the
        // 64-register budget of two 512-thread CTAs per SM, 6.2 -> 5.0 G queries/s.)
        for (uint32_t r = tid; r < st.count; r += THREADS) {
            Desc d;
            load_sector(reinterpret_cast<const Unit16*>(ix.desc + st.lo + r), d.a, d.b);
            const Quad skip = load_quad(ix.skips + st.lo + r);
            stage_record<WIDE>(st, ix, r, d, skip, origin, body_lo, body_units, const_cast<uint32_t*>(&ctrl[2]), wp.aux_cap);
        }
        if (WIDE) __syncthreads();
        for (uint32_t blk = tid; blk < body_units / 2u; blk += THREADS) {
            const uint32_t what = WIDE ? lds8(st.kinds + blk) : static_cast<uint32_t>(BLOCK_DENSE2);
            if (what == BLOCK_UNUSED) continue;
            Quad lo, hi;
            load_sector(ix.bodies + body_lo + 2u * blk, lo, hi);
            stage_block(st, what, blk, lo, hi);
        }
        if (WIDE) {
            const uint32_t wide = ctrl[2] < wp.aux_cap ? ctrl[2] : wp.aux_cap;
            for (uint32_t a = tid; a < wide; a += THREADS) stage_wide_shortcuts(st, a);
        }
        __syncthreads();
        while (at < q_end) {
            uint32_t next_at = 0, q_next = 0;
            if (lane == 0) next_at = q_begin + atomicAdd(const_cast<uint32_t*>(&ctrl[1]), 32u);
            next_at = __shfl_sync(0xFFFFFFFFu, next_at, 0);
            if (next_at + lane < q_end) {
                q_next = __ldg(perm + next_at + lane);
                if (wp.prefetch) prefetch_row(patterns + static_cast<size_t>(q_next) * k, k);
            }
            const bool mine = at + lane < q_end;
            WindowQuery q;
            q.idx = 0; q.start = 0; q.end = 0; q.i = 0; q.status = mine && k != 0 ? QUERY_ACTIVE : QUERY_NONE;
            for (uint32_t seg = 0; seg < k; seg += SEGMENT) {
                if (!__any_sync(0xFFFFFFFFu, q.status == QUERY_ACTIVE)) break;
                const uint32_t n_seg = k - seg < SEGMENT ? k - seg : SEGMENT;
                load_tile<T>(patterns, q.status == QUERY_ACTIVE ? q_cur : NO_QUERY, k, seg, n_seg, aligned && n_seg % (32u / sizeof(T)) == 0, tile, origin,
                             st.count, lane);
                if (n_seg < SEGMENT) sts16(slot + n_seg * TILE_LINE, NODE_OUTSIDE);  // the line after a short segment
                __syncwarp();
                if (q.status == QUERY_ACTIVE) {
                    if (seg == 0) window_find(st, lds16(slot), k, q);
                    if (q.status == QUERY_ACTIVE) window_extend<WIDE>(st, slot, seg, n_seg, k, q);
                }
                __syncwarp();  // the tile is rewritten in the next round
            }
            if (mine) {
                if (q.status == QUERY_DEFER || q.status == QUERY_ACTIVE) {
                    deferred[atomicAdd(&counters[1], 1u)] = q_cur;
                } else {
                    const bool found = q.status == QUERY_FOUND;
                    gbwt_b200_state result;
                    result.node = found ? q.idx + origin : 0u; result.start = found ? q.start : 0u; result.end = found ? q.end : 0u;
                    store_state(out + q_cur, result);
                }
            }
            at = next_at; q_cur = q_next;
        }
    }
}

// ---- path extraction from record windows ----------------------------------------------------------------------------
// Checkpointed extraction (kernels.cuh: k_extract_checkpointed) walks segment j of every sequence with one lane, each
// lane loading the records it meets from L1 / L2 / HBM: 62 instructions per node at 24 warps per SM, a third of the issue
// slots busy, every step an L2 round trip. But the lanes that walk segment j of neighbouring sequences walk the SAME
// records -- that is what a pangenome is. Here a CTA takes segment j of 512 sequences, stages the window of records its
// lanes are in (the staging of the search kernel above: one 16-byte entry per record, one 4-byte entry per 16 positions
// of a bitvector) and every lane steps through it from shared memory; when most lanes have left the window the CTA
// stages the next one. A lane that cannot take a step from the window (its node is not staged, a record format the
// window does not decode, the end of a sequence) takes that step from the global layout instead, so the result never
// depends on where the windows fall. Every node is still produced by an LF step (Record::lf, src/bwt.rs:480-496).
// A lane parks up to 64 nodes between flushes, as 16-bit differences from the first node of the row (a walk stays near
// where it is; a node that does not fit ends the round early): rows of 64 nodes leave as 512 contiguous bytes, and 256-byte
// pieces from 150 k rows at a time were what bound the first version (DRAM wrote 54.6 GB at 2.6 TB/s, every piece a page
// of its own). Row stride: 33 words.
constexpr uint32_t EXTRACT_TILE_NODES = 64, EXTRACT_TILE_STRIDE = 33;

// One LF step from the global layout: GBWT::forward (src/gbwt.rs:222-229). (offset << 32) | node, 0 = None. Out of line
// (and therefore without the 256-bit inline-asm load, see DESIGN.md): the rare step must not weigh on the walk's registers.
__device__ __noinline__ uint64_t global_forward(const RecordDesc* descs, const Unit16* bodies, const Edge* edges, uint32_t base, uint32_t records,
                                                uint32_t node, uint32_t offset) {
    const uint32_t rec = node - base;
    if (node < base + 1u || rec >= records) return 0;
    Desc d;
    d.a = load_quad(reinterpret_cast<const Unit16*>(descs + rec));
    d.b = load_quad(reinterpret_cast<const Unit16*>(descs + rec) + 1);
    const uint32_t fmt = d.fmt();
    if (fmt == FMT_EMPTY || offset >= d.total_len()) return 0;
    IndexView view;  // the scans only look at the bodies and the edge lists
    view.desc = descs; view.bodies = bodies; view.edges = edges; view.endmarker = nullptr;
    view.records = records; view.offset = base; view.alphabet_size = 0; view.sequences = 0; view.endmarker_len = 0;
    view.bidirectional = 0; view.skips = nullptr; view.edges_valid = 1; view.walk_limit = 0; view.stage_body = nullptr;
    uint32_t symbol, rank_i;
    if (fmt == FMT_SINGLE) {
        symbol = 0; rank_i = offset;
    } else if (fmt == FMT_DENSE2) {
        // (the block with two 128-bit loads: the 256-bit inline-asm load must not appear in a function that is not inlined)
        uint32_t blk = offset / DENSE_BITS;
        if (blk >= d.body_len()) blk = d.body_len() - 1;
        DenseBlock block;
        block.lo = load_quad(bodies + d.body() + 2 * blk);
        block.hi = load_quad(bodies + d.body() + 2 * blk + 1);
        const uint32_t ones = dense_block_rank1(block, offset - blk * DENSE_BITS, symbol);
        rank_i = symbol ? ones : offset - ones;
    } else {
        symbol = symbol_at_runs(view, d, offset);
        if (symbol == NO_SYMBOL) return 0;
        FlipSet fs;
        fs.lt = 0; fs.extra = NO_SYMBOL;
        Ranks r;
        r.at_start = r.at_end = r.flipped = 0;
        rank_runs_inline<false>(view, d, symbol, fs, offset, offset, r);
        rank_i = r.at_start;
    }
    const Edge e = edge_at(view, d, symbol);
    if (e.node == 0) return 0;  // successor is the endmarker: the sequence ends (src/bwt.rs:485-486)
    return (static_cast<uint64_t>(e.offset + rank_i) << 32) | e.node;
}

struct ExtractLane {
    uint32_t node, offset;  // current position
    uint32_t left;          // nodes of the segment still to be emitted (0 = done)
    uint32_t parked;        // nodes in the tile row
    uint32_t row_base;      // the tile row holds node - row_base
    bool moved;             // has taken a step from this window
};

__device__ __forceinline__ bool fits_row(uint32_t node, uint32_t row_base) { return node - row_base + 0x8000u < 0x10000u; }
__device__ __forceinline__ int32_t lds16_signed(uint32_t a) {
    int32_t v;
    asm volatile("ld.shared.s16 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}

// As many steps as the tile row has room for. The inner loop only knows the common step (the node's record is staged
// and decoded, and so is the record it leads to) and leaves for anything else, which is sorted out per lane below: a
// lane whose step leads out of the staged range waits for the next window if it has moved in this one, and otherwise
// takes the step from the global layout, as it does for records the window does not decode and at the end of a
// sequence -- every window moves every lane. Returns true if the lane is waiting.
__device__ __forceinline__ bool extract_round(const Staged& st, uint32_t origin, ExtractLane& ln, uint32_t row, const RecordDesc* descs,
                                              const Unit16* bodies, const Edge* edges, uint32_t base, uint32_t records) {
    uint32_t node = ln.node, offset = ln.offset, left = ln.left, at_row = row + 2u * ln.parked;
    const uint32_t row_end = row + 2u * (EXTRACT_TILE_NODES - 1u);  // room for two nodes below this address
    if (ln.parked == 0) ln.row_base = node;
    const uint32_t row_base = ln.row_base;
    bool waiting = false, moved = ln.moved, full = false;  // full: a node does not fit the row (16-bit differences)
    for (;;) {
        bool leaves = false;  // the inner loop left because the step leads out of the staged range (or the node is not staged)
        while (left != 0 && at_row < row_end) {
            const uint32_t idx = node - origin;
            if (idx >= st.count) { leaves = true; break; }
            const uint4 h = lds128(st.rec + 16u * idx);
            const uint32_t kind = h.y >> 16, total = h.y & 0xFFFFu;
            if ((kind >= KIND_WIDE && kind != KIND_SINGLE) || offset >= total) break;  // not decoded here / GBWT::forward -> None
            uint32_t b = 0, r = offset;
            if (kind != KIND_SINGLE) {
                const uint32_t w = lds32(st.ranks + 4u * (kind + (offset >> 4)));
                const uint32_t sh = offset & 15u;
                b = (w >> (16u + sh)) & 1u;
                const uint32_t ones = (w & 0xFFFFu) + static_cast<uint32_t>(__popc((w >> 16) & ~(0xFFFFFFFFu << sh)));
                r = b ? ones : offset - ones;
            }
            const uint32_t target = b ? h.x >> 16 : h.x & 0xFFFFu, hop = b ? h.w : h.z;
            if (target == NODE_OUTSIDE) { leaves = true; break; }
            if (!fits_row(node, row_base)) { full = true; break; }  // (only with nodes parked before it: the row starts again here)
            if (!fits_row(target + origin, row_base)) break;        // (a far jump: one node at a time, below)
            sts16(at_row, node - row_base);
            if ((hop & 0xFFFFu) != NODE_OUTSIDE) {
                // two nodes: the successor is a single-edge record (layout.h, IndexView::skips)
                if (left > 1) sts16(at_row + 2u, target + origin - row_base);
                at_row += left > 1 ? 4u : 2u;
                node = (hop & 0xFFFFu) + origin; offset = (hop >> 16) + r;
                left = left > 2 ? left - 2 : 0;
            } else {
                at_row += 2u;
                node = target + origin; offset = lds16(st.offs + 4u * idx + 2u * b) + r;
                left -= 1;
            }
            moved = true;
        }
        if (left == 0 || at_row >= row_end || full) break;
        if (leaves && moved) { waiting = true; break; }
        // one step from the global layout
        if (!fits_row(node, row_base)) break;  // (the row is written out and starts again at this node)
        sts16(at_row, node - row_base);
        at_row += 2u;
        const uint64_t next = global_forward(descs, bodies, edges, base, records, node, offset);
        if (next == 0) { left = 0; break; }
        node = static_cast<uint32_t>(next); offset = static_cast<uint32_t>(next >> 32);
        left -= 1;
        moved = true;
    }
    ln.node = node; ln.offset = offset; ln.left = left; ln.parked = (at_row - row) / 2u; ln.moved = moved;
    return waiting;
}

template <int THREADS, int CTAS>
__global__ void __launch_bounds__(THREADS, CTAS) k_extract_window(IndexView ix, CheckpointView cv, WindowPlan wp, const uint64_t* __restrict__ ids, size_t m,
                                                                const uint64_t* __restrict__ out_offsets, uint64_t base_offset,
                                                                uint64_t* __restrict__ nodes, uint64_t* __restrict__ lengths,
                                                                uint32_t* __restrict__ counters) {
    constexpr unsigned FULL = 0xFFFFFFFFu;
    extern __shared__ __align__(128) unsigned char smem[];
    // ctrl: [0] work ticket, [2] lowest record of an active lane, [3] highest, [4] lanes walking towards higher records
    volatile uint32_t* ctrl = reinterpret_cast<volatile uint32_t*>(smem);
    const uint32_t tid = threadIdx.x, lane = tid & 31u;
    const uint32_t base = static_cast<uint32_t>(ix.offset), records = static_cast<uint32_t>(ix.records);
    Staged st;
    st.rec = smem_addr(smem) + SMEM_HEADER;
    st.offs = st.rec + 16u * wp.max_records;
    st.aux = st.offs + 4u * wp.max_records;
    st.kinds = st.aux;
    st.ranks = st.aux;
    uint32_t tiles = st.ranks + (wp.body_cap / 2u) * 48u;
    asm volatile("" : "+r"(st.rec), "+r"(st.offs), "+r"(st.ranks), "+r"(tiles));
    const uint32_t tile = tiles + (tid >> 5) * (32u * EXTRACT_TILE_STRIDE * 4u), row = tile + lane * (EXTRACT_TILE_STRIDE * 4u);
    const RecordDesc* const descs = ix.desc;
    const Unit16* const bodies = ix.bodies;
    const Edge* const edges = ix.edges;
    const uint64_t blocks = (m + THREADS - 1) / THREADS;
    const uint64_t items = blocks * cv.max_segments;
    for (;;) {
        __syncthreads();
        if (tid == 0) ctrl[0] = atomicAdd(&counters[0], 1u);
        __syncthreads();
        const uint64_t item = ctrl[0];
        if (item >= items) break;
        const uint64_t j = item / blocks, i = (item - j * blocks) * THREADS + tid;
        // this lane's segment, if it has one (as in k_extract_checkpointed)
        ExtractLane ln;
        ln.node = 0; ln.offset = 0; ln.left = 0; ln.parked = 0; ln.row_base = 0; ln.moved = false;
        uint64_t* dst = nodes;
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
                    ln.node = raw.x; ln.offset = raw.y;
                    const uint64_t index = (static_cast<uint64_t>(raw.w) << 32) | raw.z;
                    uint64_t end = len;
                    if (j + 1 < count) {
                        const uint4 next = __ldg(reinterpret_cast<const uint4*>(cv.table + first + j + 1));
                        end = (static_cast<uint64_t>(next.w) << 32) | next.z;
                    }
                    if (end > cap) end = cap;  // nothing beyond the caller's slot is written
                    const uint64_t todo = end > index ? end - index : 0;
                    ln.left = todo < 0xFFFFFFFFull ? static_cast<uint32_t>(todo) : 0xFFFFFFFFu;
                    dst = nodes + (lo - base_offset) + index;
                }
            }
        }
        // windows until every lane is done
        for (;;) {
            // where the active lanes are, and which way they walk (node identifiers follow the graph's topological order:
            // a forward node leads to higher records, a reverse node to lower ones; only a matter of speed if not)
            __syncthreads();
            if (tid == 0) { ctrl[2] = 0xFFFFFFFFu; ctrl[3] = 0; ctrl[4] = 0; ctrl[5] = 0; ctrl[6] = 0; }
            __syncthreads();
            if (ln.left != 0) {
                const uint32_t rec = ln.node - base;
                atomicMin(const_cast<uint32_t*>(&ctrl[2]), rec);
                atomicMax(const_cast<uint32_t*>(&ctrl[3]), rec);
                atomicAdd(const_cast<uint32_t*>(&ctrl[(ln.node & 1u) == 0 ? 4 : 5]), 1u);
            }
            __syncthreads();
            const uint32_t lowest = ctrl[2], highest = ctrl[3], up = ctrl[4], down = ctrl[5];
            if (up + down == 0) break;
            const uint32_t behind = STAGE_GRANULE;  // records kept behind the slowest lane
            uint32_t lo;
            if (up >= down) lo = lowest > behind ? lowest - behind : 0u;
            else lo = highest + behind + 1u > wp.max_records ? highest + behind + 1u - wp.max_records : 0u;
            lo &= ~(STAGE_GRANULE - 1u);
            st.lo = lo;
            const uint32_t hi = lo + wp.max_records < records ? lo + wp.max_records : records;
            st.count = hi - lo;
            const uint32_t origin = base + lo;
            const uint32_t body_lo = __ldg(ix.stage_body + lo / STAGE_GRANULE);
            const uint32_t body_hi = __ldg(ix.stage_body + (hi + STAGE_GRANULE - 1u) / STAGE_GRANULE);
            const uint32_t body_units = body_hi - body_lo < wp.body_cap ? body_hi - body_lo : wp.body_cap;
            for (uint32_t r = tid; r < st.count; r += THREADS) {
                Desc d;
                load_sector(reinterpret_cast<const Unit16*>(ix.desc + lo + r), d.a, d.b);
                const Quad skip = load_quad(ix.skips + lo + r);
                stage_record<false>(st, ix, r, d, skip, origin, body_lo, body_units, nullptr, 0);
            }
            for (uint32_t blk = tid; blk < body_units / 2u; blk += THREADS) {
                Quad blo, bhi;
                load_sector(ix.bodies + body_lo + 2u * blk, blo, bhi);
                stage_block(st, BLOCK_DENSE2, blk, blo, bhi);
            }
            __syncthreads();
            ln.moved = false;
            // rounds in this window: walk, write the tile out. No barrier between rounds (the warps of a CTA would otherwise
            // all walk and then all write): a warp leaves for the next window when all of its walkers wait for it, or when an
            // eighth of the CTA's walkers do (ctrl[6], which only grows while a window lasts).
            uint32_t reported = 0;
            for (;;) {
                const bool waiting = extract_round(st, origin, ln, row, descs, bodies, edges, base, records);
                __syncwarp();
                // all rows of the warp out, one after the other: up to 512 contiguous bytes per row, 256 per store instruction
                const uint64_t row_addr = reinterpret_cast<uint64_t>(dst);
#pragma unroll 4
                for (uint32_t r = 0; r < 32; r++) {
                    const uint32_t n = __shfl_sync(FULL, ln.parked, r);
                    const uint32_t first = __shfl_sync(FULL, ln.row_base, r);
                    const uint32_t a_lo = __shfl_sync(FULL, static_cast<uint32_t>(row_addr), r);
                    const uint32_t a_hi = __shfl_sync(FULL, static_cast<uint32_t>(row_addr >> 32), r);
                    uint64_t* to = reinterpret_cast<uint64_t*>((static_cast<uint64_t>(a_hi) << 32) | a_lo);
                    if (cv.discard) continue;
                    const uint32_t at = tile + r * (EXTRACT_TILE_STRIDE * 4u) + 2u * lane;
                    if (lane < n) __stcs(to + lane, static_cast<uint64_t>(first + static_cast<uint32_t>(lds16_signed(at))));
                    if (lane + 32u < n) __stcs(to + lane + 32u, static_cast<uint64_t>(first + static_cast<uint32_t>(lds16_signed(at + 64u))));
                }
                __syncwarp();
                dst += ln.parked;
                ln.parked = 0;
                const unsigned walkers = __ballot_sync(FULL, ln.left != 0), waiters = __ballot_sync(FULL, ln.left != 0 && waiting);
                if (walkers == waiters) break;  // (nobody left who could move in this window)
                const uint32_t stalled = static_cast<uint32_t>(__popc(waiters));
                if (lane == 0 && stalled > reported) atomicAdd(const_cast<uint32_t*>(&ctrl[6]), stalled - reported);
                reported = stalled > reported ? stalled : reported;
                if (8u * ctrl[6] >= up + down) break;
            }
        }
    }
}

// Pattern reader of the kernels that keep the chunk in registers (the general loop for deferred queries and the plain
// 32-bit kernels): same interface, no shared memory.
template <class T>
struct PlainRowReader {
    const T* p;
    __device__ __forceinline__ bool node(uint32_t i, uint32_t& out) {
        const uint64_t v = __ldg(p + i);
        out = static_cast<uint32_t>(v);
        return (v >> 32) == 0;
    }
};

// ---- bidirectional search from record windows ------------------------------------------------------------------------
// bd_find(path[first]) + extend_forward over path(first, end) + extend_backward over path[start, first) (the driver of
// src/gbwt/tests.rs:352-361 over src/gbwt.rs:311-384), with the records in shared memory like the search above. The batch
// is sorted by the window of path[first]; a warp takes 32 searches, reads the nodes path[start, end) of each into a tile of
// 32 lines (window indexes, one line per position; longer subpaths go to the general kernel) and every lane runs the two
// phases on it: forward extensions up the tile, then -- a backward extension by x is a forward extension of the flipped
// state by flip(x), src/gbwt.rs:362-367 -- the same loop down the tile on the other strand's records, which lie next to
// this strand's in record order. Per step the half being extended moves like GBWT::extend, the other half's range start
// moves by the number of positions of the range whose successor precedes the extension in the reverse order
// (Record::bd_follow, src/bwt.rs:621-656): for a record with two edges that is all the ones, all the zeros or nothing,
// depending on the edge taken and on whether the two successors are the two orientations of one node. Records the window
// does not decode, nodes it does not hold and subpaths longer than the tile put the search on the deferred list.
constexpr uint32_t BD_TILE_LINES = 32, BD_TILE_BYTES = (BD_TILE_LINES + 2u) * TILE_LINE;  // one sentinel line either side

// The extensions of one search in ONE loop: `fwd` forward extensions by the tile lines above the anchor, then `bwd` backward
// extensions by the lines below it, which are forward extensions of the flipped state by the flipped nodes
// (src/gbwt.rs:362-367). Half `a` is the one being extended (at window index a_idx), `b` the other one: when a lane has
// made its forward extensions it swaps the halves and walks down. The lanes of a warp share the loop whatever phase each
// is in, so a warp spends max(fwd + bwd) iterations on its 32 searches; as two loops, one per phase, it spent
// max(fwd) + max(bwd), nearly twice that on subpaths with the anchor anywhere (profiles/r2_bd_window_ncu.txt: 10 of
// 32 lanes active in the loops). Returns QUERY_ACTIVE when all extensions were made; `flipped` says which half `a` is then.
__device__ __forceinline__ uint32_t bd_window_extend(const Staged& st, uint32_t origin, uint32_t at_anchor, uint32_t fwd, uint32_t bwd,
                                                     uint32_t& a_idx, uint32_t& a_start, uint32_t& a_end, uint32_t& b_idx, uint32_t& b_start,
                                                     bool& flipped) {
    const uint32_t parity = origin & 1u;
    uint32_t left = fwd, later = bwd, pat = at_anchor + TILE_LINE;
    int32_t line = static_cast<int32_t>(TILE_LINE);
    uint32_t flip = 0;  // 1 in the backward phase
    uint32_t status = QUERY_ACTIVE;
    for (;;) {
        // (selects, not branches: the lanes of a warp are in different phases and must not part ways over this)
        const bool turn = left == 0;
        if (turn && later == 0) break;
        // a lane that has made its forward extensions: the other half's range has the same size; it becomes the half to extend
        const uint32_t size = a_end - a_start, o_idx = a_idx, o_start = a_start;
        a_idx = turn ? b_idx : a_idx; b_idx = turn ? o_idx : b_idx;
        a_start = turn ? b_start : a_start; b_start = turn ? o_start : b_start;
        a_end = a_start + size;
        left = turn ? later : left; later = turn ? 0u : later; flip = turn ? 1u : flip;
        line = turn ? -static_cast<int32_t>(TILE_LINE) : line; pat = turn ? at_anchor - TILE_LINE : pat;
        const uint4 h = lds128(st.rec + 16u * a_idx);
        uint32_t x1 = lds16(pat), x2 = left > 1 ? lds16(pat + line) : NODE_OUTSIDE;
        // backward: flip(node) as a window index -- the other orientation's record is the neighbour (node ^ 1); forward: as it is
        x1 = x1 == NODE_OUTSIDE ? x1 : ((x1 + parity) ^ flip) - parity;
        x2 = x2 == NODE_OUTSIDE ? x2 : ((x2 + parity) ^ flip) - parity;
        if (x1 >= st.count) x1 = NODE_OUTSIDE;
        if (x2 >= st.count) x2 = NODE_OUTSIDE;
        if (x1 == NODE_OUTSIDE) { status = QUERY_DEFER; break; }
        const uint32_t total = h.y & 0xFFFFu, kind = h.y >> 16;
        const uint32_t s = a_start < total ? a_start : total, e = a_end < total ? a_end : total;
        if (s >= e) { status = kind == KIND_DEFER ? QUERY_DEFER : QUERY_NONE; break; }  // (as in window_extend)
        const uint32_t t0 = h.x & 0xFFFFu, t1 = h.x >> 16;
        uint32_t b = 0, rs = s, re = e, moved = 0;
        if (kind < KIND_WIDE) {
            b = x1 == t1 ? 1u : 0u;
            if (x1 != t0 && b == 0) { status = QUERY_NONE; break; }
            if (t0 == NODE_OUTSIDE || t1 == NODE_OUTSIDE) { status = QUERY_DEFER; break; }  // (cannot tell whether the successors are one node's two orientations)
            const uint32_t last = e - 1u;
            const uint32_t ws = lds32(st.ranks + 4u * (kind + (s >> 4))), we = lds32(st.ranks + 4u * (kind + (last >> 4)));
            const uint32_t ones_s = (ws & 0xFFFFu) + static_cast<uint32_t>(__popc((ws >> 16) & ~(0xFFFFFFFFu << (s & 15u))));
            const uint32_t ones_e = (we & 0xFFFFu) + static_cast<uint32_t>(__popc((we >> 16) & ~(0xFFFFFFFEu << (last & 15u))));
            rs = b ? ones_s : s - ones_s;
            re = b ? ones_e : e - ones_e;
            if (rs >= re) { status = QUERY_NONE; break; }
            // Record::bd_follow's second value: edge 0 is preceded (in the reverse order) by edge 1 only when both lead to the
            // same node and edge 0 to its forward orientation; edge 1 by edge 0 unless that is the case
            const bool paired = t1 == t0 + 1u && ((t0 + origin) & 1u) == 0;
            const uint32_t ones = ones_e - ones_s, zeros = (e - s) - ones;
            moved = b == 0 ? (paired ? ones : 0u) : (paired ? 0u : zeros);
        } else if (kind == KIND_SINGLE) {
            if (x1 != t0) { status = QUERY_NONE; break; }
        } else {
            status = kind == KIND_EMPTY ? QUERY_NONE : QUERY_DEFER;
            break;
        }
        b_start += moved;
        const uint32_t hop = b ? h.w : h.z;
        uint32_t offset;
        if (x2 == (hop & 0xFFFFu) && x2 != NODE_OUTSIDE) {
            // two extensions at once: the second one is over a single-edge record, which moves neither range start
            offset = hop >> 16; a_idx = x2; pat += 2 * line; left -= 2;
        } else {
            offset = lds16(st.offs + 4u * a_idx + 2u * b); a_idx = x1; pat += line; left -= 1;
        }
        a_start = offset + rs; a_end = offset + re;
    }
    flipped = flip != 0;
    return status;
}

template <int THREADS, int CTAS>
__global__ void __launch_bounds__(THREADS, CTAS) k_bd_window(IndexView ix, WindowPlan wp, const uint64_t* __restrict__ nodes,
                                                              const uint64_t* __restrict__ offsets, uint64_t base_offset,
                                                              const uint64_t* __restrict__ first, const uint64_t* __restrict__ start,
                                                              const uint64_t* __restrict__ end, const uint32_t* __restrict__ perm,
                                                              const uint4* __restrict__ packed, const uint32_t* __restrict__ bucket_end,
                                                              gbwt_b200_bdstate* __restrict__ out, uint32_t* __restrict__ deferred,
                                                              uint32_t* __restrict__ counters) {
    constexpr unsigned FULL = 0xFFFFFFFFu;
    (void)offsets; (void)first; (void)start; (void)end;  // (read by the placement step, which left what is needed in `packed`)
    extern __shared__ __align__(128) unsigned char smem[];
    volatile uint32_t* ctrl = reinterpret_cast<volatile uint32_t*>(smem);  // [0] window ticket, [1] next query slot
    const uint32_t tid = threadIdx.x, lane = tid & 31u;
    const uint32_t base = static_cast<uint32_t>(ix.offset), records = static_cast<uint32_t>(ix.records);
    Staged st;
    st.rec = smem_addr(smem) + SMEM_HEADER;
    st.offs = st.rec + 16u * wp.max_records;
    st.aux = st.offs + 4u * wp.max_records;
    st.kinds = st.aux;
    st.ranks = st.aux;
    uint32_t tile = st.ranks + (wp.body_cap / 2u) * 48u + (tid >> 5) * BD_TILE_BYTES;
    asm volatile("" : "+r"(st.rec), "+r"(st.offs), "+r"(st.ranks), "+r"(tile));
    const uint32_t slot = tile + 2u * lane;  // line 0 is the sentinel below the first node, data in lines 1 .. 32
    sts16(slot, NODE_OUTSIDE);
    for (;;) {
        __syncthreads();
        if (tid == 0) { ctrl[0] = atomicAdd(&counters[0], 1u); ctrl[1] = 0; }
        __syncthreads();
        const uint32_t w = ctrl[0];
        if (w >= wp.windows) break;
        uint32_t q_begin, q_end;
        if (wp.direct_cap != 0) {  // (one-pass placement: window w owns perm / packed [w cap, (w + 1) cap), bucket_end[w] = its count)
            const uint32_t filled = __ldg(bucket_end + w);
            q_begin = w * wp.direct_cap;
            q_end = q_begin + (filled < wp.direct_cap ? filled : wp.direct_cap);
        } else {
            q_begin = w == 0 ? 0u : __ldg(bucket_end + w - 1u);
            q_end = __ldg(bucket_end + w);
        }
        if (q_begin >= q_end) continue;
        uint32_t at = 0;
        if (lane == 0) at = q_begin + atomicAdd(const_cast<uint32_t*>(&ctrl[1]), 32u);
        at = __shfl_sync(FULL, at, 0);
        const uint32_t r0 = w << wp.wshift;
        st.lo = r0 > wp.margin ? r0 - wp.margin : 0u;
        const uint32_t want_hi = r0 + (1u << wp.wshift) + wp.margin;
        const uint32_t hi = want_hi < records ? want_hi : records;
        st.count = hi - st.lo;
        const uint32_t origin = base + st.lo;
        const uint32_t body_lo = __ldg(ix.stage_body + st.lo / STAGE_GRANULE);
        const uint32_t body_hi = __ldg(ix.stage_body + (hi + STAGE_GRANULE - 1u) / STAGE_GRANULE);
        const uint32_t body_units = body_hi - body_lo < wp.body_cap ? body_hi - body_lo : wp.body_cap;
        for (uint32_t r = tid; r < st.count; r += THREADS) {
            Desc d;
            load_sector(reinterpret_cast<const Unit16*>(ix.desc + st.lo + r), d.a, d.b);
            const Quad skip = load_quad(ix.skips + st.lo + r);
            stage_record<false>(st, ix, r, d, skip, origin, body_lo, body_units, nullptr, 0);
        }
        for (uint32_t blk = tid; blk < body_units / 2u; blk += THREADS) {
            Quad blo, bhi;
            load_sector(ix.bodies + body_lo + 2u * blk, blo, bhi);
            stage_block(st, BLOCK_DENSE2, blk, blo, bhi);
        }
        __syncthreads();
        while (at < q_end) {
            const bool mine = at + lane < q_end;
            const uint32_t q = mine ? __ldg(perm + at + lane) : 0u;
            // this lane's search: nodes path[begin, finish) of its path, bd_find at `anchor`
            uint32_t status = QUERY_NONE, length = 0, anchor = 0;
            const uint64_t* row = nullptr;
            if (mine) {
                const uint4 rec = __ldg(packed + at + lane);
                if (rec.z != 0) {  // (else None, like query_bd_search_fast)
                    status = rec.z <= BD_TILE_LINES ? QUERY_ACTIVE : QUERY_DEFER;
                    length = rec.z; anchor = rec.w;
                    row = nodes + ((static_cast<uint64_t>(rec.y) << 32) | rec.x);
                }
            }
            // the tile: line 1 + t = node t of every row's subpath, NODE_OUTSIDE beyond its end; one row per iteration, lanes = positions
            const unsigned long long my_row = reinterpret_cast<unsigned long long>(status == QUERY_ACTIVE ? row : nullptr);
            // (eight rows requested before the first one is narrowed: the rows of a sorted batch are scattered over HBM)
#pragma unroll 1
            for (uint32_t r0 = 0; r0 < 32; r0 += 8) {
                uint64_t loaded[8];
                bool have[8];
#pragma unroll
                for (uint32_t j = 0; j < 8; j++) {
                    const uint64_t* p = reinterpret_cast<const uint64_t*>(__shfl_sync(FULL, my_row, r0 + j));
                    const uint32_t n = __shfl_sync(FULL, length, r0 + j);
                    have[j] = p != nullptr;
                    loaded[j] = 0;
                    if (have[j] && lane < n) loaded[j] = __ldg(p + lane);
                }
#pragma unroll
                for (uint32_t j = 0; j < 8; j++) {
                    // (beyond the end of a subpath `loaded` is node 0, which is no record of any window: NODE_OUTSIDE)
                    if (have[j]) sts16(tile + ((1u + lane) * TILE_PITCH + r0 + j) * 2u, loaded[j] == 0 ? NODE_OUTSIDE : pattern_index(loaded[j], origin, st.count));
                }
            }
            if (status == QUERY_ACTIVE) sts16(slot + (1u + BD_TILE_LINES) * TILE_LINE, NODE_OUTSIDE);
            __syncwarp();
            uint32_t f_idx = 0, f_start = 0, f_end = 0, r_idx = 0, r_start = 0, r_end = 0;
            if (status == QUERY_ACTIVE) {
                // bd_find (src/gbwt.rs:311-324)
                const uint32_t at_anchor = slot + (1u + anchor) * TILE_LINE;
                const uint32_t x0 = lds16(at_anchor);
                const uint32_t parity = origin & 1u;
                const uint32_t x0_flip = x0 == NODE_OUTSIDE ? x0 : ((x0 + parity) ^ 1u) - parity;
                if (x0 == NODE_OUTSIDE || x0 + st.lo == 0 || x0_flip >= st.count) status = QUERY_DEFER;
                else {
                    const uint2 h = lds64(st.rec + 16u * x0);
                    const uint32_t kind = h.y >> 16, total = h.y & 0xFFFFu;
                    if (kind == KIND_DEFER) status = QUERY_DEFER;
                    else if (kind == KIND_EMPTY || total == 0) status = QUERY_NONE;
                    else {
                        // `a` starts as the forward half, `b` as the reverse half
                        uint32_t a_idx = x0, a_start = 0, a_end = total, b_idx = x0_flip, b_start = 0;
                        bool flipped = false;
                        status = bd_window_extend(st, origin, at_anchor, length - anchor - 1u, anchor, a_idx, a_start, a_end, b_idx, b_start, flipped);
                        const uint32_t b_end = b_start + (a_end - a_start);
                        f_idx = flipped ? b_idx : a_idx; f_start = flipped ? b_start : a_start; f_end = flipped ? b_end : a_end;
                        r_idx = flipped ? a_idx : b_idx; r_start = flipped ? a_start : b_start; r_end = flipped ? a_end : b_end;
                    }
                }
            }
            __syncwarp();  // the tile is rewritten for the next 32 searches
            if (mine) {
                if (status == QUERY_DEFER) {
                    deferred[atomicAdd(&counters[1], 1u)] = q;
                } else {
                    const bool found = status == QUERY_ACTIVE;
                    gbwt_b200_bdstate result;
                    result.forward.node = found ? f_idx + origin : 0u; result.forward.start = found ? f_start : 0u; result.forward.end = found ? f_end : 0u;
                    result.reverse.node = found ? r_idx + origin : 0u; result.reverse.start = found ? r_start : 0u; result.reverse.end = found ? r_end : 0u;
                    out[q] = result;
                }
            }
            if (lane == 0) at = q_begin + atomicAdd(const_cast<uint32_t*>(&ctrl[1]), 32u);
            at = __shfl_sync(FULL, at, 0);
        }
    }
}

// The placement step of the sort for bidirectional searches (see find_window.h).
__global__ void __launch_bounds__(BLOCK_THREADS) k_bd_place(const uint32_t* __restrict__ keys, size_t n, uint32_t* __restrict__ cursor,
                                                             uint32_t* __restrict__ perm, const uint64_t* __restrict__ offsets, uint64_t base_offset,
                                                             const uint64_t* __restrict__ first, const uint64_t* __restrict__ start,
                                                             const uint64_t* __restrict__ end, uint4* __restrict__ packed) {
    for (size_t q = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; q < n; q += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const uint64_t lo = __ldg(offsets + q), hi = __ldg(offsets + q + 1);
        const uint64_t len = hi > lo ? hi - lo : 0;
        const uint64_t f = __ldg(first + q), s = __ldg(start + q), e = __ldg(end + q);
        uint4 rec = make_uint4(0u, 0u, 0u, 0u);
        if (s <= f && f < e && e <= len && len <= 0xFFFFFFFFull) {
            const uint64_t at = (lo - base_offset) + s;
            rec = make_uint4(static_cast<uint32_t>(at), static_cast<uint32_t>(at >> 32), static_cast<uint32_t>(e - s), static_cast<uint32_t>(f - s));
        }
        const uint32_t slot = atomicAdd(cursor + __ldg(keys + q), 1u);
        perm[slot] = static_cast<uint32_t>(q);
        packed[slot] = rec;
    }
}

// The same in one pass (see k_window_place_direct): the window of path[first] is computed here, every window owns `cap`
// slots, a search that finds its window full goes to the deferred list.
__global__ void __launch_bounds__(BLOCK_THREADS) k_bd_place_direct(IndexView ix, uint32_t wshift, const uint64_t* __restrict__ nodes, size_t n,
                                                                    uint32_t cap, uint32_t* __restrict__ filled, uint32_t* __restrict__ perm,
                                                                    const uint64_t* __restrict__ offsets, uint64_t base_offset,
                                                                    const uint64_t* __restrict__ first, const uint64_t* __restrict__ start,
                                                                    const uint64_t* __restrict__ end, uint4* __restrict__ packed,
                                                                    uint32_t* __restrict__ deferred, uint32_t* __restrict__ counters) {
    for (size_t q = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; q < n; q += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const uint64_t lo = __ldg(offsets + q), hi = __ldg(offsets + q + 1);
        const uint64_t len = hi > lo ? hi - lo : 0;
        const uint64_t f = __ldg(first + q), s = __ldg(start + q), e = __ldg(end + q);
        uint4 rec = make_uint4(0u, 0u, 0u, 0u);
        uint32_t b = 0;
        if (s <= f && f < e && e <= len && len <= 0xFFFFFFFFull) {
            const uint64_t at = (lo - base_offset) + s;
            rec = make_uint4(static_cast<uint32_t>(at), static_cast<uint32_t>(at >> 32), static_cast<uint32_t>(e - s), static_cast<uint32_t>(f - s));
            uint64_t record;
            if (record_of(ix, __ldg(nodes + (lo - base_offset) + f), record)) b = static_cast<uint32_t>(record >> wshift);
        }
        const uint32_t slot = atomicAdd(filled + b, 1u);
        if (slot < cap) {
            perm[static_cast<size_t>(b) * cap + slot] = static_cast<uint32_t>(q);
            packed[static_cast<size_t>(b) * cap + slot] = rec;
        } else {
            deferred[atomicAdd(&counters[1], 1u)] = static_cast<uint32_t>(q);
        }
    }
}

// The deferred searches, by the general loop.
__global__ void __launch_bounds__(BLOCK_THREADS) k_bd_deferred(IndexView ix, const uint64_t* __restrict__ nodes, const uint64_t* __restrict__ offsets,
                                                                uint64_t base_offset, const uint64_t* __restrict__ first,
                                                                const uint64_t* __restrict__ start, const uint64_t* __restrict__ end,
                                                                const uint32_t* __restrict__ deferred, const uint32_t* __restrict__ counters,
                                                                gbwt_b200_bdstate* __restrict__ out) {
    const uint32_t n = counters[1];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t q = __ldg(deferred + i);
        const uint64_t lo = __ldg(offsets + q), hi = __ldg(offsets + q + 1);
        gbwt_b200_bdstate result;
        query_bd_search_fast<true>(ix, nodes + (lo - base_offset), hi > lo ? hi - lo : 0, __ldg(first + q), __ldg(start + q), __ldg(end + q), result);
        out[q] = result;
    }
}

// The deferred queries, by the general rounds loop (every record format, every edge case).
template <class T>
__global__ void __launch_bounds__(BLOCK_THREADS) k_find_deferred(IndexView ix, const T* __restrict__ patterns,
                                                                  const uint32_t* __restrict__ deferred, const uint32_t* __restrict__ counters,
                                                                  uint32_t k, gbwt_b200_state* __restrict__ out) {
    const uint32_t n = counters[1];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t q = __ldg(deferred + i);
        PlainRowReader<T> rd{patterns + static_cast<size_t>(q) * k};
        gbwt_b200_state result;
        query_find_extend_rounds<true>(ix, rd, k, result);
        store_state(out + q, result);
    }
}

// One-pass placement: the batch is not sorted exactly; every window owns `cap` slots (twice its share of the batch) and a
// query takes the next free slot of the window of its first node -- one pass over the first nodes, one returning atomic,
// no keys array, no scan. A query that finds its window full goes to the deferred list (a batch that crowds one part of
// the graph is then mostly answered by the general kernel, as it would be without windows).
template <class T>
__global__ void __launch_bounds__(BLOCK_THREADS) k_window_place_direct(IndexView ix, uint32_t wshift, const T* __restrict__ patterns, size_t n, size_t k,
                                                                        uint32_t cap, uint32_t* __restrict__ filled, uint32_t* __restrict__ slots,
                                                                        uint32_t* __restrict__ deferred, uint32_t* __restrict__ counters) {
    for (size_t q = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; q < n; q += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const uint64_t node = first_node(patterns, q, k);
        uint64_t rec;
        const uint32_t b = record_of(ix, node, rec) ? static_cast<uint32_t>(rec >> wshift) : 0u;
        const uint32_t at = atomicAdd(filled + b, 1u);
        if (at < cap) slots[static_cast<size_t>(b) * cap + at] = static_cast<uint32_t>(q);
        else deferred[atomicAdd(&counters[1], 1u)] = static_cast<uint32_t>(q);
    }
}

template <class T>
__global__ void __launch_bounds__(BLOCK_THREADS) k_window_keys(IndexView ix, uint32_t wshift, const T* __restrict__ patterns, size_t n,
                                                                size_t k, uint32_t* __restrict__ keys, uint32_t* __restrict__ counts) {
    for (size_t q = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; q < n; q += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const uint64_t node = first_node(patterns, q, k);
        uint64_t rec;
        const uint32_t b = record_of(ix, node, rec) ? static_cast<uint32_t>(rec >> wshift) : 0u;
        keys[q] = b;
        atomicAdd(counts + 1 + b, 1u);
    }
}

// Plain kernels for 32-bit pattern nodes: the general rounds loop, with or without the locality permutation.
template <bool RUNS>
__global__ void __launch_bounds__(BLOCK_THREADS) k_find_extend_u32(IndexView ix, const uint32_t* __restrict__ patterns,
                                                                    const uint32_t* __restrict__ perm, size_t n, size_t k,
                                                                    gbwt_b200_state* __restrict__ out) {
    GBWT_FOR_EACH_QUERY(q, n, perm) {
        gbwt_b200_state result;
        PlainRowReader<uint32_t> rd{patterns + q * k};
        query_find_extend_rounds<RUNS>(ix, rd, static_cast<uint32_t>(k), result);
        store_state(out + q, result);
    }
}

int env_or(const char* name, int fallback) {
    const char* e = std::getenv(name);
    return e ? std::atoi(e) : fallback;
}

template <class T, int THREADS, int CTAS>
int launch_window_variant(const IndexView& ix, const WindowPlan& plan, const T* patterns, const uint32_t* perm,
                          const uint32_t* bucket_end, size_t k, gbwt_b200_state* out, uint32_t* deferred, uint32_t* counters,
                          int sm_count, cudaStream_t stream) {
    auto kernel = plan.wide ? k_find_window<T, THREADS, CTAS, true> : k_find_window<T, THREADS, CTAS, false>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(plan.smem_bytes));
    if (e != cudaSuccess) return static_cast<int>(e);
    const unsigned grid = static_cast<unsigned>(std::min<uint64_t>(plan.windows, static_cast<uint64_t>(sm_count) * CTAS));
    kernel<<<grid, THREADS, plan.smem_bytes, stream>>>(ix, plan, patterns, perm, bucket_end, static_cast<uint32_t>(k), out, deferred, counters);
    return static_cast<int>(cudaGetLastError());
}

}  // namespace

bool plan_windows(const IndexView& ix, uint64_t body_units, double edge_span, bool wide, uint32_t pattern_len, WindowPlan& plan) {
    plan.wide = wide ? 1u : 0u;
    if (!ix.edges_valid || ix.records < 2 || ix.stage_body == nullptr) return false;
    // Shared memory per CTA (two CTAs of 512 threads per SM by default): 40 bytes per staged record, the pattern
    // columns, and what is left holds the bitvectors (48 bytes per 32-byte block of the global layout).
    const uint32_t threads = static_cast<uint32_t>(env_or("GBWT_B200_WINDOW_THREADS", 512));
    const uint32_t smem_kb = static_cast<uint32_t>(env_or("GBWT_B200_WINDOW_SMEM_KB", threads >= 1024 ? 224 : (threads >= 512 ? 112 : 55)));
    uint32_t window = static_cast<uint32_t>(env_or("GBWT_B200_WINDOW", threads >= 1024 ? 1024 : (threads >= 512 ? 512 : 256)));
    // the records a pattern moves away from its first one (3 records per edge on a chain of bi-allelic sites: 96 for 32 nodes)
    plan.edge_span = static_cast<float>(edge_span);
    plan.body_units = body_units;
    const uint32_t travelled = static_cast<uint32_t>(std::min(256.0, std::max(64.0, std::max<uint32_t>(pattern_len, 16) * edge_span)));
    uint32_t margin = static_cast<uint32_t>(env_or("GBWT_B200_WINDOW_MARGIN", static_cast<int>(travelled)));
    if (threads != 256 && threads != 512 && threads != 1024) return false;
    if (window < STAGE_GRANULE || (window & (window - 1)) != 0 || smem_kb > 226 || smem_kb < 16) return false;
    margin = (margin + STAGE_GRANULE - 1) / STAGE_GRANULE * STAGE_GRANULE;
    plan.wshift = 0;
    while ((1u << plan.wshift) < window) plan.wshift++;
    plan.margin = margin;
    plan.max_records = window + 2 * margin;
    plan.aux_cap = plan.wide ? plan.max_records / 4 : 0;  // wide records the window can hold (32 bytes each); the rest are deferred
    const uint64_t fixed = window_smem_bytes(plan.max_records, 0, threads, plan.aux_cap);
    const uint64_t budget = static_cast<uint64_t>(smem_kb) * 1024;
    if (fixed + 4096 > budget) return false;
    plan.body_cap = static_cast<uint32_t>((budget - fixed - 16) / 49) * 2;  // 48 bytes of entries + one kind byte per block
    // no point in reserving more than the average window needs several times over
    const uint64_t avg_units = body_units * plan.max_records / std::max<uint64_t>(1, ix.records);
    plan.body_cap = static_cast<uint32_t>(std::min<uint64_t>(plan.body_cap, std::max<uint64_t>(256, 4 * avg_units + 64))) & ~1u;
    plan.windows = static_cast<uint32_t>(((ix.records - 1) >> plan.wshift) + 1);
    plan.threads = threads;
    plan.prefetch = static_cast<uint32_t>(env_or("GBWT_B200_WINDOW_PREFETCH", 0));
    plan.fine = static_cast<uint32_t>(std::min<int>(std::max(0, env_or("GBWT_B200_WINDOW_FINE", 0)), static_cast<int>(plan.wshift)));
    plan.smem_bytes = window_smem_bytes(plan.max_records, plan.body_cap, threads, plan.aux_cap);
    return true;
}

template <class T>
void launch_window_keys(const IndexView& ix, const WindowPlan& plan, const T* patterns, size_t n, size_t k, uint32_t* keys,
                        uint32_t* counts, unsigned grid, cudaStream_t stream) {
    k_window_keys<T><<<grid, BLOCK_THREADS, 0, stream>>>(ix, plan.wshift - plan.fine, patterns, n, k, keys, counts);
}

template <class T>
void launch_window_place_direct(const IndexView& ix, const WindowPlan& plan, const T* patterns, size_t n, size_t k, uint32_t* filled,
                                uint32_t* slots, uint32_t* deferred, uint32_t* counters, unsigned grid, cudaStream_t stream) {
    k_window_place_direct<T><<<grid, BLOCK_THREADS, 0, stream>>>(ix, plan.wshift, patterns, n, k, plan.direct_cap, filled, slots, deferred, counters);
}

template <class T>
int launch_find_window(const IndexView& ix, const WindowPlan& plan, const T* patterns, const uint32_t* perm,
                       const uint32_t* bucket_end, size_t n, size_t k, gbwt_b200_state* out, uint32_t* deferred,
                       uint32_t* counters, int sm_count, cudaStream_t stream) {
    (void)n;
    if (plan.threads == 1024) return launch_window_variant<T, 1024, 1>(ix, plan, patterns, perm, bucket_end, k, out, deferred, counters, sm_count, stream);
    if (plan.threads == 256) return launch_window_variant<T, 256, 4>(ix, plan, patterns, perm, bucket_end, k, out, deferred, counters, sm_count, stream);
    return launch_window_variant<T, 512, 2>(ix, plan, patterns, perm, bucket_end, k, out, deferred, counters, sm_count, stream);
}

template <class T>
void launch_find_deferred(const IndexView& ix, const T* patterns, const uint32_t* deferred, const uint32_t* counters, size_t k,
                          gbwt_b200_state* out, unsigned grid, cudaStream_t stream) {
    k_find_deferred<T><<<grid, BLOCK_THREADS, 0, stream>>>(ix, patterns, deferred, counters, static_cast<uint32_t>(k), out);
}

// Checkpointed extraction from record windows (k_extract_window): the search plan's window with the margins dropped (the
// walks only move one way) and a tile of output rows. False: the plan does not fit this index / GPU.
bool plan_extract_windows(const WindowPlan& search, size_t sequences, WindowPlan& plan) {
    plan = search;
    // 1024 lanes per SM: two CTAs of 512 lanes (measured on config 5: 18.2 ms against 19.3 for one CTA of 1024 lanes, whose
    // window is twice as long but whose warps all restage at the same time), and smaller CTAs for smaller batches, so that the
    // lanes of a CTA are all at work (128 sequences, the share of one of 8 GPUs on config 5: 225 G LF steps/s with four CTAs
    // of 128 lanes per SM, 210 with CTAs of 256, 195 with a quarter-full CTA of 512, 168 for the one-lane walks; 256
    // sequences: 283 with half-full CTAs of 512, 277 with CTAs of 256). GBWT_B200_EXTRACT_WINDOW_THREADS overrides.
    uint32_t threads = sequences >= 192 ? 512u : 128u;
    const int knob = env_or("GBWT_B200_EXTRACT_WINDOW_THREADS", 0);
    if (knob == 128 || knob == 256 || knob == 512 || knob == 1024) threads = static_cast<uint32_t>(knob);
    plan.threads = threads;
    plan.aux_cap = 0; plan.wide = 0;
    const uint32_t tile_bytes = (plan.threads / 32u) * 32u * EXTRACT_TILE_STRIDE * 4u;
    const uint32_t budget = plan.threads >= 256 ? 224u * plan.threads : 56u * 1024u;  // (four CTAs of 128 lanes per SM: a window needs room)
    // records per window: what is left after the tile, at ~(20 + 48 * bodies per record) bytes per record
    const double per_record = RECORD_BYTES + 48.0 * 0.5 * static_cast<double>(search.body_units) / std::max<double>(1.0, static_cast<double>(search.windows) * (1u << search.wshift));
    uint32_t max_records = static_cast<uint32_t>((budget - SMEM_HEADER - tile_bytes) / (per_record * 1.15));
    max_records &= ~(STAGE_GRANULE - 1u);
    if (max_records < 4 * STAGE_GRANULE) return false;
    plan.max_records = max_records;
    plan.margin = 0;
    const uint32_t fixed = SMEM_HEADER + max_records * RECORD_BYTES + tile_bytes;
    plan.body_cap = ((budget - fixed) / 48u) * 2u;
    plan.smem_bytes = fixed + (plan.body_cap / 2u) * 48u;
    return true;
}

int launch_extract_window(const IndexView& ix, const CheckpointView& cv, const WindowPlan& plan, const uint64_t* ids, size_t m,
                          const uint64_t* out_offsets, uint64_t base_offset, uint64_t* nodes, uint64_t* lengths, uint32_t* counters, int sm_count,
                          cudaStream_t stream) {
    auto kernel = plan.threads == 1024 ? k_extract_window<1024, 1> : (plan.threads == 512 ? k_extract_window<512, 2> :
                  (plan.threads == 256 ? k_extract_window<256, 4> : k_extract_window<128, 4>));
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(plan.smem_bytes));
    if (e != cudaSuccess) return static_cast<int>(e);
    const uint64_t items = ((m + plan.threads - 1) / plan.threads) * static_cast<uint64_t>(cv.max_segments);
    const unsigned grid = static_cast<unsigned>(std::min<uint64_t>(items, static_cast<uint64_t>(sm_count) * (plan.threads >= 256 ? 1024u / plan.threads : 4u)));
    kernel<<<grid, plan.threads, plan.smem_bytes, stream>>>(ix, cv, plan, ids, m, out_offsets, base_offset, nodes, lengths, counters);
    return static_cast<int>(cudaGetLastError());
}

// Bidirectional searches from record windows (k_bd_window) + the deferred ones by the general loop. The plan is the search
// plan with a tile of 34 lines per warp; false from plan_bd_windows: it does not fit.
bool plan_bd_windows(const WindowPlan& search, WindowPlan& plan) {
    plan = search;
    if (plan.threads != 512) return false;
    plan.aux_cap = 0; plan.wide = 0;
    const uint32_t fixed = SMEM_HEADER + plan.max_records * RECORD_BYTES + (plan.threads / 32u) * BD_TILE_BYTES;
    const uint32_t budget = 112u * 1024u;
    if (fixed + 8192u > budget) return false;
    plan.body_cap = std::min<uint32_t>(search.body_cap, ((budget - fixed) / 48u) * 2u);
    plan.smem_bytes = fixed + (plan.body_cap / 2u) * 48u;
    return true;
}

void launch_bd_place(const uint32_t* keys, size_t n, uint32_t* cursor, uint32_t* perm, const uint64_t* offsets, uint64_t base_offset,
                     const uint64_t* first, const uint64_t* start, const uint64_t* end, uint4* packed, unsigned grid, cudaStream_t stream) {
    k_bd_place<<<grid, BLOCK_THREADS, 0, stream>>>(keys, n, cursor, perm, offsets, base_offset, first, start, end, packed);
}

void launch_bd_place_direct(const IndexView& ix, const WindowPlan& plan, const uint64_t* nodes, size_t n, uint32_t* filled, uint32_t* perm,
                            const uint64_t* offsets, uint64_t base_offset, const uint64_t* first, const uint64_t* start, const uint64_t* end,
                            uint4* packed, uint32_t* deferred, uint32_t* counters, unsigned grid, cudaStream_t stream) {
    k_bd_place_direct<<<grid, BLOCK_THREADS, 0, stream>>>(ix, plan.wshift, nodes, n, plan.direct_cap, filled, perm, offsets, base_offset, first, start, end,
                                                          packed, deferred, counters);
}

int launch_bd_window(const IndexView& ix, const WindowPlan& plan, const uint64_t* nodes, const uint64_t* offsets, uint64_t base_offset,
                     const uint64_t* first, const uint64_t* start, const uint64_t* end, const uint32_t* perm, const uint4* packed,
                     const uint32_t* bucket_end, gbwt_b200_bdstate* out, uint32_t* deferred, uint32_t* counters, int sm_count,
                     cudaStream_t stream) {
    auto kernel = k_bd_window<512, 2>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(plan.smem_bytes));
    if (e != cudaSuccess) return static_cast<int>(e);
    const unsigned grid = static_cast<unsigned>(std::min<uint64_t>(plan.windows, static_cast<uint64_t>(sm_count) * 2));
    kernel<<<grid, 512, plan.smem_bytes, stream>>>(ix, plan, nodes, offsets, base_offset, first, start, end, perm, packed, bucket_end, out, deferred,
                                                   counters);
    e = cudaGetLastError();
    if (e != cudaSuccess) return static_cast<int>(e);
    k_bd_deferred<<<static_cast<unsigned>(sm_count) * 4, BLOCK_THREADS, 0, stream>>>(ix, nodes, offsets, base_offset, first, start, end, deferred, counters, out);
    return static_cast<int>(cudaGetLastError());
}

void launch_find_extend_u32(const IndexView& ix, bool runs, const uint32_t* patterns, const uint32_t* perm, size_t n, size_t k,
                            gbwt_b200_state* out, unsigned grid, cudaStream_t stream) {
    if (runs) k_find_extend_u32<true><<<grid, BLOCK_THREADS, 0, stream>>>(ix, patterns, perm, n, k, out);
    else k_find_extend_u32<false><<<grid, BLOCK_THREADS, 0, stream>>>(ix, patterns, perm, n, k, out);
}

template void launch_window_place_direct<uint64_t>(const IndexView&, const WindowPlan&, const uint64_t*, size_t, size_t, uint32_t*, uint32_t*, uint32_t*,
                                                   uint32_t*, unsigned, cudaStream_t);
template void launch_window_place_direct<uint32_t>(const IndexView&, const WindowPlan&, const uint32_t*, size_t, size_t, uint32_t*, uint32_t*, uint32_t*,
                                                   uint32_t*, unsigned, cudaStream_t);
template void launch_window_keys<uint64_t>(const IndexView&, const WindowPlan&, const uint64_t*, size_t, size_t, uint32_t*, uint32_t*, unsigned, cudaStream_t);
template void launch_window_keys<uint32_t>(const IndexView&, const WindowPlan&, const uint32_t*, size_t, size_t, uint32_t*, uint32_t*, unsigned, cudaStream_t);
template int launch_find_window<uint64_t>(const IndexView&, const WindowPlan&, const uint64_t*, const uint32_t*, const uint32_t*, size_t, size_t,
                                          gbwt_b200_state*, uint32_t*, uint32_t*, int, cudaStream_t);
template int launch_find_window<uint32_t>(const IndexView&, const WindowPlan&, const uint32_t*, const uint32_t*, const uint32_t*, size_t, size_t,
                                          gbwt_b200_state*, uint32_t*, uint32_t*, int, cudaStream_t);
template void launch_find_deferred<uint64_t>(const IndexView&, const uint64_t*, const uint32_t*, const uint32_t*, size_t, gbwt_b200_state*, unsigned, cudaStream_t);
template void launch_find_deferred<uint32_t>(const IndexView&, const uint32_t*, const uint32_t*, const uint32_t*, size_t, gbwt_b200_state*, unsigned, cudaStream_t);

}  // namespace gbwt_b200
