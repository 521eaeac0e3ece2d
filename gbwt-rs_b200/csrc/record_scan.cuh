// record_scan.cuh -- per-record primitives on the device layout (layout.h): descriptor fetch, edge lookup,
// rank of a symbol at one or two positions (the core of Record::follow / bd_follow / lf, gbwt-rs
// src/bwt.rs:480-496, 595-656) and the GBWT-level steps built from them (src/gbwt.rs:213-229, 269-384).
//
// Everything here is one-lane code: one thread owns one query. The functions are __host__ __device__ so
// that tests/hostsim can run exactly this logic on the CPU against the oracle when no GPU is present;
// the product library only ever calls them from kernels (kernels.cu).
#pragma once
#include <stdint.h>

#include "../../include/gbwt_b200.h"
#include "layout.h"

namespace gbwt_b200 {

#if defined(__CUDA_ARCH__)
#define GBWT_LDG(p) __ldg(p)
#define GBWT_POPC(x) __popc(x)
#else
#define GBWT_LDG(p) (*(p))
#define GBWT_POPC(x) __builtin_popcount(x)
#endif

struct Quad { uint32_t x, y, z, w; };

// One 128-bit read-only load (LDG.E.128.CONSTANT on the device).
GBWT_HD Quad load_quad(const Unit16* p) {
    Quad q;
#if defined(__CUDA_ARCH__)
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(p));
    q.x = v.x; q.y = v.y; q.z = v.z; q.w = v.w;
#else
    q.x = p->x; q.y = p->y; q.z = p->z; q.w = p->w;
#endif
    return q;
}

// One 256-bit read-only load of a 32-byte-aligned sector (LDG.E.256.CONSTANT on sm_100a): descriptors and
// dense blocks are exactly one sector, so each costs a single load instruction and a single L1 wavefront.
GBWT_HD void load_sector(const Unit16* p, Quad& lo, Quad& hi) {
#if defined(__CUDA_ARCH__) && defined(GBWT_EXP_LD128)
    lo = load_quad(p);
    hi = load_quad(p + 1);
#elif defined(__CUDA_ARCH__) && defined(GBWT_EXP_CG)
    asm volatile("ld.global.cg.v8.u32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(lo.x), "=r"(lo.y), "=r"(lo.z), "=r"(lo.w), "=r"(hi.x), "=r"(hi.y), "=r"(hi.z), "=r"(hi.w)
                 : "l"(p));
#elif defined(__CUDA_ARCH__)
    asm volatile("ld.global.nc.v8.u32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(lo.x), "=r"(lo.y), "=r"(lo.z), "=r"(lo.w), "=r"(hi.x), "=r"(hi.y), "=r"(hi.z), "=r"(hi.w)
                 : "l"(p));
#else
    lo = load_quad(p);
    hi = load_quad(p + 1);
#endif
}

// A descriptor held in eight registers: a = {total_len, meta, w0, w1}, b = {body, body_len, w2, w3}.
struct Desc {
    Quad a, b;
    GBWT_HD uint32_t total_len() const { return a.x; }
    GBWT_HD uint32_t fmt() const { return (a.y >> 16) & 0xFF; }
    GBWT_HD bool inline_edges() const { return ((a.y >> 24) & DESC_INLINE_EDGES) != 0; }
    // 0 = the run body has no checkpoints, else log2(positions per checkpoint) + 1 (layout.h)
    GBWT_HD uint32_t checkpoints() const { return (a.y >> (24 + DESC_CKPT_SHIFT)) & DESC_CKPT_MASK; }
    GBWT_HD uint32_t sigma() const { return inline_edges() ? (a.y & 0xFFFF) : a.w; }
    GBWT_HD uint32_t edge_base() const { return a.z; }
    GBWT_HD uint32_t node0() const { return a.z; }
    GBWT_HD uint32_t offset0() const { return a.w; }
    GBWT_HD uint32_t node1() const { return b.z; }
    GBWT_HD uint32_t offset1() const { return b.w; }
    GBWT_HD uint32_t magic() const { return b.z; }
    GBWT_HD uint32_t body() const { return b.x; }
    GBWT_HD uint32_t body_len() const { return b.y; }
};

GBWT_HD Desc load_desc(const IndexView& ix, uint64_t rec) {
    Desc d;
    load_sector(reinterpret_cast<const Unit16*>(ix.desc + rec), d.a, d.b);
    return d;
}

// GBWT::node_to_record + BWT::record (src/gbwt.rs:150-152, src/bwt.rs:124-130): false = None.
GBWT_HD bool record_of(const IndexView& ix, uint64_t node, uint64_t& rec) {
    if (node < ix.offset) return false;  // Rust's wrapping subtraction lands beyond BWT::len()
    rec = node - ix.offset;
    return rec < ix.records;
}

GBWT_HD Edge edge_at(const IndexView& ix, const Desc& d, uint32_t rank) {
    Edge e;
    if (d.inline_edges()) {
        e.node = rank == 0 ? d.node0() : d.node1();
        e.offset = rank == 0 ? d.offset0() : d.offset1();
    } else {
        const Edge* p = ix.edges + d.edge_base() + rank;
        e.node = GBWT_LDG(&p->node);
        e.offset = GBWT_LDG(&p->offset);
    }
    return e;
}

// The symbols that bd_follow counts towards the reverse range (src/bwt.rs:646-648): v with
// flip(successor(v)) < flip(node). The edge list is sorted, so that set is {v < lt} plus possibly `extra`.
struct FlipSet {
    uint32_t lt, extra;
    GBWT_HD bool has(uint32_t v) const { return v < lt || v == extra; }
};

// Record::edge_to (src/bwt.rs:543-555). Returns false when `node` is not a successor.
template <bool BD>
GBWT_HD bool find_edge(const IndexView& ix, const Desc& d, uint64_t node, uint32_t& rank, uint32_t& edge_offset,
                       FlipSet& fs) {
    const uint32_t sigma = d.sigma();
    if (d.inline_edges()) {
        if (node == d.node0()) { rank = 0; edge_offset = d.offset0(); }
        else if (sigma == 2 && node == d.node1()) { rank = 1; edge_offset = d.offset1(); }
        else return false;
    } else {
        uint32_t low = 0, high = sigma;
        bool found = false;
        while (low < high) {
            uint32_t mid = low + (high - low) / 2;
            Edge e = edge_at(ix, d, mid);
            if (node < e.node) high = mid;
            else if (node == e.node) { rank = mid; edge_offset = e.offset; found = true; break; }
            else low = mid + 1;
        }
        if (!found) return false;
    }
    if (BD) {
        fs.lt = rank;
        fs.extra = NO_SYMBOL;
        if ((node & 1) != 0 && rank > 0 && edge_at(ix, d, rank - 1).node == node - 1) fs.lt = rank - 1;
        if ((node & 1) == 0 && rank + 1 < sigma && edge_at(ix, d, rank + 1).node == node + 1) fs.extra = rank + 1;
    }
    return true;
}

// |[off, off + len) ∩ [0, x)| = support::intersect(..).len() of src/bwt.rs:605-607.
GBWT_HD uint32_t covered(uint32_t x, uint32_t off, uint32_t len) {
    uint32_t t = x - (x < off ? x : off);
    return t < len ? t : len;
}

struct Ranks {
    uint32_t at_start, at_end;  // occurrences of the symbol in [0, start) and [0, end)
    uint32_t flipped;           // positions of [start, end) whose symbol is in the FlipSet (bd only)
};

// ---- FMT_DENSE2 ---------------------------------------------------------------------------------
struct DenseBlock { Quad lo, hi; };

GBWT_HD DenseBlock load_dense_block(const Unit16* body, uint32_t blk) {
    DenseBlock b;
    load_sector(body + 2 * blk, b.lo, b.hi);
    return b;
}

// Ones in the block's payload bits [0, r), r <= 192, plus the ones before the block; `bit` = payload bit r
// (0 when r == 192). One sub-count and one masked 64-bit popcount (layout.h).
GBWT_HD uint32_t dense_block_rank1(const DenseBlock& b, uint32_t r, uint32_t& bit) {
    uint32_t j = r >> 6;
    if (j > 2) j = 2;
    const uint32_t p = r - 64 * j;  // 0..64 bits of 64-bit word j
    const uint32_t w_lo = j == 0 ? b.lo.z : (j == 1 ? b.hi.x : b.hi.z);
    const uint32_t w_hi = j == 0 ? b.lo.w : (j == 1 ? b.hi.y : b.hi.w);
    const uint32_t sub = j == 0 ? 0u : (j == 1 ? (b.lo.y & 0xFFu) : ((b.lo.y >> 8) & 0xFFu));
    const uint32_t m_lo = p >= 32 ? 0xFFFFFFFFu : ((1u << p) - 1u);
    const uint32_t m_hi = p <= 32 ? 0u : (p >= 64 ? 0xFFFFFFFFu : ((1u << (p - 32)) - 1u));
    bit = p < 32 ? ((w_lo >> p) & 1u) : (p < 64 ? ((w_hi >> (p - 32)) & 1u) : 0u);
    return b.lo.x + sub + GBWT_POPC(w_lo & m_lo) + GBWT_POPC(w_hi & m_hi);
}

// Ones in [0, i) of a dense body; i <= total_len. `bit` receives the symbol at position i (0 if i == total).
GBWT_HD uint32_t dense_rank1(const Unit16* body, uint32_t blocks, uint32_t i, uint32_t& bit) {
    uint32_t blk = i / DENSE_BITS;
    if (blk >= blocks) blk = blocks - 1;
    const DenseBlock b = load_dense_block(body, blk);
    return dense_block_rank1(b, i - blk * DENSE_BITS, bit);
}

// rank1(start) and rank1(end), start <= end <= total_len; one block load when both fall in the same block.
GBWT_HD void dense_rank1_pair(const Unit16* body, uint32_t blocks, uint32_t start, uint32_t end, uint32_t& ones_s,
                              uint32_t& ones_e) {
    uint32_t blk_s = start / DENSE_BITS, blk_e = end / DENSE_BITS;
    if (blk_s >= blocks) blk_s = blocks - 1;
    if (blk_e >= blocks) blk_e = blocks - 1;
    uint32_t bit;
    const DenseBlock bs = load_dense_block(body, blk_s);
    ones_s = dense_block_rank1(bs, start - blk_s * DENSE_BITS, bit);
    if (blk_e == blk_s) {
        ones_e = dense_block_rank1(bs, end - blk_e * DENSE_BITS, bit);
    } else {
        const DenseBlock be = load_dense_block(body, blk_e);
        ones_e = dense_block_rank1(be, end - blk_e * DENSE_BITS, bit);
    }
}

// ---- run formats ------------------------------------------------------------------------------------
template <bool BD>
GBWT_HD void add_run(uint32_t value, uint32_t len, uint32_t symbol, const FlipSet& fs, uint32_t start, uint32_t end,
                     uint32_t& off, Ranks& r) {
    const uint32_t cs = covered(start, off, len), ce = covered(end, off, len);
    if (value == symbol) { r.at_start += cs; r.at_end += ce; }
    if (BD) { if (fs.has(value)) r.flipped += ce - cs; }
    off += len;
}

// Sum of the four byte products a_i * b_i (IDP4A on the device).
GBWT_HD uint32_t dot4(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
    return __dp4a(a, b, 0u);
#else
    uint32_t s = 0;
    for (int i = 0; i < 4; i++) s += ((a >> (8 * i)) & 0xFF) * ((b >> (8 * i)) & 0xFF);
    return s;
#endif
}

// 0x01 in every byte of x that is zero; exact for bytes <= 0x7F.
GBWT_HD uint32_t zero_bytes(uint32_t x) { return (((x + 0x7F7F7F7Fu) & 0x80808080u) ^ 0x80808080u) >> 7; }

// RUN8 body whose alphabet size is a power of two <= 128 (the common outdegree 2 and 4): four runs are decoded
// per 32-bit word with byte-parallel arithmetic -- lengths L = (w >> t) + 1 and values V = w & (sigma - 1) per
// byte, sums with dot products. A word that lies entirely before `start` or entirely inside [start, end) only
// adds its totals; the at most two words that straddle a boundary take the byte-by-byte path.
template <bool BD>
GBWT_HD void rank_runs8_pow2(const Unit16* body, uint32_t n, uint32_t sigma, uint32_t symbol, const FlipSet& fs,
                             uint32_t start, uint32_t end, Ranks& r) {
#if defined(__CUDA_ARCH__)
    const uint32_t t = 31u - static_cast<uint32_t>(__clz(sigma));
#else
    const uint32_t t = 31u - static_cast<uint32_t>(__builtin_clz(sigma));
#endif
    const uint32_t len_mask = (0xFFu >> t) * 0x01010101u, val_mask = (sigma - 1u) * 0x01010101u;
    const uint32_t sym_bytes = symbol * 0x01010101u;
    const uint32_t lt_add = (0x80u - (fs.lt < 128u ? fs.lt : 128u)) * 0x01010101u;
    const uint32_t extra_bytes = (fs.extra < 128u ? fs.extra : 0x7Fu) * 0x01010101u;
    const bool has_extra = fs.extra < sigma;
    uint32_t off = 0;
    for (uint32_t base = 0; base < n && off < end; base += 16) {
        const Quad q = load_quad(body + (base >> 4));
        const uint32_t words[4] = {q.x, q.y, q.z, q.w};
GBWT_UNROLL
        for (uint32_t j = 0; j < 4; j++) {
            const uint32_t first = base + 4 * j;
            if (first < n && off < end) {
                const uint32_t w = words[j];
                const uint32_t lens = ((w >> t) & len_mask) + 0x01010101u, vals = w & val_mask;
                const uint32_t total = dot4(lens, 0x01010101u);
                const bool whole = n - first >= 4;
                if (whole && (off + total <= start || (off >= start && off + total <= end))) {
                    const uint32_t count = dot4(lens, zero_bytes(vals ^ sym_bytes));
                    r.at_end += count;
                    if (off + total <= start) {
                        r.at_start += count;
                    } else if (BD) {
                        uint32_t in_set = (((vals + lt_add) & 0x80808080u) ^ 0x80808080u) >> 7;
                        if (has_extra) in_set |= zero_bytes(vals ^ extra_bytes);
                        r.flipped += dot4(lens, in_set);
                    }
                    off += total;
                } else {
                    const uint32_t nb = n - first < 4 ? n - first : 4;
                    for (uint32_t b = 0; b < nb; b++) {
                        const uint32_t byte = (w >> (8 * b)) & 0xFF;
                        add_run<BD>(byte & (sigma - 1u), (byte >> t) + 1u, symbol, fs, start, end, off, r);
                    }
                }
            }
        }
    }
}

// ---- FMT_DENSE4 (layout.h): two bits per position ---------------------------------------------------------
// Occurrences of `symbol` among the first r (<= 16) two-bit fields of w.
GBWT_HD uint32_t dense4_matches(uint32_t w, uint32_t symbol, uint32_t r) {
    const uint32_t y = w ^ (symbol * 0x55555555u);
    uint32_t t = ~(y | (y >> 1)) & 0x55555555u;
    t = r >= 16 ? t : (t & ((1u << (2 * r)) - 1u));
    return GBWT_POPC(t);
}

// Occurrences of `symbol` in [0, i) of a DENSE4 body, i <= total_len.
GBWT_HD uint32_t dense4_rank(const Unit16* body, uint32_t blocks, uint32_t symbol, uint32_t i) {
    uint32_t blk = i / DENSE4_POSITIONS;
    if (blk >= blocks) blk = blocks - 1;
    const uint32_t r = i - blk * DENSE4_POSITIONS;  // 0 .. 64
    const Quad head = load_quad(body + 2 * blk), codes = load_quad(body + 2 * blk + 1);
    const uint32_t c1 = head.x, c2 = head.y & ~DENSE4_TAG, c3 = head.z;
    uint32_t count = symbol == 0 ? blk * DENSE4_POSITIONS - c1 - c2 - c3 : (symbol == 1 ? c1 : (symbol == 2 ? c2 : c3));
    const uint32_t w[4] = {codes.x, codes.y, codes.z, codes.w};
GBWT_UNROLL
    for (uint32_t j = 0; j < 4; j++) {
        if (r > 16 * j) count += dense4_matches(w[j], symbol, r - 16 * j);
    }
    return count;
}

GBWT_HD uint32_t dense4_symbol(const Unit16* body, uint32_t i) {
    const uint32_t blk = i / DENSE4_POSITIONS, at = i % DENSE4_POSITIONS;
    const Quad codes = load_quad(body + 2 * blk + 1);
    const uint32_t w = (at >> 4) == 0 ? codes.x : ((at >> 4) == 1 ? codes.y : ((at >> 4) == 2 ? codes.z : codes.w));
    return (w >> (2 * (at & 15u))) & 3u;
}

// ---- checkpointed run bodies (layout.h) ---------------------------------------------------------------
// A long run body carries a table of checkpoints behind its runs: one every P = 2^shift positions, runs split there
// at load time so that a run starts exactly at the checkpoint. Entry j - 1 (position j P) holds, in `stride` words,
// C_v = the number of positions before j P with a symbol <= v for v = 0 .. sigma - 2 and, in word sigma - 1, the
// index of the run that starts at j P. A rank is then one table entry plus a scan of at most one interval's runs
// instead of a scan from the start of the body (the reference scans from the start: src/bwt.rs:603-613 over
// RLEIter, src/support.rs:1413-1430).
struct RunCheckpoint {
    uint32_t run, offset;   // where the scan starts: run index and the position that run starts at
    uint32_t count, flip;   // occurrences of the symbol / of the FlipSet symbols before `offset`
};

GBWT_HD uint32_t run_units(uint32_t fmt, uint32_t n) {
    return fmt == FMT_RUN8 ? (n + 15u) >> 4 : (fmt == FMT_RUN32 ? (n + 3u) >> 2 : (n + 1u) >> 1);
}

template <bool BD>
GBWT_HD RunCheckpoint load_checkpoint(const Unit16* body, const Desc& d, uint32_t symbol, const FlipSet& fs, uint32_t pos) {
    RunCheckpoint c;
    c.run = 0; c.offset = 0; c.count = 0; c.flip = 0;
    const uint32_t shift = d.checkpoints() - 1u;
    const uint32_t last = (d.total_len() - 1u) >> shift;  // checkpoints 1 .. last exist
    uint32_t j = pos >> shift;
    if (j > last) j = last;
    if (j == 0) return c;
    const uint32_t sigma = d.sigma(), stride = (sigma + 3u) & ~3u;
    const uint32_t* table = reinterpret_cast<const uint32_t*>(body + ((run_units(d.fmt(), d.body_len()) + 1u) & ~1u)) + static_cast<size_t>(j - 1u) * stride;
    c.offset = j << shift;
    c.run = GBWT_LDG(table + sigma - 1u);
    // C_{sigma - 1} is the position itself
    const uint32_t upto = symbol + 1u < sigma ? GBWT_LDG(table + symbol) : c.offset;
    const uint32_t below = symbol > 0 ? GBWT_LDG(table + symbol - 1u) : 0u;
    c.count = upto - below;
    if (BD) {
        if (fs.lt > 0) c.flip = fs.lt < sigma ? GBWT_LDG(table + fs.lt - 1u) : c.offset;
        if (fs.extra < sigma) {
            const uint32_t e_upto = fs.extra + 1u < sigma ? GBWT_LDG(table + fs.extra) : c.offset;
            c.flip += e_upto - (fs.extra > 0 ? GBWT_LDG(table + fs.extra - 1u) : 0u);
        }
    }
    return c;
}

// Adds to c.count / c.flip the occurrences in [c.offset, pos), scanning from run c.run.
template <bool BD>
GBWT_HD void scan_runs_to(const Unit16* body, const Desc& d, uint32_t symbol, const FlipSet& fs, uint32_t pos, RunCheckpoint& c) {
    const uint32_t n = d.body_len(), fmt = d.fmt();
    uint32_t off = c.offset;
    if (fmt == FMT_RUN8) {
        const uint32_t sigma = d.sigma();
        const uint32_t magic = d.inline_edges() ? 32769u : d.magic();  // inline edges + runs => sigma == 2
        for (uint32_t base = c.run & ~15u; base < n && off < pos; base += 16) {
            const Quad q = load_quad(body + (base >> 4));
            const uint32_t words[4] = {q.x, q.y, q.z, q.w};
GBWT_UNROLL
            for (uint32_t j = 0; j < 16; j++) {
                if (base + j >= c.run && base + j < n && off < pos) {
                    const uint32_t b = (words[j >> 2] >> (8 * (j & 3))) & 0xFF;
                    const uint32_t quot = (b * magic) >> 16, value = b - quot * sigma;
                    const uint32_t part = pos - off < quot + 1 ? pos - off : quot + 1;
                    if (value == symbol) c.count += part;
                    if (BD) { if (fs.has(value)) c.flip += part; }
                    off += quot + 1;
                }
            }
        }
    } else if (fmt == FMT_RUN32) {
        for (uint32_t base = c.run & ~3u; base < n && off < pos; base += 4) {
            const Quad q = load_quad(body + (base >> 2));
            const uint32_t words[4] = {q.x, q.y, q.z, q.w};
GBWT_UNROLL
            for (uint32_t j = 0; j < 4; j++) {
                if (base + j >= c.run && base + j < n && off < pos) {
                    const uint32_t value = words[j] & 0xFF, len = (words[j] >> 8) + 1;
                    const uint32_t part = pos - off < len ? pos - off : len;
                    if (value == symbol) c.count += part;
                    if (BD) { if (fs.has(value)) c.flip += part; }
                    off += len;
                }
            }
        }
    } else {  // FMT_RUN64
        for (uint32_t run = c.run; run < n && off < pos; run++) {
            const Quad q = load_quad(body + (run >> 1));
            const uint32_t value = (run & 1) ? q.z : q.x, len = (run & 1) ? q.w : q.y;
            const uint32_t part = pos - off < len ? pos - off : len;
            if (value == symbol) c.count += part;
            if (BD) { if (fs.has(value)) c.flip += part; }
            off += len;
        }
    }
}

// rank(start), rank(end) and the flipped count of [start, end) on a checkpointed body.
template <bool BD>
GBWT_HD void rank_runs_checkpointed(const IndexView& ix, const Desc& d, uint32_t symbol, const FlipSet& fs, uint32_t start,
                                    uint32_t end, Ranks& r) {
    const Unit16* body = ix.bodies + d.body();
    RunCheckpoint cs = load_checkpoint<BD>(body, d, symbol, fs, start);
    scan_runs_to<BD>(body, d, symbol, fs, start, cs);
    r.at_start = r.at_end = cs.count;
    if (end != start) {
        RunCheckpoint ce = load_checkpoint<BD>(body, d, symbol, fs, end);
        scan_runs_to<BD>(body, d, symbol, fs, end, ce);
        r.at_end = ce.count;
        if (BD) r.flipped = ce.flip - cs.flip;
    }
}

// Scans the runs of a RUN8 / RUN32 / RUN64 body up to `end` (the reference's early exit, src/bwt.rs:610-612).
// Not inlined on the device: the scan loops would otherwise set the register budget (and the occupancy) of
// the kernels whose common case is the register-light dense / single-edge step.
template <bool BD>
GBWT_HD void rank_runs_inline(const IndexView& ix, const Desc& d, uint32_t symbol, const FlipSet& fs, uint32_t start,
                              uint32_t end, Ranks& r) {
    if (d.fmt() == FMT_DENSE4) {
        const Unit16* body4 = ix.bodies + d.body();
        const uint32_t blocks = d.body_len();
        r.at_start = dense4_rank(body4, blocks, symbol, start);
        r.at_end = end != start ? dense4_rank(body4, blocks, symbol, end) : r.at_start;
        if (BD && end != start) {
            for (uint32_t v = 0; v < d.sigma(); v++)
                if (fs.has(v)) r.flipped += dense4_rank(body4, blocks, v, end) - dense4_rank(body4, blocks, v, start);
        }
        return;
    }
    if (d.checkpoints() != 0) { rank_runs_checkpointed<BD>(ix, d, symbol, fs, start, end, r); return; }
    const Unit16* body = ix.bodies + d.body();
    const uint32_t n = d.body_len();
    const uint32_t fmt = d.fmt();
    uint32_t off = 0;
    if (fmt == FMT_RUN8 && d.sigma() <= 128 && (d.sigma() & (d.sigma() - 1)) == 0) {
        rank_runs8_pow2<BD>(body, n, d.sigma(), symbol, fs, start, end, r);
    } else if (fmt == FMT_RUN8) {
        const uint32_t sigma = d.sigma();
        const uint32_t magic = d.inline_edges() ? 32769u : d.magic();  // inline edges + runs => sigma == 2
        for (uint32_t base = 0; base < n && off < end; base += 16) {
            const Quad q = load_quad(body + (base >> 4));
            const uint32_t words[4] = {q.x, q.y, q.z, q.w};
            const uint32_t nb = n - base < 16 ? n - base : 16;
GBWT_UNROLL
            for (uint32_t j = 0; j < 16; j++) {
                if (j < nb) {
                    const uint32_t b = (words[j >> 2] >> (8 * (j & 3))) & 0xFF;
                    const uint32_t quot = (b * magic) >> 16;
                    add_run<BD>(b - quot * sigma, quot + 1, symbol, fs, start, end, off, r);
                }
            }
        }
    } else if (fmt == FMT_RUN32) {
        for (uint32_t base = 0; base < n && off < end; base += 4) {
            const Quad q = load_quad(body + (base >> 2));
            const uint32_t words[4] = {q.x, q.y, q.z, q.w};
            const uint32_t nb = n - base < 4 ? n - base : 4;
GBWT_UNROLL
            for (uint32_t j = 0; j < 4; j++) {
                if (j < nb) add_run<BD>(words[j] & 0xFF, (words[j] >> 8) + 1, symbol, fs, start, end, off, r);
            }
        }
    } else {  // FMT_RUN64
        for (uint32_t base = 0; base < n && off < end; base += 2) {
            const Quad q = load_quad(body + (base >> 1));
            add_run<BD>(q.x, q.y, symbol, fs, start, end, off, r);
            if (base + 1 < n) add_run<BD>(q.z, q.w, symbol, fs, start, end, off, r);
        }
    }
}

template <bool BD>
GBWT_HD_NOINLINE void rank_runs(const IndexView& ix, const Desc& d, uint32_t symbol, const FlipSet& fs, uint32_t start,
                                uint32_t end, Ranks& r) {
    rank_runs_inline<BD>(ix, d, symbol, fs, start, end, r);
}

// Symbol at position i (< total_len) of a run body: the first pass of Record::lf (src/bwt.rs:483-484).
GBWT_HD uint32_t symbol_at_runs(const IndexView& ix, const Desc& d, uint32_t i) {
    const Unit16* body = ix.bodies + d.body();
    const uint32_t n = d.body_len();
    const uint32_t fmt = d.fmt();
    uint32_t off = 0, symbol = NO_SYMBOL, first = 0;
    if (fmt == FMT_DENSE4) return i < d.total_len() ? dense4_symbol(body, i) : NO_SYMBOL;
    if (d.checkpoints() != 0 && i < d.total_len()) {
        // start at the checkpoint before position i (word sigma - 1 of its entry: the run that starts there)
        const uint32_t shift = d.checkpoints() - 1u, j = i >> shift;
        if (j > 0) {
            const uint32_t sigma = d.sigma(), stride = (sigma + 3u) & ~3u;
            const uint32_t* table = reinterpret_cast<const uint32_t*>(body + ((run_units(fmt, n) + 1u) & ~1u)) + static_cast<size_t>(j - 1u) * stride;
            first = GBWT_LDG(table + sigma - 1u);
            off = j << shift;
        }
    }
    if (fmt == FMT_RUN8) {
        const uint32_t sigma = d.sigma();
        const uint32_t magic = d.inline_edges() ? 32769u : d.magic();  // inline edges + runs => sigma == 2
        for (uint32_t base = first & ~15u; base < n && symbol == NO_SYMBOL; base += 16) {
            const Quad q = load_quad(body + (base >> 4));
            const uint32_t words[4] = {q.x, q.y, q.z, q.w};
            const uint32_t nb = n - base < 16 ? n - base : 16;
GBWT_UNROLL
            for (uint32_t j = 0; j < 16; j++) {
                if (j < nb && base + j >= first) {
                    const uint32_t b = (words[j >> 2] >> (8 * (j & 3))) & 0xFF;
                    const uint32_t quot = (b * magic) >> 16;
                    if (symbol == NO_SYMBOL && i - off < quot + 1) symbol = b - quot * sigma;
                    off += quot + 1;
                }
            }
        }
    } else if (fmt == FMT_RUN32) {
        for (uint32_t base = first & ~3u; base < n && symbol == NO_SYMBOL; base += 4) {
            const Quad q = load_quad(body + (base >> 2));
            const uint32_t words[4] = {q.x, q.y, q.z, q.w};
            const uint32_t nb = n - base < 4 ? n - base : 4;
GBWT_UNROLL
            for (uint32_t j = 0; j < 4; j++) {
                if (j < nb && base + j >= first) {
                    const uint32_t len = (words[j] >> 8) + 1;
                    if (symbol == NO_SYMBOL && i - off < len) symbol = words[j] & 0xFF;
                    off += len;
                }
            }
        }
    } else {
        for (uint32_t run = first; run < n && symbol == NO_SYMBOL; run++) {
            const Quad q = load_quad(body + (run >> 1));
            const uint32_t value = (run & 1) ? q.z : q.x, len = (run & 1) ? q.w : q.y;
            if (i - off < len) symbol = value;
            off += len;
        }
    }
    return symbol;
}

// rank_symbol(start), rank_symbol(end) and, for BD, the flipped count, for any body format.
// `start` <= `end`; both are clamped to the record length (ranks saturate there).
// RUNS = false compiles the run-length formats out: the host picks that instantiation for indexes that hold
// none (IndexView::run_records == 0), so the scan loops do not set the register budget of the dense path.
// INLINE_SCAN: the run scan is inlined into the caller (for callers that are themselves out of line).
template <bool BD, bool RUNS = true, bool INLINE_SCAN = false>
GBWT_HD Ranks rank_pair(const IndexView& ix, const Desc& d, uint32_t symbol, const FlipSet& fs, uint32_t start,
                        uint32_t end) {
    Ranks r;
    r.at_start = r.at_end = r.flipped = 0;
    const uint32_t total = d.total_len();
    if (start > total) start = total;
    if (end > total) end = total;
    const uint32_t fmt = d.fmt();
    if (fmt == FMT_SINGLE) {
        r.at_start = start; r.at_end = end;
        if (BD) r.flipped = fs.has(0) ? end - start : 0;
    } else if (fmt == FMT_DENSE2) {
        uint32_t ones_s, ones_e;
        dense_rank1_pair(ix.bodies + d.body(), d.body_len(), start, end, ones_s, ones_e);
        r.at_start = symbol ? ones_s : start - ones_s;
        r.at_end = symbol ? ones_e : end - ones_e;
        if (BD) {
            const uint32_t ones = ones_e - ones_s, zeros = (end - start) - ones;
            r.flipped = (fs.has(0) ? zeros : 0) + (fs.has(1) ? ones : 0);
        }
    } else if (RUNS) {
        if (INLINE_SCAN) rank_runs_inline<BD>(ix, d, symbol, fs, start, end, r);
        else rank_runs<BD>(ix, d, symbol, fs, start, end, r);
    }
    return r;
}

// ---- GBWT-level steps (on the ABI value types of include/gbwt_b200.h) ---------------------------------

GBWT_HD void set_none(gbwt_b200_state& s) { s.node = 0; s.start = 0; s.end = 0; }
GBWT_HD void set_none(gbwt_b200_bdstate& s) { set_none(s.forward); set_none(s.reverse); }
GBWT_HD void set_none(gbwt_b200_pos& p) { p.node = 0; p.offset = 0; }

// GBWT::find, src/gbwt.rs:269-281. The length comes from the descriptor instead of Record::len()'s scan.
GBWT_HD bool gbwt_find(const IndexView& ix, uint64_t node, gbwt_b200_state& out) {
    set_none(out);
    uint64_t rec;
    if (node < ix.offset + 1 || !record_of(ix, node, rec)) return false;
    const Desc d = load_desc(ix, rec);
    if (d.fmt() == FMT_EMPTY || d.total_len() == 0) return false;
    out.node = node; out.end = d.total_len();
    return true;
}

// Record::follow / bd_follow on the record of `from` (src/bwt.rs:595-656) as used by GBWT::extend and
// bd_internal (src/gbwt.rs:292-304, 370-384). `flipped` is bd_follow's second return value.
template <bool BD>
GBWT_HD bool gbwt_follow(const IndexView& ix, uint64_t from, uint64_t start, uint64_t end, uint64_t node,
                         gbwt_b200_state& out, uint64_t& flipped) {
    set_none(out);
    flipped = 0;
    uint64_t rec;
    if (node < ix.offset + 1 || start >= end || !record_of(ix, from, rec)) return false;
    const Desc d = load_desc(ix, rec);
    if (d.fmt() == FMT_EMPTY) return false;
    uint32_t rank = 0, edge_offset = 0;
    FlipSet fs;
    fs.lt = 0; fs.extra = NO_SYMBOL;
    if (!find_edge<BD>(ix, d, node, rank, edge_offset, fs)) return false;
    const uint32_t total = d.total_len();
    const uint32_t s = start > total ? total : static_cast<uint32_t>(start);
    const uint32_t e = end > total ? total : static_cast<uint32_t>(end);
    const Ranks r = rank_pair<BD>(ix, d, rank, fs, s, e);
    if (r.at_start >= r.at_end) return false;
    out.node = node;
    out.start = static_cast<uint64_t>(edge_offset) + r.at_start;
    out.end = static_cast<uint64_t>(edge_offset) + r.at_end;
    flipped = r.flipped;
    return true;
}

// GBWT::extend, src/gbwt.rs:292-304.
GBWT_HD bool gbwt_extend(const IndexView& ix, const gbwt_b200_state& state, uint64_t node, gbwt_b200_state& out) {
    uint64_t flipped;
    return gbwt_follow<false>(ix, state.node, state.start, state.end, node, out, flipped);
}

// GBWT::bd_find, src/gbwt.rs:311-324.
GBWT_HD bool gbwt_bd_find(const IndexView& ix, uint64_t node, gbwt_b200_bdstate& out) {
    set_none(out);
    gbwt_b200_state st;
    if (!gbwt_find(ix, node, st)) return false;
    out.forward = st;
    out.reverse.node = node ^ 1; out.reverse.start = st.start; out.reverse.end = st.end;
    return true;
}

// GBWT::extend_forward + bd_internal, src/gbwt.rs:339-347, 370-384. `out` may alias `state`.
GBWT_HD bool gbwt_extend_forward(const IndexView& ix, const gbwt_b200_bdstate& state, uint64_t node,
                                 gbwt_b200_bdstate& out) {
    const gbwt_b200_state reverse = state.reverse;
    gbwt_b200_state fwd;
    uint64_t flipped;
    if (!gbwt_follow<true>(ix, state.forward.node, state.forward.start, state.forward.end, node, fwd, flipped)) {
        set_none(out);
        return false;
    }
    out.forward = fwd;
    out.reverse.node = reverse.node;
    out.reverse.start = reverse.start + flipped;
    out.reverse.end = out.reverse.start + (fwd.end - fwd.start);
    return true;
}

// GBWT::extend_backward, src/gbwt.rs:362-367: flip, extend forward with the flipped node, flip back.
GBWT_HD bool gbwt_extend_backward(const IndexView& ix, const gbwt_b200_bdstate& state, uint64_t node,
                                  gbwt_b200_bdstate& out) {
    gbwt_b200_bdstate flipped_state;
    flipped_state.forward = state.reverse;
    flipped_state.reverse = state.forward;
    gbwt_b200_bdstate res;
    if (!gbwt_extend_forward(ix, flipped_state, node ^ 1, res)) { set_none(out); return false; }
    out.forward = res.reverse;
    out.reverse = res.forward;
    return true;
}

// Record::lf at `offset` of the record whose descriptor is `d` (src/bwt.rs:480-496). False = None.
GBWT_HD bool lf_in_record(const IndexView& ix, const Desc& d, uint64_t offset, gbwt_b200_pos& out) {
    set_none(out);
    const uint32_t fmt = d.fmt();
    if (fmt == FMT_EMPTY || offset >= d.total_len()) return false;
    const uint32_t i = static_cast<uint32_t>(offset);
    uint32_t symbol, rank_i;
    if (fmt == FMT_SINGLE) {
        symbol = 0; rank_i = i;
    } else if (fmt == FMT_DENSE2) {
        const uint32_t ones = dense_rank1(ix.bodies + d.body(), d.body_len(), i, symbol);
        rank_i = symbol ? ones : i - ones;
    } else {
        symbol = symbol_at_runs(ix, d, i);
        if (symbol == NO_SYMBOL) return false;
        FlipSet fs;
        fs.lt = 0; fs.extra = NO_SYMBOL;
        Ranks r;
        r.at_start = r.at_end = r.flipped = 0;
        rank_runs<false>(ix, d, symbol, fs, i, i, r);
        rank_i = r.at_start;
    }
    const Edge e = edge_at(ix, d, symbol);
    if (e.node == 0) return false;  // successor is the endmarker: the sequence ends (src/bwt.rs:485-486)
    out.node = e.node; out.offset = static_cast<uint64_t>(e.offset) + rank_i;
    return true;
}

// GBWT::forward + Record::lf, src/gbwt.rs:222-229, src/bwt.rs:480-496. False = None.
GBWT_HD bool gbwt_forward(const IndexView& ix, const gbwt_b200_pos& pos, gbwt_b200_pos& out) {
    set_none(out);
    uint64_t rec;
    if (pos.node < ix.offset + 1 || !record_of(ix, pos.node, rec)) return false;
    return lf_in_record(ix, load_desc(ix, rec), pos.offset, out);
}

// GBWT::start, src/gbwt.rs:213-219.
GBWT_HD bool gbwt_start(const IndexView& ix, uint64_t id, gbwt_b200_pos& out) {
    set_none(out);
    if (id >= ix.endmarker_len) return false;
    const uint32_t node = GBWT_LDG(&ix.endmarker[id].node);
    if (node == 0) return false;
    out.node = node; out.offset = GBWT_LDG(&ix.endmarker[id].offset);
    return true;
}

// ---- backward navigation (src/gbwt.rs:236-250, src/bwt.rs:502-584) ------------------------------------

// Number of occurrences of `symbol` in the whole record.
GBWT_HD uint32_t count_symbol(const IndexView& ix, const Desc& d, uint32_t symbol) {
    FlipSet fs;
    fs.lt = 0; fs.extra = NO_SYMBOL;
    const uint32_t total = d.total_len();
    return rank_pair<false>(ix, d, symbol, fs, total, total).at_end;
}

// Position of the k-th (0-based) occurrence of `symbol`; false if there are not that many.
GBWT_HD bool select_symbol(const IndexView& ix, const Desc& d, uint32_t symbol, uint32_t k, uint32_t& pos) {
    const uint32_t fmt = d.fmt();
    const uint32_t total = d.total_len();
    if (fmt == FMT_SINGLE) { pos = k; return k < total; }
    const Unit16* body = ix.bodies + d.body();
    const uint32_t n = d.body_len();
    if (fmt == FMT_DENSE2) {
        // last block whose prefix count of `symbol` is <= k
        uint32_t lo = 0, hi = n;
        while (hi - lo > 1) {
            const uint32_t mid = lo + (hi - lo) / 2;
            const uint32_t ones = load_quad(body + 2 * mid).x;
            const uint32_t before = symbol ? ones : mid * DENSE_BITS - ones;
            if (before <= k) lo = mid; else hi = mid;
        }
        const Quad a = load_quad(body + 2 * lo), b = load_quad(body + 2 * lo + 1);
        const uint32_t w[6] = {a.z, a.w, b.x, b.y, b.z, b.w};
        uint32_t need = k - (symbol ? a.x : lo * DENSE_BITS - a.x);
        for (uint32_t j = 0; j < 6; j++) {
            uint32_t bits = symbol ? w[j] : ~w[j];
            const uint32_t c = GBWT_POPC(bits);
            if (need < c) {
                for (uint32_t t = 0; t < need; t++) bits &= bits - 1;
                uint32_t bit = 0;
                while (!((bits >> bit) & 1u)) bit++;
                pos = lo * DENSE_BITS + 32 * j + bit;
                return pos < total;
            }
            need -= c;
        }
        return false;
    }
    if (fmt == FMT_DENSE4) {
        // last block whose prefix count of `symbol` is <= k, then position by position
        uint32_t lo = 0, hi = n;
        while (hi - lo > 1) {
            const uint32_t mid = lo + (hi - lo) / 2;
            if (dense4_rank(body, n, symbol, mid * DENSE4_POSITIONS) <= k) lo = mid; else hi = mid;
        }
        uint32_t seen4 = dense4_rank(body, n, symbol, lo * DENSE4_POSITIONS);
        for (uint32_t p = lo * DENSE4_POSITIONS; p < total && p < (lo + 1) * DENSE4_POSITIONS; p++) {
            if (dense4_symbol(body, p) == symbol) {
                if (seen4 == k) { pos = p; return true; }
                seen4++;
            }
        }
        return false;
    }
    uint32_t off = 0, seen = 0;
    if (fmt == FMT_RUN8) {
        const uint32_t sigma = d.sigma();
        const uint32_t magic = d.inline_edges() ? 32769u : d.magic();
        for (uint32_t base = 0; base < n; base += 16) {
            const Quad q = load_quad(body + (base >> 4));
            const uint32_t words[4] = {q.x, q.y, q.z, q.w};
            const uint32_t nb = n - base < 16 ? n - base : 16;
            for (uint32_t j = 0; j < nb; j++) {
                const uint32_t b = (words[j >> 2] >> (8 * (j & 3))) & 0xFF;
                const uint32_t quot = (b * magic) >> 16;
                if (b - quot * sigma == symbol) {
                    if (k - seen < quot + 1) { pos = off + (k - seen); return true; }
                    seen += quot + 1;
                }
                off += quot + 1;
            }
        }
    } else if (fmt == FMT_RUN32) {
        for (uint32_t base = 0; base < n; base += 4) {
            const Quad q = load_quad(body + (base >> 2));
            const uint32_t words[4] = {q.x, q.y, q.z, q.w};
            const uint32_t nb = n - base < 4 ? n - base : 4;
            for (uint32_t j = 0; j < nb; j++) {
                const uint32_t len = (words[j] >> 8) + 1;
                if ((words[j] & 0xFF) == symbol) {
                    if (k - seen < len) { pos = off + (k - seen); return true; }
                    seen += len;
                }
                off += len;
            }
        }
    } else {
        for (uint32_t base = 0; base < n; base++) {
            const Quad q = load_quad(body + (base >> 1));
            const uint32_t value = (base & 1) ? q.z : q.x, len = (base & 1) ? q.w : q.y;
            if (value == symbol) {
                if (k - seen < len) { pos = off + (k - seen); return true; }
                seen += len;
            }
            off += len;
        }
    }
    return false;
}

// Record::predecessor_at (src/bwt.rs:502-540) on the record of flip(node): walks the successors in the order
// of the flipped nodes (adjacent edges to the two orientations of one node swap places, :521-525).
GBWT_HD bool predecessor_at(const IndexView& ix, const Desc& d, uint32_t i, uint64_t& predecessor) {
    const uint32_t sigma = d.sigma();
    uint32_t offset = 0;
    for (uint32_t j = 0; j < sigma;) {
        const bool pair = j + 1 < sigma && edge_at(ix, d, j).node / 2 == edge_at(ix, d, j + 1).node / 2;
        const uint32_t order[2] = {pair ? j + 1 : j, j};
        const uint32_t steps = pair ? 2 : 1;
        for (uint32_t t = 0; t < steps; t++) {
            const uint32_t v = order[t];
            offset += count_symbol(ix, d, v);
            if (offset > i) {
                const uint32_t node = edge_at(ix, d, v).node;
                if (node == 0) return false;
                predecessor = node ^ 1;
                return true;
            }
        }
        j += steps;
    }
    return false;
}

// GBWT::backward, src/gbwt.rs:236-250 (the caller has checked is_bidirectional()).
GBWT_HD bool gbwt_backward(const IndexView& ix, const gbwt_b200_pos& pos, gbwt_b200_pos& out) {
    const uint64_t node = pos.node, offset = pos.offset;
    set_none(out);
    uint64_t rec;
    if (node <= ix.offset + 1 || !record_of(ix, node ^ 1, rec)) return false;
    const Desc rev = load_desc(ix, rec);
    if (rev.fmt() == FMT_EMPTY || offset >= rev.total_len()) return false;
    uint64_t predecessor;
    if (!predecessor_at(ix, rev, static_cast<uint32_t>(offset), predecessor)) return false;
    if (!record_of(ix, predecessor, rec)) return false;
    const Desc pred = load_desc(ix, rec);
    if (pred.fmt() == FMT_EMPTY) return false;
    // Record::offset_to, src/bwt.rs:558-584
    uint32_t rank = 0, edge_offset = 0;
    FlipSet fs;
    if (!find_edge<false>(ix, pred, node, rank, edge_offset, fs)) return false;
    if (edge_offset > offset) return false;
    const uint64_t k = offset - edge_offset;
    uint32_t where;
    if (k > 0xFFFFFFFFull || !select_symbol(ix, pred, rank, static_cast<uint32_t>(k), where)) return false;
    out.node = predecessor; out.offset = where;
    return true;
}

// ---- all extensions of a state (GBZ::follow_forward / follow_backward, src/gbz.rs:519-544, 1223-1231) --------

// Every non-empty single-node extension of `state` in edge order (EdgeIter, src/gbz.rs:835-861: an edge to the
// endmarker is skipped), each computed like GBWT::bd_internal (src/gbwt.rs:370-384); backward = the same on the
// flipped state with the results flipped back. Writes at most `cap` states and returns their number, or
// UINT64_MAX where the reference returns None (GBZ::has_node fails or the record does not exist).
GBWT_HD uint64_t gbwt_follow_all(const IndexView& ix, const gbwt_b200_bdstate& state, bool backward,
                                 gbwt_b200_bdstate* out, uint64_t cap) {
    const gbwt_b200_state fwd = backward ? state.reverse : state.forward;
    const gbwt_b200_state rev = backward ? state.forward : state.reverse;
    // GBZ::has_node (src/gbz.rs:286-289): the forward orientation is in the alphabet and has a record
    const uint64_t forward_node = fwd.node & ~1ull;
    uint64_t rec;
    if (!(forward_node > ix.offset && forward_node < ix.alphabet_size) || !record_of(ix, forward_node, rec)) return ~0ull;
    if (load_desc(ix, rec).fmt() == FMT_EMPTY) return ~0ull;
    if (!record_of(ix, fwd.node, rec)) return ~0ull;
    const Desc d = load_desc(ix, rec);
    if (d.fmt() == FMT_EMPTY) return ~0ull;
    const uint32_t sigma = d.sigma();
    const uint32_t total = d.total_len();
    uint64_t n = 0;
    if (fwd.start >= fwd.end) return 0;  // bd_follow: an empty range has no extensions
    const uint32_t s = fwd.start > total ? total : static_cast<uint32_t>(fwd.start);
    const uint32_t e = fwd.end > total ? total : static_cast<uint32_t>(fwd.end);
    for (uint32_t rank = 0; rank < sigma; rank++) {
        const Edge edge = edge_at(ix, d, rank);
        if (edge.node == 0) continue;  // EdgeIter::new skips the endmarker (always rank 0); bd_follow rejects it too
        FlipSet fs;
        fs.lt = rank; fs.extra = NO_SYMBOL;
        if ((edge.node & 1) != 0 && rank > 0 && edge_at(ix, d, rank - 1).node == edge.node - 1) fs.lt = rank - 1;
        if ((edge.node & 1) == 0 && rank + 1 < sigma && edge_at(ix, d, rank + 1).node == edge.node + 1) fs.extra = rank + 1;
        const Ranks r = rank_pair<true>(ix, d, rank, fs, s, e);
        if (r.at_start >= r.at_end) continue;
        gbwt_b200_bdstate next;
        next.forward.node = edge.node;
        next.forward.start = static_cast<uint64_t>(edge.offset) + r.at_start;
        next.forward.end = static_cast<uint64_t>(edge.offset) + r.at_end;
        next.reverse.node = rev.node;
        next.reverse.start = rev.start + r.flipped;
        next.reverse.end = next.reverse.start + (r.at_end - r.at_start);
        if (backward) { const gbwt_b200_state t = next.forward; next.forward = next.reverse; next.reverse = t; }
        if (n < cap) out[n] = next;
        n++;
    }
    return n;
}

// ---- whole queries ---------------------------------------------------------------------------------

// ---- find + extends for one pattern -------------------------------------------------------------------
// The loop of src/bin/benchmark.rs:161-167, i.e. GBWT::find (src/gbwt.rs:269-281) then GBWT::extend /
// Record::follow (src/gbwt.rs:292-304, src/bwt.rs:595-616) per node. Same results as chaining gbwt_find /
// gbwt_extend, arranged for the GPU: the range lives in two 32-bit registers and every descriptor is loaded
// once, with a single 256-bit load.

// Pattern readers hand out node i as 32 bits plus a validity flag: every node of a loaded index is below 2^32
// (layout.h), so a pattern node above that can never match and the hot loop never touches 64-bit node ids.
struct PlainReader {
    const uint64_t* p;
    GBWT_HD bool node(uint32_t i, uint32_t& out) {
        const uint64_t v = GBWT_LDG(p + i);
        out = static_cast<uint32_t>(v);
        return (v >> 32) == 0;
    }
};

// Step on a single-edge record: every position maps to edge 0.
GBWT_HD bool follow_single(const Desc& d, uint32_t next, uint32_t& start, uint32_t& end) {
    const uint32_t total = d.total_len();
    const uint32_t s = d.offset0() + (start < total ? start : total), e = d.offset0() + (end < total ? end : total);
    if (next != d.node0() || s >= e) return false;
    start = s; end = e;
    return true;
}

// Step on a record with a body.
template <bool RUNS, bool INLINE_SCAN = false>
GBWT_HD bool follow_body(const IndexView& ix, const Desc& d, uint32_t next, uint32_t& start, uint32_t& end) {
    uint32_t rank = 0, edge_offset = 0;
    FlipSet fs;
    fs.lt = 0; fs.extra = NO_SYMBOL;
    if (!find_edge<false>(ix, d, next, rank, edge_offset, fs)) return false;
    const Ranks r = rank_pair<false, RUNS, INLINE_SCAN>(ix, d, rank, fs, start, end);
    if (r.at_start >= r.at_end) return false;
    start = edge_offset + r.at_start; end = edge_offset + r.at_end;
    return true;
}

// Descriptor of the record of `node` (32-bit arithmetic; the caller has checked node >= first_node); false =
// BWT::record() is None.
GBWT_HD bool record_desc32(const IndexView& ix, uint32_t node, Desc& d) {
    const uint32_t rec = node - static_cast<uint32_t>(ix.offset);
    if (rec >= ix.records) return false;
    d = load_desc(ix, rec);
    return d.fmt() != FMT_EMPTY;
}

// The loop runs in rounds: any number of single-edge records (a few instructions each), then one record with
// a body, so that the lanes of a warp meet again at the expensive rank step instead of diverging on the record
// format (measured on B200 with tools/exp_find.py: 1.2x for dense bodies, 1.9x for run-length bodies over
// the straight per-node chain). Counters, nodes and ranges are all 32-bit.
template <bool RUNS, class Reader>
GBWT_HD void query_find_extend_rounds(const IndexView& ix, Reader& rd, uint32_t k, gbwt_b200_state& out) {
    set_none(out);
    if (k == 0) return;
    const uint64_t first_node = ix.offset + 1;
    uint32_t node;
    Desc d;
    // GBWT::find on pattern node 0 (src/gbwt.rs:269-281)
    if (!rd.node(0, node) || node < first_node || !record_desc32(ix, node, d) || d.total_len() == 0) return;
    uint32_t start = 0, end = d.total_len();
    uint32_t i = 1;
    while (i < k) {
        bool dead = false;
        while (i < k && d.fmt() == FMT_SINGLE) {
            uint32_t next;
            if (!rd.node(i, next) || next < first_node || !follow_single(d, next, start, end)) { dead = true; break; }
            node = next; i++;
            if (i < k && !record_desc32(ix, node, d)) { dead = true; break; }
        }
        if (dead) return;
        if (i >= k) break;
        uint32_t next;
        if (!rd.node(i, next) || next < first_node || !follow_body<RUNS>(ix, d, next, start, end)) return;
        node = next; i++;
        if (i < k && !record_desc32(ix, node, d)) return;
    }
    out.node = node; out.start = start; out.end = end;
}

// Patterns of 2^32 nodes or more cannot be stored anywhere near a GPU; they are reported as None.
GBWT_HD void query_find_extend(const IndexView& ix, const uint64_t* pattern, uint64_t k, gbwt_b200_state& out) {
    PlainReader rd;
    rd.p = pattern;
    if (k > 0xFFFFFFFFull) { set_none(out); return; }
    query_find_extend_rounds<true>(ix, rd, static_cast<uint32_t>(k), out);
}

// bd_find(path[first]), extend_forward over path(first, end), extend_backward over path[start, first) in
// descending order: the reference's test driver, src/gbwt/tests.rs:352-361.
// Same results as chaining gbwt_bd_find / gbwt_extend_forward / gbwt_extend_backward, arranged like
// query_find_extend_rounds: 32-bit nodes and ranges, one descriptor load per step, rounds of single-edge records
// followed by one record with a body. A backward extension by `node` is a forward extension of the flipped state
// by flip(node) (src/gbwt.rs:362-367), so both phases run the same loop on swapped halves of the state.
struct Half32 { uint32_t node, start, end; };

// Extends `a` (the half being extended; `d` is the descriptor of a.node) by `x` and moves `b` (the other half)
// like bd_internal (src/gbwt.rs:370-384). False = None.
template <bool RUNS>
GBWT_HD bool bd_step(const IndexView& ix, const Desc& d, uint32_t x, Half32& a, Half32& b) {
    uint32_t flipped = 0;
    if (d.fmt() == FMT_SINGLE) {
        // the only edge has rank 0; no other symbol can precede it, so the reverse range keeps its start
        if (!follow_single(d, x, a.start, a.end)) return false;
    } else {
        uint32_t rank = 0, edge_offset = 0;
        FlipSet fs;
        fs.lt = 0; fs.extra = NO_SYMBOL;
        if (!find_edge<true>(ix, d, x, rank, edge_offset, fs)) return false;
        const Ranks r = rank_pair<true, RUNS>(ix, d, rank, fs, a.start, a.end);
        if (r.at_start >= r.at_end) return false;
        a.start = edge_offset + r.at_start; a.end = edge_offset + r.at_end;
        flipped = r.flipped;
    }
    a.node = x;
    b.start += flipped;
    b.end = b.start + (a.end - a.start);
    return true;
}

// Runs `count` extensions of `a` by the nodes path[from], path[from + step], ... (xor `flip` for the backward
// phase). Rounds: single-edge records, then one record with a body.
template <bool RUNS>
GBWT_HD bool bd_run(const IndexView& ix, const uint64_t* path, uint32_t from, int32_t step, uint32_t count, uint32_t flip,
                    Half32& a, Half32& b) {
    if (count == 0) return true;
    const uint64_t first_node = ix.offset + 1;
    Desc d;
    if (!record_desc32(ix, a.node, d)) return false;  // like BWT::record(node_to_record(..)), no first_node test here
    uint32_t at = from, left = count;
    while (left > 0) {
        bool dead = false;
        while (left > 0 && d.fmt() == FMT_SINGLE) {
            const uint64_t v = GBWT_LDG(path + at) ^ flip;
            if ((v >> 32) != 0 || v < first_node || !bd_step<RUNS>(ix, d, static_cast<uint32_t>(v), a, b)) { dead = true; break; }
            at += step; left--;
            if (left > 0 && !record_desc32(ix, a.node, d)) { dead = true; break; }
        }
        if (dead) return false;
        if (left == 0) break;
        const uint64_t v = GBWT_LDG(path + at) ^ flip;
        if ((v >> 32) != 0 || v < first_node || !bd_step<RUNS>(ix, d, static_cast<uint32_t>(v), a, b)) return false;
        at += step; left--;
        if (left > 0 && !record_desc32(ix, a.node, d)) return false;
    }
    return true;
}

template <bool RUNS>
GBWT_HD void query_bd_search_fast(const IndexView& ix, const uint64_t* path, uint64_t len, uint64_t first, uint64_t start,
                                  uint64_t end, gbwt_b200_bdstate& out) {
    set_none(out);
    if (!(start <= first && first < end && end <= len) || len > 0xFFFFFFFFull) return;
    const uint64_t v = GBWT_LDG(path + first);
    Desc d;
    // bd_find (src/gbwt.rs:311-324)
    if ((v >> 32) != 0 || v < ix.offset + 1 || !record_desc32(ix, static_cast<uint32_t>(v), d) || d.total_len() == 0) return;
    Half32 fwd, rev;
    fwd.node = static_cast<uint32_t>(v); fwd.start = 0; fwd.end = d.total_len();
    rev.node = fwd.node ^ 1u; rev.start = 0; rev.end = fwd.end;
    const uint32_t f = static_cast<uint32_t>(first);
    if (!bd_run<RUNS>(ix, path, f + 1, 1, static_cast<uint32_t>(end - first - 1), 0u, fwd, rev)) return;
    if (f > start && !bd_run<RUNS>(ix, path, f - 1, -1, static_cast<uint32_t>(first - start), 1u, rev, fwd)) return;
    out.forward.node = fwd.node; out.forward.start = fwd.start; out.forward.end = fwd.end;
    out.reverse.node = rev.node; out.reverse.start = rev.start; out.reverse.end = rev.end;
}

GBWT_HD void query_bd_search(const IndexView& ix, const uint64_t* path, uint64_t len, uint64_t first, uint64_t start,
                             uint64_t end, gbwt_b200_bdstate& out) {
    query_bd_search_fast<true>(ix, path, len, first, start, end, out);
}

// GBWT::sequence(id).collect() (src/gbwt.rs:253-261, 557-568): writes at most `cap` nodes and returns the
// full length, or UINT64_MAX when sequence() is None (id >= sequences()).
GBWT_HD uint64_t walk_sequence(const IndexView& ix, uint64_t id, uint64_t* out, uint64_t cap) {
    if (id >= ix.sequences) return ~0ull;
    uint64_t n = 0;
    gbwt_b200_pos pos;
    bool some = gbwt_start(ix, id, pos);
    while (some && n <= ix.walk_limit) {  // (the limit only ever matters for a damaged index with a cycle)
        if (n < cap) out[n] = pos.node;
        n++;
        gbwt_b200_pos next;
        some = gbwt_forward(ix, pos, next);
        pos = next;
    }
    return n;
}

// locate(node, offset) (gbwt_b200.h; the C++ GBWT's locate(node, i) is the model): the walk Record::lf takes from the
// position until it meets a locate sample; the answer is the sample's sequence and its index minus the steps taken.
// Per step the record's sample range and its descriptor are requested together: most records hold no sample, and the
// descriptor is what the LF step needs next. The walk never uses the two-hop shortcuts (IndexView::skips): they step over
// the middle node, and a sample there would be missed. False (and {UINT64_MAX, UINT64_MAX}) where the position does not
// exist, and where no sample is met within lv.max_steps steps (a damaged index: a consistent one always meets one).
// `steps` receives the number of LF steps taken.
GBWT_HD bool gbwt_locate(const IndexView& ix, const LocateView& lv, uint64_t node, uint64_t offset, gbwt_b200_occurrence& out,
                         uint64_t& steps) {
    out.sequence = ~0ull; out.index = ~0ull;
    steps = 0;
    uint64_t rec;
    // (offsets are 32-bit in the layout: a larger one must not be truncated onto a sampled offset)
    if (node < ix.offset + 1 || !record_of(ix, node, rec) || offset > 0xFFFFFFFFull) return false;
    gbwt_b200_pos pos;
    pos.node = node; pos.offset = offset;
    for (uint64_t s = 0;; s++) {
        const uint32_t lo = GBWT_LDG(lv.first + rec), hi = GBWT_LDG(lv.first + rec + 1);
        const Desc d = load_desc(ix, rec);
        if (lo < hi) {
            // samples of a record are sorted by offset: the last one at or below this offset
            const uint32_t i = static_cast<uint32_t>(pos.offset);
            uint32_t a = lo, b = hi;
            while (b - a > 1) {
                const uint32_t mid = a + (b - a) / 2;
                if (GBWT_LDG(&lv.samples[mid].offset) <= i) a = mid; else b = mid;
            }
            if (GBWT_LDG(&lv.samples[a].offset) == i) {
                const uint64_t index = GBWT_LDG(&lv.samples[a].index);
                steps = s;
                if (index < s) return false;  // (a damaged index)
                out.sequence = GBWT_LDG(&lv.samples[a].seq);
                out.index = index - s;
                return true;
            }
        }
        if (s >= lv.max_steps) { steps = s; return false; }
        gbwt_b200_pos next;
        // (also the validity test of the first position: no record, an empty one, or an offset past its end -> None)
        if (!lf_in_record(ix, d, pos.offset, next) || !record_of(ix, next.node, rec) || next.node < ix.offset + 1) { steps = s; return false; }
        pos = next;
    }
}

// ---- ranges of sequences (gbwt_b200_ranges.h) ----------------------------------------------------------------------

// support::COMPLEMENT, src/support.rs:87-98, as arithmetic (a 256-entry table indexed per lane would serialise in
// the constant cache): both cases of A/C/G/T map to the upper-case complement, every other byte to 'N'.
GBWT_HD uint32_t complement_base(uint32_t c) {
    const uint32_t u = c & 0xDFu;  // 'a'..'z' -> 'A'..'Z'; no other byte lands on A, C, G or T
    uint32_t r = 'N';
    r = (u == 'A') ? 'T' : r;
    r = (u == 'C') ? 'G' : r;
    r = (u == 'G') ? 'C' : r;
    r = (u == 'T') ? 'A' : r;
    return r;
}

// The path checkpoint (CheckpointView) a walk to node number j of sequence s starts from, as a slot of the table. Slot k
// of a sequence holds the first flush of the build walk at or after node k 2^shift, which is at most 31 nodes later
// (flushes are at most 32 nodes apart, intervals at least 64): so it is slot min(j >> shift, count - 1), or the one before
// when that one lies beyond j. The caller has checked j < seq_len[s], so the sequence has slot 0 (node 0).
GBWT_HD uint32_t checkpoint_slot(const CheckpointView& cv, uint32_t shift, uint64_t s, uint64_t j) {
    const uint32_t first = GBWT_LDG(cv.first + s), count = GBWT_LDG(cv.first + s + 1) - first;
    uint64_t k = j >> shift;
    if (k >= count) k = count - 1;
    if (k > 0 && GBWT_LDG(&cv.table[first + k].index) > j) k--;
    return first + static_cast<uint32_t>(k);
}

// Position of the checkpoint in `slot`; `index` receives its node number.
GBWT_HD gbwt_b200_pos checkpoint_pos(const CheckpointView& cv, uint32_t slot, uint64_t& index) {
    gbwt_b200_pos p;
    p.node = GBWT_LDG(&cv.table[slot].node);
    p.offset = GBWT_LDG(&cv.table[slot].offset);
    index = GBWT_LDG(&cv.table[slot].index);
    return p;
}

// seek(s, j): the position of node number j of GBWT::sequence(s), i.e. GBWT::start(s) followed by j GBWT::forward steps
// (src/gbwt.rs:213-229). With checkpoints (cv.table != nullptr) the walk starts from the checkpoint at or before j, at
// most 2^shift + 31 steps away; without, from start(s). False (and None) when s >= sequences() or j >= the length of s.
// No walk takes more than walk_limit steps, so a damaged index terminates. `steps` receives the LF steps taken.
GBWT_HD bool gbwt_seek(const IndexView& ix, const CheckpointView& cv, uint32_t shift, uint64_t s, uint64_t j, gbwt_b200_pos& out,
                       uint64_t& steps) {
    set_none(out);
    steps = 0;
    if (s >= ix.sequences) return false;
    gbwt_b200_pos pos;
    uint64_t at = 0;
    if (cv.table != nullptr) {
        if (j >= GBWT_LDG(cv.seq_len + s)) return false;
        pos = checkpoint_pos(cv, checkpoint_slot(cv, shift, s, j), at);
    } else if (!gbwt_start(ix, s, pos)) {
        return false;
    }
    for (; at < j; at++) {
        gbwt_b200_pos next;
        if (steps >= ix.walk_limit || !gbwt_forward(ix, pos, next)) return false;
        pos = next;
        steps++;
    }
    out = pos;
    return true;
}

}  // namespace gbwt_b200
