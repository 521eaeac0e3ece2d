// layout_builder.cpp -- see layout_builder.h and layout.h.
#include "layout_builder.h"

#include <algorithm>
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <type_traits>
#include <vector>
#ifdef _OPENMP
#include <omp.h>
#endif

#include "../../include/gbwt_b200.h"

namespace gbwt_b200 {
namespace {

// Decoder for one record in the reference encoding. Follows ByteCodeIter::next (src/support.rs:1151-1164)
// and RLEIter::next (src/support.rs:1413-1430) with RLE::sanitize (src/support.rs:1292-1296).
struct RecordReader {
    const uint8_t* p;
    uint64_t n, at = 0;
    uint64_t sigma = 0, threshold = 0;
    uint32_t sigma32 = 0, magic = 0;  // byte / sigma by multiplication (layout.h: div_magic), not by a 64-bit division per run
    bool bad = false;

    RecordReader(const uint8_t* bytes, uint64_t len) : p(bytes), n(len) {}

    // A varint of more than ten bytes, or one whose tenth byte does not fit 64 bits, is damaged input.
    bool varint(uint64_t& v) {
        v = 0;
        for (unsigned shift = 0; at < n; shift += 7) {
            uint8_t b = p[at++];
            if (shift >= 64 || (shift == 63 && (b & 0x7E) != 0)) { bad = true; return false; }
            v += static_cast<uint64_t>(b & 0x7F) << shift;
            if (!(b & 0x80)) return true;
        }
        return false;
    }
    void begin_runs(uint64_t s) {
        sigma = s;
        threshold = (s < 255) ? 256 / s : 0;
        if (s >= 1 && s < 255) { sigma32 = static_cast<uint32_t>(s); magic = div_magic(sigma32); }
    }
    // One run of the reference's sequence; false at the end of the record (or on a truncated run).
    bool run(uint64_t& value, uint64_t& len) {
        if (at >= n) return false;
        if (sigma >= 255) {
            uint64_t l;
            if (!varint(value) || !varint(l) || l == ~0ull) { bad = true; return false; }
            len = l + 1;
        } else {
            const uint32_t b = p[at++], q = (b * magic) >> 16;  // q = b / sigma for b < 256, sigma <= 256
            value = b - q * sigma32;
            len = q + 1;
            if (len == threshold) {
                uint64_t extra;
                if (!varint(extra) || extra > ~0ull - len) { bad = true; return false; }
                len += extra;
            }
        }
        return true;
    }
};

// (no default member initialisers: an array of plans is sized without being cleared, plan_record() starts from Plan{} = all
// zero = an empty record, status OK)
struct Plan {
    uint64_t sigma, total, runs, run8, run32, header_end;
    uint64_t count01[2];  // occurrences of symbols 0 and 1 (what the two-hop shortcuts are checked against)
    uint8_t fmt;
    uint8_t ckpt;         // 0, or log2(positions per checkpoint) + 1 for a run body with a checkpoint table (layout.h)
    uint32_t units;       // body size in 16-byte units
    int status;
};
static_assert(std::is_trivially_default_constructible<Plan>::value && FMT_EMPTY == 0 && GBWT_B200_OK == 0, "Plan{} is the plan of an empty record");

// Tuning / test knobs for the checkpoint tables (layout.h): GBWT_B200_CKPT=0 disables them, GBWT_B200_CKPT_MIN_RUNS and
// GBWT_B200_CKPT_INTERVAL_RUNS override when a body gets one and how many runs lie between two checkpoints.
struct CheckpointPolicy {
    uint64_t min_runs = CKPT_MIN_RUNS, interval_runs = CKPT_RUNS_PER_INTERVAL;
    bool enabled = true;
    CheckpointPolicy() {
        if (const char* e = std::getenv("GBWT_B200_CKPT")) enabled = std::atoi(e) != 0;
        if (const char* e = std::getenv("GBWT_B200_CKPT_MIN_RUNS")) min_runs = static_cast<uint64_t>(std::max(0, std::atoi(e)));
        if (const char* e = std::getenv("GBWT_B200_CKPT_INTERVAL_RUNS")) interval_runs = static_cast<uint64_t>(std::max(1, std::atoi(e)));
    }
};

inline uint64_t run_units_of(uint8_t fmt, uint64_t n) {
    return fmt == FMT_RUN8 ? (n + 15) / 16 : (fmt == FMT_RUN32 ? (n + 3) / 4 : (n + 1) / 2);
}

inline uint64_t ceil_div(uint64_t a, uint64_t b) { return (a + b - 1) / b; }

// Pass 1: size every candidate format and pick one.
Plan plan_record(const uint8_t* bytes, uint64_t len, int policy, const CheckpointPolicy& cp) {
    Plan pl{};
    if (len == 0) return pl;  // Record::new: empty slice -> None (src/bwt.rs:342)
    RecordReader rd(bytes, len);
    if (!rd.varint(pl.sigma)) { pl.status = GBWT_B200_E_INVALID_DATA; return pl; }
    if (pl.sigma == 0) return pl;  // decompress_edges: sigma == 0 -> None (src/bwt.rs:381)
    if (pl.sigma > 0xFFFFFFFFull) { pl.status = GBWT_B200_E_RANGE; return pl; }
    // room[b] = how many positions edge b can still send before offset_b + rank passes 2^32 - 1: the kernels add edge
    // offsets and ranks in 32 bits. A consistent index never runs out (offset_b + count_b <= the target's length < 2^32).
    // (one buffer per thread, reused from record to record; every edge takes at least two bytes of the record)
    if (pl.sigma > (len - rd.at) / 2) { pl.status = GBWT_B200_E_INVALID_DATA; return pl; }
    thread_local std::vector<uint64_t> room;
    room.resize(pl.sigma);
    uint64_t node = 0;
    for (uint64_t i = 0; i < pl.sigma; i++) {
        uint64_t delta, off;
        if (!rd.varint(delta) || !rd.varint(off)) { pl.status = GBWT_B200_E_INVALID_DATA; return pl; }
        node += delta;
        if (node > 0xFFFFFFFFull || off > 0xFFFFFFFFull) { pl.status = GBWT_B200_E_RANGE; return pl; }
        room[i] = 0xFFFFFFFFull - off;
    }
    pl.header_end = rd.at;
    rd.begin_runs(pl.sigma);
    const uint64_t max8 = pl.sigma <= 256 ? std::max<uint64_t>(1, 256 / pl.sigma) : 0;
    uint64_t value, rl;
    while (rd.run(value, rl)) {
        if (value >= pl.sigma) { pl.status = GBWT_B200_E_INVALID_DATA; return pl; }
        // a run longer than the 32-bit layout (a crafted length near 2^64 would wrap the sums below)
        if (rl == 0 || rl > 0xFFFFFFFFull) { pl.status = GBWT_B200_E_RANGE; return pl; }
        if (rl > room[value]) { pl.status = GBWT_B200_E_RANGE; return pl; }
        room[value] -= rl;
        pl.total += rl;
        if (value < 2) pl.count01[value] += rl;
        pl.runs++;
        if (max8) pl.run8 += ceil_div(rl, max8);
        pl.run32 += ceil_div(rl, RUN32_MAX_LEN);
        if (pl.total > 0xFFFFFFFFull) { pl.status = GBWT_B200_E_RANGE; return pl; }
    }
    if (rd.bad) { pl.status = GBWT_B200_E_INVALID_DATA; return pl; }
    if (pl.sigma == 1) { pl.fmt = FMT_SINGLE; return pl; }
    uint64_t best = ~0ull;
    if (pl.sigma <= 256) {
        best = ceil_div(pl.run8, 16); pl.fmt = FMT_RUN8;
        uint64_t u32 = ceil_div(pl.run32 * 4, 16);
        if (u32 < best) { best = u32; pl.fmt = FMT_RUN32; }
    } else {
        best = ceil_div(pl.runs * 8, 16); pl.fmt = FMT_RUN64;
    }
    // (a damaged file can hold a record with edges but no runs: it must not become a dense body of zero blocks)
    if (pl.sigma == 2 && policy == GBWT_B200_LAYOUT_AUTO && pl.total > 0) {
        // A dense record answers rank with one 32-byte block however long it is, so it is preferred
        // unless it would more than triple the footprint of a body that already spans several sectors. (A body of a
        // few dozen runs is a short scan and stays as it is; it is the body of a hundred runs -- low-frequency alleles
        // over a thousand haplotypes -- that would otherwise cost every rank a table entry and a scan.)
        uint64_t dense = 2 * ceil_div(pl.total, DENSE_BITS);
        if (dense <= std::max<uint64_t>(4, 3 * best)) { best = dense; pl.fmt = FMT_DENSE2; }
    }
    best = (best + 1) & ~1ull;  // every body starts on a 32-byte sector boundary (256-bit loads)
    uint64_t dense4_units = 0;
    if ((pl.sigma == 3 || pl.sigma == 4) && policy == GBWT_B200_LAYOUT_AUTO && pl.total > 0 && pl.total < (uint64_t(1) << 31))
        dense4_units = 2 * ceil_div(pl.total, DENSE4_POSITIONS);
    // Checkpoints for a long run body: one every P positions with about interval_runs runs in between, P a power of two
    // doubled until the table is no larger than the runs themselves. Runs are split at the checkpoints, at most one
    // more run each, which the body is sized for.
    const uint64_t fmt_runs = pl.fmt == FMT_RUN8 ? pl.run8 : (pl.fmt == FMT_RUN32 ? pl.run32 : pl.runs);
    if (cp.enabled && pl.fmt >= FMT_RUN8 && pl.sigma <= CKPT_MAX_SIGMA && fmt_runs > cp.min_runs && pl.total > 1) {
        const uint64_t stride_units = (pl.sigma + 3) / 4;
        uint32_t shift = 1;
        while (shift < 30 && (uint64_t(1) << shift) * fmt_runs < cp.interval_runs * pl.total) shift++;
        uint64_t entries = (pl.total - 1) >> shift;
        while (shift < 30 && entries * stride_units > run_units_of(pl.fmt, fmt_runs + entries)) { shift++; entries = (pl.total - 1) >> shift; }
        if (entries > 0) {
            pl.ckpt = static_cast<uint8_t>(shift + 1);
            best = ((run_units_of(pl.fmt, fmt_runs + entries) + 1) & ~1ull) + ((entries * stride_units + 1) & ~1ull);
        }
    }
    // Three or four symbols: two bits per position answer a rank from one 32-byte block, preferred under the same rule
    // as the bitvector of a two-symbol record (unless it more than triples a body that already spans several sectors).
    if (dense4_units != 0 && dense4_units <= std::max<uint64_t>(4, 3 * best)) { best = dense4_units; pl.fmt = FMT_DENSE4; pl.ckpt = 0; }
    if (best > 0xFFFFFFFFull) { pl.status = GBWT_B200_E_RANGE; return pl; }
    pl.units = static_cast<uint32_t>(best);
    return pl;
}

// Pass 2: write the descriptor, edges and body of one record.
void emit_record(const uint8_t* bytes, uint64_t len, const Plan& pl, uint64_t body_unit, uint64_t edge_index,
                 RecordDesc& d, uint64_t* bodies, Edge* edges) {
    std::memset(&d, 0, sizeof(d));
    d.fmt = pl.fmt;
    if (pl.fmt == FMT_EMPTY) return;
    d.body = static_cast<uint32_t>(body_unit);
    d.total_len = static_cast<uint32_t>(pl.total);
    d.sigma16 = static_cast<uint16_t>(std::min<uint64_t>(pl.sigma, 65535));
    RecordReader rd(bytes, len);
    uint64_t sigma;
    rd.varint(sigma);
    uint64_t node = 0;
    if (sigma <= 2) {
        d.flags |= DESC_INLINE_EDGES;
        for (uint64_t i = 0; i < sigma; i++) {
            uint64_t delta, off;
            rd.varint(delta); rd.varint(off);
            node += delta;
            uint32_t* w = i == 0 ? d.w01 : d.w23;
            w[0] = static_cast<uint32_t>(node);
            w[1] = static_cast<uint32_t>(off);
        }
    } else {
        d.w01[0] = static_cast<uint32_t>(edge_index);
        d.w01[1] = static_cast<uint32_t>(sigma);
        d.w23[0] = sigma <= 256 ? div_magic(static_cast<uint32_t>(sigma)) : 0;
        for (uint64_t i = 0; i < sigma; i++) {
            uint64_t delta, off;
            rd.varint(delta); rd.varint(off);
            node += delta;
            edges[edge_index + i] = Edge{static_cast<uint32_t>(node), static_cast<uint32_t>(off)};
        }
    }
    rd.begin_runs(sigma);
    uint8_t* body = reinterpret_cast<uint8_t*>(bodies + 2 * body_unit);
    uint64_t value, rl;
    switch (pl.fmt) {
    case FMT_SINGLE:
        break;
    case FMT_DENSE2: {
        uint64_t blocks = ceil_div(pl.total, DENSE_BITS);
        d.body_len = static_cast<uint32_t>(blocks);
        uint32_t* words = reinterpret_cast<uint32_t*>(body);
        uint64_t pos = 0;
        while (rd.run(value, rl)) {
            if (value == 1) {
                for (uint64_t i = pos; i < pos + rl && i < pl.total; i++) {
                    uint64_t blk = i / DENSE_BITS, bit = i % DENSE_BITS;
                    words[blk * 8 + 2 + bit / 32] |= 1u << (bit % 32);
                }
            }
            pos += rl;
        }
        uint32_t ones = 0;
        for (uint64_t b = 0; b < blocks; b++) {
            uint32_t* w = words + b * 8;
            w[0] = ones;
            const uint32_t c0 = static_cast<uint32_t>(__builtin_popcount(w[2]) + __builtin_popcount(w[3]));
            const uint32_t c1 = c0 + static_cast<uint32_t>(__builtin_popcount(w[4]) + __builtin_popcount(w[5]));
            w[1] = c0 | (c1 << 8);
            ones += c1 + static_cast<uint32_t>(__builtin_popcount(w[6]) + __builtin_popcount(w[7]));
        }
        break;
    }
    case FMT_DENSE4: {
        const uint64_t blocks = ceil_div(pl.total, DENSE4_POSITIONS);
        d.body_len = static_cast<uint32_t>(blocks);
        uint32_t* words = reinterpret_cast<uint32_t*>(body);
        uint64_t pos = 0;
        while (rd.run(value, rl)) {
            for (uint64_t i = pos; i < pos + rl && i < pl.total; i++) {
                const uint64_t blk = i / DENSE4_POSITIONS, at = i % DENSE4_POSITIONS;
                words[blk * 8 + 4 + at / 16] |= static_cast<uint32_t>(value) << (2 * (at % 16));
            }
            pos += rl;
        }
        uint32_t before[4] = {0, 0, 0, 0};
        for (uint64_t b = 0; b < blocks; b++) {
            uint32_t* w = words + b * 8;
            w[0] = before[1]; w[1] = before[2] | DENSE4_TAG; w[2] = before[3];
            const uint64_t here = std::min<uint64_t>(DENSE4_POSITIONS, pl.total - b * DENSE4_POSITIONS);
            for (uint64_t at = 0; at < here; at++) before[(w[4 + at / 16] >> (2 * (at % 16))) & 3u]++;
        }
        break;
    }
    case FMT_RUN8:
    case FMT_RUN32:
    case FMT_RUN64: {
        // The reference's run sequence, re-encoded: runs are split at the format's maximal length and, with a
        // checkpoint table, at every multiple of P (a rank only depends on the sums of |run ∩ range| per symbol, which
        // splitting a run does not change).
        const uint64_t max_len = pl.fmt == FMT_RUN8 ? std::max<uint64_t>(1, 256 / sigma) : (pl.fmt == FMT_RUN32 ? RUN32_MAX_LEN : 0xFFFFFFFFull);
        const uint64_t per_unit = pl.fmt == FMT_RUN8 ? 16 : (pl.fmt == FMT_RUN32 ? 4 : 2);
        const uint32_t shift = pl.ckpt ? pl.ckpt - 1u : 0;
        const uint64_t interval = pl.ckpt ? (uint64_t(1) << shift) : ~0ull;
        const uint64_t entries = pl.ckpt ? (pl.total - 1) >> shift : 0;
        const uint64_t stride = (sigma + 3) / 4 * 4;
        const uint64_t table_units = (entries * stride / 4 + 1) & ~1ull;
        const uint64_t cap = (static_cast<uint64_t>(pl.units) - table_units) * per_unit;  // runs the body was sized for
        std::vector<uint32_t> counts(pl.ckpt ? sigma : 0, 0), table(entries * stride, 0);
        uint32_t* out32 = reinterpret_cast<uint32_t*>(body);
        uint64_t n = 0, pos = 0, next_checkpoint = interval, written = 0;
        while (rd.run(value, rl)) {
            while (rl > 0 && n < cap) {
                const uint64_t piece = std::min(std::min(rl, max_len), next_checkpoint - pos);
                if (pl.fmt == FMT_RUN8) body[n] = static_cast<uint8_t>(value + sigma * (piece - 1));
                else if (pl.fmt == FMT_RUN32) out32[n] = static_cast<uint32_t>(value) | (static_cast<uint32_t>(piece - 1) << 8);
                else { out32[2 * n] = static_cast<uint32_t>(value); out32[2 * n + 1] = static_cast<uint32_t>(piece); }
                n++;
                rl -= piece; pos += piece;
                if (pl.ckpt) {
                    counts[value] += static_cast<uint32_t>(piece);
                    if (pos == next_checkpoint && written < entries) {
                        uint32_t* e = table.data() + written * stride;
                        uint32_t upto = 0;
                        for (uint64_t v = 0; v + 1 < sigma; v++) { upto += counts[v]; e[v] = upto; }
                        e[sigma - 1] = static_cast<uint32_t>(n);  // the next run starts at this checkpoint
                        written++;
                        next_checkpoint += interval;
                    }
                }
            }
        }
        d.body_len = static_cast<uint32_t>(n);
        if (pl.ckpt && written == entries) {
            d.flags |= static_cast<uint8_t>(pl.ckpt << DESC_CKPT_SHIFT);
            uint32_t* dst = reinterpret_cast<uint32_t*>(body) + 4 * ((run_units_of(pl.fmt, n) + 1) & ~1ull);
            std::memcpy(dst, table.data(), table.size() * sizeof(uint32_t));
        }
        break;
    }
    default:
        break;
    }
}

}  // namespace

int build_layout(const ParsedGBWT& in, int policy, HostLayout& out, std::string& err) {
    if (policy != GBWT_B200_LAYOUT_AUTO && policy != GBWT_B200_LAYOUT_RUNS) {
        err = "unknown layout policy"; return GBWT_B200_E_ARGUMENT;
    }
    const uint64_t R = in.record_starts.size();
    if (in.alphabet_size > (1ull << 32) || R > 0xFFFFFFFFull) {
        err = "alphabet does not fit the 32-bit device layout"; return GBWT_B200_E_RANGE;
    }
    // BWT::len() is the number of record starts; GBWT ids are mapped with node - offset (src/gbwt.rs:150-152).
    auto rec_len = [&](uint64_t i) { return (i + 1 < R ? in.record_starts[i + 1] : in.bwt_len) - in.record_starts[i]; };

    // Load-time work: use the host's processors (GBWT_B200_BUILD_THREADS overrides), not OMP_NUM_THREADS, which
    // launchers such as torchrun pin to 1.
    int threads = 1;
#ifdef _OPENMP
    threads = omp_get_num_procs();
#endif
    if (const char* e = std::getenv("GBWT_B200_BUILD_THREADS")) threads = std::max(1, std::atoi(e));
    (void)threads;
    // (80 bytes per record, every one of them written by the pass below: no point in one thread clearing them first)
    BigVector<Plan> plans;
    plans.resize(R);
    const CheckpointPolicy checkpoint_policy;
    std::atomic<int> status{GBWT_B200_OK};
#pragma omp parallel for schedule(dynamic, 4096) num_threads(threads)
    for (int64_t i = 0; i < static_cast<int64_t>(R); i++) {
        plans[i] = plan_record(in.bwt + in.record_starts[i], rec_len(i), policy, checkpoint_policy);
        if (plans[i].status != GBWT_B200_OK) status.store(plans[i].status);
    }
    if (status.load() != GBWT_B200_OK) {
        err = status.load() == GBWT_B200_E_RANGE ? "a record does not fit the 32-bit device layout" : "BWT: malformed record";
        return status.load();
    }
    // Where every record's body and edge list go: prefix sums over the plans, by blocks of records (sums of the blocks in
    // parallel, a scan over the few block sums, then the prefixes inside every block in parallel).
    BigVector<uint64_t> body_at, edge_at;
    body_at.resize(R + 1); edge_at.resize(R + 1);
    {
        const uint64_t block = uint64_t(1) << 16, blocks = (R + block - 1) / block;
        std::vector<uint64_t> block_body(blocks + 1, 0), block_edge(blocks + 1, 0), block_total(blocks, 0), block_ckpt(blocks, 0);
        std::vector<uint64_t> block_fmt(blocks * FMT_COUNT, 0);
#pragma omp parallel for schedule(static) num_threads(threads)
        for (int64_t b = 0; b < static_cast<int64_t>(blocks); b++) {
            uint64_t body = 0, edge = 0, total = 0, ckpt = 0;
            for (uint64_t i = b * block; i < std::min(R, (b + 1) * block); i++) {
                body += plans[i].units;
                edge += plans[i].sigma > 2 ? plans[i].sigma : 0;
                block_fmt[b * FMT_COUNT + plans[i].fmt]++;
                if (plans[i].ckpt != 0) ckpt++;
                total += plans[i].total;
            }
            block_body[b + 1] = body; block_edge[b + 1] = edge; block_total[b] = total; block_ckpt[b] = ckpt;
        }
        for (uint64_t b = 0; b < blocks; b++) {
            block_body[b + 1] += block_body[b]; block_edge[b + 1] += block_edge[b];
            out.total_length += block_total[b]; out.checkpointed_records += block_ckpt[b];
            for (int f = 0; f < FMT_COUNT; f++) out.format_counts[f] += block_fmt[b * FMT_COUNT + f];
        }
#pragma omp parallel for schedule(static) num_threads(threads)
        for (int64_t b = 0; b < static_cast<int64_t>(blocks); b++) {
            uint64_t body = block_body[b], edge = block_edge[b];
            for (uint64_t i = b * block; i < std::min(R, (b + 1) * block); i++) {
                body_at[i] = body; edge_at[i] = edge;
                body += plans[i].units;
                edge += plans[i].sigma > 2 ? plans[i].sigma : 0;
            }
        }
        body_at[R] = block_body[blocks]; edge_at[R] = block_edge[blocks];
    }
    if (body_at[R] > 0xFFFFFFFFull || edge_at[R] > 0xFFFFFFFFull) {
        err = "index does not fit the 32-bit device layout"; return GBWT_B200_E_RANGE;
    }
    // (sized without clearing -- see UninitAllocator -- and cleared by all threads: whoever clears a page also maps it)
    auto clear_all = [&](void* p, size_t bytes) {
        const size_t piece = size_t(1) << 22, pieces = (bytes + piece - 1) / piece;
        unsigned char* at = static_cast<unsigned char*>(p);
#pragma omp parallel for schedule(static) num_threads(threads)
        for (int64_t j = 0; j < static_cast<int64_t>(pieces); j++) std::memset(at + j * piece, 0, std::min(piece, bytes - j * piece));
    };
    out.desc.resize(R);
    clear_all(out.desc.data(), R * sizeof(RecordDesc));
    out.bodies.resize(2 * body_at[R] + 2);
    clear_all(out.bodies.data(), out.bodies.size() * sizeof(uint64_t));
    out.edges.assign(edge_at[R] + 1, Edge{0, 0});
#pragma omp parallel for schedule(dynamic, 4096) num_threads(threads)
    for (int64_t i = 0; i < static_cast<int64_t>(R); i++) {
        emit_record(in.bwt + in.record_starts[i], rec_len(i), plans[i], body_at[i], edge_at[i], out.desc[i],
                    out.bodies.data(), out.edges.data());
    }

    // Pass 3: edge targets are checked once here so that a path walk can follow them without bounds tests, and the
    // two-hop shortcuts over single-edge successors are filled in (layout.h, IndexView::skips).
    out.skips.resize(2 * R + 2);
    clear_all(out.skips.data(), out.skips.size() * sizeof(uint64_t));
    std::atomic<bool> edges_valid{true};
    auto has_record = [&](uint64_t node) { return node > in.offset && node - in.offset < R; };
#pragma omp parallel for schedule(dynamic, 4096) num_threads(threads)
    for (int64_t i = 0; i < static_cast<int64_t>(R); i++) {
        const RecordDesc& d = out.desc[i];
        if (d.fmt == FMT_EMPTY) continue;
        if (!(d.flags & DESC_INLINE_EDGES)) {
            for (uint64_t e = 0; e < plans[i].sigma; e++) {
                const uint32_t node = out.edges[edge_at[i] + e].node;
                if (node != 0 && !has_record(node)) edges_valid.store(false);
            }
            continue;
        }
        uint32_t* skip = reinterpret_cast<uint32_t*>(out.skips.data() + 2 * i);
        for (uint64_t b = 0; b < plans[i].sigma; b++) {
            const uint32_t* w = b == 0 ? d.w01 : d.w23;
            if (w[0] == 0) continue;
            if (!has_record(w[0])) { edges_valid.store(false); continue; }
            const RecordDesc& v = out.desc[w[0] - in.offset];
            if (v.fmt != FMT_SINGLE || v.w01[0] == 0 || !has_record(v.w01[0])) continue;
            // The shortcut replaces the step on v: Record::follow / lf there clamp to v's length (src/bwt.rs:605-607,
            // 484), which only leaves the positions alone if everything u sends over this edge lies inside v. Always
            // true in a consistent index; on a damaged one the shortcut is simply not made.
            if (static_cast<uint64_t>(w[1]) + plans[i].count01[b] > v.total_len) continue;
            const uint64_t offset = static_cast<uint64_t>(w[1]) + v.w01[1];
            if (offset > 0xFFFFFFFFull) continue;
            skip[2 * b] = v.w01[0];
            skip[2 * b + 1] = static_cast<uint32_t>(offset);
        }
    }
    out.edges_valid = edges_valid.load();

    // Staging table of the window kernels (layout.h, IndexView::stage_body): where the bodies of every
    // STAGE_GRANULE-th record start, so that a CTA can size the bulk copy of a record window without reading
    // descriptors first. Bodies lie in record order, so a window of records owns one contiguous range of units.
    {
        const uint64_t entries = R / STAGE_GRANULE + 2;
        out.stage_body.assign(entries, static_cast<uint32_t>(body_at[R]));
        for (uint64_t j = 0; j * STAGE_GRANULE <= R; j++) out.stage_body[j] = static_cast<uint32_t>(body_at[j * STAGE_GRANULE]);
    }
    // How local the graph is in record order: the share of edges whose target lies within STAGE_LOCAL records. The
    // window kernels are only worth launching when a pattern mostly stays near its first record.
    {
        uint64_t edges_seen = 0, edges_near = 0, span = 0;
#pragma omp parallel for schedule(static) num_threads(threads) reduction(+ : edges_seen, edges_near, span)
        for (int64_t i = 0; i < static_cast<int64_t>(R); i++) {
            const RecordDesc& d = out.desc[i];
            if (d.fmt == FMT_EMPTY) continue;
            auto tally = [&](uint32_t node) {
                if (node == 0) return;
                edges_seen++;
                const int64_t delta = static_cast<int64_t>(node) - static_cast<int64_t>(in.offset) - i;
                if (delta >= -static_cast<int64_t>(STAGE_LOCAL) && delta <= static_cast<int64_t>(STAGE_LOCAL)) { edges_near++; span += static_cast<uint64_t>(delta < 0 ? -delta : delta); }
            };
            if (d.flags & DESC_INLINE_EDGES) {
                tally(d.w01[0]);
                if (plans[i].sigma == 2) tally(d.w23[0]);
            } else {
                for (uint64_t e = 0; e < plans[i].sigma; e++) tally(out.edges[edge_at[i] + e].node);
            }
        }
        out.edges_total = edges_seen;
        out.edges_local = edges_near;
        out.edges_local_span = span;
    }

    // Endmarker: Record::decompress of record 0 (src/bwt.rs:465-475, src/gbwt.rs:413-414).
    out.endmarker.clear();
    if (R > 0) {
        if (plans[0].fmt == FMT_EMPTY) { err = "GBWT: missing endmarker record"; return GBWT_B200_E_INVALID_DATA; }
        RecordReader rd(in.bwt + in.record_starts[0], rec_len(0));
        uint64_t sigma;
        rd.varint(sigma);
        std::vector<Edge> e(sigma);
        uint64_t node = 0;
        for (uint64_t i = 0; i < sigma; i++) {
            uint64_t delta, off;
            rd.varint(delta); rd.varint(off);
            node += delta;
            e[i] = Edge{static_cast<uint32_t>(node), static_cast<uint32_t>(off)};
        }
        rd.begin_runs(sigma);
        out.endmarker.reserve(plans[0].total);
        uint64_t value, rl;
        while (rd.run(value, rl)) {
            for (uint64_t j = 0; j < rl; j++) { out.endmarker.push_back(e[value]); e[value].offset++; }
        }
    }
    return GBWT_B200_OK;
}

}  // namespace gbwt_b200
