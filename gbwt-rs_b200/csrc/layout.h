// layout.h -- the device-resident GBWT layout (shared by the host builder and the kernels).
//
// The reference keeps the BWT as one byte vector of variable-length ByteCode/RLE records located by
// an Elias-Fano select (gbwt-rs src/bwt.rs:96-130) and re-decodes the edge list into a heap Vec on
// every access (src/bwt.rs:378-395). Here every record gets
//   * one 32-byte descriptor (= one HBM sector) holding what `find`, `edge_to` and the scan need, with
//     the edge list inline when the outdegree is <= 2, and
//   * a 16-byte-aligned body in one of five formats chosen per record at load time so that a rank query
//     touches as few sectors as possible and never needs a serial varint decode.
// All formats are semantically equal to the reference's run sequence: len / lf / follow / bd_follow
// only depend on the sums of |run ∩ range| per symbol (src/bwt.rs:449-496, 595-656), which are invariant
// under splitting a run, and on the symbol at a position.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define GBWT_HD __host__ __device__ __forceinline__
#define GBWT_HD_NOINLINE __host__ __device__ __noinline__
#else
#define GBWT_HD inline
#define GBWT_HD_NOINLINE inline
#endif
#if defined(__CUDA_ARCH__)
#define GBWT_UNROLL _Pragma("unroll")
#else
#define GBWT_UNROLL
#endif

namespace gbwt_b200 {

enum BodyFormat : uint8_t {
    FMT_EMPTY = 0,   // sigma == 0: BWT::record() is None (src/bwt.rs:342, 381)
    FMT_SINGLE = 1,  // sigma == 1: every position maps to edge 0, no body needed
    FMT_DENSE2 = 2,  // sigma == 2: plain bitvector, 32-byte blocks {u32 ones_before, u32 sub-counts, 192 bits}
    FMT_RUN8 = 3,    // one byte per run: value + sigma * (len - 1), len <= max(1, 256 / sigma); no escapes
    FMT_RUN32 = 4,   // one u32 per run: value | (len - 1) << 8, sigma <= 256, len <= 2^24
    FMT_RUN64 = 5,   // two u32 per run: value, len
    FMT_DENSE4 = 6,  // sigma == 3 or 4: two bits per position, 32-byte blocks {counts of symbols 1, 2, 3 before the block, -, 64 positions}
    FMT_COUNT = 7
};

// Dense block for three or four symbols = one 32-byte sector: words 0-2 = occurrences of symbols 1, 2, 3 before the
// block (word 1 has bit 31 set, which tells a staged DENSE4 block from a DENSE2 block; the format is only used for records
// shorter than 2^31), word 3 unused, words 4-7 = 64 positions of two bits each (position p -> word 4 + p / 16, bits
// 2 (p % 16)). A rank is one block and at most four masked 32-bit match counts.
constexpr uint32_t DENSE4_POSITIONS = 64;
constexpr uint32_t DENSE4_TAG = 0x80000000u;

// Dense block = one 32-byte sector: word 0 = ones before the block, word 1 = ones in payload bits [0, 64) in
// bits 0-7 and ones in [0, 128) in bits 8-15, words 2-7 = 192 payload bits (position p -> word 2 + p / 32,
// bit p % 32). rank needs the block, one sub-count and ONE masked 64-bit popcount.
constexpr uint32_t DENSE_BITS = 192;
constexpr uint32_t DENSE_WORDS = 6;
constexpr uint8_t DESC_INLINE_EDGES = 1;    // w[] = {node0, offset0, node1, offset1}
// Checkpointed run bodies: flags bits 1-5 hold log2(P) + 1 when a table of checkpoints follows the runs of a RUN8 /
// RUN32 / RUN64 body (0: none). The table starts on the next 32-byte boundary after the runs; entry j - 1 describes
// position j P (j = 1 .. (total_len - 1) / P), in (sigma + 3) / 4 * 4 words: words 0 .. sigma - 2 = the number of
// positions before j P with a symbol <= v, word sigma - 1 = the index of the run that starts at j P (the builder
// splits runs at multiples of P). Only for records with at most CKPT_MAX_SIGMA edges and more than CKPT_MIN_RUNS runs.
constexpr uint32_t DESC_CKPT_SHIFT = 1, DESC_CKPT_MASK = 31;
constexpr uint32_t CKPT_MAX_SIGMA = 64, CKPT_MIN_RUNS = 32, CKPT_RUNS_PER_INTERVAL = 32;
constexpr uint32_t RUN32_MAX_LEN = 1u << 24;
constexpr uint32_t NO_SYMBOL = 0xFFFFFFFFu;
// Window kernels (find_window.cuh): record windows are staged into shared memory in multiples of STAGE_GRANULE
// records; STAGE_LOCAL is the distance (in records) within which an edge counts as local.
constexpr uint32_t STAGE_GRANULE = 32;
constexpr uint32_t STAGE_LOCAL = 128;

// One record. 32 bytes, 32-byte aligned: a single sector, fetched with one 256-bit load, gives everything
// but the body.
struct alignas(32) RecordDesc {
    uint32_t total_len;  // Record::len(), src/bwt.rs:449-455
    uint16_t sigma16;    // min(sigma, 65535)
    uint8_t fmt;         // BodyFormat
    uint8_t flags;
    // DESC_INLINE_EDGES: w = {node0, offset0, node1, offset1} (node1 unused when sigma == 1)
    // otherwise:         w = {first edge index into IndexView::edges, sigma, magic = 65536 / sigma + 1, 0}
    uint32_t w01[2];
    uint32_t body;       // offset of the body in 16-byte units (always even: bodies are 32-byte aligned)
    uint32_t body_len;   // RUN8: bytes; RUN32 / RUN64: runs; DENSE2: 32-byte blocks
    uint32_t w23[2];
};
static_assert(sizeof(RecordDesc) == 32, "descriptor must be one sector");

// One 16-byte unit of body storage (loaded with a single 128-bit access on the device).
struct alignas(16) Unit16 { uint32_t x, y, z, w; };

// Edge (node, offset), src/bwt.rs:63-69, narrowed to 32 bits.
struct Edge { uint32_t node, offset; };

// Everything a kernel needs; passed by value.
struct IndexView {
    const RecordDesc* desc;   // [records]
    const Unit16* bodies;     // 16-byte units
    const Edge* edges;        // edge lists of records with sigma > 2
    const Edge* endmarker;    // [endmarker_len] decompressed endmarker record (src/gbwt.rs:413-414)
    uint64_t records;         // BWT::len()
    uint64_t offset;          // alphabet offset (src/gbwt.rs:127-129)
    uint64_t alphabet_size;
    uint64_t sequences;
    uint64_t endmarker_len;
    uint32_t bidirectional;
    // Path-walk accelerator (K0 pass 3), one 16-byte unit per record with inline edges: {n0, o0, n1, o1}. When the
    // successor v_b over edge b is a single-edge record (LF(v_b, j) = (w, p + j)), n_b = w and o_b = offset_b + p,
    // so LF(LF(u, i)) = (n_b, o_b + rank_b(i)) without touching v_b's record; n_b = 0 where that does not apply.
    const Unit16* skips;
    uint32_t edges_valid;     // every edge of every record leads to the endmarker or to a node with a record
    // Sum of Record::len() over all records: no sequence of a consistent index visits more nodes than that. Walks
    // stop there, so that a damaged index with a cycle cannot keep a kernel running for ever (the reference's
    // iterator would not terminate on such an index).
    uint64_t walk_limit;
    // Body offset (16-byte units) of record j * STAGE_GRANULE for j = 0 .. records / STAGE_GRANULE + 1 (the entries
    // past the last record hold the total): bodies lie in record order, so the bodies of a record window are the
    // contiguous range between two entries.
    const uint32_t* stage_body;
};

// Path checkpoints (kernels.cuh: k_build_checkpoints): the position of about every `interval`-th node of every sequence,
// so that a sequence can be extracted as independent segments.
struct Checkpoint { uint32_t node, offset; uint64_t index; };  // position of node number `index` of a sequence
static_assert(sizeof(Checkpoint) == 16, "checkpoints are loaded with one vector load");
struct CheckpointView {
    const Checkpoint* table;
    const uint32_t* first;     // [sequences + 1]: slots of sequence s are table[first[s] .. first[s + 1])
    const uint64_t* seq_len;   // [sequences]
    uint32_t max_segments;     // most checkpoints any sequence has
    uint32_t discard;          // measurement only (GBWT_B200_EXTRACT_DISCARD=1): walk, but do not store the nodes
    uint32_t lookahead;        // records ahead of the walks at which a warp touches the index once per round (0 = off)
};

// Node labels of the graph in HBM: label i = bytes[starts[i] .. starts[i + 1]) (Graph::sequence, src/graph.rs:124-126).
struct GraphView {
    const uint64_t* starts;  // [sequences + 1]
    const uint8_t* bytes;
    uint64_t sequences;
};

// Locate samples (kernels.cuh: k_build_locate, locate.cu): (sequence, index) at some positions of every sequence, indexed
// by BWT position. The samples of record r are samples[first[r] .. first[r + 1]), sorted by offset.
struct LocateSample { uint32_t offset, seq; uint64_t index; };  // position (record, offset) is node `index` of sequence `seq`
static_assert(sizeof(LocateSample) == 16, "samples are loaded with one vector load");
struct LocateView {
    const uint32_t* first;          // [records + 1]
    const LocateSample* samples;
    uint64_t max_steps;             // LF steps after which a walk gives up (none): the sample bound plus slack
};

// Magic multiplier for q = b / sigma, 0 <= b < 256, 1 <= sigma <= 256: q = (b * magic) >> 16.
GBWT_HD uint32_t div_magic(uint32_t sigma) { return 65536u / sigma + 1u; }

}  // namespace gbwt_b200
