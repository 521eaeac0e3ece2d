/*
 * gbwt_b200.h -- C ABI of the B200-native GBWT search / LF engine (libgbwt_b200.so).
 *
 * The reference (gbwt-rs, crate `gbz` 0.5.1) exposes no FFI; its boundary for this path is the
 * public Rust API of `GBWT` (src/gbwt.rs), plus, for the rows next to the path, `GBZ::follow_*` and
 * `GBZ::sequence` (src/gbz.rs) and `extract_sequence` (src/bin/gbz-extract.rs). Every entry point below is
 * the batched form of one of those functions and cites the one it replaces. A scalar crate call is a batch of one.
 *
 * Conventions
 *  - All integers are 64-bit like the crate's `usize`; nothing is truncated at the boundary. The device
 *    layout stores node ids, offsets and record lengths in 32 bits, so an index whose alphabet size
 *    exceeds 2^32 (a node id above 2^32 - 1) or whose record length reaches 2^32 is rejected at load
 *    with GBWT_B200_E_RANGE (it could not fit a B200's HBM either: one 32-byte record descriptor per
 *    node). So is an index in which some edge b of a record has offset_b + count_b > 2^32 - 1, count_b
 *    being the number of the record's positions with symbol b: the kernels add edge offsets and ranks in
 *    32 bits. A consistent index never has one (offset_b + count_b is at most the length of b's record).
 *  - `Option::None` is encoded in-band: a SearchState with start >= end is None and is canonicalised to
 *    {0,0,0} (the reference guarantees Some => non-empty range, src/bwt.rs:615, 448); a None Pos is {0,0}
 *    (a Some Pos never has node == ENDMARKER, src/gbwt.rs:213-219, src/bwt.rs:485-486).
 *  - Where the reference panics (assert!) the call returns a non-zero status and writes nothing:
 *    GBWT_B200_E_NOT_BIDIRECTIONAL for src/gbwt.rs:237, 312, 340.
 *  - Host entry points take plain host pointers (pageable or pinned; pinned memory is copied
 *    asynchronously and overlapped with the kernels). `_device` entry points take device pointers valid
 *    on the index's device and a CUDA stream handle (cudaStream_t passed as void*, NULL = default
 *    stream); they only enqueue work.
 *  - An index handle is immutable after creation (gbwt_b200_index_attach_graph excepted) and may be used from
 *    many host threads at once, like the `Sync` reference type (src/gbwt.rs:95-102). The only thing queries
 *    leave behind is the length of the sequences they have walked, kept in device memory so that later
 *    extractions can walk them from both ends. There is no CPU fallback: every query entry point runs CUDA
 *    kernels on the device chosen at creation.
 *  - Damaged input is rejected with GBWT_B200_E_INVALID_DATA; no C++ exception crosses this boundary.
 */
#ifndef GBWT_B200_H
#define GBWT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define GBWT_B200_API __declspec(dllexport)
#else
#define GBWT_B200_API __attribute__((visibility("default")))
#endif

/* ---- status codes ----------------------------------------------------------------------------- */
enum {
    GBWT_B200_OK = 0,
    GBWT_B200_E_INVALID_DATA = 1,      /* io::ErrorKind::InvalidData of src/gbwt.rs:404-429, src/bwt.rs:179-181 */
    GBWT_B200_E_IO = 2,                /* file could not be read */
    GBWT_B200_E_RANGE = 3,             /* a value does not fit the 32-bit device layout */
    GBWT_B200_E_NOT_BIDIRECTIONAL = 4, /* the reference's assert! at src/gbwt.rs:237, 312, 340 */
    GBWT_B200_E_CUDA = 5,              /* CUDA runtime error; see gbwt_b200_last_error() */
    GBWT_B200_E_ARGUMENT = 6,          /* NULL handle / pointer, bad layout policy, ... */
    GBWT_B200_E_NO_DEVICE = 7,         /* no CUDA device: there is deliberately no CPU fallback */
    GBWT_B200_E_NO_GRAPH = 8,          /* node sequences requested from an index that has no graph (not a GBZ) */
    GBWT_B200_E_NO_SAMPLES = 9         /* locate on an index created without GBWT_B200_LAYOUT_LOCATE */
};

/* ---- value types ------------------------------------------------------------------------------ */
/* Pos, src/bwt.rs:63-69. */
typedef struct { uint64_t node, offset; } gbwt_b200_pos;
/* SearchState, src/gbwt.rs:454-474: last matched node + half-open offset range. */
typedef struct { uint64_t node, start, end; } gbwt_b200_state;
/* BidirectionalState, src/gbwt.rs:484-528. */
typedef struct { gbwt_b200_state forward, reverse; } gbwt_b200_bdstate;
/* What locate answers for one BWT position: node number `index` (from 0) of GBWT::sequence(`sequence`). {UINT64_MAX,
 * UINT64_MAX} where there is no such position. */
typedef struct { uint64_t sequence, index; } gbwt_b200_occurrence;

typedef struct gbwt_b200_index gbwt_b200_index;

/* How record bodies are laid out in HBM (see DESIGN.md "Device layout"). */
enum {
    GBWT_B200_LAYOUT_AUTO = 0, /* per record: the format that touches the fewest bytes per query */
    GBWT_B200_LAYOUT_RUNS = 1, /* run-length bodies only (the reference's runs, escape-free re-encoding) */
    /* Flags, or-ed into the policy. Path checkpoints: while the index is created, one walk over every sequence records
     * its length and its position at every few hundredth node, so that sequence()/extract afterwards run as
     * independent segments instead of one dependent chain per sequence (results identical; see DESIGN.md).
     * Built by default for indexes of 4 Mi path nodes or more. */
    GBWT_B200_LAYOUT_CHECKPOINTS = 0x100,    /* build them whatever the size */
    GBWT_B200_LAYOUT_NO_CHECKPOINTS = 0x200, /* never build them (extraction walks whole chains) */
    /* Locate samples (opt-in): while the index is created, one walk over every sequence samples its positions, so that
     * gbwt_b200_locate can turn a BWT position into (sequence, index). Without this flag no locate entry point works
     * (GBWT_B200_E_NO_SAMPLES) and nothing else changes. See "locate" below and DESIGN.md. */
    GBWT_B200_LAYOUT_LOCATE = 0x400
};

/* ---- construction (replaces GBWT::load / serialize::load_from, src/gbwt.rs:402-438; the embedded
 *      GBWT of a GBZ file, src/gbz.rs:678-690) ---------------------------------------------------- */
GBWT_B200_API int gbwt_b200_index_load_file(const char* path, int device, int layout_policy, gbwt_b200_index** out);
/* `bytes` is a Simple-SDS GBWT image or a GBZ image (the embedded GBWT is used). */
GBWT_B200_API int gbwt_b200_index_from_bytes(const void* bytes, size_t len, int device, int layout_policy,
                                            gbwt_b200_index** out);
/* Raw parts: header fields, concatenated record bytes in the reference encoding (src/bwt.rs:241-253)
 * and the start offset of each of the `records` records (what BWT::record_bytes selects, src/bwt.rs:116-121). */
GBWT_B200_API int gbwt_b200_index_from_parts(uint64_t sequences, uint64_t size, uint64_t offset, uint64_t alphabet_size,
                                            uint64_t flags, const uint8_t* bwt_bytes, uint64_t bwt_len,
                                            const uint64_t* record_starts, uint64_t records, int device,
                                            int layout_policy, gbwt_b200_index** out);
/* Node labels for an index built from parts (the Graph half of a GBZ, src/gbz.rs:678-696; Graph::sequences,
 * src/graph.rs:84-89): label i = label_bytes[label_starts[i] .. label_starts[i+1]) belongs to original-graph node
 * first_node / 2 + i. Checks what GBZ::load checks (bidirectional index, sequence count). Not thread-safe
 * against queries running on the same handle. Indexes loaded from a GBZ image have their graph already. */
GBWT_B200_API int gbwt_b200_index_attach_graph(gbwt_b200_index* index, uint64_t sequences, const uint64_t* label_starts,
                                              const uint8_t* label_bytes);
/* The way back (GBWT::serialize, src/gbwt.rs:388-400): the index as a Simple-SDS GBWT image that the reference
 * crate and the C++ tools can load. Records are re-encoded from the device layout in the reference encoding with
 * maximal runs (BWTBuilder::append, src/bwt.rs:241-253), so the BWT of a file written by the reference comes back
 * byte for byte. What is not on the accelerated path is kept on the host as it was loaded and written back whole: the
 * tags (with `source` set to "jltsiren/gbwt-rs" and in key order, which is what the reference writes after a load,
 * src/gbwt.rs:404-405), the document-array samples and the metadata. `*image` is allocated by the library:
 * gbwt_b200_free(). */
GBWT_B200_API int gbwt_b200_index_serialize(const gbwt_b200_index* index, void** image, size_t* len);
GBWT_B200_API int gbwt_b200_index_save_file(const gbwt_b200_index* index, const char* path);
/* GBZ::serialize (src/gbz.rs:662-671): GBZ header (version 2), tags, the GBWT image above, the Graph. The Graph section
 * of an index loaded from a GBZ image is written back as it was read (node labels, segment names, node-to-segment
 * mapping; the reference would re-compress the labels with Zstandard -- both forms load in the reference); labels given
 * with gbwt_b200_index_attach_graph are written as a version-3 Graph without translation. GBWT_B200_E_NO_GRAPH
 * without node labels. */
GBWT_B200_API int gbwt_b200_index_serialize_gbz(const gbwt_b200_index* index, void** image, size_t* len);
GBWT_B200_API int gbwt_b200_index_save_gbz_file(const gbwt_b200_index* index, const char* path);
/* Build once, replicate over NVLink (multi-GPU jobs: one process per GPU, the same index on every GPU). The exporting
 * process describes its index in a small blob (scalars, the carried tags / metadata, one CUDA IPC handle per device
 * array; gbwt_b200_free() it); every other process of the node imports it: the arrays are copied device to device from
 * the exporter's GPU into the importer's `device`. The exporter must keep its index alive until the imports are done.
 * The imported handle is independent afterwards and answers exactly like one built from the same image. */
GBWT_B200_API int gbwt_b200_index_export_ipc(const gbwt_b200_index* index, void** blob, size_t* len);
GBWT_B200_API int gbwt_b200_index_import_ipc(const void* blob, size_t len, int device, gbwt_b200_index** out);
GBWT_B200_API void gbwt_b200_free(void* p);
GBWT_B200_API void gbwt_b200_index_destroy(gbwt_b200_index* index);
/* Message of the last failure on the calling thread (never NULL). */
GBWT_B200_API const char* gbwt_b200_last_error(void);

/* ---- statistics (src/gbwt.rs:105-175) ---------------------------------------------------------- */
GBWT_B200_API uint64_t gbwt_b200_len(const gbwt_b200_index* index);             /* GBWT::len */
GBWT_B200_API uint64_t gbwt_b200_sequences(const gbwt_b200_index* index);       /* GBWT::sequences */
GBWT_B200_API uint64_t gbwt_b200_alphabet_size(const gbwt_b200_index* index);   /* GBWT::alphabet_size */
GBWT_B200_API uint64_t gbwt_b200_alphabet_offset(const gbwt_b200_index* index); /* GBWT::alphabet_offset */
GBWT_B200_API uint64_t gbwt_b200_effective_size(const gbwt_b200_index* index);  /* GBWT::effective_size */
GBWT_B200_API uint64_t gbwt_b200_first_node(const gbwt_b200_index* index);      /* GBWT::first_node */
GBWT_B200_API int gbwt_b200_has_node(const gbwt_b200_index* index, uint64_t id); /* GBWT::has_node */
GBWT_B200_API int gbwt_b200_is_bidirectional(const gbwt_b200_index* index);     /* GBWT::is_bidirectional */
GBWT_B200_API int gbwt_b200_device(const gbwt_b200_index* index);
GBWT_B200_API int gbwt_b200_has_graph(const gbwt_b200_index* index);            /* loaded from a GBZ / graph attached */
GBWT_B200_API uint64_t gbwt_b200_graph_sequences(const gbwt_b200_index* index); /* Graph::sequences, src/graph.rs:112-114 */
GBWT_B200_API uint64_t gbwt_b200_graph_bytes(const gbwt_b200_index* index);     /* HBM held by the node labels */
GBWT_B200_API uint64_t gbwt_b200_skip_bytes(const gbwt_b200_index* index);      /* HBM held by the path-walk shortcuts */
/* Records whose run-length body carries a checkpoint table: a rank on them reads one table entry and scans one interval
 * of runs, where RLEIter (src/support.rs:1413-1430, used by Record::follow / lf, src/bwt.rs:480-496, 595-656) scans from
 * the start of the record. */
GBWT_B200_API uint64_t gbwt_b200_run_checkpoint_records(const gbwt_b200_index* index);
/* Records with three or four edges held as two bits per position (counted with the dense records in the breakdown of
 * gbwt_b200_device_bytes). */
GBWT_B200_API uint64_t gbwt_b200_dense4_records(const gbwt_b200_index* index);
/* Bytes of HBM held by the index (including the path-walk shortcuts and node labels, reported separately
 * below), and a breakdown: [0] descriptors, [1] bodies, [2] edge lists, [3] endmarker; [4..9] number of records per body format (empty, single-edge, dense, run8, run32, run64). */
GBWT_B200_API uint64_t gbwt_b200_device_bytes(const gbwt_b200_index* index, uint64_t breakdown[10]);
/* Path checkpoints of this index: [0] present, [1] interval (nodes), [2] entries, [3] bytes of HBM, [4] microseconds the
 * build walk took on the device, [5] most segments any sequence has. */
GBWT_B200_API void gbwt_b200_checkpoint_info(const gbwt_b200_index* index, uint64_t info[6]);
/* The record-window search kernel's plan for this index and its counters (development / tests): [0] can run, [1] is
 * the default for sorted batches, [2] records per window, [3] margin, [4] body units staged, [5] threads per CTA,
 * [6] shared memory per CTA, [7] windows, [8] edges, [9] edges to nearby records, and -- only counted when
 * GBWT_B200_WINDOW_STATS=1 -- [10] queries sent through windows, [11] queries the windows deferred to the general kernel,
 * [12] device time of the window kernel launches in nanoseconds, [13] number of those launches. */
GBWT_B200_API void gbwt_b200_window_info(const gbwt_b200_index* index, uint64_t info[14]);

/* Locate samples of this index: [0] present, [1] interval (positions of a sequence), [2] samples, [3] bytes of HBM, [4]
 * microseconds the build took on the device, and -- only counted when GBWT_B200_LOCATE_STATS=1 -- [5] LF steps taken by
 * locate walks. */
GBWT_B200_API void gbwt_b200_locate_info(const gbwt_b200_index* index, uint64_t info[6]);

/* ---- unidirectional search -------------------------------------------------------------------- */
/* GBWT::find (src/gbwt.rs:269-281) for n nodes. */
GBWT_B200_API int gbwt_b200_find(const gbwt_b200_index* index, const uint64_t* nodes, size_t n, gbwt_b200_state* out);
/* GBWT::extend (src/gbwt.rs:292-304): out[i] = extend(states[i], nodes[i]). out may alias states. */
GBWT_B200_API int gbwt_b200_extend(const gbwt_b200_index* index, const gbwt_b200_state* states, const uint64_t* nodes,
                                  size_t n, gbwt_b200_state* out);
/* find(p[0]) followed by extend over p[1..k) (the loop of src/bin/benchmark.rs:161-167) for n patterns of
 * k nodes each, row-major. k == 0 yields None. */
GBWT_B200_API int gbwt_b200_find_extend(const gbwt_b200_index* index, const uint64_t* patterns, size_t n, size_t k,
                                       gbwt_b200_state* out);
/* The same for callers that hold 32-bit node identifiers (every node of a loaded index is below 2^32, see
 * GBWT_B200_E_RANGE): half the bytes over PCIe per query. Results are identical to gbwt_b200_find_extend on the
 * widened patterns; a Rust caller with Vec<usize> paths (src/bin/benchmark.rs:155-169) narrows once on its side. */
GBWT_B200_API int gbwt_b200_find_extend_u32(const gbwt_b200_index* index, const uint32_t* patterns, size_t n, size_t k,
                                           gbwt_b200_state* out);
/* Same for ragged patterns: pattern q = nodes[offsets[q] .. offsets[q+1]). */
GBWT_B200_API int gbwt_b200_find_extend_ragged(const gbwt_b200_index* index, const uint64_t* nodes,
                                              const uint64_t* offsets, size_t n, gbwt_b200_state* out);

/* ---- bidirectional search --------------------------------------------------------------------- */
/* GBWT::bd_find (src/gbwt.rs:311-324). */
GBWT_B200_API int gbwt_b200_bd_find(const gbwt_b200_index* index, const uint64_t* nodes, size_t n, gbwt_b200_bdstate* out);
/* GBWT::extend_forward (src/gbwt.rs:339-347). */
GBWT_B200_API int gbwt_b200_extend_forward(const gbwt_b200_index* index, const gbwt_b200_bdstate* states,
                                          const uint64_t* nodes, size_t n, gbwt_b200_bdstate* out);
/* GBWT::extend_backward (src/gbwt.rs:362-367). */
GBWT_B200_API int gbwt_b200_extend_backward(const gbwt_b200_index* index, const gbwt_b200_bdstate* states,
                                           const uint64_t* nodes, size_t n, gbwt_b200_bdstate* out);
/* Fused search: for path q = nodes[offsets[q] .. offsets[q+1]), bd_find(path[first[q]]), extend_forward over
 * path[first+1 .. end), then extend_backward over path[start .. first) in descending order
 * (the reference's own test driver, src/gbwt/tests.rs:352-361). Requires start <= first < end <= len. */
GBWT_B200_API int gbwt_b200_bd_search(const gbwt_b200_index* index, const uint64_t* nodes, const uint64_t* offsets,
                                     const uint64_t* first, const uint64_t* start, const uint64_t* end, size_t n,
                                     gbwt_b200_bdstate* out);

/* GBZ::follow_forward / follow_backward with StateIter (src/gbz.rs:519-544, 1211-1249), at the GBWT level: all
 * non-empty single-node extensions of each state, in edge order (EdgeIter, src/gbz.rs:835-861). counts[i] receives
 * the number of extensions of state i, UINT64_MAX where the reference returns None (no such node). When `out` is
 * not NULL the extensions of state i are written to out[out_offsets[i] ..], at most
 * out_offsets[i+1] - out_offsets[i] of them; call once with out == NULL to size the output. */
GBWT_B200_API int gbwt_b200_follow(const gbwt_b200_index* index, const gbwt_b200_bdstate* states, size_t n, int backward,
                                  const uint64_t* out_offsets, gbwt_b200_bdstate* out, uint64_t* counts);

/* ---- sequence navigation ---------------------------------------------------------------------- */
/* GBWT::start (src/gbwt.rs:213-219). */
GBWT_B200_API int gbwt_b200_start(const gbwt_b200_index* index, const uint64_t* seq_ids, size_t n, gbwt_b200_pos* out);
/* GBWT::forward (src/gbwt.rs:222-229). */
GBWT_B200_API int gbwt_b200_forward(const gbwt_b200_index* index, const gbwt_b200_pos* positions, size_t n,
                                   gbwt_b200_pos* out);
/* GBWT::backward (src/gbwt.rs:236-250). */
GBWT_B200_API int gbwt_b200_backward(const gbwt_b200_index* index, const gbwt_b200_pos* positions, size_t n,
                                    gbwt_b200_pos* out);
/* Length of GBWT::sequence(id) (src/gbwt.rs:253-261, 557-568); UINT64_MAX where sequence() is None
 * (id >= sequences()). */
GBWT_B200_API int gbwt_b200_sequence_lengths(const gbwt_b200_index* index, const uint64_t* seq_ids, size_t m,
                                            uint64_t* lengths);
/* GBWT::sequence(id).collect() for m sequences: sequence i is written to nodes[out_offsets[i] ..], at most
 * out_offsets[i+1] - out_offsets[i] nodes (what is left of a longer slot is unspecified); lengths[i] receives the
 * full length (UINT64_MAX for None), so a caller that does not know the lengths can size the output with
 * gbwt_b200_sequence_lengths first. On a bidirectional index, sequences whose length an earlier call has measured
 * are walked from both ends at once (sequence id ^ 1 is the same path on the other strand); the two halves are
 * compared at the node where they meet and a sequence is redone from the front if they differ. */
GBWT_B200_API int gbwt_b200_extract(const gbwt_b200_index* index, const uint64_t* seq_ids, size_t m,
                                   const uint64_t* out_offsets, uint64_t* nodes, uint64_t* lengths);

/* ---- locate: which sequences, and where on them (beyond the reference crate) -------------------------------------
 * The reference crate has no locate: it carries the document-array samples of a GBWT file as opaque bytes
 * (src/gbwt.rs:100, 417). The model is the C++ GBWT's `locate(node, i)` and `locate(state)` (gbwt/gbwt.h, backed by
 * its DASamples). The answer is defined by what the crate does provide: position (node, i) with node >= first_node()
 * and i < Record::len() lies on exactly one sequence s, as node number j (from 0) of GBWT::sequence(s) -- the j-th
 * position that GBWT::start(s) and j GBWT::forward steps reach (src/gbwt.rs:213-229, 253-261, 557-568). locate(node, i)
 * = {s, j}. {UINT64_MAX, UINT64_MAX} where no such position exists: node == ENDMARKER or below first_node(), a node
 * without a record or with an empty record, i >= len, and, on a damaged index, a walk that meets no sample within its
 * bound. Requires an index created with GBWT_B200_LAYOUT_LOCATE (GBWT_B200_E_NO_SAMPLES otherwise).
 * How: the samples hold (sequence, index) at every 2^shift-th node of every sequence (GBWT_B200_LOCATE_SHIFT, default
 * 10) and at its last node; a position walks forward with Record::lf until it meets one, then subtracts its steps. */
GBWT_B200_API int gbwt_b200_locate(const gbwt_b200_index* index, const gbwt_b200_pos* positions, size_t n,
                                  gbwt_b200_occurrence* out);
/* The occurrences of a SearchState {node, start, end}: locate of (node, start) .. (node, end - 1), in offset order,
 * end - start of them, none for a None state. counts[i] = end - start (0 for None), so a caller can size the output
 * without a first call; the occurrences of state i are written to out[out_offsets[i] ..], at most
 * out_offsets[i+1] - out_offsets[i] of them (what is left of a longer slot is unspecified). out may be NULL (counts
 * only). The C++ GBWT's locate(state) is the sorted, deduplicated set of the .sequence fields of this answer. */
GBWT_B200_API int gbwt_b200_locate_states(const gbwt_b200_index* index, const gbwt_b200_state* states, size_t n,
                                         const uint64_t* out_offsets, gbwt_b200_occurrence* out, uint64_t* counts);

/* ---- node sequences (GBZ files only; GBWT_B200_E_NO_GRAPH otherwise) ------------------------------ */
/* GBZ::sequence_len / GBZ::sequence (src/gbz.rs:292-306) for n original-graph node identifiers: lengths[i] is the
 * label length, UINT64_MAX where the reference returns None (GBZ::has_node is false, src/gbz.rs:286-289). */
GBWT_B200_API int gbwt_b200_node_sequence_lengths(const gbwt_b200_index* index, const uint64_t* node_ids, size_t n,
                                                 uint64_t* lengths);
/* Label i is written to bytes[out_offsets[i] ..], at most out_offsets[i+1] - out_offsets[i] bytes. */
GBWT_B200_API int gbwt_b200_node_sequences(const gbwt_b200_index* index, const uint64_t* node_ids, size_t n,
                                          const uint64_t* out_offsets, uint8_t* bytes, uint64_t* lengths);
/* extract_sequence (src/bin/gbz-extract.rs:173-189) over GBZ::path (src/gbz.rs:461-466) for m GBWT sequence ids
 * (= support::encode_path(path_id, orientation), src/support.rs:247-249): the labels of the nodes on the path,
 * reverse-complemented for reverse-oriented nodes (support::reverse_complement, src/support.rs:104-110), then
 * the `endmarker` byte. lengths[i] = length of the full result including the endmarker, UINT64_MAX where
 * GBZ::path is None (id >= sequences()). An index with path checkpoints (GBWT_B200_LAYOUT_CHECKPOINTS, the default for long
 * sequences) and node labels spells every sequence as independent segments and answers the lengths from a table. */
GBWT_B200_API int gbwt_b200_dna_lengths(const gbwt_b200_index* index, const uint64_t* seq_ids, size_t m, uint64_t* lengths);
/* Result i is written to bytes[out_offsets[i] ..], at most out_offsets[i+1] - out_offsets[i] bytes. */
GBWT_B200_API int gbwt_b200_extract_dna(const gbwt_b200_index* index, const uint64_t* seq_ids, size_t m, uint8_t endmarker,
                                       const uint64_t* out_offsets, uint8_t* bytes, uint64_t* lengths);

/* ---- device-pointer entry points (inputs and outputs already resident in HBM) ------------------- */
GBWT_B200_API int gbwt_b200_find_extend_device(const gbwt_b200_index* index, const uint64_t* d_patterns, size_t n,
                                              size_t k, gbwt_b200_state* d_out, void* stream);
GBWT_B200_API int gbwt_b200_find_extend_u32_device(const gbwt_b200_index* index, const uint32_t* d_patterns, size_t n,
                                                  size_t k, gbwt_b200_state* d_out, void* stream);
GBWT_B200_API int gbwt_b200_find_extend_ragged_device(const gbwt_b200_index* index, const uint64_t* d_nodes,
                                                     const uint64_t* d_offsets, size_t n, gbwt_b200_state* d_out,
                                                     void* stream);
GBWT_B200_API int gbwt_b200_find_device(const gbwt_b200_index* index, const uint64_t* d_nodes, size_t n,
                                       gbwt_b200_state* d_out, void* stream);
GBWT_B200_API int gbwt_b200_extend_device(const gbwt_b200_index* index, const gbwt_b200_state* d_states,
                                         const uint64_t* d_nodes, size_t n, gbwt_b200_state* d_out, void* stream);
GBWT_B200_API int gbwt_b200_bd_find_device(const gbwt_b200_index* index, const uint64_t* d_nodes, size_t n,
                                          gbwt_b200_bdstate* d_out, void* stream);
GBWT_B200_API int gbwt_b200_bd_extend_device(const gbwt_b200_index* index, const gbwt_b200_bdstate* d_states,
                                            const uint64_t* d_nodes, size_t n, int backward,
                                            gbwt_b200_bdstate* d_out, void* stream);
GBWT_B200_API int gbwt_b200_bd_search_device(const gbwt_b200_index* index, const uint64_t* d_nodes,
                                            const uint64_t* d_offsets, const uint64_t* d_first, const uint64_t* d_start,
                                            const uint64_t* d_end, size_t n, gbwt_b200_bdstate* d_out, void* stream);
GBWT_B200_API int gbwt_b200_follow_device(const gbwt_b200_index* index, const gbwt_b200_bdstate* d_states, size_t n,
                                         int backward, const uint64_t* d_out_offsets, gbwt_b200_bdstate* d_out,
                                         uint64_t* d_counts, void* stream);
GBWT_B200_API int gbwt_b200_forward_device(const gbwt_b200_index* index, const gbwt_b200_pos* d_positions, size_t n,
                                          gbwt_b200_pos* d_out, void* stream);
GBWT_B200_API int gbwt_b200_sequence_lengths_device(const gbwt_b200_index* index, const uint64_t* d_seq_ids, size_t m,
                                                   uint64_t* d_lengths, void* stream);
GBWT_B200_API int gbwt_b200_extract_device(const gbwt_b200_index* index, const uint64_t* d_seq_ids, size_t m,
                                          const uint64_t* d_out_offsets, uint64_t* d_nodes, uint64_t* d_lengths,
                                          void* stream);

GBWT_B200_API int gbwt_b200_locate_device(const gbwt_b200_index* index, const gbwt_b200_pos* d_positions, size_t n,
                                         gbwt_b200_occurrence* d_out, void* stream);
GBWT_B200_API int gbwt_b200_locate_states_device(const gbwt_b200_index* index, const gbwt_b200_state* d_states, size_t n,
                                                const uint64_t* d_out_offsets, gbwt_b200_occurrence* d_out,
                                                uint64_t* d_counts, void* stream);

/* ---- utilities -------------------------------------------------------------------------------- */
/* Page-locked host buffers for the host entry points (cudaHostAlloc / cudaFreeHost). */
GBWT_B200_API int gbwt_b200_dna_lengths_device(const gbwt_b200_index* index, const uint64_t* d_seq_ids, size_t m,
                                              uint64_t* d_lengths, void* stream);
GBWT_B200_API int gbwt_b200_extract_dna_device(const gbwt_b200_index* index, const uint64_t* d_seq_ids, size_t m,
                                              uint8_t endmarker, const uint64_t* d_out_offsets, uint8_t* d_bytes,
                                              uint64_t* d_lengths, void* stream);
GBWT_B200_API void* gbwt_b200_host_alloc(size_t bytes);
GBWT_B200_API void gbwt_b200_host_free(void* p);
/* Number of kernels this library has launched in the calling process (for bench.py's gpu_launches). */
GBWT_B200_API uint64_t gbwt_b200_kernel_launches(void);
GBWT_B200_API const char* gbwt_b200_version(void);

#ifdef __cplusplus
}
#endif
#endif /* GBWT_B200_H */
