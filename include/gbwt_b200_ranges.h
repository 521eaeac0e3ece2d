/*
 * gbwt_b200_ranges.h -- ranges of sequences: seek to node j of a path, and extract a range of its nodes or of its DNA
 * (libgbwt_b200.so; beyond the reference crate, like locate in gbwt_b200.h).
 *
 * Every answer is a slice of something gbwt_b200.h already returns:
 *  - seek(s, j) is the position of node number j (from 0) of GBWT::sequence(s): GBWT::start(s) followed by j GBWT::forward
 *    steps (src/gbwt.rs:213-229, 253-261). It is None ({0, 0}) when s >= sequences() or j >= the length of s. It is the
 *    inverse of locate: locate(seek(s, j)) = {s, j}.
 *  - The node range (s, start, end) is extract(s)[start .. min(end, len)).
 *  - The DNA range (s, start, end) is bytes [start, min(end, L)) of extract_dna(s) without its endmarker, L = dna_lengths(s) - 1.
 *    Reverse-oriented nodes are reverse-complemented as in extract_dna. An odd sequence id is the same path on the other
 *    strand, so range [start, end) on the other strand is s ^ 1 at [len - end, len - start).
 * A range with start >= min(end, len) is empty (a start above the end, or beyond the sequence, is not an error).
 * lengths[i] = max(0, min(end, len) - start) in nodes or bytes (the full clipped size), UINT64_MAX where the sequence is None.
 * Result i is written to out[out_offsets[i] ..], at most out_offsets[i+1] - out_offsets[i] elements (what is left of a longer
 * slot is unspecified), and nothing is written outside out[out_offsets[0] .. out_offsets[m]); out_offsets[0] may be above 0.
 * A caller can size slot i as end - start without a first call.
 *
 * How: the path checkpoints of the index (GBWT_B200_LAYOUT_CHECKPOINTS; gbwt_b200_checkpoint_info) hold the position of about
 * every interval-th node of every sequence, and, with node labels, the DNA offset of each. A seek walks at most about one
 * interval from the checkpoint before node j; a range is cut at the checkpoints it crosses into pieces walked in parallel.
 * Without checkpoints (or without DNA checkpoints, GBWT_B200_DNA_CHECKPOINTS=0) every walk starts at GBWT::start. No walk
 * runs past the total length of the index, so a damaged index terminates. Ranges add nothing to the index.
 *
 * Errors: the index checks come first and launch nothing (GBWT_B200_E_NO_GRAPH for DNA ranges without node labels). Device
 * calls take absolute offsets and slots like those of gbwt_b200.h; an empty device batch (n == 0 or m == 0) returns
 * GBWT_B200_OK, launches nothing and may pass NULL pointers.
 */
#ifndef GBWT_B200_RANGES_H
#define GBWT_B200_RANGES_H

#include "gbwt_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* out[q] = seek(seq_ids[q], indexes[q]). */
GBWT_B200_API int gbwt_b200_seek(const gbwt_b200_index* index, const uint64_t* seq_ids, const uint64_t* indexes, size_t n,
                                gbwt_b200_pos* out);
/* Node range i = (seq_ids[i], starts[i], ends[i]) to nodes[out_offsets[i] ..]. */
GBWT_B200_API int gbwt_b200_extract_ranges(const gbwt_b200_index* index, const uint64_t* seq_ids, const uint64_t* starts,
                                          const uint64_t* ends, size_t m, const uint64_t* out_offsets, uint64_t* nodes,
                                          uint64_t* lengths);
/* DNA range i = (seq_ids[i], starts[i], ends[i]) to bytes[out_offsets[i] ..]. */
GBWT_B200_API int gbwt_b200_extract_dna_ranges(const gbwt_b200_index* index, const uint64_t* seq_ids, const uint64_t* starts,
                                              const uint64_t* ends, size_t m, const uint64_t* out_offsets, uint8_t* bytes,
                                              uint64_t* lengths);

/* The same with device pointers on the caller's stream (cudaStream_t as void*, NULL = default stream). */
GBWT_B200_API int gbwt_b200_seek_device(const gbwt_b200_index* index, const uint64_t* d_seq_ids, const uint64_t* d_indexes,
                                       size_t n, gbwt_b200_pos* d_out, void* stream);
GBWT_B200_API int gbwt_b200_extract_ranges_device(const gbwt_b200_index* index, const uint64_t* d_seq_ids,
                                                 const uint64_t* d_starts, const uint64_t* d_ends, size_t m,
                                                 const uint64_t* d_out_offsets, uint64_t* d_nodes, uint64_t* d_lengths,
                                                 void* stream);
GBWT_B200_API int gbwt_b200_extract_dna_ranges_device(const gbwt_b200_index* index, const uint64_t* d_seq_ids,
                                                     const uint64_t* d_starts, const uint64_t* d_ends, size_t m,
                                                     const uint64_t* d_out_offsets, uint8_t* d_bytes, uint64_t* d_lengths,
                                                     void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GBWT_B200_RANGES_H */
