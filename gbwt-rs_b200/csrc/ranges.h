// ranges.h -- launchers of ranges.cu (gbwt_b200_seek, gbwt_b200_extract_ranges, gbwt_b200_extract_dna_ranges).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/gbwt_b200.h"
#include "layout.h"

namespace gbwt_b200 {

// Path checkpoints as the range walks see them: cv.table == nullptr means none (every walk starts at GBWT::start).
// out[q] = seek(ids[q], indexes[q]).
cudaError_t launch_seek(const IndexView& ix, const CheckpointView& cv, uint32_t shift, const uint64_t* ids, const uint64_t* indexes,
                        uint64_t n, gbwt_b200_pos* out, int sm_count, cudaStream_t s);

// Nodes [starts[i], min(ends[i], len)) of sequence ids[i] to nodes[out_offsets[i] - base ..], cut to the slot;
// lengths[i] = the full clipped size (UINT64_MAX where the sequence is None; may be null).
cudaError_t launch_range_nodes(const IndexView& ix, const CheckpointView& cv, uint32_t shift, const uint64_t* ids, const uint64_t* starts,
                               const uint64_t* ends, uint64_t m, const uint64_t* out_offsets, uint64_t base, uint64_t* nodes,
                               uint64_t* lengths, int sm_count, cudaStream_t s);

// The same in DNA bytes (extract_dna without the endmarker). With DNA checkpoints, dna_at[slot] = bytes of the sequence before
// the checkpoint's node and dna_len[id] = the sequence's DNA length plus one; cv.table == nullptr: neither is read.
cudaError_t launch_range_dna(const IndexView& ix, const GraphView& graph, const CheckpointView& cv, const uint64_t* dna_at,
                             const uint64_t* dna_len, const uint64_t* ids, const uint64_t* starts, const uint64_t* ends, uint64_t m,
                             const uint64_t* out_offsets, uint64_t base, uint8_t* bytes, uint64_t* lengths, int sm_count,
                             cudaStream_t s);

}  // namespace gbwt_b200
