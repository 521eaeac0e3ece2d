// locate.h -- launchers of locate.cu (gbwt_b200_locate*, the sample table's sort).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/gbwt_b200.h"
#include "layout.h"

namespace gbwt_b200 {

// Sorts `count` samples emitted by the build walk (keys = record << 32 | offset) into a table: `table` receives them in key
// order, first[r] (r = 0 .. records) the first slot of record r. Scratch space comes from the stream-ordered pool.
cudaError_t locate_sort_samples(uint64_t* keys, LocateSample* samples, uint64_t count, uint64_t records, LocateSample* table,
                                uint32_t* first, int sm_count, cudaStream_t s);

// out[q] = locate(positions[q]). `steps` (may be null): the LF steps of all walks are added to it.
cudaError_t launch_locate(const IndexView& ix, const LocateView& lv, const gbwt_b200_pos* positions, uint64_t n,
                          gbwt_b200_occurrence* out, unsigned long long* steps, int sm_count, cudaStream_t s);

// The occurrences of states[0 .. n): counts[q] = end - start (may be null); with out != null, the first
// min(end - start, out_offsets[q + 1] - out_offsets[q]) of them go to out[out_offsets[q] - base ..].
cudaError_t launch_locate_states(const IndexView& ix, const LocateView& lv, const gbwt_b200_state* states, uint64_t n,
                                 const uint64_t* out_offsets, uint64_t base, gbwt_b200_occurrence* out, uint64_t* counts,
                                 unsigned long long* steps, int sm_count, cudaStream_t s);

}  // namespace gbwt_b200
