// build.h -- the GBWT of a set of paths, built on the device (build.cu; gbwt_b200_build_image in gbwt_b200_build.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

namespace gbwt_b200 {

// The statuses of build_gbwt_image from host arrays (offsets absolute, n >= 1), before anything is copied; on success
// `records` = the number of records of the GBWT.
int build_check_paths(const uint64_t* nodes, const uint64_t* offsets, uint64_t n, bool bidirectional, uint64_t& records, std::string& err);
// Device memory a build of `paths` paths with `path_nodes` nodes in all takes, without the sort's temporary storage:
// about 36 bytes per position (nodes + sequences) and 28 per record.
uint64_t build_device_bytes(uint64_t paths, uint64_t path_nodes, bool bidirectional, uint64_t records);

// Path q = d_nodes[d_offsets[q] .. d_offsets[q+1]), q < n, read on stream s of the current device. With `bidirectional`,
// sequence 2q = path q and 2q+1 = its reverse with every node flipped; otherwise sequence q = path q. On success `image`
// is the Simple-SDS GBWT file of the sequences. `extra_bytes`: device memory the caller already holds for the inputs,
// counted into info[3]. info (may be null): positions sorted, doubling rounds, device microseconds, peak device bytes.
// Returns a GBWT_B200_* status; `err` says why when it is not OK. Everything allocated here is freed before it returns.
int build_gbwt_image(const uint64_t* d_nodes, const uint64_t* d_offsets, uint64_t n, bool bidirectional, uint64_t extra_bytes,
                     cudaStream_t s, std::vector<uint8_t>& image, uint64_t* info, std::string& err);

}  // namespace gbwt_b200
