// insert.h -- new paths inserted into a loaded GBWT, on the device (insert.cu; gbwt_b200_insert_image in
// gbwt_b200_insert.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "layout.h"

namespace gbwt_b200 {

// The index the paths go into: its device layout and the header fields the layout does not hold.
struct InsertTarget {
    IndexView view;
    uint64_t size = 0;         // GBWT::len()
    uint64_t edges_total = 0;  // edges of all records
    uint64_t body_bytes = 0;   // bytes of body storage
};

// Path q = d_nodes[d_offsets[q] .. d_offsets[q+1]), q < n, read on stream s of the index's device (the current one). On
// success `image` is the Simple-SDS GBWT file of A's sequences followed by the new ones: path q is sequence
// A.sequences + q, or A.sequences + 2q and its reverse + 1 when A is bidirectional. `extra_bytes`: device memory the caller
// already holds for the inputs, counted into info[3]. info (may be null): positions of the new sequences, doubling
// rounds, device microseconds, peak device bytes, the longest new sequence, microseconds of the insertion walk.
// Returns a GBWT_B200_* status; `err` says why when it is not OK. Everything allocated here is freed before it returns.
int insert_gbwt_image(const InsertTarget& a, const uint64_t* d_nodes, const uint64_t* d_offsets, uint64_t n, uint64_t extra_bytes,
                      cudaStream_t s, std::vector<uint8_t>& image, uint64_t* info, std::string& err);

}  // namespace gbwt_b200
