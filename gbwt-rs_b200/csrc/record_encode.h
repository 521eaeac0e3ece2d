// record_encode.h -- the byte encoding of BWT records (ByteCode::write, gbwt-rs src/support.rs:1063-1070; RLE::write,
// src/support.rs:1225-1248), shared by the host writer (layout_writer.cpp) and the device builder (build.cu).
#pragma once
#include <stdint.h>

#include "layout.h"

namespace gbwt_b200 {

// Either counts or writes: the two passes of an encoder share one code path.
struct ByteSink {
    uint8_t* at = nullptr;
    uint64_t n = 0;
    GBWT_HD void byte(uint8_t b) { if (at != nullptr) at[n] = b; n++; }
    GBWT_HD void varint(uint64_t v) {  // 7 bits per byte, least significant first, bit 7 = more to come
        while (v > 0x7F) { byte(static_cast<uint8_t>((v & 0x7F) | 0x80)); v >>= 7; }
        byte(static_cast<uint8_t>(v));
    }
};

// RLE::write_unchecked for one maximal run.
GBWT_HD void put_run(ByteSink& out, uint64_t sigma, uint64_t value, uint64_t len) {
    if (sigma >= 255) { out.varint(value); out.varint(len - 1); return; }
    const uint64_t threshold = 256 / sigma;
    if (len < threshold) { out.byte(static_cast<uint8_t>(value + sigma * (len - 1))); return; }
    out.byte(static_cast<uint8_t>(value + sigma * (threshold - 1)));
    out.varint(len - threshold);
}

// The header of a record (BWTBuilder::append, gbwt-rs src/bwt.rs:241-253): the outdegree, then (node delta, offset) per
// edge in node order; edge(e) returns the EdgeValue of edge e < sigma.
struct EdgeValue { uint64_t node, offset; };
template <class EdgeAt>
GBWT_HD void put_edges(ByteSink& out, uint64_t sigma, EdgeAt edge) {
    out.varint(sigma);
    uint64_t previous = 0;
    for (uint64_t e = 0; e < sigma; e++) {
        const EdgeValue x = edge(e);
        out.varint(x.node - previous);
        out.varint(x.offset);
        previous = x.node;
    }
}

}  // namespace gbwt_b200
