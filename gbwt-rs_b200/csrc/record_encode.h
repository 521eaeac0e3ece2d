// record_encode.h -- the byte encoding of BWT records (ByteCode::write, gbwt-rs src/support.rs:1063-1070; RLE::write,
// src/support.rs:1225-1248), shared by the host writer (layout_writer.cpp) and the device builder (build.cu); and the
// run iterator over the bodies of the device layout, shared by the writer and the device insertion (insert.cu).
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

// Feeds the runs of a body (layout.h) to `emit(value, len)` in order, possibly split (a checkpointed body splits runs at
// its checkpoints; the caller merges). `bodies` = the start of the body storage (IndexView::bodies).
template <class Emit>
GBWT_HD void for_each_run(const RecordDesc& d, const void* bodies, Emit emit) {
    const uint8_t* body = static_cast<const uint8_t*>(bodies) + 16 * static_cast<uint64_t>(d.body);
    switch (d.fmt) {
    case FMT_SINGLE:
        if (d.total_len > 0) emit(0, d.total_len);
        break;
    case FMT_DENSE2: {
        const uint32_t* words = reinterpret_cast<const uint32_t*>(body);
        uint64_t run_value = 0, run_len = 0;
        for (uint64_t i = 0; i < d.total_len; i++) {
            const uint64_t blk = i / DENSE_BITS, bit = i % DENSE_BITS;
            const uint64_t v = (words[blk * 8 + 2 + bit / 32] >> (bit % 32)) & 1u;
            if (run_len > 0 && v != run_value) { emit(run_value, run_len); run_len = 0; }
            run_value = v; run_len++;
        }
        if (run_len > 0) emit(run_value, run_len);
        break;
    }
    case FMT_DENSE4: {
        const uint32_t* words = reinterpret_cast<const uint32_t*>(body);
        uint64_t run_value = 0, run_len = 0;
        for (uint64_t i = 0; i < d.total_len; i++) {
            const uint64_t blk = i / DENSE4_POSITIONS, at = i % DENSE4_POSITIONS;
            const uint64_t v = (words[blk * 8 + 4 + at / 16] >> (2 * (at % 16))) & 3u;
            if (run_len > 0 && v != run_value) { emit(run_value, run_len); run_len = 0; }
            run_value = v; run_len++;
        }
        if (run_len > 0) emit(run_value, run_len);
        break;
    }
    case FMT_RUN8: {
        const uint64_t sigma = (d.flags & DESC_INLINE_EDGES) ? d.sigma16 : d.w01[1];
        for (uint64_t i = 0; i < d.body_len; i++) emit(body[i] % sigma, body[i] / sigma + 1);
        break;
    }
    case FMT_RUN32: {
        const uint32_t* w = reinterpret_cast<const uint32_t*>(body);
        for (uint64_t i = 0; i < d.body_len; i++) emit(w[i] & 0xFFu, static_cast<uint64_t>(w[i] >> 8) + 1);
        break;
    }
    case FMT_RUN64: {
        const uint32_t* w = reinterpret_cast<const uint32_t*>(body);
        for (uint64_t i = 0; i < d.body_len; i++) emit(w[2 * i], w[2 * i + 1]);
        break;
    }
    default:
        break;
    }
}

}  // namespace gbwt_b200
