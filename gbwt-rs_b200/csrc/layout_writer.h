// layout_writer.h -- the way back: turns the device layout of layout.h into a Simple-SDS GBWT image that the
// reference (and this library) can load again (SURVEY.md 8(f) next-4; GBWT::serialize, gbwt-rs src/gbwt.rs:388-400;
// BWT::serialize, src/bwt.rs:170-174; the record encoding of BWTBuilder::append, src/bwt.rs:241-253, with
// RLE::write, src/support.rs:1225-1248, and ByteCode::write, src/support.rs:1063-1070). Host code, run on demand.
//
// Records are re-encoded from the layout, not kept from the input: edges from the descriptor / edge lists, runs from
// the body with adjacent runs of one value merged (the layout may have split them; maximal runs are what the
// reference's builders write). What is not on the accelerated path -- tags, document-array samples, metadata, the Graph
// section of a GBZ -- is written back as it was loaded (`Carried`); like the reference's loader (src/gbwt.rs:404-405,
// src/gbz.rs:680-681) the `source` tag is set to "jltsiren/gbwt-rs" and the tags are written in key order.
#pragma once
#include <cstdint>
#include <string>
#include <utility>
#include <vector>

#include "layout.h"

namespace gbwt_b200 {

struct LayoutArrays {
    const RecordDesc* desc = nullptr;
    uint64_t records = 0;
    const uint64_t* bodies = nullptr;  // 16-byte units as pairs of words
    const Edge* edges = nullptr;
};

struct GBWTHeaderFields {
    uint64_t sequences = 0, size = 0, offset = 0, alphabet_size = 0, flags = 0;
};

// What the loader carried through (sds_loader.h, ParsedGBWT); empty members = absent.
struct Carried {
    std::vector<std::pair<std::string, std::string>> tags, gbz_tags;
    std::vector<uint8_t> da_samples, metadata, graph_section;
};

// The concatenated records in the reference encoding and the start offset of each.
int encode_bwt(const LayoutArrays& in, std::vector<uint8_t>& data, std::vector<uint64_t>& record_starts, std::string& err);

// A complete GBWT file image: header, tags, BWT (Elias-Fano index + data), DA samples, Option<Metadata>.
int write_gbwt_image(const GBWTHeaderFields& header, const LayoutArrays& in, const Carried& carried, std::vector<uint8_t>& image,
                     std::string& err);
// The same from records already encoded: data[0 .. data_len) with record r at starts[r].
void write_gbwt_image(const GBWTHeaderFields& header, const uint8_t* data, uint64_t data_len, const std::vector<uint64_t>& starts,
                      const Carried& carried, std::vector<uint8_t>& image);

// A complete GBZ file image (GBZ::serialize, src/gbz.rs:662-671): header, tags, the GBWT image, the Graph section --
// the one that was loaded, or (for labels attached with gbwt_b200_index_attach_graph) a version-3 Graph written from
// label_starts[0 .. sequences] / label_bytes without segment names (Graph::serialize, src/graph.rs:284-294, with
// StringArray::serialize, src/support.rs:601-622, for the sequences).
int write_gbz_image(const GBWTHeaderFields& header, const LayoutArrays& in, const Carried& carried, const uint64_t* label_starts,
                    uint64_t sequences, const uint8_t* label_bytes, std::vector<uint8_t>& image, std::string& err);

}  // namespace gbwt_b200
