// layout_writer.cpp -- see layout_writer.h.
#include "layout_writer.h"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>

#ifdef _OPENMP
#include <omp.h>
#endif

#include "../../include/gbwt_b200.h"
#include "record_encode.h"

namespace gbwt_b200 {
namespace {

constexpr uint64_t GBWT_TAG = 0x6B376B37ull, GBWT_VERSION = 5;
constexpr uint64_t FLAG_BIDIRECTIONAL = 1, FLAG_METADATA = 2, FLAG_SIMPLE_SDS = 4;
constexpr uint64_t GBZ_TAG = 0x205A4247ull, GBZ_VERSION = 2, GRAPH_TAG = 0x6B3764AFull, FLAG_GRAPH_SIMPLE_SDS = 2;

// One record in the encoding of BWTBuilder::append: sigma, (node delta, offset) per edge, maximal runs.
void put_record(ByteSink& out, const RecordDesc& d, const LayoutArrays& in) {
    if (d.fmt == FMT_EMPTY) { out.varint(0); return; }
    const bool inline_edges = (d.flags & DESC_INLINE_EDGES) != 0;
    const uint64_t sigma = inline_edges ? d.sigma16 : d.w01[1];
    put_edges(out, sigma, [&](uint64_t e) {
        if (inline_edges) return e == 0 ? EdgeValue{d.w01[0], d.w01[1]} : EdgeValue{d.w23[0], d.w23[1]};
        return EdgeValue{in.edges[d.w01[0] + e].node, in.edges[d.w01[0] + e].offset};
    });
    uint64_t run_value = 0, run_len = 0;
    for_each_run(d, in.bodies, [&](uint64_t value, uint64_t len) {
        if (run_len > 0 && value != run_value) { put_run(out, sigma, run_value, run_len); run_len = 0; }
        run_value = value; run_len += len;
    });
    if (run_len > 0) put_run(out, sigma, run_value, run_len);
}

int build_threads() {
    int threads = 1;
#ifdef _OPENMP
    threads = omp_get_num_procs();
#endif
    if (const char* e = std::getenv("GBWT_B200_BUILD_THREADS")) threads = std::max(1, std::atoi(e));
    return threads;
}

// ---- Simple-SDS containers (SURVEY.md App. A) ----------------------------------------------------------------------

struct WordSink {
    std::vector<uint8_t>& out;
    void word(uint64_t v) { const size_t at = out.size(); out.resize(at + 8); std::memcpy(out.data() + at, &v, 8); }
    void words(const std::vector<uint64_t>& v) { const size_t at = out.size(); out.resize(at + 8 * v.size()); if (!v.empty()) std::memcpy(out.data() + at, v.data(), 8 * v.size()); }
    void bytes(const uint8_t* p, uint64_t n) {  // Vec<u8>: length, then the bytes padded to a whole element
        word(n);
        const size_t at = out.size();
        out.resize(at + (n + 7) / 8 * 8, 0);
        if (n > 0) std::memcpy(out.data() + at, p, n);
    }
};

// SparseVector (Elias-Fano): universe, high BitVector (ones, RawVector, three absent supports), low IntVector.
void put_sparse(WordSink& w, uint64_t universe, const std::vector<uint64_t>& values) {
    const uint64_t ones = values.size();
    uint64_t width = 1;
    if (ones > 0 && ones <= universe) {
        const double ideal = std::round(std::log2(static_cast<double>(universe) * std::log(2.0) / static_cast<double>(ones)));
        width = ideal < 1.0 ? 1 : static_cast<uint64_t>(ideal);
    }
    const uint64_t mask = width < 64 ? (1ull << width) - 1 : ~0ull;
    const uint64_t buckets = (width < 64 ? universe >> width : 0) + ((universe & mask) != 0 ? 1 : 0);
    const uint64_t high_len = ones + buckets;
    std::vector<uint64_t> high((high_len + 63) / 64, 0), low((ones * width + 63) / 64, 0);
    for (uint64_t j = 0; j < ones; j++) {
        const uint64_t v = values[j], hp = (width < 64 ? v >> width : 0) + j;
        high[hp / 64] |= 1ull << (hp % 64);
        const uint64_t lv = v & mask, bit = j * width;
        low[bit / 64] |= lv << (bit % 64);
        if (bit % 64 + width > 64) low[bit / 64 + 1] |= lv >> (64 - bit % 64);
    }
    w.word(universe);
    w.word(ones); w.word(high_len); w.word(high.size()); w.words(high);
    w.word(0); w.word(0); w.word(0);
    w.word(ones); w.word(width); w.word(ones * width); w.word(low.size()); w.words(low);
}

// StringArray::serialize (src/support.rs:601-622): start offsets (no sentinel), alphabet, packed characters.
void put_string_array(WordSink& w, const std::vector<uint64_t>& starts, const uint8_t* bytes, uint64_t total) {
    const std::basic_string<unsigned char> all(bytes, bytes + total);
    put_sparse(w, starts.empty() ? 0 : starts.back() + 1, starts);
    bool present[256] = {false};
    for (unsigned char c : all) present[c] = true;
    uint8_t alphabet[256], pack[256] = {0};
    uint64_t sigma = 0;
    for (int c = 0; c < 256; c++) if (present[c]) { pack[c] = static_cast<uint8_t>(sigma); alphabet[sigma++] = static_cast<uint8_t>(c); }
    w.bytes(alphabet, sigma);
    uint64_t width = 1;
    while (sigma > 1 && ((sigma - 1) >> width) != 0) width++;
    std::vector<uint64_t> packed((all.size() * width + 63) / 64, 0);
    for (uint64_t i = 0; i < all.size(); i++) {
        const uint64_t v = pack[static_cast<unsigned char>(all[i])], bit = i * width;
        packed[bit / 64] |= v << (bit % 64);
        if (bit % 64 + width > 64) packed[bit / 64 + 1] |= v >> (64 - bit % 64);
    }
    w.word(all.size()); w.word(width); w.word(all.size() * width); w.word(packed.size()); w.words(packed);
}

// Tags: a StringArray of [key, value, ...].
void put_tags(WordSink& w, const std::vector<std::string>& strings) {
    std::vector<uint64_t> starts;
    std::string all;
    for (const std::string& s : strings) { starts.push_back(all.size()); all += s; }
    put_string_array(w, starts, reinterpret_cast<const uint8_t*>(all.data()), all.size());
}

}  // namespace

int encode_bwt(const LayoutArrays& in, std::vector<uint8_t>& data, std::vector<uint64_t>& record_starts, std::string& err) {
    if (in.records > 0 && (in.desc == nullptr || in.bodies == nullptr || in.edges == nullptr)) {
        err = "null layout"; return GBWT_B200_E_ARGUMENT;
    }
    const int threads = build_threads();
    (void)threads;
    std::vector<uint64_t> sizes(in.records + 1, 0);
#pragma omp parallel for schedule(dynamic, 4096) num_threads(threads)
    for (int64_t i = 0; i < static_cast<int64_t>(in.records); i++) {
        ByteSink count;
        put_record(count, in.desc[i], in);
        sizes[i + 1] = count.n;
    }
    record_starts.resize(in.records);
    for (uint64_t i = 0; i < in.records; i++) { record_starts[i] = sizes[i]; sizes[i + 1] += sizes[i]; }
    data.assign(sizes[in.records], 0);
#pragma omp parallel for schedule(dynamic, 4096) num_threads(threads)
    for (int64_t i = 0; i < static_cast<int64_t>(in.records); i++) {
        ByteSink write;
        write.at = data.data() + record_starts[i];
        put_record(write, in.desc[i], in);
    }
    return GBWT_B200_OK;
}

namespace {

// Tags as the reference writes them after a load: `source` = "jltsiren/gbwt-rs", keys in order (a BTreeMap).
std::vector<std::string> linearize_tags(std::vector<std::pair<std::string, std::string>> tags) {
    bool have_source = false;
    for (auto& kv : tags) if (kv.first == "source") { kv.second = "jltsiren/gbwt-rs"; have_source = true; }
    if (!have_source) tags.emplace_back("source", "jltsiren/gbwt-rs");
    std::sort(tags.begin(), tags.end());
    std::vector<std::string> flat;
    for (const auto& kv : tags) { flat.push_back(kv.first); flat.push_back(kv.second); }
    return flat;
}

void append_bytes(std::vector<uint8_t>& out, const std::vector<uint8_t>& bytes) { out.insert(out.end(), bytes.begin(), bytes.end()); }

}  // namespace

int write_gbwt_image(const GBWTHeaderFields& header, const LayoutArrays& in, const Carried& carried, std::vector<uint8_t>& image,
                     std::string& err) {
    std::vector<uint8_t> data;
    std::vector<uint64_t> starts;
    const int rc = encode_bwt(in, data, starts, err);
    if (rc != GBWT_B200_OK) return rc;
    write_gbwt_image(header, data.data(), data.size(), starts, carried, image);
    return GBWT_B200_OK;
}

void write_gbwt_image(const GBWTHeaderFields& header, const uint8_t* data, uint64_t data_len, const std::vector<uint64_t>& starts,
                      const Carried& carried, std::vector<uint8_t>& image) {
    image.clear();
    image.reserve(data_len + data_len / 4 + carried.da_samples.size() + carried.metadata.size() + 4096);
    WordSink w{image};
    const bool has_metadata = carried.metadata.size() > 8;  // Option<Metadata>: more than the size word
    w.word(GBWT_TAG | (GBWT_VERSION << 32));
    w.word(header.sequences); w.word(header.size); w.word(header.offset); w.word(header.alphabet_size);
    w.word((header.flags & FLAG_BIDIRECTIONAL) | FLAG_SIMPLE_SDS | (has_metadata ? FLAG_METADATA : 0));
    put_tags(w, linearize_tags(carried.tags));
    put_sparse(w, data_len, starts);
    w.bytes(data, data_len);
    if (carried.da_samples.empty()) w.word(0);  // an empty Vec<u64>
    else append_bytes(image, carried.da_samples);
    if (!has_metadata) w.word(0);               // Option<Metadata>: None
    else append_bytes(image, carried.metadata);
}

int write_gbz_image(const GBWTHeaderFields& header, const LayoutArrays& in, const Carried& carried, const uint64_t* label_starts,
                    uint64_t sequences, const uint8_t* label_bytes, std::vector<uint8_t>& image, std::string& err) {
    std::vector<uint8_t> gbwt;
    const int rc = write_gbwt_image(header, in, carried, gbwt, err);
    if (rc != GBWT_B200_OK) return rc;
    image.clear();
    image.reserve(gbwt.size() + carried.graph_section.size() + 4096);
    WordSink w{image};
    w.word(GBZ_TAG | (GBZ_VERSION << 32));
    w.word(0);  // GBZ flags
    put_tags(w, linearize_tags(carried.gbz_tags));
    append_bytes(image, gbwt);
    if (!carried.graph_section.empty()) { append_bytes(image, carried.graph_section); return GBWT_B200_OK; }
    if (label_starts == nullptr || (label_starts[sequences] > 0 && label_bytes == nullptr)) { err = "no node labels to write"; return GBWT_B200_E_NO_GRAPH; }
    // Graph, version 3 (sequences as a plain StringArray), no translation
    uint64_t nodes = 0;
    for (uint64_t i = 0; i < sequences; i++) if (label_starts[i + 1] > label_starts[i]) nodes++;
    w.word(GRAPH_TAG | (uint64_t(3) << 32));
    w.word(nodes);
    w.word(FLAG_GRAPH_SIMPLE_SDS);
    std::vector<uint64_t> starts(label_starts, label_starts + sequences);
    put_string_array(w, starts, label_bytes, label_starts[sequences]);
    put_string_array(w, {}, nullptr, 0);  // segment names: none
    put_sparse(w, 0, {});                 // node-to-segment mapping: empty
    return GBWT_B200_OK;
}

}  // namespace gbwt_b200
