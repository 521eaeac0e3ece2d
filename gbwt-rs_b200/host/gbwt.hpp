// gbwt.hpp -- header-only C++17 mirror of the gbwt-rs `GBWT` API (src/gbwt.rs) over the C ABI of
// include/gbwt_b200.h. Same method names, argument meaning and error behaviour as the crate:
//   Option<T>  -> std::optional<T>;   assert! panics -> std::logic_error;   io::Error -> std::runtime_error.
// Scalar methods are batches of one; the *_batch methods are what a throughput-oriented caller uses.
// The Rust toolchain is not available in the build image, so this stands where the crate's host side would
// (INTEGRATION.md shows the equivalent Rust shim).
#pragma once
#include <cstddef>
#include <cstdint>
#include <optional>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "../../include/gbwt_b200.h"
#include "../../include/gbwt_b200_build.h"
#include "../../include/gbwt_b200_ranges.h"

namespace gbwt_b200_host {

constexpr std::size_t ENDMARKER = 0;  // src/lib.rs:59

// src/bwt.rs:63-69
struct Pos {
    std::size_t node = 0, offset = 0;
    bool operator==(const Pos& o) const { return node == o.node && offset == o.offset; }
};

// src/gbwt.rs:454-474. `range` is half-open like Rust's Range<usize>.
struct SearchState {
    std::size_t node = 0;
    std::pair<std::size_t, std::size_t> range{0, 0};
    std::size_t len() const { return range.second - range.first; }
    bool is_empty() const { return range.second <= range.first; }
    bool operator==(const SearchState& o) const { return node == o.node && range == o.range; }
};

// src/gbwt.rs:484-528
struct BidirectionalState {
    SearchState forward, reverse;
    std::size_t len() const { return forward.len(); }
    bool is_empty() const { return forward.is_empty(); }
    BidirectionalState flip() const { return BidirectionalState{reverse, forward}; }
    // (node id, is_reverse) of the first / last node on the path, src/gbwt.rs:517-527
    std::pair<std::size_t, bool> from() const { std::size_t n = reverse.node ^ 1; return {n / 2, (n & 1) != 0}; }
    std::pair<std::size_t, bool> to() const { return {forward.node / 2, (forward.node & 1) != 0}; }
};

class GBWT {
public:
    // serialize::load_from (src/gbwt.rs:402-438): a Simple-SDS GBWT file or a GBZ file (its embedded GBWT).
    static GBWT load(const std::string& path, int device = 0, int layout = GBWT_B200_LAYOUT_AUTO) {
        gbwt_b200_index* h = nullptr;
        check(gbwt_b200_index_load_file(path.c_str(), device, layout, &h));
        return GBWT(h);
    }
    static GBWT from_bytes(const void* bytes, std::size_t len, int device = 0, int layout = GBWT_B200_LAYOUT_AUTO) {
        gbwt_b200_index* h = nullptr;
        check(gbwt_b200_index_from_bytes(bytes, len, device, layout, &h));
        return GBWT(h);
    }
    // From the parts GBWT::load assembles (src/gbwt.rs:402-438; BWT::load, src/bwt.rs:176-185): header fields, the
    // concatenated record bytes and the start offset of every record.
    static GBWT from_parts(std::size_t sequences, std::size_t size, std::size_t offset, std::size_t alphabet_size, uint64_t flags,
                           const std::vector<uint8_t>& bwt, const std::vector<uint64_t>& record_starts, int device = 0,
                           int layout = GBWT_B200_LAYOUT_AUTO) {
        gbwt_b200_index* h = nullptr;
        check(gbwt_b200_index_from_parts(sequences, size, offset, alphabet_size, flags, bwt.data(), bwt.size(), record_starts.data(),
                                         record_starts.size(), device, layout, &h));
        return GBWT(h);
    }
    // The Simple-SDS GBWT file of the paths, built on the device (gbwt_b200_build.h; beyond the crate, which has no builder).
    // bidirectional: sequence 2q = path q, 2q+1 = its reverse with every node flipped.
    static std::vector<uint8_t> build_image(const std::vector<std::vector<uint64_t>>& paths, bool bidirectional = true, int device = 0) {
        std::vector<uint64_t> nodes, offsets{0};
        for (const auto& p : paths) { nodes.insert(nodes.end(), p.begin(), p.end()); offsets.push_back(nodes.size()); }
        void* image = nullptr;
        std::size_t len = 0;
        check(gbwt_b200_build_image(nodes.data(), offsets.data(), paths.size(), bidirectional ? 1 : 0, device, &image, &len, nullptr));
        return take(image, len);
    }
    // The GBWT of the paths: build_image loaded with from_bytes.
    static GBWT build(const std::vector<std::vector<uint64_t>>& paths, bool bidirectional = true, int device = 0,
                      int layout = GBWT_B200_LAYOUT_AUTO) {
        const std::vector<uint8_t> image = build_image(paths, bidirectional, device);
        return from_bytes(image.data(), image.size(), device, layout);
    }
    // serialize::serialize_to (src/gbwt.rs:388-400): the Simple-SDS GBWT file, tags, DA samples and metadata as loaded.
    void save(const std::string& path) const { check(gbwt_b200_index_save_file(h_, path.c_str())); }
    std::vector<uint8_t> serialize() const {
        void* image = nullptr;
        std::size_t len = 0;
        check(gbwt_b200_index_serialize(h_, &image, &len));
        return take(image, len);
    }
    // GBZ::serialize (src/gbz.rs:662-671); throws std::runtime_error for an index without node labels.
    void save_gbz(const std::string& path) const { check(gbwt_b200_index_save_gbz_file(h_, path.c_str())); }
    std::vector<uint8_t> serialize_gbz() const {
        void* image = nullptr;
        std::size_t len = 0;
        check(gbwt_b200_index_serialize_gbz(h_, &image, &len));
        return take(image, len);
    }
    GBWT(GBWT&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
    GBWT& operator=(GBWT&& o) noexcept { if (this != &o) { reset(); h_ = o.h_; o.h_ = nullptr; } return *this; }
    GBWT(const GBWT&) = delete;
    GBWT& operator=(const GBWT&) = delete;
    ~GBWT() { reset(); }
    const gbwt_b200_index* handle() const { return h_; }

    // Statistics, src/gbwt.rs:105-175.
    std::size_t len() const { return gbwt_b200_len(h_); }
    bool is_empty() const { return len() == 0; }
    std::size_t sequences() const { return gbwt_b200_sequences(h_); }
    std::size_t alphabet_size() const { return gbwt_b200_alphabet_size(h_); }
    std::size_t alphabet_offset() const { return gbwt_b200_alphabet_offset(h_); }
    std::size_t effective_size() const { return gbwt_b200_effective_size(h_); }
    std::size_t first_node() const { return gbwt_b200_first_node(h_); }
    std::size_t node_to_record(std::size_t node) const { return node - alphabet_offset(); }
    std::size_t record_to_node(std::size_t record) const { return record + alphabet_offset(); }
    bool has_node(std::size_t id) const { return gbwt_b200_has_node(h_, id) != 0; }
    bool is_bidirectional() const { return gbwt_b200_is_bidirectional(h_) != 0; }
    // Where the index lives and what it holds there (no counterpart in the crate).
    int device() const { return gbwt_b200_device(h_); }
    std::size_t device_bytes() const { uint64_t breakdown[10]; return gbwt_b200_device_bytes(h_, breakdown); }
    bool has_checkpoints() const { uint64_t info[6]; gbwt_b200_checkpoint_info(h_, info); return info[0] != 0; }
    static std::string version() { return gbwt_b200_version(); }

    // Sequence navigation, src/gbwt.rs:213-261.
    std::optional<Pos> start(std::size_t id) const {
        uint64_t in = id;
        gbwt_b200_pos out;
        check(gbwt_b200_start(h_, &in, 1, &out));
        return to_pos(out);
    }
    std::optional<Pos> forward(Pos pos) const {
        gbwt_b200_pos in{pos.node, pos.offset}, out;
        check(gbwt_b200_forward(h_, &in, 1, &out));
        return to_pos(out);
    }
    std::optional<Pos> backward(Pos pos) const {  // panics (throws) if the index is not bidirectional
        gbwt_b200_pos in{pos.node, pos.offset}, out;
        check(gbwt_b200_backward(h_, &in, 1, &out));
        return to_pos(out);
    }
    // GBWT::sequence(id).collect(): nullopt iff id >= sequences().
    std::optional<std::vector<std::size_t>> sequence(std::size_t id) const {
        if (id >= sequences()) return std::nullopt;
        auto paths = extract({static_cast<uint64_t>(id)});
        return std::vector<std::size_t>(paths.second.begin(), paths.second.end());
    }

    // locate (beyond the crate; the C++ GBWT's locate is the model, include/gbwt_b200.h): (sequence, index) of a position,
    // nullopt where there is no such position; the occurrences of a state in offset order. Needs an index created with
    // GBWT_B200_LAYOUT_LOCATE (throws otherwise).
    std::optional<std::pair<std::size_t, std::size_t>> locate(Pos pos) const {
        gbwt_b200_pos in{pos.node, pos.offset};
        gbwt_b200_occurrence out;
        check(gbwt_b200_locate(h_, &in, 1, &out));
        if (out.sequence == UINT64_MAX) return std::nullopt;
        return std::make_pair(static_cast<std::size_t>(out.sequence), static_cast<std::size_t>(out.index));
    }
    std::vector<std::pair<std::size_t, std::size_t>> locate(const SearchState& state) const {
        const gbwt_b200_state in = from_state(state);
        const uint64_t n = state.range.second > state.range.first ? state.range.second - state.range.first : 0;
        const uint64_t offsets[2] = {0, n};
        std::vector<gbwt_b200_occurrence> raw(n);
        uint64_t count = 0;
        check(gbwt_b200_locate_states(h_, &in, 1, offsets, raw.data(), &count));
        std::vector<std::pair<std::size_t, std::size_t>> out;
        for (const auto& o : raw) out.emplace_back(static_cast<std::size_t>(o.sequence), static_cast<std::size_t>(o.index));
        return out;
    }

    // Ranges of sequences (beyond the crate, include/gbwt_b200_ranges.h). seek: the position of node number j of
    // sequence(seq), nullopt where there is none. sequence_range: sequence(seq)[start .. min(end, len)); dna_range: bytes
    // [start, min(end, L)) of path_dna(seq) without its endmarker. Both are nullopt iff seq >= sequences(); a start at or
    // beyond the end gives an empty result.
    std::optional<Pos> seek(std::size_t seq, std::size_t j) const {
        uint64_t id = seq, index = j;
        gbwt_b200_pos out;
        check(gbwt_b200_seek(h_, &id, &index, 1, &out));
        return to_pos(out);
    }
    std::optional<std::vector<std::size_t>> sequence_range(std::size_t seq, std::size_t start, std::size_t end) const {
        auto raw = range<uint64_t>(gbwt_b200_extract_ranges, seq, start, end);
        if (!raw) return std::nullopt;
        return std::vector<std::size_t>(raw->begin(), raw->end());
    }
    std::optional<std::string> dna_range(std::size_t seq, std::size_t start, std::size_t end) const {
        auto raw = range<uint8_t>(gbwt_b200_extract_dna_ranges, seq, start, end);
        if (!raw) return std::nullopt;
        return std::string(raw->begin(), raw->end());
    }

    // Subpath search, src/gbwt.rs:269-304.
    std::optional<SearchState> find(std::size_t node) const {
        uint64_t in = node;
        gbwt_b200_state out;
        check(gbwt_b200_find(h_, &in, 1, &out));
        return to_state(out);
    }
    std::optional<SearchState> extend(const SearchState& state, std::size_t node) const {
        gbwt_b200_state in = from_state(state), out;
        uint64_t n = node;
        check(gbwt_b200_extend(h_, &in, &n, 1, &out));
        return to_state(out);
    }

    // Bidirectional search, src/gbwt.rs:311-384. Throw std::logic_error where the reference panics.
    std::optional<BidirectionalState> bd_find(std::size_t node) const {
        uint64_t in = node;
        gbwt_b200_bdstate out;
        check(gbwt_b200_bd_find(h_, &in, 1, &out));
        return to_bd(out);
    }
    std::optional<BidirectionalState> extend_forward(const BidirectionalState& state, std::size_t node) const {
        gbwt_b200_bdstate in{from_state(state.forward), from_state(state.reverse)}, out;
        uint64_t n = node;
        check(gbwt_b200_extend_forward(h_, &in, &n, 1, &out));
        return to_bd(out);
    }
    std::optional<BidirectionalState> extend_backward(const BidirectionalState& state, std::size_t node) const {
        gbwt_b200_bdstate in{from_state(state.forward), from_state(state.reverse)}, out;
        uint64_t n = node;
        check(gbwt_b200_extend_backward(h_, &in, &n, 1, &out));
        return to_bd(out);
    }

    // GBZ::follow_forward / follow_backward (src/gbz.rs:519-544): all non-empty single-node extensions of a state
    // in edge order; nullopt where the reference returns None (the node does not exist).
    std::optional<std::vector<BidirectionalState>> follow_forward(const BidirectionalState& state) const { return follow(state, 0); }
    std::optional<std::vector<BidirectionalState>> follow_backward(const BidirectionalState& state) const { return follow(state, 1); }

    // Node sequences and DNA-level extraction (GBZ files). GBZ::sequence / sequence_len (src/gbz.rs:292-306):
    // nullopt where the graph has no such node; throws std::runtime_error for an index without a graph.
    bool has_graph() const { return gbwt_b200_has_graph(h_) != 0; }
    std::optional<std::size_t> sequence_len(std::size_t node_id) const {
        uint64_t id = node_id, len = 0;
        check(gbwt_b200_node_sequence_lengths(h_, &id, 1, &len));
        if (len == UINT64_MAX) return std::nullopt;
        return static_cast<std::size_t>(len);
    }
    std::optional<std::string> node_sequence(std::size_t node_id) const {
        auto len = sequence_len(node_id);
        if (!len) return std::nullopt;
        std::string out(*len, '\0');
        uint64_t id = node_id, got = 0;
        const uint64_t offsets[2] = {0, *len};
        check(gbwt_b200_node_sequences(h_, &id, 1, offsets, reinterpret_cast<uint8_t*>(out.data()), &got));
        return out;
    }
    // extract_sequence of src/bin/gbz-extract.rs:173-189 for GBWT sequence ids (= encode_path(path, orientation)):
    // (offsets, bytes); every result ends with `endmarker`; a None path contributes an empty slice.
    std::pair<std::vector<uint64_t>, std::string> extract_dna(const std::vector<uint64_t>& ids, uint8_t endmarker = 0) const {
        std::vector<uint64_t> lengths(ids.size()), offsets(ids.size() + 1, 0);
        check(gbwt_b200_dna_lengths(h_, ids.data(), ids.size(), lengths.data()));
        for (std::size_t i = 0; i < ids.size(); i++) offsets[i + 1] = offsets[i] + (lengths[i] == UINT64_MAX ? 0 : lengths[i]);
        std::string bytes(offsets.back(), '\0');
        check(gbwt_b200_extract_dna(h_, ids.data(), ids.size(), endmarker, offsets.data(), reinterpret_cast<uint8_t*>(bytes.data()), lengths.data()));
        return {std::move(offsets), std::move(bytes)};
    }
    std::optional<std::string> path_dna(std::size_t seq_id, uint8_t endmarker = 0) const {
        if (seq_id >= sequences()) return std::nullopt;
        return extract_dna({static_cast<uint64_t>(seq_id)}, endmarker).second;
    }

    // Batched forms (what the kernels are for). Results use the C ABI value types; None = empty range.
    std::vector<gbwt_b200_state> find_extend_batch(const std::vector<uint64_t>& patterns, std::size_t k) const {
        std::size_t n = k ? patterns.size() / k : 0;
        std::vector<gbwt_b200_state> out(n);
        check(gbwt_b200_find_extend(h_, patterns.data(), n, k, out.data()));
        return out;
    }
    // The same with 32-bit node identifiers (half the bytes over PCIe; a node >= 2^32 has no record in an index that loads).
    std::vector<gbwt_b200_state> find_extend_batch(const std::vector<uint32_t>& patterns, std::size_t k) const {
        std::size_t n = k ? patterns.size() / k : 0;
        std::vector<gbwt_b200_state> out(n);
        check(gbwt_b200_find_extend_u32(h_, patterns.data(), n, k, out.data()));
        return out;
    }
    // Patterns of different lengths: pattern q = nodes[offsets[q] .. offsets[q + 1]).
    std::vector<gbwt_b200_state> find_extend_ragged(const std::vector<uint64_t>& nodes, const std::vector<uint64_t>& offsets) const {
        std::vector<gbwt_b200_state> out(offsets.empty() ? 0 : offsets.size() - 1);
        check(gbwt_b200_find_extend_ragged(h_, nodes.data(), offsets.data(), out.size(), out.data()));
        return out;
    }
    std::vector<gbwt_b200_bdstate> bd_search_batch(const std::vector<uint64_t>& nodes, const std::vector<uint64_t>& offsets,
                                                   const std::vector<uint64_t>& first, const std::vector<uint64_t>& start,
                                                   const std::vector<uint64_t>& end) const {
        std::vector<gbwt_b200_bdstate> out(first.size());
        check(gbwt_b200_bd_search(h_, nodes.data(), offsets.data(), first.data(), start.data(), end.data(), first.size(), out.data()));
        return out;
    }
    // (offsets, nodes) of the given sequences; a None sequence contributes an empty slice.
    std::pair<std::vector<uint64_t>, std::vector<uint64_t>> extract(const std::vector<uint64_t>& ids) const {
        std::vector<uint64_t> lengths(ids.size()), offsets(ids.size() + 1, 0);
        check(gbwt_b200_sequence_lengths(h_, ids.data(), ids.size(), lengths.data()));
        for (std::size_t i = 0; i < ids.size(); i++) offsets[i + 1] = offsets[i] + (lengths[i] == UINT64_MAX ? 0 : lengths[i]);
        std::vector<uint64_t> nodes(offsets.back());
        check(gbwt_b200_extract(h_, ids.data(), ids.size(), offsets.data(), nodes.data(), lengths.data()));
        return {std::move(offsets), std::move(nodes)};
    }

private:
    // One range: a call with an empty slot for its length, then one into a slot of that size.
    template <class T, class Fn>
    std::optional<std::vector<T>> range(Fn fn, std::size_t seq, std::size_t start, std::size_t end) const {
        uint64_t id = seq, s = start, e = end, len = 0;
        const uint64_t none[2] = {0, 0};
        check(fn(h_, &id, &s, &e, 1, none, nullptr, &len));
        if (len == UINT64_MAX) return std::nullopt;
        std::vector<T> out(len);
        const uint64_t offsets[2] = {0, len};
        check(fn(h_, &id, &s, &e, 1, offsets, out.data(), &len));
        return out;
    }
    std::optional<std::vector<BidirectionalState>> follow(const BidirectionalState& state, int backward) const {
        gbwt_b200_bdstate in{from_state(state.forward), from_state(state.reverse)};
        uint64_t count = 0;
        check(gbwt_b200_follow(h_, &in, 1, backward, nullptr, nullptr, &count));
        if (count == UINT64_MAX) return std::nullopt;
        std::vector<gbwt_b200_bdstate> raw(count);
        const uint64_t offsets[2] = {0, count};
        check(gbwt_b200_follow(h_, &in, 1, backward, offsets, raw.data(), &count));
        std::vector<BidirectionalState> out;
        for (const auto& r : raw) out.push_back(*to_bd(r));
        return out;
    }
    static std::vector<uint8_t> take(void* image, std::size_t len) {
        const uint8_t* p = static_cast<const uint8_t*>(image);
        std::vector<uint8_t> out(p, p + len);
        gbwt_b200_free(image);
        return out;
    }
    explicit GBWT(gbwt_b200_index* h) : h_(h) {}
    void reset() { if (h_) gbwt_b200_index_destroy(h_); h_ = nullptr; }
    static void check(int rc) {
        if (rc == GBWT_B200_OK) return;
        std::string msg = gbwt_b200_last_error();
        if (rc == GBWT_B200_E_NOT_BIDIRECTIONAL) throw std::logic_error(msg);  // assert!, src/gbwt.rs:237, 312, 340
        throw std::runtime_error("gbwt_b200 error " + std::to_string(rc) + ": " + msg);
    }
    static gbwt_b200_state from_state(const SearchState& s) { return gbwt_b200_state{s.node, s.range.first, s.range.second}; }
    static std::optional<SearchState> to_state(const gbwt_b200_state& s) {
        if (s.end <= s.start) return std::nullopt;
        return SearchState{static_cast<std::size_t>(s.node), {static_cast<std::size_t>(s.start), static_cast<std::size_t>(s.end)}};
    }
    static std::optional<BidirectionalState> to_bd(const gbwt_b200_bdstate& s) {
        auto f = to_state(s.forward), r = to_state(s.reverse);
        if (!f) return std::nullopt;
        return BidirectionalState{*f, r ? *r : SearchState{}};
    }
    static std::optional<Pos> to_pos(const gbwt_b200_pos& p) {
        if (p.node == ENDMARKER) return std::nullopt;
        return Pos{static_cast<std::size_t>(p.node), static_cast<std::size_t>(p.offset)};
    }
    gbwt_b200_index* h_ = nullptr;
};

}  // namespace gbwt_b200_host
