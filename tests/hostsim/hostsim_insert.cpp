// hostsim_insert.cpp -- TEST-ONLY harness: runs the product's insertion step (insert_step.h) on the CPU over the product's
// device layout (K0) of an index A, with A's incoming-edge table made here the way insert.cu makes it, so that the alpha of
// every new entry can be checked against brute-force sort keys in `-m "not gpu"` tests. Nothing in libgbwt_b200.so links
// or calls it; it is built only by tests/test_hostsim_insert.py.
#include <algorithm>
#include <cstdio>
#include <string>
#include <utility>
#include <vector>

#include "../../gbwt-rs_b200/csrc/insert_step.h"
#include "../../gbwt-rs_b200/csrc/layout_builder.h"
#include "../../gbwt-rs_b200/csrc/sds_loader.h"

using namespace gbwt_b200;

struct InsertSim {
    HostLayout layout;
    IndexView view;
    ParsedGBWT parsed;
    std::vector<uint64_t> keys;
    std::vector<uint32_t> offs;
};

extern "C" {

InsertSim* hi_load(const uint8_t* bytes, size_t len, int policy, char* err, size_t errlen) {
    InsertSim* h = new InsertSim();
    std::string msg;
    int rc = parse_gbwt_image(bytes, len, h->parsed, msg);
    if (rc == GBWT_B200_OK) rc = build_layout(h->parsed, policy, h->layout, msg);
    if (rc != GBWT_B200_OK) {
        if (err && errlen) std::snprintf(err, errlen, "%d: %s", rc, msg.c_str());
        delete h;
        return nullptr;
    }
    IndexView& v = h->view;
    v.desc = h->layout.desc.data();
    v.bodies = reinterpret_cast<const Unit16*>(h->layout.bodies.data());
    v.edges = h->layout.edges.data();
    v.endmarker = h->layout.endmarker.data();
    v.records = h->layout.desc.size();
    v.offset = h->parsed.offset;
    v.alphabet_size = h->parsed.alphabet_size;
    v.sequences = h->parsed.sequences;
    v.endmarker_len = h->layout.endmarker.size();
    v.bidirectional = (h->parsed.flags & GBWT_FLAG_BIDIRECTIONAL) != 0;
    v.skips = reinterpret_cast<const Unit16*>(h->layout.skips.data());
    v.edges_valid = h->layout.edges_valid ? 1 : 0;
    v.walk_limit = h->layout.total_length;
    v.stage_body = nullptr;
    h->parsed.bwt = nullptr;
    // the incoming-edge table of k_insert_a_edges: (v << 32 | u, offset) for every edge u -> v, sorted
    std::vector<std::pair<uint64_t, uint32_t>> table;
    for (uint64_t r = 0; r < v.records; r++) {
        const Desc d = load_desc(v, r);
        if (d.fmt() == FMT_EMPTY) continue;
        const uint64_t u = r == 0 ? 0 : r + v.offset;
        for (uint32_t k = 0; k < d.sigma(); k++) {
            const Edge e = edge_at(v, d, k);
            table.emplace_back((static_cast<uint64_t>(e.node) << 32) | u, e.offset);
        }
    }
    std::sort(table.begin(), table.end());
    for (const auto& t : table) { h->keys.push_back(t.first); h->offs.push_back(t.second); }
    return h;
}

void hi_free(InsertSim* h) { delete h; }

// Sequence q = nodes[offsets[q] .. offsets[q+1]), q < n (already in both orientations when A is bidirectional):
// alpha[offsets[q] + k] = alpha of its entry at node k, as the walk of k_insert_walk computes it.
void hi_alpha(const InsertSim* h, const uint64_t* nodes, const uint64_t* offsets, size_t n, uint64_t* alpha) {
    const InEdges in{h->keys.data(), h->offs.data(), h->keys.size()};
    for (size_t q = 0; q < n; q++) {
        uint64_t w = 0, a = h->view.sequences;
        for (uint64_t i = offsets[q]; i < offsets[q + 1]; i++) {
            a = insert_step(h->view, in, w, a, nodes[i]);
            alpha[i] = a;
            w = nodes[i];
        }
    }
}

// before_A(v, w) for each pair.
void hi_before(const InsertSim* h, const uint64_t* v, const uint64_t* w, size_t n, uint64_t* out) {
    const InEdges in{h->keys.data(), h->offs.data(), h->keys.size()};
    for (size_t i = 0; i < n; i++) out[i] = insert_before(h->view, in, v[i], w[i]);
}

}  // extern "C"
