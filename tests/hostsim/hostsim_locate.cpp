// hostsim_locate.cpp -- TEST-ONLY harness: runs the product's locate walk (record_scan.cuh: gbwt_locate) on the CPU over
// the product's device layout (K0), with a sample table the test supplies, so that the walk can be checked against the
// oracle's document array in `-m "not gpu"` tests. Nothing in libgbwt_b200.so links or calls it; it is built only by
// tests/test_hostsim_locate.py.
#include <cstdio>
#include <string>

#include "../../gbwt-rs_b200/csrc/layout_builder.h"
#include "../../gbwt-rs_b200/csrc/record_scan.cuh"
#include "../../gbwt-rs_b200/csrc/sds_loader.h"

using namespace gbwt_b200;

struct LocateSim {
    HostLayout layout;
    IndexView view;
    ParsedGBWT parsed;
};

extern "C" {

LocateSim* hl_load(const uint8_t* bytes, size_t len, int policy, char* err, size_t errlen) {
    LocateSim* h = new LocateSim();
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
    return h;
}

void hl_free(LocateSim* h) { delete h; }
uint64_t hl_records(const LocateSim* h) { return h->layout.desc.size(); }
uint64_t hl_walk_limit(const LocateSim* h) { return h->layout.total_length; }

// out[q] = locate(positions[q]) with the table (first[records + 1], samples), steps[q] = LF steps taken.
void hl_locate(const LocateSim* h, const uint32_t* first, const LocateSample* samples, uint64_t max_steps,
               const gbwt_b200_pos* positions, size_t n, gbwt_b200_occurrence* out, uint64_t* steps) {
    LocateView lv;
    lv.first = first; lv.samples = samples; lv.max_steps = max_steps;
    for (size_t q = 0; q < n; q++) gbwt_locate(h->view, lv, positions[q].node, positions[q].offset, out[q], steps[q]);
}

}  // extern "C"
