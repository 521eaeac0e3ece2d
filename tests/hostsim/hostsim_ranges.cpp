// hostsim_ranges.cpp -- TEST-ONLY harness: runs the product's seek walk (record_scan.cuh: gbwt_seek) on the CPU over the
// product's device layout (K0), with a path-checkpoint table the test supplies, so that the walk can be checked against the
// oracle's start + forward in `-m "not gpu"` tests. Nothing in libgbwt_b200.so links or calls it; it is built only by
// tests/test_hostsim_ranges.py.
#include <cstdio>
#include <string>

#include "../../gbwt-rs_b200/csrc/layout_builder.h"
#include "../../gbwt-rs_b200/csrc/record_scan.cuh"
#include "../../gbwt-rs_b200/csrc/sds_loader.h"

using namespace gbwt_b200;

struct RangeSim {
    HostLayout layout;
    IndexView view;
    ParsedGBWT parsed;
};

extern "C" {

RangeSim* hr_load(const uint8_t* bytes, size_t len, int policy, char* err, size_t errlen) {
    RangeSim* h = new RangeSim();
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

void hr_free(RangeSim* h) { delete h; }

// out[q] = seek(ids[q], indexes[q]) with the checkpoint table (table, first[sequences + 1], seq_len) at interval 2^shift, or
// from start() when table is null; steps[q] = LF steps taken.
void hr_seek(const RangeSim* h, const Checkpoint* table, const uint32_t* first, const uint64_t* seq_len, uint32_t shift,
             const uint64_t* ids, const uint64_t* indexes, size_t n, gbwt_b200_pos* out, uint64_t* steps) {
    CheckpointView cv{};
    cv.table = table; cv.first = first; cv.seq_len = seq_len;
    for (size_t q = 0; q < n; q++) gbwt_seek(h->view, cv, shift, ids[q], indexes[q], out[q], steps[q]);
}

}  // extern "C"
