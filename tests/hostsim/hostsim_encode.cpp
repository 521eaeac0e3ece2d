// hostsim_encode.cpp -- TEST-ONLY: the record encoder of record_encode.h (shared by the host writer and the device builder)
// compiled for the CPU, so tests/test_hostsim_encode.py can compare it with tests/gbwt_builder.py without a GPU.
#include <cstdint>

#include "../../gbwt-rs_b200/csrc/record_encode.h"

using namespace gbwt_b200;

// Record = sigma edges (node, offset) and `runs` runs (value, length), as uint64 pairs; out == nullptr counts the bytes.
extern "C" uint64_t he_encode_record(const uint64_t* edges, uint64_t sigma, const uint64_t* runs, uint64_t count, uint8_t* out) {
    ByteSink sink;
    sink.at = out;
    put_edges(sink, sigma, [&](uint64_t e) { return EdgeValue{edges[2 * e], edges[2 * e + 1]}; });
    for (uint64_t r = 0; r < count; r++) put_run(sink, sigma, runs[2 * r], runs[2 * r + 1]);
    return sink.n;
}
