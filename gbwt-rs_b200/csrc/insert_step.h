// insert_step.h -- the insertion walk of insert.cu (gbwt_b200_insert_image) as one-lane host/device code, so that
// tests/hostsim can run it on the CPU against the brute-force sort keys of tests/gbwt_builder.py.
//
// An index A gets new sequences S. For an entry e of S in record w, alpha(e) is the number of A entries of w that sort
// before e. Along a new sequence x_0 .. x_{L-1} (x_{-1} = the endmarker, alpha = A's sequence count in record 0):
//   alpha(e_k) = before_A(x_k, x_{k-1}) + rank_A(x_{k-1}, alpha(e_{k-1}), x_k)
// rank_A(w, i, v) = the entries among the first i of A's record w whose successor is v (0 without a record or an edge);
// before_A(v, w) = A's entries of record v whose predecessor is below w: the offset of A's first edge u -> v with u >= w,
// len_A(v) when there is none, 0 when A has no record v. Where A has the edge w -> v, its offset is before_A(v, w), so
// the step reads w's record alone; otherwise rank_A is 0 and before_A comes from A's incoming edges.
#pragma once
#include <stdint.h>

#include "record_scan.cuh"

namespace gbwt_b200 {

// A's edges u -> v as key v << 32 | u (u = 0: the endmarker record), sorted, with the edge's offset in v's record.
struct InEdges {
    const uint64_t* keys;
    const uint32_t* offs;
    uint64_t count;
};

// A's record of node w (w = 0: the endmarker record); false when A has no such record or it is empty.
GBWT_HD bool insert_record(const IndexView& ix, uint64_t w, Desc& d) {
    if (w != 0 && (w <= ix.offset || w - ix.offset >= ix.records)) return false;
    const uint64_t rec = w == 0 ? 0 : w - ix.offset;
    if (rec >= ix.records) return false;
    d = load_desc(ix, rec);
    return d.fmt() != FMT_EMPTY;
}

// before_A(v, w), v != 0.
GBWT_HD uint64_t insert_before(const IndexView& ix, const InEdges& in, uint64_t v, uint64_t w) {
    Desc d;
    if (!insert_record(ix, v, d)) return 0;
    const uint64_t key = (v << 32) | w;
    uint64_t lo = 0, hi = in.count;
    while (lo < hi) {
        const uint64_t mid = lo + (hi - lo) / 2;
        if (in.keys[mid] < key) lo = mid + 1; else hi = mid;
    }
    if (lo < in.count && (in.keys[lo] >> 32) == v) return in.offs[lo];
    return d.total_len();
}

// alpha of the entry at v that follows the entry at w whose alpha is `alpha`.
GBWT_HD uint64_t insert_step(const IndexView& ix, const InEdges& in, uint64_t w, uint64_t alpha, uint64_t v) {
    Desc d;
    if (insert_record(ix, w, d)) {
        uint32_t rank = 0, edge_offset = 0;
        FlipSet fs;
        fs.lt = 0; fs.extra = NO_SYMBOL;
        if (find_edge<false>(ix, d, v, rank, edge_offset, fs)) {
            const uint32_t i = alpha > d.total_len() ? d.total_len() : static_cast<uint32_t>(alpha);
            return static_cast<uint64_t>(edge_offset) + rank_pair<false>(ix, d, rank, fs, i, i).at_start;
        }
    }
    return insert_before(ix, in, v, w);
}

}  // namespace gbwt_b200
