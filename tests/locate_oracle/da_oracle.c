/* da_oracle.c -- TEST-ONLY: the document array of a GBWT, built with the CPU oracle's GBWT::start / GBWT::forward
 * (oracle/gbwt_oracle.c) and nothing else, as the truth that locate is checked against. No sampling is involved.
 *
 * Position (node, i) of record r = node - alphabet_offset lies in slot first[r] + i; da_build walks every sequence s
 * from start(s) with forward and writes (s, j) into the slot of its j-th position. Built by tests/locate_oracle.py. */
#include <stdint.h>
#include <stdlib.h>

#include "../../oracle/gbwt_oracle.h"

/* first[0 .. records]: slot of the first position of every record (records without positions, the endmarker's and
 * those below first_node() have none). Returns the number of slots. */
uint64_t da_layout(const orc_gbwt* g, uint64_t* first) {
    const uint64_t records = orc_bwt_records(g), offset = orc_alphabet_offset(g), first_node = orc_first_node(g);
    uint64_t at = 0;
    for (uint64_t r = 0; r < records; r++) {
        first[r] = at;
        const int64_t len = orc_record_len(g, r);
        if (r + offset >= first_node && len > 0) at += (uint64_t)len;
    }
    first[records] = at;
    return at;
}

/* Fills seq[] / idx[] (UINT64_MAX where no sequence visits a slot). Returns 0, or -1 if a slot is visited twice, a walk
 * leaves the layout, or a walk runs longer than there are slots (the array would not be a bijection). */
int da_build(const orc_gbwt* g, const uint64_t* first, uint64_t* seq, uint64_t* idx) {
    const uint64_t records = orc_bwt_records(g), offset = orc_alphabet_offset(g), slots = first[records];
    for (uint64_t k = 0; k < slots; k++) { seq[k] = UINT64_MAX; idx[k] = UINT64_MAX; }
    for (uint64_t s = 0; s < orc_sequences(g); s++) {
        orc_pos pos;
        int some = orc_start(g, s, &pos);
        for (uint64_t j = 0; some; j++) {
            if (j >= slots || pos.node < offset) return -1;
            const uint64_t r = pos.node - offset;
            if (r >= records || pos.offset >= first[r + 1] - first[r]) return -1;
            const uint64_t k = first[r] + pos.offset;
            if (seq[k] != UINT64_MAX) return -1;
            seq[k] = s; idx[k] = j;
            orc_pos next;
            some = orc_forward(g, pos, &next);
            pos = next;
        }
    }
    return 0;
}
