/*
 * gbwt_b200_build.h -- build a GBWT from haplotype paths on the device (libgbwt_b200.so; beyond the reference crate, which
 * has no builder: gbwt-rs src/bwt.rs:207-210. The model is the C++ GBWT's construction).
 *
 * The result is a Simple-SDS GBWT file image, the one GBWT.from_parts(<its header fields and records>).serialize() writes:
 * the header, the tags {source: jltsiren/gbwt-rs}, the BWT (Elias-Fano record starts and the records with maximal runs),
 * an empty DA-sample vector and no metadata. gbwt_b200_index_from_bytes loads it; the C++ tools and the crate read it.
 * The visits to a node are sorted by their reversed prefixes, ties at the start of a sequence broken by sequence id.
 * Header: offset = min node - 1 and alphabet_size = max node + 1 (over both orientations when bidirectional), sequences =
 * n or 2n, size = sum of (length + 1). Paths that are all empty give record 0 alone.
 *
 * How: prefix doubling of the reversed prefixes with CUB radix sorts of 32-bit ranks, then edges, runs and record bytes
 * from scans, all on the device; the host writes the file around the record bytes.
 *
 * Statuses (checked before anything is launched; the device variant checks with reductions it reads back):
 *  - GBWT_B200_E_ARGUMENT: n == 0; a null pointer with a non-empty input; offsets that decrease; node 0; node 1 when
 *    bidirectional (its flip is the endmarker).
 *  - GBWT_B200_E_RANGE: a node >= 2^32 (as in the device layout), or nodes + sequences >= 2^32.
 *  - GBWT_B200_E_CUDA: the working set does not fit the free device memory (checked before the first allocation;
 *    gbwt_b200_last_error() gives the need and the free amount), or a CUDA error.
 * Nothing stays allocated on the device after a call, whatever its status.
 *
 * Limits of this version:
 *  - ranks are 32 bits: nodes + sequences must be below 2^32;
 *  - device memory: about 36 bytes per position (nodes + sequences) and 28 bytes per record, plus the sort's temporary
 *    storage. A path set that does not fit is refused; it can be built in pieces by inserting paths into a loaded index
 *    (gbwt_b200_insert.h, included here).
 */
#ifndef GBWT_B200_BUILD_H
#define GBWT_B200_BUILD_H

#include "gbwt_b200.h"
#include "gbwt_b200_insert.h"

#ifdef __cplusplus
extern "C" {
#endif

/* A Simple-SDS GBWT image of the given paths: path q = nodes[offsets[q] .. offsets[q+1]), n paths, offsets absolute.
 * bidirectional != 0: sequence 2q = path q, 2q+1 = its reverse with every node flipped (support::reverse_path), and
 * the BIDIRECTIONAL flag; otherwise sequence q = path q. *image is allocated by the library: gbwt_b200_free().
 * info may be NULL: [0] positions sorted (nodes + sequences), [1] doubling rounds, [2] device microseconds,
 * [3] peak device bytes. */
GBWT_B200_API int gbwt_b200_build_image(const uint64_t* nodes, const uint64_t* offsets, size_t n, int bidirectional, int device,
                                        void** image, size_t* len, uint64_t info[4]);
/* The same from device arrays, read on `stream` (cudaStream_t as void*, NULL = default stream) of `device`. Blocks until
 * the image is on the host. */
GBWT_B200_API int gbwt_b200_build_image_device(const uint64_t* d_nodes, const uint64_t* d_offsets, size_t n, int bidirectional,
                                               int device, void* stream, void** image, size_t* len, uint64_t info[4]);

#ifdef __cplusplus
}
#endif
#endif /* GBWT_B200_BUILD_H */
