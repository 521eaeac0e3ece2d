/*
 * gbwt_b200_insert.h -- insert haplotype paths into a loaded GBWT on the device (libgbwt_b200.so; beyond the reference
 * crate, which has no builder). Included by gbwt_b200_build.h; gbwt_b200.h does not include it.
 *
 * Index A has nA sequences. With n new paths P, path q adds sequence nA + 2q and its flipped reverse nA + 2q + 1 when A is
 * bidirectional, otherwise sequence nA + q. The result is a Simple-SDS GBWT image, byte for byte
 * gbwt_b200_build_image(paths(A) + P, bidirectional = A's flag), where paths(A) = A's sequences (its even sequences when
 * bidirectional):
 *  - header: sequences = nA + new sequences; size = A's size + new nodes + new sequences; offset = min(A's offset, min new
 *    node - 1); alphabet_size = max(A's, max new node + 1), over both orientations when bidirectional; A's BIDIRECTIONAL
 *    flag. These equal the build's whenever A's header is the one its nodes give (every built image and the fixtures).
 *  - written like the build: tags {source: jltsiren/gbwt-rs}, an empty DA-sample vector and no metadata. A's metadata and
 *    DA samples no longer describe the sequences, so they are dropped.
 *  - A is not modified, and answers exactly as before during and after the call.
 * Two indexes merge by passing the paths of B (gbwt_b200_extract_device) as P.
 *
 * How: the new paths are sorted alone (the build's prefix doubling); a walk along each new sequence, one lane per
 * sequence, finds where each of its visits falls among A's (the rank primitives on A's records and a table of A's
 * incoming edges); then one thread per record merges the new visits into A's runs, read in place from the device layout.
 * A's records are never expanded or re-sorted. Device memory beside A's layout: about 36 bytes per new position, about 36
 * per edge of A, a few words per record of the result and the result's bytes; none of it grows with A's length.
 *
 * Statuses (checked before anything is launched; the device variant checks with reductions it reads back):
 *  - GBWT_B200_E_ARGUMENT: a null index or pointer; n == 0; offsets that decrease; node 0; node 1 when A is bidirectional.
 *  - GBWT_B200_E_RANGE: a node >= 2^32; new nodes + new sequences >= 2^32; a record of the result of 2^32 positions or more.
 *  - GBWT_B200_E_CUDA: the working set does not fit the free device memory (gbwt_b200_last_error() gives the need and the
 *    free amount), or a CUDA error.
 * Nothing stays allocated on the device after a call, whatever its status.
 */
#ifndef GBWT_B200_INSERT_H
#define GBWT_B200_INSERT_H

#include "gbwt_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* The image of A's sequences followed by the paths: path q = nodes[offsets[q] .. offsets[q+1]), n paths, offsets absolute,
 * on the index's device. *image is allocated by the library: gbwt_b200_free(). info may be NULL: [0] new positions (nodes +
 * sequences), [1] doubling rounds, [2] device microseconds, [3] peak device bytes, [4] the longest new sequence (the
 * walk's dependent chain), [5] microseconds of the insertion walk. */
GBWT_B200_API int gbwt_b200_insert_image(const gbwt_b200_index* index, const uint64_t* nodes, const uint64_t* offsets, size_t n,
                                         void** image, size_t* len, uint64_t info[6]);
/* The same from device arrays on the index's device, read on `stream` (cudaStream_t as void*, NULL = default stream).
 * Blocks until the image is on the host. */
GBWT_B200_API int gbwt_b200_insert_image_device(const gbwt_b200_index* index, const uint64_t* d_nodes, const uint64_t* d_offsets, size_t n,
                                                void* stream, void** image, size_t* len, uint64_t info[6]);

#ifdef __cplusplus
}
#endif
#endif /* GBWT_B200_INSERT_H */
