// msfm_internal.h — entry points shared between the translation units of libmsfm_match.so (not exported, not part of the
// C ABI): what the multi-GPU engine (msfm_multi.cc) needs from the single-GPU context beyond include/msfm_match.h.
#pragma once
#include <cuda_runtime.h>

#include "../../include/msfm_match.h"

#define MSFM_HIDDEN __attribute__((visibility("hidden")))

extern "C" {

// Destination of one batch's matches: called once per batch, after the per-pair counts are known, with the index of the
// batch's first match in the call's concatenated list.  Returns 0 and the host pointers the batch is copied to (good may
// come back null: flags not wanted), or non-zero when there is no room.
typedef int (*msfm_sink_fn)(void *user, int64_t first_match, int64_t n_matches, int32_t (**matches)[2], uint8_t **good);

// msfm_match_pairs with the match buffers supplied batch by batch through `sink` (offsets [n_pairs + 1] and ok [n_pairs]
// are plain host arrays).
MSFM_HIDDEN msfm_status msfm_internal_match_pairs_sink(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const msfm_params *params,
                                                       int64_t *offsets, int32_t *ok, int want_good, msfm_sink_fn sink, void *user);
// The images become usable once the work queued on `stream` so far has completed (a collective wrote their rows there):
// leaves an upload mark recorded on that stream.
MSFM_HIDDEN msfm_status msfm_internal_mark_on_stream(msfm_ctx *ctx, int32_t n, const int32_t *image_ids, cudaStream_t stream);

}  // extern "C"
