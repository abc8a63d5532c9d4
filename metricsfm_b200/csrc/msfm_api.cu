// msfm_api.cu — implementation of the C ABI declared in include/msfm_match.h.
//
// Host side of the B200-native matcher: the packed descriptor table (HBM arena + per-image TMA tensor maps), the
// per-batch work-list builder / pair scheduler for one GPU, and the launch sequence
//   match_pairs_kernel (tcgen05)  ->  finalize_kernel  ->  scan_counts_kernel  ->  gather_matches_kernel  ->  D2H.
// There is deliberately no CPU or non-sm_100 fallback: msfm_create fails with MSFM_ERR_UNSUPPORTED elsewhere.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <type_traits>
#include <vector>

#include <cuda.h>
#include <cuda_runtime.h>

#include "../../include/msfm_match.h"
#include "aux_kernels.cuh"
#include "geo_kernels.cuh"
#include "match_kernel.cuh"
#include "msfm_internal.h"

namespace {

using msfm::kAlignRows;
using msfm::kDim;
using msfm::PairDesc;
using msfm::WorkItem;

// Kernel configuration of this build (see DESIGN.md §kernels).
constexpr int kStrips = 4;   // query strips (128 rows each) per work item
constexpr int kTileN = 64;   // reference rows per tile (UMMA N)
constexpr int kStages = 8;   // B-tile ring depth
constexpr int kTbufs = 2;    // TMEM accumulator buffers per strip
using KCfg = msfm::MatchKernelCfg<kStrips, kTileN, kStages, kTbufs>;
constexpr int kItemRows = kStrips * msfm::kStripRows;

// The instantiations of the matching kernel, (DEBUG, COLLECT, GATE): every combination but a debug build of the
// collect pass, for which `debug` is ignored.
using MatchKernelFn = void (*)(msfm::MatchKernelParams);
using msfm::GateKind;
template <bool DEBUG, bool COLLECT>
MatchKernelFn match_kernel(GateKind gate) {
    if (gate == GateKind::none) return msfm::match_pairs_kernel<kStrips, kTileN, kStages, kTbufs, DEBUG, COLLECT, GateKind::none>;
    if (gate == GateKind::epipolar) return msfm::match_pairs_kernel<kStrips, kTileN, kStages, kTbufs, DEBUG, COLLECT, GateKind::epipolar>;
    return msfm::match_pairs_kernel<kStrips, kTileN, kStages, kTbufs, DEBUG, COLLECT, GateKind::homography>;
}
MatchKernelFn match_kernel(bool debug, bool collect, GateKind gate) {
    return collect ? match_kernel<false, true>(gate) : debug ? match_kernel<true, false>(gate) : match_kernel<false, false>(gate);
}

// Per-batch scratch bounds (rows).  16 Mi query rows -> 256 MiB kNN scratch + 128 MiB match scratch.
constexpr int64_t kBatchMaxQueryRows = 16ll << 20;
constexpr int64_t kBatchMaxQueryRowsMutual = 16ll << 20;  // mutual: + 128 B of gathered candidate row per query row
constexpr int64_t kBatchMaxPairs = 16384;
constexpr int64_t kBatchMaxRefRows = 16ll << 20;  // mutual: 8 B of column table per reference row of the batch
// msfm_knn2_pairs exact mode: every query row goes through the collect pass (~10 events per row on unit-norm SIFT at
// 8192 rows, p99 28), so its batches are smaller and its event list holds 16 events per row: 1 Mi rows -> 16 Mi events
// x 24 B = 400 MB.  An overflow stays correct (brute force) but must not be the common case.
constexpr int64_t kBatchMaxQueryRowsExact = 1ll << 20;
constexpr int64_t kExactEventsPerRow = 16;

struct DeviceBuf {
    void *ptr = nullptr;
    size_t bytes = 0;
};

struct ImageSlot {
    bool present = false;
    bool has_float = false;  // float rows retained (keep_float context, msfm_upload_f32)
    float scale = 0.0f;      // quantisation scale of the float upload
    int32_t rows = 0;
    int32_t rows_padded = 0;
    int64_t off = 0;
    uint64_t ready_seq = 0;  // upload mark that covers this image (0: its rows were in place when the upload call returned)
};

struct UploadMark {
    uint64_t seq;
    cudaEvent_t ev;
};

struct Extent {
    int64_t off, rows;
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

}  // namespace

struct msfm_ctx {
    int device = 0;
    int num_sms = 0;
    cudaStream_t stream = nullptr;         // matching: plans, kernels, result copies
    cudaStream_t upload_stream = nullptr;  // table changes: packer launches, tensor maps, pad rows (overlaps matching)
    cudaStream_t copy_stream = nullptr;    // host->device copies of every table upload: they never queue behind a packer
                                           // launch that is waiting for an SM (the matching kernel is persistent)
    cudaEvent_t ev_copy = nullptr;
    cudaStream_t d2h_stream = nullptr;     // match lists of batch k go back to the host under batch k+1's kernels
    cudaEvent_t ev_d2h0 = nullptr, ev_d2h1 = nullptr;  // brackets of the list copy in flight (timed)
    bool d2h_in_flight = false;
    struct StageBuf { void *ptr; size_t bytes; cudaEvent_t done; };
    std::vector<StageBuf> stage_pool;      // float rows of plain-context msfm_upload_f32* calls, until their packers have run
    std::vector<UploadMark> marks;         // asynchronous uploads still to be ordered before matching launches
    std::vector<cudaEvent_t> event_pool;
    uint64_t upload_seq = 0, waited_seq = 0;
    int32_t max_images = 0;
    int64_t arena_rows = 0;
    int64_t rows_high_water = 0;  // bump pointer
    std::vector<Extent> free_list;
    uint8_t *desc = nullptr;
    int32_t *norms = nullptr;  // column-key arena: ckey = -8*||row||^2 + (7 - row%8), see match_kernel.cuh
    float *fdesc = nullptr;    // keep_float: the callers' float rows, same row offsets as `desc` (512 B per row)
    float *resid = nullptr;    // keep_float: quantisation residual ||scale*x - q|| per row (pack_f32_kernel), same offsets
    float *img_rmax = nullptr; // keep_float: [max_images] largest residual per image (0 after release)
    bool own_arena = false;
    CUtensorMap *d_maps = nullptr;
    CUtensorMap *h_maps = nullptr;  // pinned mirror of d_maps: tensor maps are uploaded without a host sync
    std::vector<ImageSlot> images;
    EncodeTiledFn encode = nullptr;

    DeviceBuf dbg_stats;  // debug flag 8: per-phase cycle counters of the matching kernel, dumped at destroy
    DeviceBuf cand_q, cand_j, cand_d0, cand_good, cand_counts, cand_desc, cand_ckeys;  // one-way candidates + gathered rows
    DeviceBuf tilemin;       // per reference tile: smallest squared norm (tile_min_kernel, refreshed per batch)
    DeviceBuf colbest, twin_counts;  // mutual check: per-pair column table (nearest claimant per reference row); [n_pairs] + routed word
    DeviceBuf band_q, band_counts;  // float regime: query rows near a ratio threshold, per pair
    DeviceBuf band_thr, band_state, band_events, band_event_keys, band_event_count;  // ... and the collect pass over them
    int64_t band_event_cap_override = -1;  // msfm_test_set_band_event_cap (tests: 0 forces the brute-force fallback)
    DeviceBuf knn_ids, knn_dists, knn_ids_b, knn_dists_b;  // msfm_knn2_pairs: FLANN-layout rows of a batch (two sets, see match_pairs_impl)
    int64_t knn_events = 0;         // last exact-mode msfm_knn2_pairs or re-scoring msfm_match_pairs: events scored by
    int32_t knn_brute_batches = 0;  // the collect path, and batches whose event list overflowed (brute force)
    bool force_twin = false;               // msfm_test_force_twin_pass
    bool no_prune = false;                 // msfm_test_disable_pruning: the forward pass keeps exact 2-NN rows for every query row
    DeviceBuf kp_xy;                       // msfm_match_pairs_guided: keypoints (x, y) per arena row (allocated on the first call)
    DeviceBuf knn, matches, good, counts, offsets, pairdesc, items, tight_matches, tight_good;
    DeviceBuf tight_matches_b, tight_good_b;  // second set: a batch's lists are copied out while the next batch is gathered
    void *h_pinned = nullptr;
    size_t h_pinned_bytes = 0;
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr, ev_k0 = nullptr, ev_k1 = nullptr, ev_k2 = nullptr, ev_k3 = nullptr,
                ev_f1 = nullptr;

    int64_t routed_index = 0;  // the routed word (pairs routed to the twin pass) sits after the per-pair twin counts
    msfm_timing timing{};
    uint32_t debug_flags = 0;  // MSFM_DEBUG_FLAGS environment variable (timing experiments)
    std::string err;
    std::mutex mu;
};

namespace {

msfm_status fail(msfm_ctx *ctx, msfm_status st, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    return st;
}

#define MSFM_CUDA(ctx, call)                                                                                   \
    do {                                                                                                       \
        cudaError_t e__ = (call);                                                                              \
        if (e__ != cudaSuccess)                                                                                \
            return fail(ctx, e__ == cudaErrorMemoryAllocation ? MSFM_ERR_OUT_OF_MEMORY : MSFM_ERR_CUDA,         \
                        "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__);          \
    } while (0)

msfm_status ensure(msfm_ctx *ctx, DeviceBuf &b, size_t bytes) {
    if (b.bytes >= bytes && b.ptr) return MSFM_OK;
    if (b.ptr) {
        MSFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        MSFM_CUDA(ctx, cudaFree(b.ptr));
        b.ptr = nullptr;
        b.bytes = 0;
    }
    size_t want = std::max<size_t>(bytes, 256);
    MSFM_CUDA(ctx, cudaMalloc(&b.ptr, want));
    b.bytes = want;
    return MSFM_OK;
}

msfm_status ensure_pinned(msfm_ctx *ctx, size_t bytes) {
    if (ctx->h_pinned_bytes >= bytes) return MSFM_OK;
    if (ctx->h_pinned) {
        MSFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        MSFM_CUDA(ctx, cudaFreeHost(ctx->h_pinned));
        ctx->h_pinned = nullptr;
        ctx->h_pinned_bytes = 0;
    }
    MSFM_CUDA(ctx, cudaMallocHost(&ctx->h_pinned, bytes));
    ctx->h_pinned_bytes = bytes;
    return MSFM_OK;
}

int64_t round_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

// First-fit over the free list, else bump.  Extents are multiples of kAlignRows.
bool arena_alloc(msfm_ctx *ctx, int64_t rows_padded, int64_t *off) {
    for (size_t i = 0; i < ctx->free_list.size(); ++i) {
        Extent &e = ctx->free_list[i];
        if (e.rows >= rows_padded) {
            *off = e.off;
            e.off += rows_padded;
            e.rows -= rows_padded;
            if (e.rows == 0) ctx->free_list.erase(ctx->free_list.begin() + i);
            return true;
        }
    }
    if (ctx->rows_high_water + rows_padded > ctx->arena_rows) return false;
    *off = ctx->rows_high_water;
    ctx->rows_high_water += rows_padded;
    return true;
}

void arena_free(msfm_ctx *ctx, int64_t off, int64_t rows_padded) {
    if (rows_padded <= 0) return;
    ctx->free_list.push_back({off, rows_padded});
    std::sort(ctx->free_list.begin(), ctx->free_list.end(), [](const Extent &a, const Extent &b) { return a.off < b.off; });
    std::vector<Extent> merged;
    for (const Extent &e : ctx->free_list) {
        if (!merged.empty() && merged.back().off + merged.back().rows == e.off) merged.back().rows += e.rows;
        else merged.push_back(e);
    }
    if (!merged.empty() && merged.back().off + merged.back().rows == ctx->rows_high_water) {
        ctx->rows_high_water = merged.back().off;
        merged.pop_back();
    }
    ctx->free_list.swap(merged);
}

// 2-D tensor map over `rows` packed rows at `base`: inner dim 128 bytes, outer dim = exact row count, so that TMA
// zero-fills rows past the end (ragged sizes need no masking of the operands); 64-row boxes, 128-byte swizzle.
CUresult encode_row_map(const msfm_ctx *ctx, void *base, int64_t rows, CUtensorMap *m) {
    memset(m, 0, sizeof *m);
    cuuint64_t dims[2] = {(cuuint64_t)kDim, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)kDim};
    cuuint32_t box[2] = {(cuuint32_t)kDim, (cuuint32_t)msfm::kBoxRows};
    cuuint32_t estr[2] = {1u, 1u};
    return ctx->encode(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                       CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}

// One tensor map per image, in the image's slot.
msfm_status write_tensor_map(msfm_ctx *ctx, int32_t image_id, int64_t off, int32_t rows) {
    CUtensorMap m;
    const CUresult r = encode_row_map(ctx, ctx->desc + off * kDim, std::max(rows, 1), &m);
    if (r != CUDA_SUCCESS) return fail(ctx, MSFM_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    // The pinned slot of this image may still be in flight from an earlier upload of the same id (release + re-upload):
    // copies on one stream execute in order, and the slot is only rewritten after msfm_release* synchronised the streams.
    ctx->h_maps[image_id] = m;
    MSFM_CUDA(ctx, cudaMemcpyAsync(ctx->d_maps + image_id, ctx->h_maps + image_id, sizeof m, cudaMemcpyHostToDevice, ctx->upload_stream));
    return MSFM_OK;
}

msfm_status check_image_id(msfm_ctx *ctx, int32_t id, bool must_exist) {
    if (id < 0 || id >= ctx->max_images) return fail(ctx, MSFM_ERR_INVALID_ARG, "image id %d outside [0, %d)", id, ctx->max_images);
    if (must_exist && !ctx->images[id].present) return fail(ctx, MSFM_ERR_NOT_FOUND, "image id %d has not been uploaded", id);
    return MSFM_OK;
}

// Every pair of a caller's list names two uploaded images.
msfm_status check_pairs(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs) {
    msfm_status st;
    for (int64_t i = 0; i < n_pairs; ++i) {
        if ((st = check_image_id(ctx, pairs[i].ref, true)) != MSFM_OK) return st;
        if ((st = check_image_id(ctx, pairs[i].query, true)) != MSFM_OK) return st;
    }
    return MSFM_OK;
}

// Upload marks whose event the main stream has waited for (or that a synchronisation has overtaken) go back to the pool.
void recycle_marks(msfm_ctx *ctx) {
    for (const UploadMark &m : ctx->marks) ctx->event_pool.push_back(m.ev);
    ctx->marks.clear();
    ctx->waited_seq = ctx->upload_seq;
}

// Order the main stream behind the upload mark `need` and every older one.
msfm_status wait_for_uploads(msfm_ctx *ctx, uint64_t need) {
    if (need <= ctx->waited_seq) return MSFM_OK;
    size_t k = 0;
    for (; k < ctx->marks.size(); ++k) {
        if (ctx->marks[k].seq > need) break;
        // marks can sit on different streams (uploads, a collective's stream): wait for each one not yet ordered
        MSFM_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->marks[k].ev, 0));
        ctx->event_pool.push_back(ctx->marks[k].ev);  // recorded and waited for: reusable in stream order
    }
    ctx->marks.erase(ctx->marks.begin(), ctx->marks.begin() + k);
    ctx->waited_seq = need;
    return MSFM_OK;
}

// Have the asynchronous uploads up to mark `need` finished?  (Host-side query; used to size batches, never for ordering.)
bool uploads_landed(msfm_ctx *ctx, uint64_t need) {
    if (need <= ctx->waited_seq) return true;
    for (const UploadMark &m : ctx->marks)
        if (m.seq <= need && cudaEventQuery(m.ev) != cudaSuccess) return false;
    return true;
}

msfm_status reserve_locked(msfm_ctx *ctx, int32_t image_id, int32_t rows, int64_t *row_offset) {
    msfm_status st = check_image_id(ctx, image_id, false);
    if (st != MSFM_OK) return st;
    if (rows < 0 || rows > MSFM_MAX_ROWS_PER_IMAGE) return fail(ctx, MSFM_ERR_INVALID_ARG, "rows %d outside [0, %d]", rows, MSFM_MAX_ROWS_PER_IMAGE);
    if (ctx->images[image_id].present) return fail(ctx, MSFM_ERR_EXISTS, "image id %d already uploaded", image_id);
    const int64_t padded = round_up(std::max(rows, 1), kAlignRows);
    int64_t off = 0;
    if (!arena_alloc(ctx, padded, &off))
        return fail(ctx, MSFM_ERR_CAPACITY, "descriptor arena full: need %lld rows, %lld of %lld in use", (long long)padded,
                    (long long)ctx->rows_high_water, (long long)ctx->arena_rows);
    ImageSlot &s = ctx->images[image_id];
    s.present = true;
    s.rows = rows;
    s.rows_padded = (int32_t)padded;
    s.off = off;
    st = write_tensor_map(ctx, image_id, off, rows);
    if (st != MSFM_OK) {
        s.present = false;
        arena_free(ctx, off, padded);
        return st;
    }
    if (row_offset) *row_offset = off;
    return MSFM_OK;
}

struct BatchPlan {
    std::vector<PairDesc> pairs;     // forward pair descriptors (only pairs with min_keypoints rows on both sides)
    std::vector<PairDesc> twins;     // mutual cross-check: candidate rows of pair p searched against its query image
    std::vector<int64_t> src_index;  // index into the caller's pair list
    std::vector<WorkItem> items;     // forward work items
    std::vector<WorkItem> twin_items;
    std::vector<PairDesc> band_twins;  // float regime: band rows of pair p searched against its reference image (collect mode)
    std::vector<WorkItem> band_items;
    bool rescoring = false;          // the caller asked for fp32 re-scoring and the context keeps float rows
    int64_t query_rows = 0;          // forward kNN rows (= candidate / match scratch rows)
    int64_t ref_rows = 0;            // sum of reference rows (= entries of the mutual check's column table)
    int64_t row_lo = INT64_MAX, row_hi = 0;  // arena rows spanned by the batch's images (tile_min_kernel's range)
    uint64_t need_seq = 0;           // newest upload mark among the batch's images
    bool big_ref = false;            // some reference image's column table does not fit in shared memory
    int64_t ops = 0;
    bool mutual = false;
    uint32_t prune_q8 = msfm::kNoPrune;  // forward pass: dead-row rule of the matching kernel (match_kernel.cuh); off = exact 2-NN rows
    bool has_empty = false;          // some pair has no work items: its kNN rows must read "absent"
    bool any_float = false;          // some pair has retained float rows on both sides (rescoring possible)
    std::vector<float> fmat;         // guided call: F (or H) of every forward pair, 9 floats each (uploaded after the
                                     // descriptors)
    msfm::EpiGate gate{};            // guided call: keypoints and t2 from the carve, the F table's device address from
                                     // run_match_stage
    GateKind gate_kind = GateKind::none;  // what the table in gate.fmat holds and which test the matching kernel applies
    const msfm::EpiGate *epi_gate() const { return gate.fmat ? &gate : nullptr; }  // null: ungated
    int64_t knn_rows() const { return mutual ? 2 * query_rows : query_rows; }
};

// The passes of the matching kernel over a batch's work items [first_item, first_item + n_items):
//   forward  2-NN of the forward pairs' query rows, with the dead-row rule `value` (prune_q8)
//   twin     2-NN of the mutual twins' candidate rows, skipped on the device unless select_candidates_kernel routed a pair
//   collect  the items are band twins: every reference row within band_thr of a band row is appended to the event list,
//            which holds `value` events
// A guided plan's gate bars the elements that fail it in every pass.
enum class Pass { forward, twin, collect };

msfm_status launch_match_kernel(msfm_ctx *ctx, Pass pass, size_t first_item, size_t n_items, uint32_t value,
                                const BatchPlan &plan) {
    const bool collect = pass == Pass::collect, twin = pass == Pass::twin;
    const msfm::EpiGate *gate = plan.epi_gate();
    msfm::MatchKernelParams kp;
    kp.maps = ctx->d_maps;
    kp.ckeys = ctx->norms;
    kp.tilemin = static_cast<const int4 *>(ctx->tilemin.ptr);
    kp.cand_ckeys = static_cast<const int32_t *>(ctx->cand_ckeys.ptr);
    kp.cand_d0 = static_cast<const int32_t *>(collect ? ctx->band_thr.ptr : ctx->cand_d0.ptr);
    kp.counts = static_cast<const int32_t *>(collect ? ctx->band_counts.ptr : ctx->twin_counts.ptr);
    kp.pairs = static_cast<const PairDesc *>(ctx->pairdesc.ptr);
    kp.items = static_cast<const WorkItem *>(ctx->items.ptr) + first_item;
    kp.n_items = (int32_t)n_items;
    if (collect) {
        kp.event_cap = value;
        kp.event_count = static_cast<unsigned int *>(ctx->band_event_count.ptr);
        kp.events = static_cast<int4 *>(ctx->band_events.ptr);
    } else {
        kp.debug_flags = ctx->debug_flags;
        kp.stats = static_cast<unsigned long long *>(ctx->dbg_stats.ptr);  // null unless MSFM_DEBUG_FLAGS & 8
        kp.knn = static_cast<int4 *>(ctx->knn.ptr);
    }
    kp.xy = gate ? gate->xy : nullptr;
    kp.fmat = gate ? gate->fmat : nullptr;
    kp.src_row = static_cast<const int32_t *>(collect ? ctx->band_q.ptr : ctx->cand_j.ptr);
    // mutual twin pass: the launch returns at once unless select_candidates_kernel routed some pair to it
    kp.routed = twin ? reinterpret_cast<const unsigned int *>(static_cast<const int32_t *>(ctx->twin_counts.ptr) + ctx->routed_index) : nullptr;
    kp.prune_q8 = (pass == Pass::forward && !ctx->no_prune) ? value : msfm::kNoPrune;
    kp.t2 = gate ? gate->t2 : 0.0f;
    const int grid = std::max(1, std::min<int>(ctx->num_sms, kp.n_items));
    match_kernel(ctx->debug_flags != 0, collect, gate ? plan.gate_kind : GateKind::none)<<<grid, KCfg::kThreads, KCfg::kSmemAlloc, ctx->stream>>>(kp);
    MSFM_CUDA(ctx, cudaGetLastError());
    ctx->timing.match_launches += 1;
    ctx->timing.total_launches += 1;
    return MSFM_OK;
}

// The candidate scratch "image" (gathered reference rows of the one-way matches) and its tensor map, which lives in
// the slot after the last image.
msfm_status ensure_cand_scratch(msfm_ctx *ctx, int64_t rows) {
    msfm_status st;
    if ((st = ensure(ctx, ctx->cand_ckeys, (size_t)rows * 4)) != MSFM_OK) return st;
    if (ctx->cand_desc.ptr && ctx->cand_desc.bytes >= (size_t)rows * kDim) return MSFM_OK;
    if ((st = ensure(ctx, ctx->cand_desc, (size_t)rows * kDim)) != MSFM_OK) return st;
    CUtensorMap m;
    const CUresult r = encode_row_map(ctx, ctx->cand_desc.ptr, (int64_t)(ctx->cand_desc.bytes / kDim), &m);
    if (r != CUDA_SUCCESS) return fail(ctx, MSFM_ERR_CUDA, "cuTensorMapEncodeTiled (candidate scratch) failed with CUresult %d", (int)r);
    MSFM_CUDA(ctx, cudaMemcpyAsync(ctx->d_maps + ctx->max_images, &m, sizeof m, cudaMemcpyHostToDevice, ctx->stream));
    MSFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return MSFM_OK;
}

// Complete the batch: twin descriptors (one per forward pair) and their work items.  Twin p searches the gathered
// candidate rows of pair p (rows [knn_off, knn_off + count_p) of the candidate scratch, count known only on the device)
// against pair p's query image; its kNN rows mirror the forward region, shifted by query_rows.
void finish_plan(msfm_ctx *ctx, BatchPlan &plan) {
    const int32_t nb = (int32_t)plan.pairs.size();
    if (plan.rescoring && plan.any_float) {
        // Band twins: the query rows of pair p that sit near a ratio threshold (gathered into rows [knn_off, knn_off +
        // band_count_p) of the candidate scratch by mark_band_kernel) against pair p's reference image, collect mode.
        const int32_t base = nb + (plan.mutual ? nb : 0);
        for (int32_t pi = 0; pi < nb; ++pi) {
            const PairDesc &f = plan.pairs[pi];
            PairDesc tw = f;
            tw.qry_img = ctx->max_images;  // candidate scratch map
            tw.qry_off = f.knn_off;        // row in cand_ckeys / band_thr
            tw.knn_off = 0;                // collect mode writes events, not kNN rows
            tw.qry_row_base = (int32_t)f.knn_off;
            tw.cand_idx = pi;
            tw.fscale2 = 0.0f;
            plan.band_twins.push_back(tw);
        }
        // items that can actually hold band rows (low row0) first, the mostly empty tail last
        for (int32_t row0 = 0, any = 1; any; row0 += kItemRows) {
            any = 0;
            for (int32_t pi = 0; pi < nb; ++pi) {
                const PairDesc &f = plan.pairs[pi];
                if (f.ref_rows > 0 && f.fscale2 > 0.0f && row0 < f.qry_rows) { plan.band_items.push_back({base + pi, row0}); any = 1; }
            }
        }
    }
    if (!plan.mutual) return;
    plan.twins.reserve(nb);
    for (int32_t pi = 0; pi < nb; ++pi) {
        const PairDesc &f = plan.pairs[pi];
        PairDesc tw;
        tw.ref_img = f.qry_img;
        tw.qry_img = ctx->max_images;  // candidate scratch map
        tw.ref_rows = f.qry_rows;
        tw.qry_rows = f.qry_rows;      // upper bound; the device reads counts[cand_idx]
        tw.ref_off = f.qry_off;
        tw.qry_off = f.knn_off;        // row in cand_ckeys
        tw.knn_off = plan.query_rows + f.knn_off;
        tw.qry_row_base = (int32_t)f.knn_off;
        tw.cand_idx = pi;
        tw.fscale2 = 0.0f;
        tw.pad_ = 0;
        tw.col_off = 0;
        plan.twins.push_back(tw);
    }
    // items that can actually hold candidates (low row0) first, the mostly empty tail last: balances the persistent CTAs
    plan.twin_items.reserve(plan.items.size());
    for (int32_t row0 = 0, any = 1; any; row0 += kItemRows) {
        any = 0;
        for (int32_t pi = 0; pi < nb; ++pi) {
            const PairDesc &f = plan.pairs[pi];
            if (f.ref_rows > 0 && row0 < f.qry_rows) { plan.twin_items.push_back({nb + pi, row0}); any = 1; }
        }
    }
}

// Upload the plan and run the forward matching launch (timed); leaves the kNN rows in scratch.  A guided plan's F table
// travels behind the pair descriptors, and its address completes plan.gate.
msfm_status run_match_stage(msfm_ctx *ctx, BatchPlan &plan) {
    msfm_status st;
    const size_t fw_bytes = plan.pairs.size() * sizeof(PairDesc);
    const size_t tw_bytes = plan.twins.size() * sizeof(PairDesc), bt_bytes = plan.band_twins.size() * sizeof(PairDesc);
    const size_t f_bytes = plan.fmat.size() * sizeof(float);
    const size_t pd_bytes = fw_bytes + tw_bytes + bt_bytes + f_bytes;
    const size_t it_fw = plan.items.size() * sizeof(WorkItem);
    const size_t it_tw = (plan.twin_items.size() + plan.band_items.size()) * sizeof(WorkItem);
    // both parts padded to whole 16-byte words for the pull kernel
    const size_t pd_pad = (pd_bytes + 15) / 16 * 16, it_pad = (it_fw + it_tw + 15) / 16 * 16;
    if ((st = ensure(ctx, ctx->pairdesc, pd_pad)) != MSFM_OK) return st;
    if ((st = ensure(ctx, ctx->items, it_pad)) != MSFM_OK) return st;
    if ((st = ensure(ctx, ctx->knn, (size_t)plan.knn_rows() * sizeof(int4))) != MSFM_OK) return st;
    if ((st = ensure(ctx, ctx->cand_counts, plan.pairs.size() * 4)) != MSFM_OK) return st;
    if ((st = ensure_pinned(ctx, pd_pad + it_pad + 64)) != MSFM_OK) return st;
    if ((st = wait_for_uploads(ctx, plan.need_seq)) != MSFM_OK) return st;  // asynchronous uploads of the batch's images
    // the pinned staging area is reused per batch: the previous batch has been synchronised by its D2H
    char *hp = static_cast<char *>(ctx->h_pinned);
    memcpy(hp, plan.pairs.data(), fw_bytes);
    if (tw_bytes) memcpy(hp + fw_bytes, plan.twins.data(), tw_bytes);
    if (bt_bytes) memcpy(hp + fw_bytes + tw_bytes, plan.band_twins.data(), bt_bytes);
    if (f_bytes) memcpy(hp + fw_bytes + tw_bytes + bt_bytes, plan.fmat.data(), f_bytes);
    plan.gate.fmat = f_bytes ? reinterpret_cast<const float *>(static_cast<const char *>(ctx->pairdesc.ptr) + fw_bytes + tw_bytes + bt_bytes) : nullptr;
    memcpy(hp + pd_pad, plan.items.data(), it_fw);
    if (!plan.twin_items.empty()) memcpy(hp + pd_pad + it_fw, plan.twin_items.data(), plan.twin_items.size() * sizeof(WorkItem));
    if (!plan.band_items.empty())
        memcpy(hp + pd_pad + it_fw + plan.twin_items.size() * sizeof(WorkItem), plan.band_items.data(), plan.band_items.size() * sizeof(WorkItem));
    {   // pulled by the SMs, not queued on the copy engine behind bulk uploads (see pull_plan_kernel)
        const size_t n16 = (pd_pad + it_pad) / 16;
        const int blocks = (int)std::max<size_t>(1, std::min<size_t>((size_t)ctx->num_sms, (n16 + 255) / 256));
        msfm::pull_plan_kernel<<<blocks, 256, 0, ctx->stream>>>(reinterpret_cast<const uint4 *>(hp), static_cast<uint4 *>(ctx->pairdesc.ptr), pd_pad / 16,
                                                               static_cast<uint4 *>(ctx->items.ptr), it_pad / 16);
        MSFM_CUDA(ctx, cudaGetLastError());
        ctx->timing.total_launches += 1;
    }
    if (plan.has_empty) MSFM_CUDA(ctx, cudaMemsetAsync(ctx->knn.ptr, 0xFF, (size_t)plan.query_rows * sizeof(int4), ctx->stream));
    if (plan.row_hi > plan.row_lo) {  // smallest norm per reference tile, over the arena rows this batch can touch
        if ((st = ensure(ctx, ctx->tilemin, (size_t)(ctx->arena_rows / msfm::kKeyTileRows + 1) * sizeof(int4))) != MSFM_OK) return st;
        const int64_t tile0 = plan.row_lo / msfm::kKeyTileRows, tile1 = (plan.row_hi + msfm::kKeyTileRows - 1) / msfm::kKeyTileRows;
        msfm::tile_min_kernel<<<(unsigned)((tile1 - tile0 + 7) / 8), 256, 0, ctx->stream>>>(ctx->norms, static_cast<int4 *>(ctx->tilemin.ptr), tile0, tile1 - tile0);
        MSFM_CUDA(ctx, cudaGetLastError());
        ctx->timing.total_launches += 1;
    }
    MSFM_CUDA(ctx, cudaEventRecord(ctx->ev_k0, ctx->stream));
    if (!plan.items.empty() && (st = launch_match_kernel(ctx, Pass::forward, 0, plan.items.size(), plan.prune_q8, plan)) != MSFM_OK) return st;
    MSFM_CUDA(ctx, cudaEventRecord(ctx->ev_k1, ctx->stream));
    ctx->timing.int8_ops += plan.ops;
    return MSFM_OK;
}

void plan_add_pair(msfm_ctx *ctx, BatchPlan &plan, int64_t src, int32_t ref, int32_t qry) {
    const ImageSlot &r = ctx->images[ref], &q = ctx->images[qry];
    PairDesc pd;
    pd.ref_img = ref;
    pd.qry_img = qry;
    pd.ref_rows = r.rows;
    pd.qry_rows = q.rows;
    pd.ref_off = r.off;
    pd.qry_off = q.off;
    pd.knn_off = plan.query_rows;
    pd.qry_row_base = 0;
    pd.cand_idx = -1;
    pd.fscale2 = (r.has_float && q.has_float && r.scale == q.scale) ? r.scale * r.scale : 0.0f;
    pd.pad_ = 0;
    pd.col_off = plan.ref_rows;
    if (r.rows > msfm::kSmemTableRows) plan.big_ref = true;
    plan.need_seq = std::max(plan.need_seq, std::max(r.ready_seq, q.ready_seq));
    plan.row_lo = std::min(plan.row_lo, std::min<int64_t>(r.off, q.off));
    plan.row_hi = std::max(plan.row_hi, std::max<int64_t>(r.off + r.rows, q.off + q.rows));
    if (pd.fscale2 > 0.0f) plan.any_float = true;
    const int32_t pidx = (int32_t)plan.pairs.size();
    plan.pairs.push_back(pd);
    plan.src_index.push_back(src);
    const bool work = r.rows > 0 && q.rows > 0;
    if (!work) plan.has_empty = true;
    if (work)
        for (int32_t row0 = 0; row0 < q.rows; row0 += kItemRows) plan.items.push_back({pidx, row0});
    plan.query_rows += q.rows;
    plan.ref_rows += r.rows;
    plan.ops += 2ll * r.rows * q.rows * kDim;
}

// Host wait for the list copy in flight (if any); its duration goes to timing.d2h_ms.
msfm_status wait_list_copy(msfm_ctx *ctx) {
    if (!ctx->d2h_in_flight) return MSFM_OK;
    ctx->d2h_in_flight = false;
    MSFM_CUDA(ctx, cudaEventSynchronize(ctx->ev_d2h1));
    float ms = 0.f;
    MSFM_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev_d2h0, ctx->ev_d2h1));
    ctx->timing.d2h_ms += ms;
    return MSFM_OK;
}

// A list copy still in flight when a call fails half-way must not outlive the call: the caller may free the
// destination buffers as soon as it sees the error.  (On success wait_list_copy has already cleared the flag.)
struct DrainListCopy {
    msfm_ctx *c;
    ~DrainListCopy() {
        if (c->d2h_in_flight) {
            cudaStreamSynchronize(c->d2h_stream);
            c->d2h_in_flight = false;
        }
    }
};

// Start copying a batch's result arrays to the host on the list-copy stream, behind the batch's last kernel (ev_f1).  The
// second range is skipped when it is empty.  wait_list_copy waits for the copy.
msfm_status start_list_copy(msfm_ctx *ctx, void *dst0, const void *src0, size_t bytes0, void *dst1, const void *src1, size_t bytes1) {
    MSFM_CUDA(ctx, cudaStreamWaitEvent(ctx->d2h_stream, ctx->ev_f1, 0));
    MSFM_CUDA(ctx, cudaEventRecord(ctx->ev_d2h0, ctx->d2h_stream));
    MSFM_CUDA(ctx, cudaMemcpyAsync(dst0, src0, bytes0, cudaMemcpyDeviceToHost, ctx->d2h_stream));
    if (bytes1) MSFM_CUDA(ctx, cudaMemcpyAsync(dst1, src1, bytes1, cudaMemcpyDeviceToHost, ctx->d2h_stream));
    MSFM_CUDA(ctx, cudaEventRecord(ctx->ev_d2h1, ctx->d2h_stream));
    ctx->d2h_in_flight = true;
    ctx->timing.d2h_bytes += (int64_t)(bytes0 + bytes1);
    return MSFM_OK;
}

msfm_status accumulate_kernel_time(msfm_ctx *ctx, cudaEvent_t e0, cudaEvent_t e1) {
    float ms = 0.f;
    MSFM_CUDA(ctx, cudaEventElapsedTime(&ms, e0, e1));
    ctx->timing.match_kernel_ms += ms;
    return MSFM_OK;
}

// Device time of a batch that has completed: the forward pass [ev_k0, ev_k1] and, when the batch recorded them, the twin
// pass [ev_k2, ev_k3] are matching-kernel time; the rest of [ev_k0, ev_f1] is finalize time.
msfm_status add_batch_times(msfm_ctx *ctx, bool twin_events) {
    float ms_all = 0.f, ms_fw = 0.f, ms_twin = 0.f;
    MSFM_CUDA(ctx, cudaEventElapsedTime(&ms_all, ctx->ev_k0, ctx->ev_f1));
    MSFM_CUDA(ctx, cudaEventElapsedTime(&ms_fw, ctx->ev_k0, ctx->ev_k1));
    if (twin_events) MSFM_CUDA(ctx, cudaEventElapsedTime(&ms_twin, ctx->ev_k2, ctx->ev_k3));
    ctx->timing.match_kernel_ms += ms_fw + ms_twin;
    ctx->timing.finalize_ms += ms_all - ms_fw - ms_twin;
    return MSFM_OK;
}

// ---- Collect stage of the float regime: the band rows of a re-scoring msfm_match_pairs, every query row of an exact
// msfm_knn2_pairs.  The caller's mark kernel gathers the rows and their thresholds into the candidate scratch; the
// matching kernel's collect pass lists every reference row under a row's threshold, the events are scored in fp32 and
// finish_band_kernel decides each row.  When the event list overflows, the dp4a brute force decides the batch instead.

// Capacity of the event list: `allowance` + 65 536, or the test override; the kernels count events in 32 bits.
size_t collect_event_cap(const msfm_ctx *ctx, size_t allowance) {
    return std::min<size_t>(ctx->band_event_cap_override >= 0 ? (size_t)ctx->band_event_cap_override : allowance + 65536, UINT32_MAX);
}

msfm_status ensure_collect_scratch(msfm_ctx *ctx, size_t rows, size_t n_pairs, size_t event_cap) {
    msfm_status st;
    if ((st = ensure(ctx, ctx->band_q, rows * 4)) != MSFM_OK) return st;
    if ((st = ensure(ctx, ctx->band_counts, n_pairs * 4)) != MSFM_OK) return st;
    if ((st = ensure(ctx, ctx->band_thr, rows * 4)) != MSFM_OK) return st;
    if ((st = ensure(ctx, ctx->band_state, rows * 16)) != MSFM_OK) return st;
    if ((st = ensure(ctx, ctx->band_events, std::max<size_t>(event_cap, 1) * 16)) != MSFM_OK) return st;
    if ((st = ensure(ctx, ctx->band_event_keys, std::max<size_t>(event_cap, 1) * 8)) != MSFM_OK) return st;
    return ensure(ctx, ctx->band_event_count, 4);
}

// The collect stage's parameters over the current batch's scratch.  The ratio rule fields are left at zero and the
// FLANN outputs null: msfm_match_pairs sets the former, msfm_knn2_pairs the latter.
msfm::BandParams collect_params(const msfm_ctx *ctx, size_t event_cap) {
    msfm::BandParams bp;
    bp.pairs = static_cast<const PairDesc *>(ctx->pairdesc.ptr);
    bp.knn = static_cast<int4 *>(ctx->knn.ptr);
    bp.ratio = bp.ratio_good = bp.max_dist_sq = bp.band = 0.0f;
    bp.reject_gt = 0;
    bp.band_q = static_cast<int32_t *>(ctx->band_q.ptr);
    bp.band_counts = static_cast<int32_t *>(ctx->band_counts.ptr);
    bp.fdesc = ctx->fdesc;
    bp.desc_arena = ctx->desc;
    bp.ckeys = ctx->norms;
    bp.band_thr = static_cast<int32_t *>(ctx->band_thr.ptr);
    bp.band_state = static_cast<unsigned long long *>(ctx->band_state.ptr);
    bp.cand_desc = static_cast<uint8_t *>(ctx->cand_desc.ptr);
    bp.cand_ckeys = static_cast<int32_t *>(ctx->cand_ckeys.ptr);
    bp.events = static_cast<const int4 *>(ctx->band_events.ptr);
    bp.event_keys = static_cast<unsigned long long *>(ctx->band_event_keys.ptr);
    bp.event_count = static_cast<const unsigned int *>(ctx->band_event_count.ptr);
    bp.event_cap = (uint32_t)event_cap;
    return bp;
}

// Everything after the mark kernel: the collect pass over the plan's band items, fp32 scoring of the events, the rows'
// decisions, and the brute force, which returns at once unless the event list overflowed.
msfm_status run_collect_pass(msfm_ctx *ctx, const BatchPlan &plan, const msfm::BandParams &bp) {
    msfm_status st;
    if (!plan.band_items.empty() &&
        (st = launch_match_kernel(ctx, Pass::collect, plan.items.size() + plan.twin_items.size(), plan.band_items.size(), bp.event_cap,
                                  plan)) != MSFM_OK)
        return st;
    const int nb = (int)plan.pairs.size();
    msfm::score_events_kernel<<<4 * ctx->num_sms, 256, 0, ctx->stream>>>(bp);
    msfm::second_events_kernel<<<4 * ctx->num_sms, 256, 0, ctx->stream>>>(bp);
    msfm::finish_band_kernel<<<nb, 256, 0, ctx->stream>>>(bp);
    const int gx = std::min(nb, 4 * ctx->num_sms);
    const int gy = std::max(1, std::min(32, (4 * ctx->num_sms + gx - 1) / gx));
    // a guided batch: the brute force applies the plan's gate as the collect pass does
    const msfm::EpiGate *gate = plan.epi_gate();
    const GateKind kind = gate ? plan.gate_kind : GateKind::none;
    const msfm::EpiGate g = gate ? *gate : msfm::EpiGate{nullptr, nullptr, 0.0f};
    if (kind == GateKind::homography)
        msfm::rescore_band_kernel<GateKind::homography><<<dim3(gx, gy), 256, 0, ctx->stream>>>(bp, nb, g);
    else if (kind == GateKind::epipolar)
        msfm::rescore_band_kernel<GateKind::epipolar><<<dim3(gx, gy), 256, 0, ctx->stream>>>(bp, nb, g);
    else
        msfm::rescore_band_kernel<GateKind::none><<<dim3(gx, gy), 256, 0, ctx->stream>>>(bp, nb, g);
    MSFM_CUDA(ctx, cudaGetLastError());
    ctx->timing.total_launches += 4;
    return MSFM_OK;
}

// `events` is the collect pass's event count, read back after the batch: more than the list holds means the brute force
// decided the batch.
void note_collect_events(msfm_ctx *ctx, unsigned int events, size_t event_cap) {
    if (events > event_cap) ctx->knn_brute_batches += 1;
    else ctx->knn_events += events;
}

// kNN of a single pair into scratch (no min_keypoints test).  Caller holds the lock.
msfm_status knn_single(msfm_ctx *ctx, int32_t ref_id, int32_t query_id, BatchPlan &plan) {
    msfm_status st;
    if ((st = check_image_id(ctx, ref_id, true)) != MSFM_OK) return st;
    if ((st = check_image_id(ctx, query_id, true)) != MSFM_OK) return st;
    plan_add_pair(ctx, plan, 0, ref_id, query_id);
    ctx->timing = msfm_timing{};
    MSFM_CUDA(ctx, cudaEventRecord(ctx->ev_begin, ctx->stream));
    if (plan.query_rows == 0) return MSFM_OK;
    return run_match_stage(ctx, plan);  // a pair without work items leaves "absent" rows (memset)
}

// Where a call's results go: per-pair offsets / ok flags in host arrays, the match lists through a sink (see msfm_internal.h).
struct OutSpec {
    int64_t *offsets = nullptr;
    int32_t *ok = nullptr;
    bool has_good = false;
    msfm_sink_fn sink = nullptr;
    void *user = nullptr;
};

// The public entry point's sink: the caller's msfm_result buffers.
struct CallerBuffers {
    int32_t (*matches)[2];
    uint8_t *good;
    int64_t capacity;
};
int caller_sink(void *user, int64_t first, int64_t n, int32_t (**m)[2], uint8_t **g) {
    const CallerBuffers *cb = static_cast<const CallerBuffers *>(user);
    if (first + n > cb->capacity) return 1;
    *m = cb->matches + first;
    *g = cb->good ? cb->good + first : nullptr;
    return 0;
}

// The gate of msfm_match_pairs_guided (epipolar: M = F) or msfm_match_pairs_guided_homography (homography: M = H), as
// the caller passed it.
struct GuidedArgs {
    GateKind kind;
    const double (*M)[9];
    float th;
    const float *const *image_xy;
    const int32_t *image_npts;
    int32_t n_images;
};

// Everything the guided entry points reject is rejected here, before any launch.  On success `fq` holds every pair's
// matrix rounded to fp32.  The image ids have been checked.
msfm_status check_guided(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const msfm_params *params, const GuidedArgs &g,
                         std::vector<float> &fq) {
    const bool homog = g.kind == GateKind::homography;
    const char *fn = homog ? "msfm_match_pairs_guided_homography" : "msfm_match_pairs_guided";
    const char *mat = homog ? "H" : "F";
    if (!std::isfinite(params->rescore_band) || params->rescore_band < 0.0f)
        return fail(ctx, MSFM_ERR_INVALID_ARG, "%s: rescore_band %g must be finite and >= 0", fn, (double)params->rescore_band);
    if (params->rescore_band > 0.0f && !ctx->fdesc)
        return fail(ctx, MSFM_ERR_INVALID_ARG, "%s: rescore_band > 0 needs a keep_float context (retained float rows)", fn);
    if (!std::isfinite(g.th) || !(g.th > 0.0f))
        return fail(ctx, MSFM_ERR_INVALID_ARG, "%s: %s %g must be finite and > 0", fn, homog ? "th_transfer" : "th_epipolar", (double)g.th);
    if (n_pairs == 0) return MSFM_OK;
    if (!g.M) return fail(ctx, MSFM_ERR_INVALID_ARG, "%s: null %s", fn, mat);
    if (!g.image_xy || !g.image_npts) return fail(ctx, MSFM_ERR_INVALID_ARG, "%s: null image_xy / image_npts", fn);
    std::vector<char> checked((size_t)std::max(g.n_images, 0), 0);
    fq.resize((size_t)n_pairs * 9);
    for (int64_t p = 0; p < n_pairs; ++p) {
        for (const int32_t i : {pairs[p].ref, pairs[p].query}) {
            if (i >= g.n_images)
                return fail(ctx, MSFM_ERR_INVALID_ARG, "%s: pair %lld names image %d, outside [0, n_images = %d)", fn,
                            (long long)p, i, g.n_images);
            if (checked[i]) continue;
            checked[i] = 1;
            const int32_t rows = ctx->images[i].rows;
            if (g.image_npts[i] != rows)
                return fail(ctx, MSFM_ERR_INVALID_ARG, "%s: image %d has %d keypoints and %d uploaded rows", fn, i,
                            g.image_npts[i], rows);
            if (rows > 0 && !g.image_xy[i]) return fail(ctx, MSFM_ERR_INVALID_ARG, "%s: image %d has no keypoints", fn, i);
            for (int64_t k = 0; k < 2ll * rows; ++k)
                if (!std::isfinite(g.image_xy[i][k]))
                    return fail(ctx, MSFM_ERR_INVALID_ARG, "%s: keypoint %lld of image %d is not finite", fn, (long long)(k / 2), i);
        }
        bool nonzero = false;
        for (int k = 0; k < 9; ++k) {
            const float f = (float)g.M[p][k];  // one rounding to nearest
            if (!std::isfinite(f))
                return fail(ctx, MSFM_ERR_INVALID_ARG, "%s: %s of pair %lld has a non-finite entry (in fp32)", fn, mat, (long long)p);
            nonzero = nonzero || f != 0.0f;
            fq[(size_t)p * 9 + k] = f;
        }
        if (!nonzero) return fail(ctx, MSFM_ERR_INVALID_ARG, "%s: %s of pair %lld is zero", fn, mat, (long long)p);
    }
    return MSFM_OK;
}

// Keypoints of the images a guided call touches, to their arena rows of ctx->kp_xy (on the matching stream).
msfm_status upload_keypoints(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const GuidedArgs &g) {
    msfm_status st;
    const bool fresh = ctx->kp_xy.ptr == nullptr;
    if ((st = ensure(ctx, ctx->kp_xy, (size_t)ctx->arena_rows * sizeof(float2))) != MSFM_OK) return st;
    if (fresh) MSFM_CUDA(ctx, cudaMemsetAsync(ctx->kp_xy.ptr, 0, ctx->kp_xy.bytes, ctx->stream));
    std::vector<char> sent((size_t)g.n_images, 0);
    for (int64_t p = 0; p < n_pairs; ++p)
        for (const int32_t i : {pairs[p].ref, pairs[p].query}) {
            if (sent[i] || ctx->images[i].rows == 0) continue;
            sent[i] = 1;
            MSFM_CUDA(ctx, cudaMemcpyAsync(static_cast<float2 *>(ctx->kp_xy.ptr) + ctx->images[i].off, g.image_xy[i],
                                           (size_t)ctx->images[i].rows * sizeof(float2), cudaMemcpyHostToDevice, ctx->stream));
        }
    return MSFM_OK;
}

// msfm_match_pairs, and the guided entry points when `guided` is set: the same batches, with the forward and twin passes
// of the matching kernel under the epipolar or homography gate and every mutual pair routed to the twin pass.
msfm_status match_pairs_impl(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const msfm_params *params, const OutSpec *out,
                             bool resident, int64_t *n_matches_total, const GuidedArgs *guided = nullptr) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n_pairs < 0 || (n_pairs > 0 && !pairs) || !params) return fail(ctx, MSFM_ERR_INVALID_ARG, "null pair list / params or negative n_pairs");
    if (!resident && (!out || !out->offsets || !out->ok || !out->sink))
        return fail(ctx, MSFM_ERR_INVALID_ARG, "msfm_result needs offsets, ok and matches buffers");
    if (!(params->ratio > 0.0f)) return fail(ctx, MSFM_ERR_INVALID_ARG, "ratio must be > 0");
    msfm_status st;
    if ((st = check_pairs(ctx, pairs, n_pairs)) != MSFM_OK) return st;
    std::vector<float> fq;  // guided: F (or H) of every pair in fp32
    if (guided && (st = check_guided(ctx, pairs, n_pairs, params, *guided, fq)) != MSFM_OK) return st;
    ctx->timing = msfm_timing{};
    DrainListCopy drain_list_copy{ctx};
    MSFM_CUDA(ctx, cudaEventRecord(ctx->ev_begin, ctx->stream));
    if (guided && (st = upload_keypoints(ctx, pairs, n_pairs, *guided)) != MSFM_OK) return st;
    const bool mutual = params->mutual != 0;
    const bool want_good = params->ratio_good > 0.0f && (resident || out->has_good);
    const int64_t max_rows = mutual ? kBatchMaxQueryRowsMutual : kBatchMaxQueryRows;
    if (params->rescore_band > 0.0f && ctx->fdesc) { ctx->knn_events = 0; ctx->knn_brute_batches = 0; }
    int64_t written = 0;  // matches written to the caller so far
    int64_t total = 0;
    if (!resident) out->offsets[0] = 0;

    // Dead-row rule of the forward pass: rho = the largest ratio any consumer tests (+ the re-scoring band, whose rows need
    // exact neighbours) rounded UP to 1/256 plus one step, so that "dead" (d0 > rho * d1) implies fl(d0/d1) > ratio under
    // both ratio rules; thresholds near or above 1 switch the rule off.
    uint32_t prune_q8 = msfm::kNoPrune;
    {
        float rmax = std::max(params->ratio, params->ratio_good);
        if (params->rescore_band > 0.0f) rmax += params->rescore_band;
        if (rmax > 0.0f && rmax < 0.97f) prune_q8 = (uint32_t)std::floor(rmax * 256.0f) + 2;
    }
    // Batches are carved (host-only work: pair descriptors + work items) one ahead, while the previous batch runs on the GPU.
    struct Carved { BatchPlan plan; int64_t first = 0, last = 0; };
    int64_t next = 0;
    auto carve = [&](Carved &c) -> bool {  // false: no pair left
        if (next >= n_pairs) return false;
        c.plan = BatchPlan();
        c.plan.mutual = mutual;
        c.plan.rescoring = params->rescore_band > 0.0f && ctx->fdesc != nullptr;
        c.plan.prune_q8 = prune_q8;
        if (guided) {
            c.plan.gate = msfm::EpiGate{static_cast<const float2 *>(ctx->kp_xy.ptr), nullptr, guided->th * guided->th};
            c.plan.gate_kind = guided->kind;
        }
        c.first = next;
        while (next < n_pairs && (int64_t)c.plan.pairs.size() < kBatchMaxPairs) {
            const ImageSlot &r = ctx->images[pairs[next].ref], &q = ctx->images[pairs[next].query];
            const bool too_few = r.rows < params->min_keypoints || q.rows < params->min_keypoints;
            if (!too_few) {
                if (!c.plan.pairs.empty() && (c.plan.query_rows + q.rows > max_rows || (mutual && c.plan.ref_rows + r.rows > kBatchMaxRefRows))) break;
                // A pair whose images are still being uploaded does not hold back the pairs before it: the batch is cut
                // there, runs on what has landed, and the transfer goes on underneath (the caller orders the list by the
                // newest image a pair needs, e.g. by staging group).
                const uint64_t need = std::max(r.ready_seq, q.ready_seq);
                if (!c.plan.pairs.empty() && need > c.plan.need_seq && !uploads_landed(ctx, need)) break;
                plan_add_pair(ctx, c.plan, next, pairs[next].ref, pairs[next].query);
                if (guided) c.plan.fmat.insert(c.plan.fmat.end(), fq.begin() + 9 * next, fq.begin() + 9 * (next + 1));
            }
            ++next;
        }
        c.last = next;
        finish_plan(ctx, c.plan);
        return true;
    };
    Carved cur, ahead;
    bool have = carve(cur);
    for (int64_t batch_no = 0; have; ++batch_no) {  // batch_no picks the set of tight list buffers (the other set may still be on its way to the host)
        BatchPlan &plan = cur.plan;
        const int64_t first = cur.first, last = cur.last;
        const int nb = (int)plan.pairs.size();
        const bool work = nb > 0 && plan.query_rows > 0;
        const size_t rows = (size_t)plan.query_rows;
        const bool float_rescoring = plan.rescoring && plan.any_float;
        // Event list: half an event per query row of the batch.  Measured on tools/float_regime_bench.py (780 pairs of
        // 8192-row unit-norm images in one batch, ratio 0.85, band 0.02): 1.14 % of the query rows are band rows, with
        // 10.05 events each under T(q), 0.73 M events against a cap of 3.26 M, no overflow
        // (profiles/float_regime_bound_1gpu.json).  Wide bands overflow it and the brute force decides the batch, with
        // the same result.
        const size_t event_cap = float_rescoring ? collect_event_cap(ctx, rows / 2) : 0;
        // (a buffer that has to grow is not the one a list copy is still reading: see wait_list_copy below)
        DeviceBuf &tm = batch_no & 1 ? ctx->tight_matches_b : ctx->tight_matches, &tg = batch_no & 1 ? ctx->tight_good_b : ctx->tight_good;
        if (work) {
            if ((st = ensure(ctx, ctx->cand_q, rows * 4)) != MSFM_OK) return st;
            if ((st = ensure(ctx, ctx->cand_j, rows * 4)) != MSFM_OK) return st;
            if ((st = ensure(ctx, ctx->cand_d0, rows * 4)) != MSFM_OK) return st;
            if ((st = ensure(ctx, ctx->cand_good, rows)) != MSFM_OK) return st;
            if ((mutual || float_rescoring) && (st = ensure_cand_scratch(ctx, plan.query_rows)) != MSFM_OK) return st;
            if (float_rescoring && (st = ensure_collect_scratch(ctx, rows, nb, event_cap)) != MSFM_OK) return st;
            if ((st = ensure(ctx, ctx->matches, rows * sizeof(int2))) != MSFM_OK) return st;
            if (want_good && (st = ensure(ctx, ctx->good, rows)) != MSFM_OK) return st;
            if ((st = ensure(ctx, ctx->counts, (size_t)nb * 4)) != MSFM_OK) return st;
            if ((st = ensure(ctx, ctx->offsets, (size_t)(nb + 1) * 8)) != MSFM_OK) return st;
            if ((st = ensure(ctx, tm, rows * sizeof(int2))) != MSFM_OK) return st;
            if (want_good && (st = ensure(ctx, tg, rows)) != MSFM_OK) return st;
            // ---- forward 2-NN
            if ((st = run_match_stage(ctx, plan)) != MSFM_OK) return st;
            // ---- float regime: rows near a ratio threshold are decided on exact fp32 distances
            if (float_rescoring) {
                MSFM_CUDA(ctx, cudaMemsetAsync(ctx->band_event_count.ptr, 0, 4, ctx->stream));
                msfm::BandParams bp = collect_params(ctx, event_cap);
                bp.ratio = params->ratio;
                bp.ratio_good = params->ratio_good;
                bp.max_dist_sq = params->max_dist_sq;
                bp.band = params->rescore_band;
                bp.reject_gt = (params->flags & MSFM_RATIO_REJECT_GT) ? 1 : 0;
                msfm::mark_band_kernel<<<nb, 1024, 0, ctx->stream>>>(bp, ctx->resid, ctx->img_rmax);
                MSFM_CUDA(ctx, cudaGetLastError());
                ctx->timing.total_launches += 1;
                // tensor pass in collect mode over the gathered band rows, then fp32 scoring of what it listed
                if ((st = run_collect_pass(ctx, plan, bp)) != MSFM_OK) return st;
            }
            // ---- ratio test -> one-way candidates; mutual check from the forward results (column table + dangerous rows),
            //      pairs too ambiguous for that are routed to the tensor twin pass
            if (mutual) {
                if ((st = ensure(ctx, ctx->colbest, plan.big_ref ? (size_t)std::max<int64_t>(plan.ref_rows, 1) * 8 : 256)) != MSFM_OK) return st;
                if ((st = ensure(ctx, ctx->twin_counts, (size_t)(nb + 1) * 4)) != MSFM_OK) return st;
                ctx->routed_index = nb;
                if (plan.big_ref) MSFM_CUDA(ctx, cudaMemsetAsync(ctx->colbest.ptr, 0xFF, (size_t)plan.ref_rows * 8, ctx->stream));
                MSFM_CUDA(ctx, cudaMemsetAsync(static_cast<int32_t *>(ctx->twin_counts.ptr) + nb, 0, 4, ctx->stream));
            }
            msfm::SelectParams sp;
            sp.pairs = static_cast<const PairDesc *>(ctx->pairdesc.ptr);
            sp.knn = static_cast<const int4 *>(ctx->knn.ptr);
            sp.ratio = params->ratio;
            sp.ratio_good = params->ratio_good;
            sp.max_dist_sq = params->max_dist_sq;
            sp.reject_gt = (params->flags & MSFM_RATIO_REJECT_GT) ? 1 : 0;
            sp.cand_q = static_cast<int32_t *>(ctx->cand_q.ptr);
            sp.cand_j = static_cast<int32_t *>(ctx->cand_j.ptr);
            sp.cand_d0 = static_cast<int32_t *>(ctx->cand_d0.ptr);
            sp.cand_good = static_cast<uint8_t *>(ctx->cand_good.ptr);
            sp.counts = static_cast<int32_t *>(ctx->cand_counts.ptr);
            sp.float_mutual = (mutual && float_rescoring) ? 1 : 0;
            sp.mutual = mutual ? 1 : 0;
            sp.force_twin = (ctx->force_twin || guided) ? 1 : 0;  // the forward-result check is not proven under a gate
            sp.colbest = static_cast<unsigned long long *>(ctx->colbest.ptr);
            sp.smem_table_rows = msfm::kSmemTableRows;
            sp.danger = static_cast<int2 *>(ctx->matches.ptr);  // the match scratch is written by the emission afterwards
            sp.twin_counts = static_cast<int32_t *>(ctx->twin_counts.ptr);
            sp.routed = reinterpret_cast<unsigned int *>(static_cast<int32_t *>(ctx->twin_counts.ptr) + nb);
            sp.desc_arena = ctx->desc;
            sp.ckeys = ctx->norms;
            sp.cand_desc = static_cast<uint8_t *>(ctx->cand_desc.ptr);
            sp.cand_ckeys = static_cast<int32_t *>(ctx->cand_ckeys.ptr);
            msfm::select_candidates_kernel<<<nb, 1024, mutual ? msfm::kSelectSmemBytes : 0, ctx->stream>>>(sp);
            MSFM_CUDA(ctx, cudaGetLastError());
            ctx->timing.total_launches += 1;
            // ---- tensor twin pass (nearest query row of every candidate's reference row) for the routed pairs only
            MSFM_CUDA(ctx, cudaEventRecord(ctx->ev_k2, ctx->stream));
            if (mutual && !plan.twin_items.empty() &&
                (st = launch_match_kernel(ctx, Pass::twin, plan.items.size(), plan.twin_items.size(), 0, plan)) != MSFM_OK)
                return st;
            MSFM_CUDA(ctx, cudaEventRecord(ctx->ev_k3, ctx->stream));
            // ---- emission, offsets, tight gather
            msfm::EmitParams ep;
            ep.pairs = sp.pairs;
            ep.knn = sp.knn;
            ep.twin_base = plan.query_rows;
            ep.cand_q = sp.cand_q;
            ep.cand_j = sp.cand_j;
            ep.cand_good = sp.cand_good;
            ep.cand_counts = sp.counts;
            ep.twin_counts = sp.twin_counts;
            ep.matches = static_cast<int2 *>(ctx->matches.ptr);
            ep.good = want_good ? static_cast<uint8_t *>(ctx->good.ptr) : nullptr;
            ep.counts = static_cast<int32_t *>(ctx->counts.ptr);
            ep.mutual = mutual ? 1 : 0;
            ep.orientation = params->orientation;
            ep.fdesc = float_rescoring ? ctx->fdesc : nullptr;
            msfm::emit_matches_kernel<<<nb, 1024, 0, ctx->stream>>>(ep);
            msfm::scan_counts_kernel<<<1, 1024, 0, ctx->stream>>>(ep.counts, nb, static_cast<int64_t *>(ctx->offsets.ptr));
            msfm::gather_matches_kernel<<<nb, 256, 0, ctx->stream>>>(
                ep.pairs, ep.counts, static_cast<const int64_t *>(ctx->offsets.ptr), ep.matches, ep.good,
                static_cast<int2 *>(tm.ptr), want_good ? static_cast<uint8_t *>(tg.ptr) : nullptr);
            MSFM_CUDA(ctx, cudaGetLastError());
            MSFM_CUDA(ctx, cudaEventRecord(ctx->ev_f1, ctx->stream));
            ctx->timing.total_launches += 3;
        }
        // ---- plan the next batch while this one runs
        have = carve(ahead);
        std::vector<int64_t> batch_offsets;
        if (work) {
            // ---- results
            batch_offsets.resize(nb + 1);
            unsigned int twin_pairs = 0, h_events = 0;
            MSFM_CUDA(ctx, cudaMemcpyAsync(batch_offsets.data(), ctx->offsets.ptr, (size_t)(nb + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
            if (mutual) MSFM_CUDA(ctx, cudaMemcpyAsync(&twin_pairs, static_cast<int32_t *>(ctx->twin_counts.ptr) + nb, 4, cudaMemcpyDeviceToHost, ctx->stream));
            if (float_rescoring) MSFM_CUDA(ctx, cudaMemcpyAsync(&h_events, ctx->band_event_count.ptr, 4, cudaMemcpyDeviceToHost, ctx->stream));
            MSFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            ctx->timing.twin_pairs += (int32_t)twin_pairs;
            if (float_rescoring) note_collect_events(ctx, h_events, event_cap);
            ctx->timing.d2h_bytes += (nb + 1) * 8;
            if ((st = add_batch_times(ctx, true)) != MSFM_OK) return st;
            const int64_t bt = batch_offsets[nb];
            total += bt;
            if ((st = wait_list_copy(ctx)) != MSFM_OK) return st;  // the previous batch's lists (copied under this batch's kernels)
            if (!resident && bt > 0) {
                int32_t (*dst_m)[2] = nullptr;
                uint8_t *dst_g = nullptr;
                if (out->sink(out->user, written, bt, &dst_m, &dst_g) != 0 || !dst_m)
                    return fail(ctx, MSFM_ERR_CAPACITY, "match buffer too small: need at least %lld entries", (long long)(written + bt));
                if (dst_g && !want_good) memset(dst_g, 0, (size_t)bt);
                // The lists leave on their own stream, ordered behind this batch's gather (ev_f1); the next batch's kernels
                // start right away on the main stream and write the OTHER set of tight buffers.  At most one list copy is
                // in flight: the previous one was waited for above, before the sink could move the host buffers.
                if ((st = start_list_copy(ctx, dst_m, tm.ptr, (size_t)bt * sizeof(int2), dst_g, tg.ptr, dst_g && want_good ? (size_t)bt : 0)) != MSFM_OK)
                    return st;
            }
        }
        // ---- host bookkeeping for pairs [first, last)
        if (!resident) {
            size_t k = 0;
            for (int64_t i = first; i < last; ++i) {
                if (k < plan.src_index.size() && plan.src_index[k] == i) {
                    const int64_t cnt = batch_offsets.empty() ? 0 : batch_offsets[k + 1] - batch_offsets[k];
                    out->ok[i] = 1;
                    out->offsets[i + 1] = out->offsets[i] + cnt;
                    ++k;
                } else {
                    out->ok[i] = 0;
                    out->offsets[i + 1] = out->offsets[i];
                }
            }
            written = out->offsets[last];
        }
        std::swap(cur, ahead);
    }
    if ((st = wait_list_copy(ctx)) != MSFM_OK) return st;
    MSFM_CUDA(ctx, cudaEventRecord(ctx->ev_end, ctx->stream));
    MSFM_CUDA(ctx, cudaEventSynchronize(ctx->ev_end));
    MSFM_CUDA(ctx, cudaEventElapsedTime(&ctx->timing.total_ms, ctx->ev_begin, ctx->ev_end));
    if (n_matches_total) *n_matches_total = total;
    return MSFM_OK;
}

// msfm_knn2_pairs (and msfm_knn2, its one-pair flags-0 form).  Per batch of consecutive pairs: the forward 2-NN without
// pruning, then either the FLANN conversion of the kNN scratch (integer distances) or, in exact mode, the collect pass
// over every query row under its bound T(q) (mark_exact_kernel), fp32 scoring of the events and the FLANN rows written
// by finish_band_kernel (rescore_band_kernel when the event list overflowed).  A batch's rows go back to the host on
// the list-copy stream under the next batch's kernels, as in match_pairs_impl.
msfm_status knn2_pairs_impl(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, uint32_t flags, int64_t *offsets, int32_t *ids,
                            float *dists, int64_t row_capacity) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n_pairs < 0 || (n_pairs > 0 && !pairs) || !offsets || !ids || !dists || row_capacity < 0)
        return fail(ctx, MSFM_ERR_INVALID_ARG, "null pair list / output buffer, negative n_pairs or negative row_capacity");
    if (flags & ~MSFM_KNN_EXACT_F32) return fail(ctx, MSFM_ERR_INVALID_ARG, "unknown flag bits 0x%x", flags & ~MSFM_KNN_EXACT_F32);
    const bool exact = (flags & MSFM_KNN_EXACT_F32) != 0;
    msfm_status st;
    if ((st = check_pairs(ctx, pairs, n_pairs)) != MSFM_OK) return st;
    int64_t rows_total = 0;
    for (int64_t i = 0; i < n_pairs; ++i) rows_total += ctx->images[pairs[i].query].rows;
    if (rows_total > row_capacity)
        return fail(ctx, MSFM_ERR_CAPACITY, "output too small: the pairs have %lld query rows, row_capacity is %lld", (long long)rows_total,
                    (long long)row_capacity);
    if (exact) {
        if (!ctx->fdesc) return fail(ctx, MSFM_ERR_INVALID_ARG, "MSFM_KNN_EXACT_F32 needs a keep_float context");
        for (int64_t i = 0; i < n_pairs; ++i) {
            const ImageSlot &r = ctx->images[pairs[i].ref], &q = ctx->images[pairs[i].query];
            if (r.rows == 0 || q.rows == 0) continue;  // nothing to score: the rows read "absent" either way
            if (!r.has_float || !q.has_float)
                return fail(ctx, MSFM_ERR_INVALID_ARG, "MSFM_KNN_EXACT_F32: pair %lld: image %d has no retained float rows (upload it with msfm_upload_f32*)",
                            (long long)i, !r.has_float ? pairs[i].ref : pairs[i].query);
            if (r.scale != q.scale)
                return fail(ctx, MSFM_ERR_INVALID_ARG, "MSFM_KNN_EXACT_F32: pair %lld: images %d and %d were quantised with different scales (%g, %g)",
                            (long long)i, pairs[i].ref, pairs[i].query, (double)r.scale, (double)q.scale);
            if (!(r.scale * r.scale > 0.0f))  // the plan marks float pairs by scale^2 > 0
                return fail(ctx, MSFM_ERR_INVALID_ARG, "MSFM_KNN_EXACT_F32: pair %lld: scale %g is too small", (long long)i, (double)r.scale);
        }
    }
    MSFM_CUDA(ctx, cudaSetDevice(ctx->device));
    offsets[0] = 0;
    for (int64_t i = 0; i < n_pairs; ++i) offsets[i + 1] = offsets[i] + ctx->images[pairs[i].query].rows;
    ctx->timing = msfm_timing{};
    if (exact) { ctx->knn_events = 0; ctx->knn_brute_batches = 0; }
    DrainListCopy drain_list_copy{ctx};
    MSFM_CUDA(ctx, cudaEventRecord(ctx->ev_begin, ctx->stream));
    const int64_t max_rows = exact ? kBatchMaxQueryRowsExact : kBatchMaxQueryRows;
    int64_t next = 0;
    auto carve = [&](BatchPlan &plan) -> bool {  // false: no pair left
        if (next >= n_pairs) return false;
        plan = BatchPlan();  // no pruning: exact 2-NN rows
        plan.rescoring = exact;
        while (next < n_pairs && (int64_t)plan.pairs.size() < kBatchMaxPairs) {
            const int64_t qr = ctx->images[pairs[next].query].rows;
            if (!plan.pairs.empty() && plan.query_rows + qr > max_rows) break;
            plan_add_pair(ctx, plan, next, pairs[next].ref, pairs[next].query);
            ++next;
        }
        finish_plan(ctx, plan);
        return true;
    };
    BatchPlan cur, ahead;
    bool have = carve(cur);
    for (int64_t batch_no = 0; have; ++batch_no) {
        BatchPlan &plan = cur;
        const int nb = (int)plan.pairs.size();
        const int64_t row_base = offsets[plan.src_index.front()];
        const bool work = plan.query_rows > 0;
        const size_t rows = (size_t)plan.query_rows;
        const size_t event_cap = exact ? collect_event_cap(ctx, rows * kExactEventsPerRow) : 0;
        DeviceBuf &oi = batch_no & 1 ? ctx->knn_ids_b : ctx->knn_ids, &od = batch_no & 1 ? ctx->knn_dists_b : ctx->knn_dists;
        if (work) {
            if ((st = ensure(ctx, oi, rows * 8)) != MSFM_OK) return st;
            if ((st = ensure(ctx, od, rows * 8)) != MSFM_OK) return st;
            if (exact) {
                if ((st = ensure_cand_scratch(ctx, plan.query_rows)) != MSFM_OK) return st;
                if ((st = ensure_collect_scratch(ctx, rows, nb, event_cap)) != MSFM_OK) return st;
            }
            // ---- forward 2-NN (exact rows: the plan carries no pruning)
            if ((st = run_match_stage(ctx, plan)) != MSFM_OK) return st;
            if (exact) {
                MSFM_CUDA(ctx, cudaMemsetAsync(ctx->band_event_count.ptr, 0, 4, ctx->stream));
                msfm::BandParams bp = collect_params(ctx, event_cap);
                bp.out_ids = static_cast<int32_t *>(oi.ptr);
                bp.out_dists = static_cast<float *>(od.ptr);
                int32_t max_q = 0;
                for (const PairDesc &pd : plan.pairs) max_q = std::max(max_q, pd.qry_rows);
                const int gy = std::max(1, std::min(64, (max_q + 255) / 256));
                msfm::mark_exact_kernel<<<dim3(nb, gy), 256, 0, ctx->stream>>>(bp, ctx->resid, ctx->img_rmax);
                MSFM_CUDA(ctx, cudaGetLastError());
                ctx->timing.total_launches += 1;
                // tensor pass in collect mode over every query row, fp32 scoring of what it listed, FLANN rows
                if ((st = run_collect_pass(ctx, plan, bp)) != MSFM_OK) return st;
            } else {
                msfm::knn_to_flann_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, ctx->stream>>>(static_cast<const int4 *>(ctx->knn.ptr), (int)rows,
                                                                                             static_cast<int32_t *>(oi.ptr), static_cast<float *>(od.ptr));
                MSFM_CUDA(ctx, cudaGetLastError());
                ctx->timing.total_launches += 1;
            }
            MSFM_CUDA(ctx, cudaEventRecord(ctx->ev_f1, ctx->stream));
        }
        // ---- plan the next batch while this one runs
        have = carve(ahead);
        if (work) {
            unsigned int h_events = 0;
            if (exact) MSFM_CUDA(ctx, cudaMemcpyAsync(&h_events, ctx->band_event_count.ptr, 4, cudaMemcpyDeviceToHost, ctx->stream));
            MSFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            if (exact) note_collect_events(ctx, h_events, event_cap);
            if ((st = add_batch_times(ctx, false)) != MSFM_OK) return st;
            if ((st = wait_list_copy(ctx)) != MSFM_OK) return st;  // the previous batch's rows (copied under this batch's kernels)
            if ((st = start_list_copy(ctx, ids + 2 * row_base, oi.ptr, rows * 8, dists + 2 * row_base, od.ptr, rows * 8)) != MSFM_OK) return st;
        }
        std::swap(cur, ahead);
    }
    if ((st = wait_list_copy(ctx)) != MSFM_OK) return st;
    MSFM_CUDA(ctx, cudaEventRecord(ctx->ev_end, ctx->stream));
    MSFM_CUDA(ctx, cudaEventSynchronize(ctx->ev_end));
    MSFM_CUDA(ctx, cudaEventElapsedTime(&ctx->timing.total_ms, ctx->ev_begin, ctx->ev_end));
    return MSFM_OK;
}

// msfm_match_pairs and msfm_match_pairs_guided: the caller's msfm_result receives the match lists.
msfm_status match_pairs_to_result(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const msfm_params *params, msfm_result *out,
                                  const GuidedArgs *guided) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return MSFM_ERR_CUDA;
    if (!out || (!out->matches && out->match_capacity > 0)) return match_pairs_impl(ctx, pairs, n_pairs, params, nullptr, false, nullptr, guided);
    CallerBuffers cb{out->matches, out->good, out->match_capacity};
    OutSpec spec;
    spec.offsets = out->offsets;
    spec.ok = out->ok;
    spec.has_good = out->good != nullptr;
    spec.sink = caller_sink;
    spec.user = &cb;
    return match_pairs_impl(ctx, pairs, n_pairs, params, &spec, false, nullptr, guided);
}

}  // namespace

// =====================================================================================================================
extern "C" {

int32_t msfm_abi_version(void) { return MSFM_ABI_VERSION; }

const char *msfm_status_string(msfm_status s) {
    switch (s) {
        case MSFM_OK: return "ok";
        case MSFM_ERR_INVALID_ARG: return "invalid argument";
        case MSFM_ERR_CUDA: return "CUDA error";
        case MSFM_ERR_OUT_OF_MEMORY: return "out of memory";
        case MSFM_ERR_NOT_FOUND: return "image not uploaded";
        case MSFM_ERR_CAPACITY: return "capacity exceeded";
        case MSFM_ERR_UNSUPPORTED: return "unsupported device (sm_100 required)";
        case MSFM_ERR_EXISTS: return "image already uploaded";
    }
    return "unknown status";
}

const char *msfm_last_error(const msfm_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

msfm_status msfm_host_alloc(size_t bytes, void **out) {
    if (!out) return MSFM_ERR_INVALID_ARG;
    *out = nullptr;
    const cudaError_t e = cudaHostAlloc(out, bytes > 0 ? bytes : 1, cudaHostAllocPortable);
    return e == cudaSuccess ? MSFM_OK : (e == cudaErrorMemoryAllocation ? MSFM_ERR_OUT_OF_MEMORY : MSFM_ERR_CUDA);
}

msfm_status msfm_host_free(void *ptr) {
    if (!ptr) return MSFM_OK;
    return cudaFreeHost(ptr) == cudaSuccess ? MSFM_OK : MSFM_ERR_CUDA;
}

msfm_status msfm_device_memory(int32_t device, int64_t *free_bytes, int64_t *total_bytes) {
    size_t f = 0, t = 0;
    if (cudaSetDevice(device) != cudaSuccess || cudaMemGetInfo(&f, &t) != cudaSuccess) return MSFM_ERR_CUDA;
    if (free_bytes) *free_bytes = (int64_t)f;
    if (total_bytes) *total_bytes = (int64_t)t;
    return MSFM_OK;
}

msfm_status msfm_create(const msfm_config *cfg, msfm_ctx **out) {
    if (!cfg || !out) return MSFM_ERR_INVALID_ARG;
    *out = nullptr;
    if (cfg->max_images <= 0 || cfg->arena_rows <= 0) return MSFM_ERR_INVALID_ARG;
    if (cfg->reserved[0] || cfg->reserved[1] || cfg->reserved[2]) return MSFM_ERR_INVALID_ARG;
    if ((cfg->external_desc_arena == nullptr) != (cfg->external_norm_arena == nullptr)) return MSFM_ERR_INVALID_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || cfg->device < 0 || cfg->device >= ndev) return MSFM_ERR_CUDA;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess) return MSFM_ERR_CUDA;
    if (prop.major != 10) return MSFM_ERR_UNSUPPORTED;  // tcgen05/TMEM path only; no fallback by design
    if (cudaSetDevice(cfg->device) != cudaSuccess) return MSFM_ERR_CUDA;

    msfm_ctx *ctx = new (std::nothrow) msfm_ctx();
    if (!ctx) return MSFM_ERR_OUT_OF_MEMORY;
    ctx->device = cfg->device;
    ctx->num_sms = prop.multiProcessorCount;
    ctx->max_images = cfg->max_images;
    ctx->arena_rows = round_up(cfg->arena_rows, kAlignRows);
    ctx->images.resize(cfg->max_images);
    if (const char *dbg = getenv("MSFM_DEBUG_FLAGS")) {
        ctx->debug_flags = (uint32_t)strtoul(dbg, nullptr, 0);
#ifndef MSFM_EXPERIMENTS
        // Bits 1, 2 and 4 skip parts of the epilogue (timing experiments, WRONG match lists): compiled in only with
        // -DMSFM_EXPERIMENTS.  A production build honours the profiling bit (8: per-phase cycle counters) and says so.
        if (ctx->debug_flags & ~8u) {
            fprintf(stderr, "[msfm] MSFM_DEBUG_FLAGS=%s ignored: result-altering experiment flags need a -DMSFM_EXPERIMENTS build\n", dbg);
            ctx->debug_flags &= 8u;
        }
#endif
    }

    auto bail = [&](msfm_status st) {
        msfm_destroy(ctx);
        return st;
    };
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn) return bail(MSFM_ERR_CUDA);
    ctx->encode = reinterpret_cast<EncodeTiledFn>(fn);
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) return bail(MSFM_ERR_CUDA);
    if (cudaStreamCreateWithFlags(&ctx->upload_stream, cudaStreamNonBlocking) != cudaSuccess) return bail(MSFM_ERR_CUDA);
    if (cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess) return bail(MSFM_ERR_CUDA);
    if (cudaEventCreateWithFlags(&ctx->ev_copy, cudaEventDisableTiming) != cudaSuccess) return bail(MSFM_ERR_CUDA);
    if (cudaStreamCreateWithFlags(&ctx->d2h_stream, cudaStreamNonBlocking) != cudaSuccess) return bail(MSFM_ERR_CUDA);
    if (cudaEventCreate(&ctx->ev_d2h0) != cudaSuccess || cudaEventCreate(&ctx->ev_d2h1) != cudaSuccess) return bail(MSFM_ERR_CUDA);
    cudaEvent_t *evs[] = {&ctx->ev_begin, &ctx->ev_end, &ctx->ev_k0, &ctx->ev_k1, &ctx->ev_k2, &ctx->ev_k3, &ctx->ev_f1};
    for (cudaEvent_t *e : evs)
        if (cudaEventCreate(e) != cudaSuccess) return bail(MSFM_ERR_CUDA);
    if (cfg->external_desc_arena) {
        if (reinterpret_cast<uintptr_t>(cfg->external_desc_arena) % 1024 != 0) return bail(MSFM_ERR_INVALID_ARG);
        ctx->desc = static_cast<uint8_t *>(cfg->external_desc_arena);
        ctx->norms = static_cast<int32_t *>(cfg->external_norm_arena);
        ctx->arena_rows = cfg->arena_rows / kAlignRows * kAlignRows;
        ctx->own_arena = false;
    } else {
        if (cudaMalloc(&ctx->desc, (size_t)ctx->arena_rows * kDim) != cudaSuccess) return bail(MSFM_ERR_OUT_OF_MEMORY);
        if (cudaMalloc(&ctx->norms, (size_t)ctx->arena_rows * 4) != cudaSuccess) return bail(MSFM_ERR_OUT_OF_MEMORY);
        ctx->own_arena = true;
    }
    if (cfg->keep_float) {
        if (cudaMalloc(&ctx->fdesc, (size_t)ctx->arena_rows * kDim * sizeof(float)) != cudaSuccess) return bail(MSFM_ERR_OUT_OF_MEMORY);
        if (cudaMalloc(&ctx->resid, (size_t)ctx->arena_rows * sizeof(float)) != cudaSuccess) return bail(MSFM_ERR_OUT_OF_MEMORY);
        if (cudaMalloc(&ctx->img_rmax, (size_t)ctx->max_images * sizeof(float)) != cudaSuccess) return bail(MSFM_ERR_OUT_OF_MEMORY);
        if (cudaMemset(ctx->img_rmax, 0, (size_t)ctx->max_images * sizeof(float)) != cudaSuccess) return bail(MSFM_ERR_CUDA);
    }
    // one tensor map per image + one for the candidate scratch
    if (cudaMalloc(&ctx->d_maps, (size_t)(ctx->max_images + 1) * sizeof(CUtensorMap)) != cudaSuccess) return bail(MSFM_ERR_OUT_OF_MEMORY);
    if (cudaMallocHost(&ctx->h_maps, (size_t)(ctx->max_images + 1) * sizeof(CUtensorMap)) != cudaSuccess) return bail(MSFM_ERR_OUT_OF_MEMORY);
    for (const bool debug : {false, true})
        for (const bool collect : {false, true})
            for (const GateKind gate : {GateKind::none, GateKind::epipolar, GateKind::homography})
                if (cudaFuncSetAttribute(match_kernel(debug, collect, gate), cudaFuncAttributeMaxDynamicSharedMemorySize, KCfg::kSmemAlloc) != cudaSuccess)
                    return bail(MSFM_ERR_CUDA);
    if (cudaFuncSetAttribute(msfm::select_candidates_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msfm::kSelectSmemBytes) != cudaSuccess)
        return bail(MSFM_ERR_CUDA);
    if (ctx->debug_flags & 8u) {
        if (cudaMalloc(&ctx->dbg_stats.ptr, 512) != cudaSuccess) return bail(MSFM_ERR_OUT_OF_MEMORY);
        ctx->dbg_stats.bytes = 512;
        cudaMemset(ctx->dbg_stats.ptr, 0, 512);
    }
    *out = ctx;
    return MSFM_OK;
}

msfm_status msfm_destroy(msfm_ctx *ctx) {
    if (!ctx) return MSFM_OK;
    cudaSetDevice(ctx->device);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    if (ctx->d2h_stream) cudaStreamSynchronize(ctx->d2h_stream);
    if (ctx->upload_stream) cudaStreamSynchronize(ctx->upload_stream);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (const msfm_ctx::StageBuf &b : ctx->stage_pool) {
        cudaFree(b.ptr);
        cudaEventDestroy(b.done);
    }
    if (ctx->ev_copy) cudaEventDestroy(ctx->ev_copy);
    if (ctx->ev_d2h0) cudaEventDestroy(ctx->ev_d2h0);
    if (ctx->ev_d2h1) cudaEventDestroy(ctx->ev_d2h1);
    if (ctx->dbg_stats.ptr) {
        unsigned long long h[64] = {0};
        cudaMemcpy(h, ctx->dbg_stats.ptr, 512, cudaMemcpyDeviceToHost);
        const double wt = h[5] ? (double)h[5] : 1.0;
        fprintf(stderr, "[msfm debug] warp-tiles %llu | hot groups/warp-tile %.3f | cycles/warp-tile: wait-acc %.1f load+thresh %.1f "
                        "phase1 %.1f phase2 %.1f\n", h[5], h[0] / wt, h[1] / wt, h[2] / wt, h[3] / wt, h[4] / wt);
        fprintf(stderr, "[msfm debug] accumulator wait of an item's first tile: %.0f cycles per warp and item (%llu warp-items)\n", h[7] ? (double)h[6] / (double)h[7] : 0.0, h[7]);
        fprintf(stderr, "[msfm debug] epilogue warps by sub-partition, cycles per warp-tile (wait | work):");
        for (int qd = 0; qd < 4; ++qd) fprintf(stderr, " q%d %.0f|%.0f", qd, h[8 + 2 * qd] / (wt / 4.0), h[9 + 2 * qd] / (wt / 4.0));
        fprintf(stderr, "\n");
        fprintf(stderr, "[msfm debug] MMA issuers, cycles per tile waiting for (B tile | accumulator buffer):");
        for (int st = 0; st < 4; ++st) fprintf(stderr, " strip%d %.0f|%.0f", st, h[40 + 2 * st] / (wt / 16.0), h[41 + 2 * st] / (wt / 16.0));
        fprintf(stderr, "\n");
        cudaFree(ctx->dbg_stats.ptr);
    }
    if (ctx->fdesc) cudaFree(ctx->fdesc);
    if (ctx->resid) cudaFree(ctx->resid);
    if (ctx->img_rmax) cudaFree(ctx->img_rmax);
    DeviceBuf *bufs[] = {&ctx->knn_ids, &ctx->knn_dists, &ctx->knn_ids_b, &ctx->knn_dists_b, &ctx->band_q, &ctx->band_counts, &ctx->band_thr, &ctx->band_state, &ctx->band_events, &ctx->band_event_keys, &ctx->band_event_count, &ctx->cand_q, &ctx->cand_j, &ctx->cand_d0, &ctx->cand_good, &ctx->cand_counts, &ctx->cand_desc, &ctx->cand_ckeys, &ctx->colbest, &ctx->twin_counts, &ctx->tilemin,
                         &ctx->kp_xy, &ctx->knn, &ctx->matches, &ctx->good, &ctx->counts, &ctx->offsets,
                         &ctx->pairdesc, &ctx->items, &ctx->tight_matches, &ctx->tight_good, &ctx->tight_matches_b, &ctx->tight_good_b};
    for (DeviceBuf *b : bufs)
        if (b->ptr) cudaFree(b->ptr);
    if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
    if (ctx->own_arena) {
        if (ctx->desc) cudaFree(ctx->desc);
        if (ctx->norms) cudaFree(ctx->norms);
    }
    if (ctx->d_maps) cudaFree(ctx->d_maps);
    if (ctx->h_maps) cudaFreeHost(ctx->h_maps);
    cudaEvent_t evs[] = {ctx->ev_begin, ctx->ev_end, ctx->ev_k0, ctx->ev_k1, ctx->ev_k2, ctx->ev_k3, ctx->ev_f1};
    for (cudaEvent_t e : evs)
        if (e) cudaEventDestroy(e);
    for (const UploadMark &m : ctx->marks) cudaEventDestroy(m.ev);
    for (cudaEvent_t e : ctx->event_pool) cudaEventDestroy(e);
    if (ctx->upload_stream) cudaStreamDestroy(ctx->upload_stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->d2h_stream) cudaStreamDestroy(ctx->d2h_stream);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return MSFM_OK;
}

// ---------------------------------------------------------------------------------------------------- table uploads
// Everything that changes the packed table (packer launches, tensor-map writes, pad rows) runs on the context's UPLOAD
// stream, so that staging overlaps matching on the main stream; the host->device copies run on the copy stream, and the
// upload stream waits for them before the packers.  The synchronous entry points wait for the upload stream before they
// return (the images are then simply "ready"); the *_async ones return at once and leave an upload mark — an event on
// the upload stream plus a sequence number stored in the images it covers.  A matching launch makes the main stream wait
// for the newest mark among the images it touches (marks complete in order).
static msfm_status finish_upload_sync(msfm_ctx *ctx) {
    MSFM_CUDA(ctx, cudaStreamSynchronize(ctx->upload_stream));
    return MSFM_OK;
}

static msfm_status leave_upload_mark(msfm_ctx *ctx, const std::vector<int32_t> &ids, cudaStream_t on = nullptr) {
    if (ids.empty()) return MSFM_OK;
    cudaEvent_t ev = nullptr;
    if (!ctx->event_pool.empty()) { ev = ctx->event_pool.back(); ctx->event_pool.pop_back(); }
    else MSFM_CUDA(ctx, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    const cudaError_t e = cudaEventRecord(ev, on ? on : ctx->upload_stream);
    if (e != cudaSuccess) {
        ctx->event_pool.push_back(ev);
        return fail(ctx, MSFM_ERR_CUDA, "cudaEventRecord failed: %s", cudaGetErrorString(e));
    }
    const uint64_t seq = ++ctx->upload_seq;
    ctx->marks.push_back({seq, ev});
    for (int32_t id : ids) ctx->images[id].ready_seq = seq;
    return MSFM_OK;
}

// Undo reserve_locked for the images of a call that failed half-way: an image must never stay "present" with unwritten rows.
static void unreserve_locked(msfm_ctx *ctx, const std::vector<int32_t> &ids) {
    for (int32_t id : ids) {
        ImageSlot &s = ctx->images[id];
        if (!s.present) continue;
        arena_free(ctx, s.off, s.rows_padded);
        s = ImageSlot{};
    }
}

// A CUDA failure after the images in `reserved` were reserved: once no copy or packer launch can still write into their
// rows, they are rolled back, and `reserved` is left empty.
static msfm_status fail_reserved(msfm_ctx *ctx, std::vector<int32_t> &reserved, cudaError_t e) {
    cudaStreamSynchronize(ctx->copy_stream);
    cudaStreamSynchronize(ctx->upload_stream);
    unreserve_locked(ctx, reserved);
    reserved.clear();
    return fail(ctx, e == cudaErrorMemoryAllocation ? MSFM_ERR_OUT_OF_MEMORY : MSFM_ERR_CUDA, "table upload failed: %s", cudaGetErrorString(e));
}

msfm_status msfm_reserve(msfm_ctx *ctx, int32_t image_id, int32_t rows, int64_t *row_offset) {
    return msfm_reserve_batch(ctx, 1, &image_id, &rows, row_offset);
}

static msfm_status reserve_batch_locked(msfm_ctx *ctx, int32_t n, const int32_t *image_ids, const int32_t *rows, int64_t *row_offsets) {
    if (n < 0 || (n > 0 && (!image_ids || !rows))) return fail(ctx, MSFM_ERR_INVALID_ARG, "msfm_reserve_batch: null argument");
    MSFM_CUDA(ctx, cudaSetDevice(ctx->device));
    msfm_status st = MSFM_OK;
    for (int32_t i = 0; i < n && st == MSFM_OK; ++i) {
        int64_t off = 0;
        if ((st = reserve_locked(ctx, image_ids[i], rows[i], &off)) != MSFM_OK) break;
        const ImageSlot &s = ctx->images[image_ids[i]];
        if (s.rows_padded > s.rows) {
            msfm::init_pad_kernel<<<8, 256, 0, ctx->upload_stream>>>(s.rows, s.rows_padded, ctx->desc + off * kDim, ctx->norms + off);
            const cudaError_t e = cudaGetLastError();
            if (e != cudaSuccess) {
                std::vector<int32_t> one{image_ids[i]};
                return fail_reserved(ctx, one, e);
            }
        }
        if (row_offsets) row_offsets[i] = off;
    }
    return st;
}

msfm_status msfm_reserve_batch(msfm_ctx *ctx, int32_t n, const int32_t *image_ids, const int32_t *rows, int64_t *row_offsets) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    const msfm_status st = reserve_batch_locked(ctx, n, image_ids, rows, row_offsets);
    // pad rows and tensor maps are in place when the call returns: a foreign writer (a collective) may fill the rows at once
    const msfm_status fin = finish_upload_sync(ctx);
    return st != MSFM_OK ? st : fin;
}

// A float staging buffer of at least `bytes` that no queued packer launch still reads: a pool buffer whose last user's
// packers have run (an event never recorded counts as complete), else a new one of at least 64 MiB.
static cudaError_t take_stage(msfm_ctx *ctx, size_t bytes, msfm_ctx::StageBuf **out) {
    for (msfm_ctx::StageBuf &b : ctx->stage_pool)
        if (b.bytes >= bytes && cudaEventQuery(b.done) == cudaSuccess) {
            *out = &b;
            return cudaSuccess;
        }
    msfm_ctx::StageBuf nb{nullptr, std::max<size_t>(bytes, (size_t)64 << 20), nullptr};
    cudaError_t e = cudaMalloc(&nb.ptr, nb.bytes);
    if (e != cudaSuccess) return e;
    if ((e = cudaEventCreateWithFlags(&nb.done, cudaEventDisableTiming)) != cudaSuccess) {
        cudaFree(nb.ptr);
        return e;
    }
    ctx->stage_pool.push_back(nb);
    *out = &ctx->stage_pool.back();
    return cudaSuccess;
}

// The one path of the five upload entry points: images [0, n) of a call, u8 or float rows `strides[i]` elements apart
// (strides null: dense rows).  `dense_only` names an entry point that refuses strided rows.
//  1. Each image is checked and reserved in turn; the first failing one ends the loop, the images before it are uploaded.
//  2. Every destination is dense: u8 rows go to the arena, float rows to the retained float rows of a keep_float context,
//     else to one staging buffer of this call.
//  3. The host->device copies are queued back to back on the copy stream, so they never wait behind a packer launch that
//     waits for an SM (the matching kernel is persistent).  Images adjacent both in host memory and in the destination
//     are one copy; strided rows are one 2-D copy each.
//  4. The packers follow on the upload stream: u8 rows are keyed in place, one launch per copy (images start on
//     multiples of kAlignRows, so row % 8 and with it the column keys do not depend on where a copy starts; only its
//     last image can have pad rows); float rows are quantised per image (each image has its own largest residual).
// A CUDA failure rolls back every image of the call.  `uploaded` receives the images queued.
extern "C++" {  // a template cannot have C linkage
template <typename T>
static msfm_status upload_locked(msfm_ctx *ctx, int32_t n, const int32_t *image_ids, const T *const *descs, const int32_t *rows,
                                 const int64_t *strides, float scale, const char *dense_only, std::vector<int32_t> &uploaded) {
    constexpr bool kFloat = std::is_same<T, float>::value;
    MSFM_CUDA(ctx, cudaSetDevice(ctx->device));
    struct Job { int32_t id; const T *src; int64_t stride; T *dst; };
    std::vector<Job> jobs;
    msfm_status st = MSFM_OK;
    for (int32_t i = 0; i < n; ++i) {
        const int64_t stride = strides ? strides[i] : kDim;
        if (stride != kDim && dense_only) { st = fail(ctx, MSFM_ERR_INVALID_ARG, "%s takes contiguous 128-byte rows only", dense_only); break; }
        if (rows[i] > 0 && !descs[i] && stride == kDim) { st = fail(ctx, MSFM_ERR_INVALID_ARG, "null descriptors"); break; }
        if ((rows[i] > 0 && !descs[i]) || stride < kDim) {
            st = fail(ctx, MSFM_ERR_INVALID_ARG, "null descriptors or stride < 128 %s", kFloat ? "floats" : "bytes");
            break;
        }
        if ((st = reserve_locked(ctx, image_ids[i], rows[i], nullptr)) != MSFM_OK) break;
        uploaded.push_back(image_ids[i]);
        jobs.push_back({image_ids[i], descs[i], stride, nullptr});
    }
    cudaError_t e = cudaSuccess;
    msfm_ctx::StageBuf *stage = nullptr;
    if (kFloat && !ctx->fdesc) {
        size_t bytes = 0;
        for (const Job &j : jobs) bytes += (size_t)ctx->images[j.id].rows * kDim * sizeof(float);
        if (bytes > 0 && (e = take_stage(ctx, bytes, &stage)) != cudaSuccess) return fail_reserved(ctx, uploaded, e);
    }
    struct Run { const T *src; int64_t stride; T *dst; int64_t off, rows, rows_padded; };
    std::vector<Run> runs;
    size_t stage_pos = 0;
    for (Job &j : jobs) {
        ImageSlot &s = ctx->images[j.id];
        if constexpr (kFloat) {
            if (ctx->fdesc) {
                j.dst = ctx->fdesc + s.off * kDim;
                if (s.rows > 0) {
                    s.has_float = true;
                    s.scale = scale;
                }
            } else {
                j.dst = static_cast<float *>(stage ? stage->ptr : nullptr) + stage_pos;
                stage_pos += (size_t)s.rows * kDim;
            }
        } else {
            j.dst = ctx->desc + s.off * kDim;
        }
        Run *last = runs.empty() ? nullptr : &runs.back();
        if (last && j.stride == kDim && last->stride == kDim && j.src == last->src + last->rows * kDim &&
            j.dst == last->dst + last->rows * kDim && last->rows + s.rows_padded < (int64_t)INT32_MAX) {
            last->rows += s.rows;
            last->rows_padded += s.rows_padded;
        } else {
            runs.push_back({j.src, j.stride, j.dst, s.off, s.rows, s.rows_padded});
        }
    }
    for (const Run &r : runs) {
        if (r.rows == 0) continue;
        e = r.stride == kDim ? cudaMemcpyAsync(r.dst, r.src, (size_t)r.rows * kDim * sizeof(T), cudaMemcpyHostToDevice, ctx->copy_stream)
                             : cudaMemcpy2DAsync(r.dst, kDim * sizeof(T), r.src, (size_t)r.stride * sizeof(T), kDim * sizeof(T), (size_t)r.rows,
                                                 cudaMemcpyHostToDevice, ctx->copy_stream);
        if (e != cudaSuccess) return fail_reserved(ctx, uploaded, e);
    }
    if (!jobs.empty()) {
        if ((e = cudaEventRecord(ctx->ev_copy, ctx->copy_stream)) != cudaSuccess) return fail_reserved(ctx, uploaded, e);
        if ((e = cudaStreamWaitEvent(ctx->upload_stream, ctx->ev_copy, 0)) != cudaSuccess) return fail_reserved(ctx, uploaded, e);
    }
    if constexpr (kFloat) {
        for (const Job &j : jobs) {
            const ImageSlot &s = ctx->images[j.id];
            const int blocks = std::max(1, std::min(4 * ctx->num_sms, (s.rows_padded + 7) / 8));
            msfm::pack_f32_kernel<<<blocks, 256, 0, ctx->upload_stream>>>(j.dst, s.rows, s.rows_padded, scale, ctx->desc + s.off * kDim, ctx->norms + s.off,
                                                                          ctx->resid ? ctx->resid + s.off : nullptr, ctx->img_rmax ? ctx->img_rmax + j.id : nullptr);
            if ((e = cudaGetLastError()) != cudaSuccess) return fail_reserved(ctx, uploaded, e);
        }
        if (stage && (e = cudaEventRecord(stage->done, ctx->upload_stream)) != cudaSuccess) return fail_reserved(ctx, uploaded, e);
    } else {
        for (const Run &r : runs) {
            const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(8 * ctx->num_sms, (r.rows_padded + 7) / 8));
            msfm::pack_u8_kernel<<<blocks, 256, 0, ctx->upload_stream>>>((int)r.rows, (int)r.rows_padded, r.dst, ctx->norms + r.off);
            if ((e = cudaGetLastError()) != cudaSuccess) return fail_reserved(ctx, uploaded, e);
        }
    }
    return st;
}
}  // extern "C++"

msfm_status msfm_upload_u8(msfm_ctx *ctx, int32_t image_id, const uint8_t *desc, int32_t rows, int64_t row_stride_bytes) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if ((rows > 0 && !desc) || row_stride_bytes < kDim) return fail(ctx, MSFM_ERR_INVALID_ARG, "null descriptors or stride < 128 bytes");
    std::vector<int32_t> uploaded;
    const msfm_status st = upload_locked(ctx, 1, &image_id, &desc, &rows, &row_stride_bytes, 0.0f, nullptr, uploaded);
    if (st != MSFM_OK) return st;
    return finish_upload_sync(ctx);  // the caller may free `desc` on return
}

msfm_status msfm_upload_u8_batch(msfm_ctx *ctx, int32_t n, const int32_t *image_ids, const uint8_t *const *descs, const int32_t *rows,
                                 const int64_t *row_stride_bytes) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n < 0 || (n > 0 && (!image_ids || !descs || !rows))) return fail(ctx, MSFM_ERR_INVALID_ARG, "msfm_upload_u8_batch: null argument");
    std::vector<int32_t> uploaded;
    const msfm_status st = upload_locked(ctx, n, image_ids, descs, rows, row_stride_bytes, 0.0f, nullptr, uploaded);
    const msfm_status fin = finish_upload_sync(ctx);  // one sync for the batch: the caller may free every `descs[i]` on return
    return st != MSFM_OK ? st : fin;
}

msfm_status msfm_upload_u8_batch_async(msfm_ctx *ctx, int32_t n, const int32_t *image_ids, const uint8_t *const *descs, const int32_t *rows,
                                       const int64_t *row_stride_bytes) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n < 0 || (n > 0 && (!image_ids || !descs || !rows))) return fail(ctx, MSFM_ERR_INVALID_ARG, "msfm_upload_u8_batch: null argument");
    std::vector<int32_t> uploaded;
    const msfm_status st = upload_locked(ctx, n, image_ids, descs, rows, row_stride_bytes, 0.0f, "msfm_upload_u8_batch_async", uploaded);
    const msfm_status mk = leave_upload_mark(ctx, uploaded);
    return st != MSFM_OK ? st : mk;
}

msfm_status msfm_sync(msfm_ctx *ctx) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    MSFM_CUDA(ctx, cudaSetDevice(ctx->device));
    MSFM_CUDA(ctx, cudaStreamSynchronize(ctx->upload_stream));
    MSFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    recycle_marks(ctx);
    return MSFM_OK;
}

msfm_status msfm_upload_f32(msfm_ctx *ctx, int32_t image_id, const float *desc, int32_t rows, int64_t row_stride_floats, float scale) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if ((rows > 0 && !desc) || row_stride_floats < kDim || !(scale > 0.0f))
        return fail(ctx, MSFM_ERR_INVALID_ARG, "null descriptors, stride < 128 floats or scale <= 0");
    std::vector<int32_t> uploaded;
    const msfm_status st = upload_locked(ctx, 1, &image_id, &desc, &rows, &row_stride_floats, scale, nullptr, uploaded);
    if (st != MSFM_OK) return st;
    return finish_upload_sync(ctx);
}

// Several float images (dense 128-float rows) without a host wait: the rows must sit in page-locked memory and stay
// valid until msfm_sync() or a later call that returns results.
msfm_status msfm_upload_f32_batch_async(msfm_ctx *ctx, int32_t n, const int32_t *image_ids, const float *const *descs, const int32_t *rows,
                                        float scale) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n < 0 || (n > 0 && (!image_ids || !descs || !rows)) || !(scale > 0.0f))
        return fail(ctx, MSFM_ERR_INVALID_ARG, "msfm_upload_f32_batch_async: null argument or scale <= 0");
    std::vector<int32_t> uploaded;
    const msfm_status st = upload_locked(ctx, n, image_ids, descs, rows, nullptr, scale, nullptr, uploaded);
    const msfm_status mk = leave_upload_mark(ctx, uploaded);
    return st != MSFM_OK ? st : mk;
}

msfm_status msfm_release(msfm_ctx *ctx, int32_t image_id) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    msfm_status st = check_image_id(ctx, image_id, true);
    if (st != MSFM_OK) return st;
    MSFM_CUDA(ctx, cudaSetDevice(ctx->device));
    MSFM_CUDA(ctx, cudaStreamSynchronize(ctx->upload_stream));
    MSFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ImageSlot &s = ctx->images[image_id];
    arena_free(ctx, s.off, s.rows_padded);
    s = ImageSlot{};
    // the next image under this id starts from a zero largest residual (the packer only raises it)
    if (ctx->img_rmax) MSFM_CUDA(ctx, cudaMemsetAsync(ctx->img_rmax + image_id, 0, sizeof(float), ctx->upload_stream));
    return MSFM_OK;
}

msfm_status msfm_release_all(msfm_ctx *ctx) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    MSFM_CUDA(ctx, cudaSetDevice(ctx->device));
    MSFM_CUDA(ctx, cudaStreamSynchronize(ctx->upload_stream));
    MSFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (ImageSlot &s : ctx->images) s = ImageSlot{};
    if (ctx->img_rmax) MSFM_CUDA(ctx, cudaMemsetAsync(ctx->img_rmax, 0, (size_t)ctx->max_images * sizeof(float), ctx->upload_stream));
    ctx->free_list.clear();
    ctx->rows_high_water = 0;
    recycle_marks(ctx);
    return MSFM_OK;
}

msfm_status msfm_image_info(const msfm_ctx *ctx_c, int32_t image_id, int32_t *rows, int64_t *row_offset) {
    msfm_ctx *ctx = const_cast<msfm_ctx *>(ctx_c);
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    msfm_status st = check_image_id(ctx, image_id, true);
    if (st != MSFM_OK) return st;
    if (rows) *rows = ctx->images[image_id].rows;
    if (row_offset) *row_offset = ctx->images[image_id].off;
    return MSFM_OK;
}

msfm_status msfm_table_ptrs(const msfm_ctx *ctx, void **desc_arena, void **norm_arena, int64_t *arena_rows, int64_t *rows_used) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    if (desc_arena) *desc_arena = ctx->desc;
    if (norm_arena) *norm_arena = ctx->norms;
    if (arena_rows) *arena_rows = ctx->arena_rows;
    if (rows_used) *rows_used = ctx->rows_high_water;
    return MSFM_OK;
}

msfm_status msfm_download_packed(msfm_ctx *ctx, int32_t image_id, uint8_t *desc_out, uint32_t *norms_out) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    msfm_status st = check_image_id(ctx, image_id, true);
    if (st != MSFM_OK) return st;
    MSFM_CUDA(ctx, cudaSetDevice(ctx->device));
    const ImageSlot &s = ctx->images[image_id];
    MSFM_CUDA(ctx, cudaStreamSynchronize(ctx->upload_stream));
    if (desc_out && s.rows) MSFM_CUDA(ctx, cudaMemcpyAsync(desc_out, ctx->desc + s.off * kDim, (size_t)s.rows * kDim, cudaMemcpyDeviceToHost, ctx->stream));
    if (norms_out && s.rows) MSFM_CUDA(ctx, cudaMemcpyAsync(norms_out, ctx->norms + s.off, (size_t)s.rows * 4, cudaMemcpyDeviceToHost, ctx->stream));
    MSFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (norms_out)  // the table stores column keys; hand back plain squared norms
        for (int32_t r = 0; r < s.rows; ++r) norms_out[r] = (uint32_t)msfm::ckey_to_norm((int32_t)norms_out[r]);
    return MSFM_OK;
}

msfm_status msfm_knn2(msfm_ctx *ctx, int32_t ref_id, int32_t query_id, int32_t *ids, float *dists) {
    // the one-pair, integer-distance form of msfm_knn2_pairs (the caller's arrays hold the query image's rows)
    const msfm_pair pair{ref_id, query_id};
    int64_t offsets[2];
    return knn2_pairs_impl(ctx, &pair, 1, 0u, offsets, ids, dists, INT64_MAX);
}

msfm_status msfm_knn2_pairs(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, uint32_t flags, int64_t *offsets, int32_t *ids,
                            float *dists, int64_t row_capacity) {
    return knn2_pairs_impl(ctx, pairs, n_pairs, flags, offsets, ids, dists, row_capacity);
}

msfm_status msfm_colbest(msfm_ctx *ctx, int32_t ref_id, int32_t query_id, int32_t *best_query, float *best_dist) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (!best_query || !best_dist) return fail(ctx, MSFM_ERR_INVALID_ARG, "null output buffer");
    MSFM_CUDA(ctx, cudaSetDevice(ctx->device));
    // best query of every reference row = nearest neighbour of that row among the query rows (roles swapped)
    BatchPlan plan;
    msfm_status st = knn_single(ctx, query_id, ref_id, plan);
    if (st != MSFM_OK) return st;
    const int m = (int)plan.query_rows;
    if (m == 0) return MSFM_OK;
    if ((st = ensure(ctx, ctx->tight_matches, (size_t)m * 4)) != MSFM_OK) return st;
    if ((st = ensure(ctx, ctx->matches, (size_t)m * 4)) != MSFM_OK) return st;
    int32_t *d_best = static_cast<int32_t *>(ctx->tight_matches.ptr);
    float *d_dist = static_cast<float *>(ctx->matches.ptr);
    msfm::knn_best_kernel<<<(m + 255) / 256, 256, 0, ctx->stream>>>(static_cast<const int4 *>(ctx->knn.ptr), m, d_best, d_dist);
    MSFM_CUDA(ctx, cudaGetLastError());
    MSFM_CUDA(ctx, cudaMemcpyAsync(best_query, d_best, (size_t)m * 4, cudaMemcpyDeviceToHost, ctx->stream));
    MSFM_CUDA(ctx, cudaMemcpyAsync(best_dist, d_dist, (size_t)m * 4, cudaMemcpyDeviceToHost, ctx->stream));
    MSFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if ((st = accumulate_kernel_time(ctx, ctx->ev_k0, ctx->ev_k1)) != MSFM_OK) return st;
    return MSFM_OK;
}

msfm_status msfm_match_pairs(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const msfm_params *params, msfm_result *out) {
    return match_pairs_to_result(ctx, pairs, n_pairs, params, out, nullptr);
}

msfm_status msfm_match_pairs_guided(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const msfm_params *params,
                                    const double (*F)[9], float th_epipolar, const float *const *image_xy,
                                    const int32_t *image_npts, int32_t n_images, msfm_result *out) {
    const GuidedArgs g{GateKind::epipolar, F, th_epipolar, image_xy, image_npts, n_images};
    return match_pairs_to_result(ctx, pairs, n_pairs, params, out, &g);
}

msfm_status msfm_match_pairs_guided_homography(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const msfm_params *params,
                                               const double (*H)[9], float th_transfer, const float *const *image_xy,
                                               const int32_t *image_npts, int32_t n_images, msfm_result *out) {
    const GuidedArgs g{GateKind::homography, H, th_transfer, image_xy, image_npts, n_images};
    return match_pairs_to_result(ctx, pairs, n_pairs, params, out, &g);
}

msfm_status msfm_internal_match_pairs_sink(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const msfm_params *params, int64_t *offsets,
                                           int32_t *ok, int want_good, msfm_sink_fn sink, void *user) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return MSFM_ERR_CUDA;
    OutSpec spec;
    spec.offsets = offsets;
    spec.ok = ok;
    spec.has_good = want_good != 0;
    spec.sink = sink;
    spec.user = user;
    return match_pairs_impl(ctx, pairs, n_pairs, params, &spec, false, nullptr);
}

msfm_status msfm_reserve_batch_async(msfm_ctx *ctx, int32_t n, const int32_t *image_ids, const int32_t *rows, int64_t *row_offsets) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    const msfm_status st = reserve_batch_locked(ctx, n, image_ids, rows, row_offsets);
    // tensor maps and pad rows are queued on the upload stream: matching launches that touch these images wait for them
    std::vector<int32_t> ids;
    for (int32_t i = 0; i < n && image_ids; ++i)
        if (image_ids[i] >= 0 && image_ids[i] < ctx->max_images && ctx->images[image_ids[i]].present) ids.push_back(image_ids[i]);
    const msfm_status mk = (st == MSFM_OK) ? leave_upload_mark(ctx, ids) : MSFM_OK;
    return st != MSFM_OK ? st : mk;
}

msfm_status msfm_internal_mark_on_stream(msfm_ctx *ctx, int32_t n, const int32_t *image_ids, cudaStream_t stream) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n < 0 || (n > 0 && !image_ids)) return fail(ctx, MSFM_ERR_INVALID_ARG, "null image list");
    MSFM_CUDA(ctx, cudaSetDevice(ctx->device));
    std::vector<int32_t> ids;
    for (int32_t i = 0; i < n; ++i) {
        const msfm_status st = check_image_id(ctx, image_ids[i], true);
        if (st != MSFM_OK) return st;
        ids.push_back(image_ids[i]);
    }
    return leave_upload_mark(ctx, ids, stream);
}

msfm_status msfm_match_pairs_resident(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const msfm_params *params,
                                      int64_t *n_matches_total) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return MSFM_ERR_CUDA;
    return match_pairs_impl(ctx, pairs, n_pairs, params, nullptr, true, n_matches_total);
}

msfm_status msfm_last_timing(const msfm_ctx *ctx, msfm_timing *out) {
    if (!ctx || !out) return MSFM_ERR_INVALID_ARG;
    *out = ctx->timing;
    return MSFM_OK;
}

msfm_status msfm_get_stream(const msfm_ctx *ctx, void **cuda_stream) {
    if (!ctx || !cuda_stream) return MSFM_ERR_INVALID_ARG;
    *cuda_stream = static_cast<void *>(ctx->stream);
    return MSFM_OK;
}

msfm_status msfm_get_upload_stream(const msfm_ctx *ctx, void **cuda_stream) {
    if (!ctx || !cuda_stream) return MSFM_ERR_INVALID_ARG;
    *cuda_stream = static_cast<void *>(ctx->upload_stream);
    return MSFM_OK;
}

msfm_status msfm_wait_event(msfm_ctx *ctx, void *cuda_event) {
    if (!ctx || !cuda_event) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    MSFM_CUDA(ctx, cudaSetDevice(ctx->device));
    MSFM_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, static_cast<cudaEvent_t>(cuda_event), 0));
    return MSFM_OK;
}

msfm_status msfm_test_disable_pruning(msfm_ctx *ctx, int32_t on) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    ctx->no_prune = on != 0;
    return MSFM_OK;
}

msfm_status msfm_test_force_twin_pass(msfm_ctx *ctx, int32_t on) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    ctx->force_twin = on != 0;
    return MSFM_OK;
}

msfm_status msfm_test_set_band_event_cap(msfm_ctx *ctx, int64_t cap) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    ctx->band_event_cap_override = cap;
    return MSFM_OK;
}

msfm_status msfm_test_last_knn_stats(msfm_ctx *ctx, int64_t *events, int32_t *brute_force_batches) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (events) *events = ctx->knn_events;
    if (brute_force_batches) *brute_force_batches = ctx->knn_brute_batches;
    return MSFM_OK;
}

// The three geometric-verification entry points share validation, staging and timing; `call` picks the model and the
// meaning of `keep`.
enum class GeoCall { verify, ransac, homography };
static msfm_status geo_impl(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const int64_t *offsets, const int32_t (*matches)[2],
                            const uint8_t *good, const float *const *image_xy, const int32_t *image_npts, int32_t n_images,
                            const msfm_geo_params *gp, int32_t *pair_ok, int32_t *pair_inliers, uint8_t *keep, double *F, GeoCall call);

msfm_status msfm_geo_verify(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const int64_t *offsets,
                            const int32_t (*matches)[2], const uint8_t *good, const float *const *image_xy,
                            const int32_t *image_npts, int32_t n_images, const msfm_geo_params *gp, int32_t *pair_ok,
                            int32_t *pair_inliers, uint8_t *keep, double *F) {
    return geo_impl(ctx, pairs, n_pairs, offsets, matches, good, image_xy, image_npts, n_images, gp, pair_ok, pair_inliers, keep, F, GeoCall::verify);
}

msfm_status msfm_geo_ransac(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const int64_t *offsets,
                            const int32_t (*matches)[2], const uint8_t *use, const float *const *image_xy,
                            const int32_t *image_npts, int32_t n_images, const msfm_geo_params *gp, int32_t *pair_ok,
                            int32_t *pair_inliers, uint8_t *inlier_mask, double *F) {
    return geo_impl(ctx, pairs, n_pairs, offsets, matches, use, image_xy, image_npts, n_images, gp, pair_ok, pair_inliers, inlier_mask, F, GeoCall::ransac);
}

msfm_status msfm_geo_homography(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const int64_t *offsets,
                                const int32_t (*matches)[2], const uint8_t *use, const float *const *image_xy,
                                const int32_t *image_npts, int32_t n_images, const msfm_geo_params *gp, int32_t *pair_ok,
                                int32_t *pair_inliers, uint8_t *inlier_mask, double *H) {
    return geo_impl(ctx, pairs, n_pairs, offsets, matches, use, image_xy, image_npts, n_images, gp, pair_ok, pair_inliers, inlier_mask, H,
                    GeoCall::homography);
}

static msfm_status geo_impl(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const int64_t *offsets, const int32_t (*matches)[2],
                            const uint8_t *good, const float *const *image_xy, const int32_t *image_npts, int32_t n_images,
                            const msfm_geo_params *gp, int32_t *pair_ok, int32_t *pair_inliers, uint8_t *keep, double *F, GeoCall call) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    const char *fn = call == GeoCall::homography ? "msfm_geo_homography" : call == GeoCall::ransac ? "msfm_geo_ransac" : "msfm_geo_verify";
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n_pairs < 0 || !gp || (n_pairs > 0 && (!pairs || !offsets || !pair_ok || !pair_inliers || !image_xy || !image_npts)))
        return fail(ctx, MSFM_ERR_INVALID_ARG, "%s: null argument", fn);
    if (n_pairs == 0) return MSFM_OK;
    const int64_t total = offsets[n_pairs];
    if (total < 0 || (total > 0 && (!matches || !good || !keep))) return fail(ctx, MSFM_ERR_INVALID_ARG, "%s: null match buffers", fn);
    MSFM_CUDA(ctx, cudaSetDevice(ctx->device));
    // keypoints of the images the pairs touch, concatenated
    std::vector<int64_t> xy_off((size_t)n_images + 1, 0);
    std::vector<char> used((size_t)n_images, 0);
    for (int64_t p = 0; p < n_pairs; ++p) {
        if (pairs[p].ref < 0 || pairs[p].ref >= n_images || pairs[p].query < 0 || pairs[p].query >= n_images)
            return fail(ctx, MSFM_ERR_INVALID_ARG, "%s: pair %lld names an image outside [0, %d)", fn, (long long)p, n_images);
        used[pairs[p].ref] = used[pairs[p].query] = 1;
    }
    for (int32_t i = 0; i < n_images; ++i) {
        if (used[i] && (image_npts[i] < 0 || (image_npts[i] > 0 && !image_xy[i])))
            return fail(ctx, MSFM_ERR_INVALID_ARG, "%s: image %d has no keypoints", fn, i);
        xy_off[i + 1] = xy_off[i] + (used[i] ? image_npts[i] : 0);
    }
    for (int64_t p = 0; p < n_pairs; ++p)
        for (int64_t k = offsets[p]; k < offsets[p + 1]; ++k)
            if (matches[k][0] < 0 || matches[k][0] >= image_npts[pairs[p].ref] || matches[k][1] < 0 || matches[k][1] >= image_npts[pairs[p].query])
                return fail(ctx, MSFM_ERR_INVALID_ARG, "%s: match %lld of pair %lld indexes past the keypoints", fn, (long long)k, (long long)p);
    const int64_t n_xy = xy_off[n_images];
    std::vector<float> xy((size_t)std::max<int64_t>(n_xy, 1) * 2);
    for (int32_t i = 0; i < n_images; ++i)
        if (used[i] && image_npts[i] > 0) memcpy(xy.data() + 2 * xy_off[i], image_xy[i], (size_t)image_npts[i] * 8);
    std::vector<int32_t> pimg((size_t)n_pairs * 2);
    for (int64_t p = 0; p < n_pairs; ++p) { pimg[2 * p] = pairs[p].ref; pimg[2 * p + 1] = pairs[p].query; }

    // per-call device buffers, released on every exit path
    struct Scratch {
        msfm_ctx *ctx;
        DeviceBuf xy, xyoff, off, m, g, pimg, ok, inl, keep, F;
        ~Scratch() {
            cudaStreamSynchronize(ctx->stream);
            for (DeviceBuf *b : {&xy, &xyoff, &off, &m, &g, &pimg, &ok, &inl, &keep, &F})
                if (b->ptr) cudaFree(b->ptr);
        }
    } d{ctx};
    msfm_status st;
    const size_t tot = (size_t)std::max<int64_t>(total, 1);
    if ((st = ensure(ctx, d.xy, xy.size() * 4)) != MSFM_OK || (st = ensure(ctx, d.xyoff, xy_off.size() * 8)) != MSFM_OK ||
        (st = ensure(ctx, d.off, (size_t)(n_pairs + 1) * 8)) != MSFM_OK || (st = ensure(ctx, d.m, tot * 8)) != MSFM_OK ||
        (st = ensure(ctx, d.g, tot)) != MSFM_OK || (st = ensure(ctx, d.pimg, pimg.size() * 4)) != MSFM_OK ||
        (st = ensure(ctx, d.ok, (size_t)n_pairs * 4)) != MSFM_OK || (st = ensure(ctx, d.inl, (size_t)n_pairs * 4)) != MSFM_OK ||
        (st = ensure(ctx, d.keep, tot)) != MSFM_OK || (st = ensure(ctx, d.F, (size_t)n_pairs * 72)) != MSFM_OK)
        return st;
    MSFM_CUDA(ctx, cudaMemcpyAsync(d.xy.ptr, xy.data(), xy.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    MSFM_CUDA(ctx, cudaMemcpyAsync(d.xyoff.ptr, xy_off.data(), xy_off.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    MSFM_CUDA(ctx, cudaMemcpyAsync(d.off.ptr, offsets, (size_t)(n_pairs + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    if (total > 0) {
        MSFM_CUDA(ctx, cudaMemcpyAsync(d.m.ptr, matches, (size_t)total * 8, cudaMemcpyHostToDevice, ctx->stream));
        MSFM_CUDA(ctx, cudaMemcpyAsync(d.g.ptr, good, (size_t)total, cudaMemcpyHostToDevice, ctx->stream));
    }
    MSFM_CUDA(ctx, cudaMemcpyAsync(d.pimg.ptr, pimg.data(), pimg.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    msfm::GeoParams kp;
    kp.offsets = static_cast<const int64_t *>(d.off.ptr);
    kp.matches = static_cast<const int2 *>(d.m.ptr);
    kp.good = static_cast<const uint8_t *>(d.g.ptr);
    kp.pair_img = static_cast<const int32_t *>(d.pimg.ptr);
    kp.xy = static_cast<const float *>(d.xy.ptr);
    kp.xy_off = static_cast<const int64_t *>(d.xyoff.ptr);
    kp.th = gp->th_epipolar;
    kp.min_points = gp->min_points;
    kp.min_inliers = gp->min_inliers;
    kp.iters = gp->iters > 0 ? gp->iters : 1024;
    kp.seed = gp->seed;
    kp.pair_base = gp->pair_index_base;
    kp.stage_b = call == GeoCall::verify ? 1 : 0;
    kp.pair_ok = static_cast<int32_t *>(d.ok.ptr);
    kp.pair_inliers = static_cast<int32_t *>(d.inl.ptr);
    kp.keep = static_cast<uint8_t *>(d.keep.ptr);
    kp.F = static_cast<double *>(d.F.ptr);
    MSFM_CUDA(ctx, cudaEventRecord(ctx->ev_k0, ctx->stream));
    const int geo_grid = (int)std::min<int64_t>(n_pairs, 8 * ctx->num_sms);
    if (call == GeoCall::homography)
        msfm::geo_homography_kernel<<<geo_grid, msfm::kGeoThreads, 0, ctx->stream>>>(kp, (int)n_pairs);
    else
        msfm::geo_verify_kernel<<<geo_grid, msfm::kGeoThreads, 0, ctx->stream>>>(kp, (int)n_pairs);
    MSFM_CUDA(ctx, cudaGetLastError());
    MSFM_CUDA(ctx, cudaEventRecord(ctx->ev_k1, ctx->stream));
    MSFM_CUDA(ctx, cudaMemcpyAsync(pair_ok, d.ok.ptr, (size_t)n_pairs * 4, cudaMemcpyDeviceToHost, ctx->stream));
    MSFM_CUDA(ctx, cudaMemcpyAsync(pair_inliers, d.inl.ptr, (size_t)n_pairs * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (total > 0) MSFM_CUDA(ctx, cudaMemcpyAsync(keep, d.keep.ptr, (size_t)total, cudaMemcpyDeviceToHost, ctx->stream));
    if (F) MSFM_CUDA(ctx, cudaMemcpyAsync(F, d.F.ptr, (size_t)n_pairs * 72, cudaMemcpyDeviceToHost, ctx->stream));
    MSFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->timing = msfm_timing{};
    MSFM_CUDA(ctx, cudaEventElapsedTime(&ctx->timing.finalize_ms, ctx->ev_k0, ctx->ev_k1));
    ctx->timing.total_launches = 1;
    return MSFM_OK;
}

msfm_status msfm_knn2_crosscheck(msfm_ctx *ctx, int32_t ref_id, int32_t query_id, int32_t *ids, float *dists) {
    if (!ctx) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (!ids || !dists) return fail(ctx, MSFM_ERR_INVALID_ARG, "null output buffer");
    msfm_status st;
    if ((st = check_image_id(ctx, ref_id, true)) != MSFM_OK) return st;
    if ((st = check_image_id(ctx, query_id, true)) != MSFM_OK) return st;
    MSFM_CUDA(ctx, cudaSetDevice(ctx->device));
    const ImageSlot &r = ctx->images[ref_id], &q = ctx->images[query_id];
    const int n = q.rows;
    if (n == 0) return MSFM_OK;
    if ((st = ensure(ctx, ctx->knn, (size_t)n * sizeof(int4))) != MSFM_OK) return st;
    if ((st = ensure(ctx, ctx->tight_matches, (size_t)n * 8)) != MSFM_OK) return st;
    if ((st = ensure(ctx, ctx->matches, (size_t)n * 8)) != MSFM_OK) return st;
    msfm::crosscheck_knn2_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(ctx->desc + r.off * kDim, ctx->norms + r.off, r.rows,
                                                                         ctx->desc + q.off * kDim, ctx->norms + q.off, n,
                                                                         static_cast<int4 *>(ctx->knn.ptr));
    int32_t *d_ids = static_cast<int32_t *>(ctx->tight_matches.ptr);
    float *d_dists = static_cast<float *>(ctx->matches.ptr);
    msfm::knn_to_flann_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(static_cast<const int4 *>(ctx->knn.ptr), n, d_ids, d_dists);
    MSFM_CUDA(ctx, cudaGetLastError());
    MSFM_CUDA(ctx, cudaMemcpyAsync(ids, d_ids, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    MSFM_CUDA(ctx, cudaMemcpyAsync(dists, d_dists, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    MSFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return MSFM_OK;
}

}  // extern "C"
