/*
 * msfm_match.h — C ABI of the B200-native pairwise SIFT-128 matcher (drop-in for MetricSfM's matching hot path).
 *
 * Plain C, plain pointers and sizes; no C++/torch/OpenCV types cross this boundary.  Every entry point returns an
 * msfm_status and never aborts or throws (the reference's cudaSift `safeCall` exit(-1)s on error,
 * SfM/thirdparty/cudasift/include/cudaSift/utils.h:17-23 — deliberately not imitated).
 *
 * Reference interfaces replaced (paths relative to /root/reference/SfM):
 *   seam S1  flann_build_index / flann_find_nearest_neighbors_index(k=2) / flann_free_index as called at
 *            src/graph/fine_matching_graph.cc:81,99,101 and src/slam_gps.cc:447,463,549
 *              -> msfm_upload_f32 / msfm_upload_u8 (build, once per image), msfm_knn2 (query), msfm_release (free)
 *   seam S2  FeatureMatching::KNNMatchingWithGeoVerify(kp1, kp2, int* id, float* dis, matches)
 *            src/feature/feature_matching.h:57-58, feature_matching.cpp:477-501 (caller-supplied kNN arrays)
 *              -> msfm_knn2 fills exactly those id/dis arrays ([2*Nquery], (nn0,nn1) interleaved, squared L2);
 *                 msfm_knn2_pairs fills them for a whole pair list, optionally exact in fp32 on float rows
 *   seam S3  bool Matcher(vector<KeyPoint>&, Mat&, vector<KeyPoint>&, Mat&, vector<pair<int,int>>&)
 *            src/feature/feature_matching.h:33-35 (KNNMatching), feature_matching_cuda_sift.h:34-36 (Run)
 *              -> msfm_match_pairs with n_pairs = 1 (host shim: metricsfm_b200/host/feature_matching_b200.h)
 *   batch    the OpenMP partner loop + serial ratio loop of FineMatchingGraph::BuildMatchGraph
 *            src/graph/fine_matching_graph.cc:87-133
 *              -> msfm_match_pairs over the whole candidate pair list (ratio 0.85 "all" + ratio_good 0.6 flags)
 *   declared GPU matchers (no call sites, semantic precedent):
 *            cudaSift::MatchSiftData  thirdparty/cudasift/include/cudaSift/sift.h:97
 *            SiftMatchGPU::SetDescriptors/GetSiftMatch(max_match, buf, distmax, ratiomax, mutual_best_match)
 *            thirdparty/siftgpu/include/siftgpu/SiftGPU.h:297-308  -> msfm_params.{max_dist_sq, ratio, mutual}
 *
 * MATCH-SPEC (SURVEY.md §8a): reference set R (M x 128), query set Q (N x 128), u8 rows.
 *   d(q,j) = sum_k (Q[q,k]-R[j,k])^2 exactly in int32; nn0 = argmin_j d (lowest j on ties);
 *   nn1 = argmin_{j != nn0} d (lowest j on ties); ids[2q..2q+1] = (nn0,nn1); dists[2q..] = ((float)d0,(float)d1);
 *   accept iff (float)d0/(float)d1 < ratio (IEEE fp32 divide, strict; NaN => reject), and, when mutual,
 *   argmin_q' d(q',nn0) == q (lowest q' on ties); a pair with M < min_keypoints or N < min_keypoints is rejected
 *   as a whole (ok = 0, no matches), like feature_matching.cpp:30-33.  Missing neighbours: id = -1, dist = +inf.
 * Float regime: float rows are quantised to u8 by the packer, so d0/d1 carries a relative error of a few 1e-3; with
 *   msfm_config.keep_float + msfm_params.rescore_band the rows near a ratio threshold are decided on the exact fp32
 *   top-2 instead (rows outside the band keep the integer decision, see msfm_params.rescore_band).
 *   msfm_knn2_pairs with MSFM_KNN_EXACT_F32 returns the kNN arrays of an fp32 matcher itself, bit for bit.
 *
 * GUIDED-SPEC (msfm_match_pairs_guided): MATCH-SPEC with the candidate set of every query row restricted to the
 *   reference rows consistent with the pair's fundamental matrix.  F is given as msfm_geo_verify writes it
 *   (double[9], row-major, p_q^T F p_r = 0 with p_r a keypoint of the reference image and p_q one of the query image,
 *   centred feature-file coordinates) and rounded once to float f[9]; t2 = th*th in fp32 (th = th_epipolar).  Every
 *   operation below is one IEEE fp32 rounding, with no fused multiply-add:
 *     query row q at (xq, yq):     a_k = ((f[k]*xq) + (f[3+k]*yq)) + f[6+k]         k = 0, 1, 2
 *     reference row j at (xj, yj): b_k = ((f[3k]*xj) + (f[3k+1]*yj)) + f[3k+2]     k = 0, 1
 *     s = ((a0*xj) + (a1*yj)) + a2,  na = (a0*a0) + (a1*a1),  nb = (b0*b0) + (b1*b1)
 *     element (q, j) is allowed iff s*s <= t2 * min(na, nb)
 *   i.e. the larger of the two squared one-sided epipolar distances is at most th^2 (msfm_geo_verify's stage-A inlier
 *   test without the division; msfm_geo_verify contracts to FMAs, so an element within rounding reach of th^2 may be
 *   decided differently there).  nn0 / nn1 are the two closest allowed reference rows (lowest index on ties); a row with
 *   fewer than two allowed rows gets id -1 / +inf and is rejected.  Ratio, ratio_good, max_dist_sq, MSFM_RATIO_REJECT_GT,
 *   orientation and the min_keypoints gate (on the images' rows) are those of MATCH-SPEC; the mutual check keeps
 *   (q, nn0) iff q is the closest allowed query row of nn0 (lowest index on ties).
 *   Float regime under the gate (rescore_band > 0 on a keep_float context, pairs whose images both keep float rows at
 *   one scale; every other pair follows the integer rule above): a query row is a band row when both of its gated
 *   quantised neighbours exist and fl(d0/d1) lies within ratio*(1 +- band) or ratio_good*(1 +- band) (the rule of
 *   msfm_params.rescore_band applied to the guided 2-NN).  A band row is decided on its exact fp32 top-2 (b0, b1) among
 *   the allowed reference rows, with the arithmetic of the float regime: squared L2 accumulated in index order with
 *   separate multiply and add, lowest index on ties; the ratio tests on fl(b0/b1), max_dist_sq on fl(b0*fl(s*s)), the
 *   match on the fp32 nearest allowed row.  Every other row keeps the integer guided decision; the allowed set is the
 *   same in both arithmetics, so a row with fewer than two allowed rows is never a band row and stays rejected.  With
 *   mutual = 1 the check is the float regime's heuristic filter of the one-way list, under the gate (not exact in fp32).
 *
 * HOMOG-SPEC (msfm_match_pairs_guided_homography): MATCH-SPEC with the candidate set of every query row restricted to the
 *   reference rows whose keypoint the pair's homography carries to within th of the query keypoint.  H is given as
 *   msfm_geo_homography writes it (double[9], row-major, p_q ~ H p_r with p_r a keypoint of the reference image and p_q
 *   one of the query image, centred feature-file coordinates) and rounded once to float h[9]; t2 = th*th in fp32
 *   (th = th_transfer).  Every operation below is one IEEE fp32 rounding, with no fused multiply-add:
 *     reference row j at (xj, yj):  U = ((h0*xj) + (h1*yj)) + h2,  V = ((h3*xj) + (h4*yj)) + h5,  W = ((h6*xj) + (h7*yj)) + h8
 *     query row q at (xq, yq):      du = U - (xq*W),  dv = V - (yq*W)
 *     element (q, j) is allowed iff (du*du) + (dv*dv) <= t2 * (W*W)
 *   i.e. the squared transfer distance |p_q - pi(H p_j)|^2 <= th^2 without the division; it does not depend on the sign
 *   of H, and W = 0 bars the element unless U = V = 0 too (only possible for a singular H).  Everything else is
 *   GUIDED-SPEC's integer rule unchanged: nn0 / nn1 are the two closest allowed reference rows (lowest index on ties), a
 *   row with fewer than two allowed rows gets id -1 / +inf and is rejected, ratio, ratio_good, max_dist_sq,
 *   MSFM_RATIO_REJECT_GT, orientation and min_keypoints as in MATCH-SPEC, and the mutual check keeps (q, nn0) iff q is
 *   the closest allowed query row of nn0.
 *   Float regime under the gate (rescore_band > 0 on a keep_float context, pairs whose images both keep float rows at
 *   one scale; every other pair follows the integer rule above): GUIDED-SPEC's float regime with this test in place of
 *   the epipolar one.  A query row is a band row when both of its gated quantised neighbours exist and fl(d0/d1) lies
 *   within ratio*(1 +- band) or ratio_good*(1 +- band).  A band row is decided on its exact fp32 top-2 (b0, b1) among
 *   the reference rows H allows, with the arithmetic of the float regime: squared L2 accumulated in index order with
 *   separate multiply and add, lowest index on ties; the ratio tests on fl(b0/b1), max_dist_sq on fl(b0*fl(s*s)), the
 *   match on the fp32 nearest allowed row.  Every other row keeps the integer H-guided decision; the allowed set is the
 *   same in both arithmetics, so a row with fewer than two allowed rows is never a band row and stays rejected.  With
 *   mutual = 1 the check is the float regime's heuristic filter of the one-way list, under the gate (not exact in fp32).
 *   Caution: at th of a few pixels the disc around pi(H p_j) seldom holds two reference keypoints at ordinary keypoint
 *   densities, and a row with fewer than two allowed rows is rejected.  The gate then keeps only rows that have a second
 *   keypoint inside the disc (e.g. a second orientation at the same location), and can keep far fewer true matches than
 *   msfm_match_pairs or the epipolar gate (DESIGN.md §8c).
 */
#ifndef MSFM_MATCH_H_
#define MSFM_MATCH_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSFM_DIM 128              /* descriptor length (SIFT-128), bytes per packed row */
#define MSFM_ABI_VERSION 3
#define MSFM_MAX_ROWS_PER_IMAGE 1000000 /* idx_max_per_image, src/basic_structs.h:171 */

typedef enum msfm_status {
    MSFM_OK = 0,
    MSFM_ERR_INVALID_ARG = 1,   /* null pointer, negative size, bad id */
    MSFM_ERR_CUDA = 2,          /* a CUDA runtime/driver call failed; see msfm_last_error */
    MSFM_ERR_OUT_OF_MEMORY = 3, /* host or device allocation failed */
    MSFM_ERR_NOT_FOUND = 4,     /* image id not uploaded */
    MSFM_ERR_CAPACITY = 5,      /* descriptor arena, image table or caller output buffer too small */
    MSFM_ERR_UNSUPPORTED = 6,   /* device is not sm_100 (no fallback path exists by design) */
    MSFM_ERR_EXISTS = 7         /* image id already uploaded (release it first) */
} msfm_status;

typedef struct msfm_ctx msfm_ctx;

typedef struct msfm_config {
    int32_t device;          /* CUDA ordinal */
    int32_t max_images;      /* image ids are 0 .. max_images-1 */
    int64_t arena_rows;      /* total packed-descriptor rows the table can hold (each image is padded to 128 rows) */
    /* Optional caller-owned device memory for the packed table (e.g. tensors a collective library fills during
     * multi-GPU replication).  Both NULL => the library allocates.  desc: arena_rows*128 bytes, 1024-byte aligned;
     * norms: arena_rows 32-bit words (an opaque per-row side table derived from the squared norms). */
    void *external_desc_arena;
    void *external_norm_arena;
    /* 1: msfm_upload_f32 also keeps the caller's float rows in HBM (512 B per row, library-owned) so that
     * msfm_match_pairs can re-score ratio-boundary rows exactly in fp32 (msfm_params.rescore_band). */
    int32_t keep_float;
    int32_t reserved[3];     /* must be zero */
} msfm_config;

typedef struct msfm_params {
    float ratio;           /* accept iff d0/d1 < ratio (strict, fp32).  Callers: 0.5 feature_matching.cpp:27;
                              0.85 / 0.6 fine_matching_graph.cc:42-43; 0.7 feature_matching_essential.cpp:31 */
    float ratio_good;      /* > 0: also flag matches with d0/d1 < ratio_good (fine_matching_graph.cc:118-123) */
    float max_dist_sq;     /* > 0: also require (float)d0 < max_dist_sq (SiftGPU distmax analogue); 0 = off */
    int32_t mutual;        /* 1: keep (q,nn0) only if q is also the best query of reference row nn0 */
    int32_t min_keypoints; /* pairs with fewer rows on either side are rejected; reference value 20 */
    int32_t orientation;   /* 0: emit (ref_index, query_index)  fine_matching_graph.cc:121,127
                              1: emit (query_index, ref_index)  feature_matching.cpp:60-61 */
    float rescore_band;    /* float regime (both images uploaded with msfm_upload_f32 on a keep_float context with the
                              same scale s; any other pair, and band 0, follows the integer rule):
                              > 0: a query row whose quantised 2-NN both exist and whose fl(d0/d1) lies within
                              ratio*(1 +- band) or ratio_good*(1 +- band) (a NaN ratio never does) is decided on
                              its exact fp32 top-2 (b0, b1) over the retained float rows (squared L2 accumulated in
                              index order like nanoflann.hpp:376-383, lowest index on ties; the candidates are found
                              under a proven bound): the ratio tests on fl(b0/b1), max_dist_sq on fl(b0*fl(s*s)), the
                              match on the fp32 nearest row.  Every other row keeps the integer decision.  The mutual
                              check of these pairs is a heuristic filter of the one-way list (not exact in fp32).
                              0 = integer rule */
    uint32_t flags;        /* MSFM_RATIO_* bits; 0 = the strict rule of MATCH-SPEC */
} msfm_params;

/* msfm_params.flags */
#define MSFM_RATIO_REJECT_GT 1u /* SLAMGPS::FeatureMatching's rule (slam_gps.cc:470-477): a row is rejected iff
                                   d0/d1 > ratio, i.e. accepted iff !(d0/d1 > ratio): non-strict, and 0/0 = NaN passes.
                                   Applies to ratio and ratio_good alike.  A missing second neighbour still rejects. */

/* One candidate pair: the kNN index is "built" on image `ref`, rows of image `query` are the queries
 * (fine_matching_graph.cc: ref = idx1, query = idx2; feature_matching.cpp:35-44: ref = image 2, query = image 1). */
typedef struct msfm_pair {
    int32_t ref;
    int32_t query;
} msfm_pair;

/* Caller-provided output of msfm_match_pairs.  matches[offsets[p] .. offsets[p+1]) belong to pair p, ascending query
 * index.  Capacity needed is at most sum over pairs of query rows (one match per query row). */
typedef struct msfm_result {
    int64_t *offsets;        /* [n_pairs + 1] */
    int32_t *ok;             /* [n_pairs] 1 = matched, 0 = rejected by the min_keypoints gate */
    int32_t (*matches)[2];   /* [match_capacity][2] */
    uint8_t *good;           /* [match_capacity] or NULL; 1 iff the match also passes ratio_good */
    int64_t match_capacity;
} msfm_result;

/* Device-side timing of the last msfm_match_pairs / msfm_knn2 call on a context (CUDA events on the library's own
 * stream).  kernel_ms covers only launches of the dominant matching kernel. */
typedef struct msfm_timing {
    float total_ms;          /* first enqueue -> last result byte landed in host memory */
    float match_kernel_ms;   /* sum over launches of the tcgen05 matching kernel */
    float finalize_ms;       /* ratio / mutual / compaction kernels */
    float d2h_ms;            /* result copies device -> host */
    int32_t match_launches;  /* number of launches of the matching kernel */
    int32_t total_launches;  /* all kernels launched by the call */
    int64_t d2h_bytes;
    int64_t int8_ops;        /* algorithmic work: sum over matched pairs of 2*M*N*128 */
    int32_t twin_pairs;      /* mutual check: pairs whose candidates had to take the tensor twin pass (the others were
                                decided from the forward results alone, DESIGN.md §4.4) */
    int32_t reserved;
} msfm_timing;

int32_t msfm_abi_version(void);
const char *msfm_status_string(msfm_status s);

/* Page-locked host memory for the staging buffers of the *_async uploads and for result buffers (a host that does not
 * link the CUDA runtime itself, like the graph driver, gets it from here).  msfm_device_memory: free / total HBM bytes. */
msfm_status msfm_host_alloc(size_t bytes, void **out);
msfm_status msfm_host_free(void *ptr);
msfm_status msfm_device_memory(int32_t device, int64_t *free_bytes, int64_t *total_bytes);

msfm_status msfm_create(const msfm_config *cfg, msfm_ctx **out);
msfm_status msfm_destroy(msfm_ctx *ctx);
/* Last error text of this context (valid until the next call on it); never NULL. */
const char *msfm_last_error(const msfm_ctx *ctx);

/* ---- descriptor packer: once per image (replaces the per-idx1 flann_build_index) ------------------------------- */
/* u8 rows, row_stride_bytes >= 128.  The library copies; the caller may free `desc` on return. */
msfm_status msfm_upload_u8(msfm_ctx *ctx, int32_t image_id, const uint8_t *desc, int32_t rows, int64_t row_stride_bytes);
/* Several images in one call: the copies and packer launches are queued back to back and the host waits once (a
 * per-image msfm_upload_u8 waits once per image).  row_stride_bytes may be NULL (contiguous 128-byte rows).  On error
 * the images before the failing one stay uploaded. */
msfm_status msfm_upload_u8_batch(msfm_ctx *ctx, int32_t n, const int32_t *image_ids, const uint8_t *const *descs,
                                 const int32_t *rows, const int64_t *row_stride_bytes);
/* Same without the host wait, for callers that stage descriptors in page-locked memory.  All table changes run on the
 * context's UPLOAD stream; a later msfm_match_pairs / msfm_knn2 launch waits (on the device, not on the host) only for the
 * uploads that cover the images it touches, so staging image group k+1 overlaps matching the pairs of groups <= k.  Every
 * `descs[i]` must stay valid and unchanged until msfm_sync() or a later call that returns results computed from it.
 * Only contiguous 128-byte rows (row_stride_bytes NULL or 128 everywhere). */
msfm_status msfm_upload_u8_batch_async(msfm_ctx *ctx, int32_t n, const int32_t *image_ids, const uint8_t *const *descs,
                                       const int32_t *rows, const int64_t *row_stride_bytes);
/* Wait for everything queued on the context's streams. */
msfm_status msfm_sync(msfm_ctx *ctx);
/* float rows (cv::Mat CV_32FC1 rows x 128, database.cc:368-370): q = min(255, max(0, rint(x*scale))).
 * scale = 1 for 512-scaled VLSIFT rows (feature_extractor_vl_sift.cpp:201-203), 512 for unit-norm rows
 * (feature_extractor_cuda_sift.cpp:75-80). */
msfm_status msfm_upload_f32(msfm_ctx *ctx, int32_t image_id, const float *desc, int32_t rows, int64_t row_stride_floats,
                            float scale);
/* Several float images (the reference's container: dense CV_32FC1 rows of 128 floats, e.g. read from <idx>_feature files
 * into page-locked staging) without a host wait; semantics of msfm_upload_u8_batch_async. */
msfm_status msfm_upload_f32_batch_async(msfm_ctx *ctx, int32_t n, const int32_t *image_ids, const float *const *descs,
                                        const int32_t *rows, float scale);
/* Reserve table space for an image whose packed rows + norms are written by someone else (a collective during
 * multi-GPU replication) at the returned row offset of the arenas.  Pad rows/norms and the image's tensor map are in
 * place when the call returns.  Order the foreign writer before matching with msfm_wait_event(). */
msfm_status msfm_reserve(msfm_ctx *ctx, int32_t image_id, int32_t rows, int64_t *row_offset);
/* Several images in one call (row_offsets may be NULL); images before a failing one stay reserved. */
msfm_status msfm_reserve_batch(msfm_ctx *ctx, int32_t n, const int32_t *image_ids, const int32_t *rows, int64_t *row_offsets);
/* Same without the host wait: pad rows and tensor maps are queued on the upload stream (msfm_get_upload_stream).  A
 * foreign writer must order itself behind that stream (an event recorded on it after this call) and matching behind
 * the writer (msfm_wait_event). */
msfm_status msfm_reserve_batch_async(msfm_ctx *ctx, int32_t n, const int32_t *image_ids, const int32_t *rows,
                                     int64_t *row_offsets);
msfm_status msfm_release(msfm_ctx *ctx, int32_t image_id);
msfm_status msfm_release_all(msfm_ctx *ctx);
msfm_status msfm_image_info(const msfm_ctx *ctx, int32_t image_id, int32_t *rows, int64_t *row_offset);
/* Device addresses of the packed table (for collectives / inspection). */
msfm_status msfm_table_ptrs(const msfm_ctx *ctx, void **desc_arena, void **norm_arena, int64_t *arena_rows,
                            int64_t *rows_used);
/* Copy an image's packed u8 rows / uint32 squared norms back to the host (tests, debugging). */
msfm_status msfm_download_packed(msfm_ctx *ctx, int32_t image_id, uint8_t *desc_out, uint32_t *norms_out);

/* ---- kNN query in FLANN layout (seams S1/S2) ------------------------------------------------------------------- */
/* ids[2*Nq], dists[2*Nq] host buffers, Nq = rows of image `query_id`.  No min_keypoints gate (FLANN has none).
 * Distances are those of the packed u8 rows (float uploads: quantised units); msfm_knn2_pairs with MSFM_KNN_EXACT_F32
 * gives the fp32 ones. */
msfm_status msfm_knn2(msfm_ctx *ctx, int32_t ref_id, int32_t query_id, int32_t *ids, float *dists);

#define MSFM_KNN_EXACT_F32 1u   /* msfm_knn2_pairs flag */

/* FLANN-layout 2-NN of every query row of every pair in one call.  Pair p's rows are rows
 * [offsets[p], offsets[p+1]) of ids/dists: ids[2r..2r+1] = (nn0, nn1), dists[2r..2r+1] = (d0, d1), missing
 * neighbour = (-1, +inf).  offsets[n_pairs+1] in query rows; ids/dists hold 2*row_capacity entries.  No min_keypoints gate.
 * flags 0: exactly msfm_knn2 per pair (squared L2 of the packed u8 rows).
 * MSFM_KNN_EXACT_F32: every pair's images must have been uploaded with msfm_upload_f32* on a keep_float context with
 *   the same scale; ids/dists are then those of an exhaustive fp32 matcher on the caller's float rows: squared L2
 *   accumulated in index order with separate multiply and add (nanoflann.hpp:376-383), in the caller's units, lowest
 *   index on ties for nn0 and nn1, bit for bit.  (A pair with an empty image needs no float rows.)  Finite rows only.
 * Errors (before any launch): INVALID_ARG for a null buffer, negative n_pairs / row_capacity, unknown flag bits, or
 * EXACT_F32 on a pair without retained float rows or with two scales (the message names the pair); the image-id
 * statuses; CAPACITY when the pairs' query rows exceed row_capacity.  msfm_last_timing: as msfm_match_pairs with
 * rescore_band (match_kernel_ms = forward launches; the collect pass counts under finalize_ms). */
msfm_status msfm_knn2_pairs(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, uint32_t flags,
                            int64_t *offsets, int32_t *ids, float *dists, int64_t row_capacity);
/* Per reference row j of ref_id: best query row (lowest index on ties) and its squared distance. */
msfm_status msfm_colbest(msfm_ctx *ctx, int32_t ref_id, int32_t query_id, int32_t *best_query, float *best_dist);

/* ---- batched pair matching (the fast path; replaces the OMP partner loop + ratio loop) ------------------------- */
msfm_status msfm_match_pairs(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const msfm_params *params,
                             msfm_result *out);
/* Same work with results left in HBM (no device->host copy): used to time the device-resident path.  n_matches_total
 * (optional) receives the total match count (one 8-byte read-back). */
msfm_status msfm_match_pairs_resident(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const msfm_params *params,
                                      int64_t *n_matches_total);

msfm_status msfm_last_timing(const msfm_ctx *ctx, msfm_timing *out);
/* The CUDA stream (cudaStream_t) every kernel and copy of this context is enqueued on, so a host harness can record
 * its own events around calls (bench.py) or order foreign work (a collective filling the table) against it. */
msfm_status msfm_get_stream(const msfm_ctx *ctx, void **cuda_stream);
/* The stream the table uploads run on (a collective that forwards freshly uploaded rows orders itself behind it). */
msfm_status msfm_get_upload_stream(const msfm_ctx *ctx, void **cuda_stream);
/* Make every later matching launch of this context wait for `cuda_event` (a cudaEvent_t recorded by the caller, e.g.
 * after a collective wrote reserved rows on its own stream).  Device-side wait; the host does not block. */
msfm_status msfm_wait_event(msfm_ctx *ctx, void *cuda_event);

/* ---- geometric verification of the matched pairs (the stage after the hot path; SURVEY.md §8f row 1) ---------- */
/* FineMatchingGraph::BuildMatchGraph verifies every pair (fine_matching_graph.cc:137-153) with
 *   A  GeoVerificationFundamental(pt_good): >= min_points good matches, F by RANSAC (7-point, error = max of the two
 *      squared point-to-epipolar-line distances <= th^2 like cv::findFundamentalMat FM_RANSAC), >= min_inliers inliers
 *      (utils/geo_verification.cc:30-58)
 *   B  GeoVerificationFundamental(pt_all, F): keep the "all" matches with |distance(p2, F p1)| < th, double arithmetic
 *      (utils/geo_verification.cc:60-79)
 * Here the whole batch runs on the GPU, one CTA per pair.  RANSAC draws are counter-based (seed, pair, hypothesis):
 * reproducible, but not OpenCV's RNG stream, so stage A agrees with the reference statistically, stage B exactly
 * given F. */
typedef struct msfm_geo_params {
    float th_epipolar;     /* 3.0  utils/geo_verification.cc:45,66 */
    int32_t min_points;    /* 30   utils/geo_verification.cc:33 */
    int32_t min_inliers;   /* 30   utils/geo_verification.cc:53 */
    int32_t iters;         /* RANSAC hypotheses per pair (each yields up to 3 models); 0 = 1024 */
    uint64_t seed;
    int64_t pair_index_base; /* added to the pair index in the RANSAC counter, so that a pair list verified in several
                                calls draws the same hypotheses as in one call */
} msfm_geo_params;
/* pairs/offsets/matches/good: the result of msfm_match_pairs with orientation 0 and ratio_good set.
 * image_xy[i]: host pointer to the centred keypoints (x, y) of image i as stored in its feature file, or NULL for
 * images no pair touches; image_npts[i] their number.  Outputs (host): pair_ok[n_pairs], pair_inliers[n_pairs]
 * (stage-A inliers among the good matches), keep[offsets[n_pairs]] (stage-B mask over the "all" matches; all zero for
 * rejected pairs), F[n_pairs][9] row-major or NULL. */
msfm_status msfm_geo_verify(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const int64_t *offsets,
                            const int32_t (*matches)[2], const uint8_t *good, const float *const *image_xy,
                            const int32_t *image_npts, int32_t n_images, const msfm_geo_params *gp, int32_t *pair_ok,
                            int32_t *pair_inliers, uint8_t *keep, double *F);

/* The RANSAC part alone, with the consensus set as a per-match mask: what the matcher family's own verification loops
 * (KNNMatchingWithGeoVerify, feature_matching.cpp:97-138: findFundamentalMat(FM_RANSAC, 3.0) then (…, 1.0), dropping
 * the outliers after each pass) consume.  `use[k]` selects the matches that take part; inlier_mask[k] = 1 iff match k
 * took part and its error is within th_epipolar of the best model.  pair_ok as in msfm_geo_verify. */
msfm_status msfm_geo_ransac(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const int64_t *offsets,
                            const int32_t (*matches)[2], const uint8_t *use, const float *const *image_xy,
                            const int32_t *image_npts, int32_t n_images, const msfm_geo_params *gp, int32_t *pair_ok,
                            int32_t *pair_inliers, uint8_t *inlier_mask, double *F);

/* msfm_geo_ransac with a homography model, p_q ~ H p_r (matches in orientation 0: reference keypoint -> query keypoint;
 * cv::findHomography(RANSAC, th) without its refinement).  gp->th_epipolar is the transfer threshold in pixels.  Shared
 * with msfm_geo_ransac: the used matches (a strided subsample above 2048, in list order), the isotropic scale
 * s = 1 / max(1, max |coordinate| of those points) in fp32, the counter-based draws from (seed, pair_index_base + p, h),
 * the winner (most inliers, then lowest hypothesis id h), and the decision: inliers of the returned H among all used
 * matches in double, pair_ok iff >= max(min_points, 4) used matches, a model exists and inliers >= min_inliers.
 * The search, step by step (hypotheses h = 0 .. iters-1, iters 0 = 1024):
 *   sample   4 distinct indices of the scaled points, drawn like msfm_geo_ransac's 7 (each slot repeats the draw until new)
 *   subset   an orientation test derived from cv::findHomography's checkSubset: for each triple {0,1,2}, {1,2,3},
 *            {0,2,3}, {0,1,3}, the product det[p_a p_b p_c] (reference, homogeneous, double) * det[...] (query) must not
 *            be negative, otherwise the sample gives no model.  Stricter than OpenCV, which also accepts a sample whose
 *            four triples all flip (a mirror); OpenCV's collinearity test (haveCollinearPoints) is not applied
 *   solver   normalised DLT: the 8 x 9 system with rows (x, y, 1, 0, 0, 0, -u x, -u y, -u) and (0, 0, 0, x, y, 1, -v x,
 *            -v y, -v) per correspondence (x, y) -> (u, v), in double, Gauss-Jordan elimination with full pivoting (as the
 *            7-point solver of msfm_geo_ransac; a pivot below 1e-12 means no model), h = the null vector with the free
 *            component 1, divided by its norm, rounded to fp32
 *   score    cv::findHomography's one-sided reprojection error |p_q - pi(H p_r)|^2 in fp32 on the scaled points,
 *            inlier iff <= (th*s)^2; a zero or non-finite w = (H p_r)_2 makes the match an outlier
 *   result   H in pixel coordinates (T^-1 H' T, T = diag(s, s, 1)), scaled so that H22 = 1 unless
 *            |H22| <= 1e-12 |H| (then to unit norm); no Levenberg-Marquardt refinement
 * inlier_mask[k] = 1 iff match k is used and its double-precision error against the returned H is <= th^2.  H[n_pairs][9]
 * row-major (zero for rejected pairs) or NULL.  Errors as msfm_geo_ransac. */
msfm_status msfm_geo_homography(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const int64_t *offsets,
                                const int32_t (*matches)[2], const uint8_t *use, const float *const *image_xy,
                                const int32_t *image_npts, int32_t n_images, const msfm_geo_params *gp,
                                int32_t *pair_ok, int32_t *pair_inliers, uint8_t *inlier_mask, double *H);

/* ---- guided re-matching of verified pairs (GUIDED-SPEC above) ------------------------------------------------- */
/* msfm_match_pairs with each query row's 2-NN searched only among the reference rows consistent with F[p] (typically
 * msfm_geo_verify's F of the pairs with pair_ok).  image_xy / image_npts / n_images as in msfm_geo_verify; image_npts[i]
 * must equal the uploaded rows of every image a pair touches.  Results, batches and msfm_last_timing as in
 * msfm_match_pairs; with mutual = 1 every pair takes the tensor twin pass (timing.twin_pairs counts them).
 * Errors (before any launch): the statuses of msfm_match_pairs, and INVALID_ARG (the message names the pair or image)
 * for a null F, image_xy or image_npts; a pair naming an image >= n_images; a touched image without keypoints, with
 * image_npts different from its uploaded rows, or with a non-finite coordinate; an F with a non-finite entry or that
 * is zero after rounding to fp32; th_epipolar not finite or not > 0; rescore_band negative or not finite, or > 0 on a
 * context without retained float rows (keep_float = 0).  rescore_band > 0 on a keep_float context: the float regime
 * under the gate (GUIDED-SPEC). */
msfm_status msfm_match_pairs_guided(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs, const msfm_params *params,
                                    const double (*F)[9], float th_epipolar,
                                    const float *const *image_xy, const int32_t *image_npts, int32_t n_images,
                                    msfm_result *out);
/* msfm_match_pairs with each query row's 2-NN searched only among the reference rows that H[p] carries to within
 * th_transfer pixels of the row's keypoint (HOMOG-SPEC above; typically msfm_geo_homography's H of the pairs with
 * pair_ok).  Arguments, results, timing and errors as msfm_match_pairs_guided with H in place of F and th_transfer in
 * place of th_epipolar.  rescore_band > 0 on a keep_float context: the float regime under the gate (HOMOG-SPEC). */
msfm_status msfm_match_pairs_guided_homography(msfm_ctx *ctx, const msfm_pair *pairs, int64_t n_pairs,
                                               const msfm_params *params, const double (*H)[9], float th_transfer,
                                               const float *const *image_xy, const int32_t *image_npts, int32_t n_images,
                                               msfm_result *out);

/* ---- GPU-side cross-check kernel (CUDA cores, dp4a); used by the tests to localise faults, never by the fast path */
msfm_status msfm_knn2_crosscheck(msfm_ctx *ctx, int32_t ref_id, int32_t query_id, int32_t *ids, float *dists);
/* Test hook: capacity of the float regime's event list (-1 = default sizing; 0 forces the brute-force fallback).
 * Applies to the rescore_band of msfm_match_pairs, msfm_match_pairs_guided and msfm_match_pairs_guided_homography and
 * to msfm_knn2_pairs' MSFM_KNN_EXACT_F32 alike. */
msfm_status msfm_test_set_band_event_cap(msfm_ctx *ctx, int64_t cap);
/* Test hook: for the last MSFM_KNN_EXACT_F32 call of msfm_knn2_pairs or the last msfm_match_pairs /
 * msfm_match_pairs_guided / msfm_match_pairs_guided_homography call with rescore_band > 0 on a keep_float context,
 * whichever came later, the events the
 * collect path scored (in a guided call: only elements the gate allows) and the batches
 * whose event list overflowed, i.e. that the brute force decided.  Either pointer may be NULL. */
msfm_status msfm_test_last_knn_stats(msfm_ctx *ctx, int64_t *events, int32_t *brute_force_batches);
/* Test hook: 1 routes every pair's mutual check through the tensor twin pass (the fallback of the bound-based check). */
msfm_status msfm_test_force_twin_pass(msfm_ctx *ctx, int32_t on);
/* Test hook: 1 switches off the forward pass's dead-row rule (rows whose two nearest neighbours already violate every
 * ratio the call tests follow only their nearest neighbour exactly); the match lists must not change. */
msfm_status msfm_test_disable_pruning(msfm_ctx *ctx, int32_t on);

#ifdef __cplusplus
}
#endif
#endif /* MSFM_MATCH_H_ */
