// aux_kernels.cuh — the small HBM-bound kernels around the matching kernel:
//   * descriptor packer (north_star subsystem 1): f32/u8 rows -> 128-byte u8 rows + uint32 squared norms
//   * finalize: ratio test (+ max-dist test, + mutual check) and ordered per-pair compaction
//   * offsets scan + tight gather of the per-pair match lists
//   * a CUDA-core dp4a brute-force kNN used only by tests as a GPU-side cross-check
#pragma once
#include <cstdint>
#include <climits>
#include <cuda_runtime.h>

#include "match_kernel.cuh"

namespace msfm {

// ------------------------------------------------------------------------------------------------ packer
// One warp per row; lane l owns bytes 4l..4l+3.  rows_padded - rows pad rows get zero bytes and kNormPad norms.
// The side table stores column keys, ckey = -8*||row||^2 + (7 - row%8) (see match_kernel.cuh), not raw norms.
// Quantisation rule (mirrored by oracle_quantize_f32): q = min(255, max(0, rint(x * scale))), NaN -> 0.
// resid (keep_float contexts, else null): per row the quantisation residual r = ||scale*x - q||_2, rounded up, and
// *rmax the largest residual of the image (the exact kNN mode's candidate bound, see exact_threshold).
__global__ void pack_f32_kernel(const float *__restrict__ src, int rows, int rows_padded, float scale,
                                uint8_t *__restrict__ dst, int32_t *__restrict__ ckeys,
                                float *__restrict__ resid = nullptr, float *__restrict__ rmax = nullptr) {
    const int warps_per_block = blockDim.x >> 5;
    const int lane = threadIdx.x & 31;
    for (int r = blockIdx.x * warps_per_block + (threadIdx.x >> 5); r < rows_padded; r += gridDim.x * warps_per_block) {
        uint32_t packed = 0, nrm = kNormPad;
        if (r < rows) {
            const float *s = src + (int64_t)r * kDim + lane * 4;
            const float f[4] = {s[0], s[1], s[2], s[3]};
            uint32_t acc = 0;
            double e2 = 0.0;  // x*scale is exact in double (24 x 24 bit significands), so is its distance to q
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                float x = rintf(f[k] * scale);
                if (!(x > 0.0f)) x = 0.0f;
                if (x > 255.0f) x = 255.0f;
                const uint32_t qv = (uint32_t)x;
                packed |= qv << (8 * k);
                acc += qv * qv;
                if (resid) {
                    const double e = (double)f[k] * (double)scale - (double)qv;
                    e2 += e * e;
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, o);
            nrm = acc;
            if (resid) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) e2 += __shfl_xor_sync(0xFFFFFFFFu, e2, o);
                if (lane == 0) {
                    const float rv = __double2float_ru(__dsqrt_ru(e2));
                    resid[r] = rv;
                    atomicMax(reinterpret_cast<int *>(rmax), __float_as_int(rv));  // >= +0: the bits order like the values
                }
            }
        }
        reinterpret_cast<uint32_t *>(dst + (int64_t)r * kDim)[lane] = packed;
        if (lane == 0) ckeys[r] = make_ckey(nrm, r);
    }
}

// u8 rows already copied to their place in the arena: keys for every row, zero bytes for the pad rows.
__global__ void pack_u8_kernel(int rows, int rows_padded, uint8_t *__restrict__ rows_inout, int32_t *__restrict__ ckeys) {
    const int warps_per_block = blockDim.x >> 5;
    const int lane = threadIdx.x & 31;
    for (int r = blockIdx.x * warps_per_block + (threadIdx.x >> 5); r < rows_padded; r += gridDim.x * warps_per_block) {
        uint32_t *row = reinterpret_cast<uint32_t *>(rows_inout + (int64_t)r * kDim);
        uint32_t nrm = kNormPad;
        if (r < rows) {
            const uint32_t packed = row[lane];
            uint32_t acc = __dp4a(packed, packed, 0u);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, o);
            nrm = acc;
        } else {
            row[lane] = 0u;
        }
        if (lane == 0) ckeys[r] = make_ckey(nrm, r);
    }
}

// Pad rows of a reserved (externally filled) image.
__global__ void init_pad_kernel(int rows, int rows_padded, uint8_t *__restrict__ dst, int32_t *__restrict__ ckeys) {
    const int warps_per_block = blockDim.x >> 5;
    const int lane = threadIdx.x & 31;
    for (int r = rows + blockIdx.x * warps_per_block + (threadIdx.x >> 5); r < rows_padded; r += gridDim.x * warps_per_block) {
        reinterpret_cast<uint32_t *>(dst + (int64_t)r * kDim)[lane] = 0u;
        if (lane == 0) ckeys[r] = make_ckey(kNormPad, r);
    }
}

// ------------------------------------------------------------------------------------------------ plan upload
// The per-batch plan (pair descriptors + work items, a few hundred KB in page-locked host memory) is PULLED by the SMs over
// PCIe instead of being copied by the host->device copy engine: that engine is a FIFO, and a plan copy queued behind the
// bulk descriptor uploads of later image groups would hold back the matching launch until all of them had finished.
// Per reference tile (kKeyTileRows rows of the arena) the smallest squared norm of its rows, for the matching kernel's pruning
// threshold (one shared-memory read per tile instead of a reduction over the tile's keys in each of the 16 epilogue warps).
// One warp per tile; recomputed per batch over the arena range the batch's images span (the column keys are written by
// the packers, by NCCL during replication, or by the caller: only at launch time is everything the batch needs in place).
__global__ void tile_min_kernel(const int32_t *__restrict__ ckeys, int4 *__restrict__ tilemin, int64_t tile0, int64_t ntiles) {
    const int lane = threadIdx.x & 31;
    const int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (i >= ntiles) return;
    const int32_t *k = ckeys + (tile0 + i) * kKeyTileRows;
    int m = k[lane];
#pragma unroll
    for (int r = 32; r < kKeyTileRows; r += 32) m = max(m, k[lane + r]);
    m = __reduce_max_sync(0xFFFFFFFFu, m);  // largest key = smallest norm
    if (lane == 0) tilemin[tile0 + i] = make_int4(ckey_to_norm(m), 0, 0, 0);
}

__global__ void pull_plan_kernel(const uint4 *__restrict__ host_src, uint4 *__restrict__ dst0, size_t n0, uint4 *__restrict__ dst1, size_t n1) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n0 + n1; i += (size_t)gridDim.x * blockDim.x) {
        const uint4 v = host_src[i];
        if (i < n0) dst0[i] = v;
        else dst1[i - n0] = v;
    }
}

// ------------------------------------------------------------------------------------------------ kNN records
// The matching kernel leaves one record {id0, id1, d0, d1} per query row, sorted (d0,id0) <= (d1,id1); an absent
// neighbour is (id -1, d INT_MAX).  load_knn() returns a record in which an id of -1 and a distance of INT_MAX always
// come together, whichever of the two was written.
__device__ __forceinline__ int4 load_knn(const int4 *__restrict__ knn, int64_t row) {
    int4 v = knn[row];
    if (v.x < 0) v.z = INT_MAX;  // rows of work-less pairs are memset to -1; seeded placeholders carry id -1
    if (v.y < 0) v.w = INT_MAX;
    if (v.z == INT_MAX) v.x = -1;
    if (v.w == INT_MAX) v.y = -1;
    return v;
}

// ------------------------------------------------------------------------------------------------ finalize
// Block-wide ordered compaction helper: returns this thread's output slot among the `keep` threads of the block
// (ascending thread index) and adds the block's total to `running` (identical in every thread).
__device__ __forceinline__ int block_rank(bool keep, int &running, int *warp_excl, int *chunk_total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const unsigned ballot = __ballot_sync(0xFFFFFFFFu, keep);
    const int prefix = __popc(ballot & ((1u << lane) - 1u));
    if (lane == 0) warp_excl[warp] = __popc(ballot);
    __syncthreads();
    if (warp == 0) {
        const int v = (lane < nwarps) ? warp_excl[lane] : 0;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int n = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o) incl += n;
        }
        warp_excl[lane] = incl - v;
        if (lane == 31) *chunk_total = incl;
    }
    __syncthreads();
    const int slot = running + warp_excl[warp] + prefix;
    running += *chunk_total;
    __syncthreads();
    return slot;
}

// ------------------------------------------------------------------------------------------------ float regime
// Float descriptors are quantised to u8 by the packer, so the ratio d0/d1 of the integer path carries a relative error
// of a few 1e-3 and rows close to a ratio threshold can land on the other side of it than an fp32 matcher would put
// them (north_star: ratio-boundary flip rate <= 1e-4 of the matches).  With the caller's float rows retained in HBM,
//   mark_band_kernel     lists, per pair, the query rows whose quantised ratio lies within +-band of a threshold
//   rescore_band_kernel  recomputes their 2-NN by exact fp32 brute force over the whole reference image (squared L2
//                        accumulated in index order with separate multiply and add, the arithmetic of
//                        nanoflann.hpp:376-383 compiled without contraction), repeats the ratio tests on those
//                        distances and overwrites the row's kNN entry with the decision
// Rows outside the band keep the integer decision: their ratio is off the threshold by many times the quantisation error.
// The fp32 work is confined to the reference rows whose QUANTISED distance is within the bound T(q) of exact_threshold
// -- only those can be fp32 top-2 neighbours, so a band row is decided on its exact fp32 top-2.  They are found by
// the matching kernel itself in "collect" mode (mark_band_kernel gathers the band rows into the candidate scratch
// image; the tensor pass lists every reference row under the per-row threshold as an event), then
//   score_events_kernel / second_events_kernel   fp32 distance per event, best and second best per band row (atomicMin
//                                                on (distance bits, reference row): lowest index wins ties)
//   finish_band_kernel                           the ratio tests on those distances, kNN entry overwritten
// rescore_band_kernel does the same search with a dp4a brute force on CUDA cores; it runs only when the event list
// overflowed (bands much wider than the recommended 0.02, inputs full of near-duplicates) and is the cross-check of the
// tests.
constexpr int kRescoredFlag = 0x40000000;  // in knn[row].x: {id0 | flag, bit0 keep | bit1 good, int d0, fp32 d0 bits}
constexpr int kRescoreRows = 16;           // band rows a CTA scores together against the reference image

struct BandParams {
    const PairDesc *pairs;
    int4 *knn;
    float ratio, ratio_good, max_dist_sq, band;
    int32_t reject_gt;     // ratio rule, see SelectParams
    int32_t *band_q;       // [forward kNN rows], pair p writes from row knn_off
    int32_t *band_counts;  // [n_pairs]
    const float *fdesc;    // retained float rows, same row offsets as the packed arena
    const uint8_t *desc_arena;
    const int32_t *ckeys;
    // collect path
    int32_t *band_thr;               // [forward kNN rows] quantised-distance threshold of each band row
    unsigned long long *band_state;  // [forward kNN rows][2] best / second best (fp32 distance bits << 32 | reference row)
    uint8_t *cand_desc;              // candidate scratch image: the band rows' packed descriptors ...
    int32_t *cand_ckeys;             // ... and their column keys
    const int4 *events;              // {band row (scratch row), reference row, pair, -} from the collect pass
    unsigned long long *event_keys;  // [event_cap]
    const unsigned int *event_count;
    uint32_t event_cap;
    // exact kNN mode (msfm_knn2_pairs with MSFM_KNN_EXACT_F32): every query row is a band row, and its fp32 (nn0, nn1,
    // d0, d1) go to these FLANN-layout arrays at row knn_off + q instead of a ratio decision into the kNN scratch
    int32_t *out_ids = nullptr;
    float *out_dists = nullptr;
};

// A quantised-distance threshold T(q) that provably holds every fp32 top-2 neighbour of query row x (the band rows of
// msfm_match_pairs and every row of the exact kNN mode).
// With s the scale, q_y the packed row of y and r_y = ||s*y - q_y|| its quantisation residual (clamping included), the
// triangle inequality gives  | s*||x-y|| - ||q_x-q_y|| | <= r_x + r_y <= r_x + R  (R: largest residual of the reference
// image).  The two quantised nearest neighbours are therefore both within s*||x-y|| <= sqrt(d1_q) + r_x + R, so the fp32
// second-nearest distance is at most that, and every fp32 top-2 row y has ||q_x-q_y|| <= sqrt(d1_q) + 2(r_x + R).
// Slack: the fp32 distance sum (128 products accumulated in order, with the rounding of the differences) is within a
// relative 130 * 2^-24 of the real value; that widens the squared bound by (1 + 130 * 2^-24)^2 < 1 + 2^-15.  The
// residuals are rounded up where they are stored and every step here rounds up, so T(q) is an upper bound.
// d1 < 0 (the reference image has fewer than two rows): every reference row is a candidate.
constexpr int kExactThrAll = 1 << 24;  // > 128 * 255^2, every quantised distance
__device__ __forceinline__ int exact_threshold(int d1, float rx, float rmax) {
    if (d1 < 0) return kExactThrAll;
    const float root = __fadd_ru(__fsqrt_ru((float)d1), __fmul_ru(2.0f, __fadd_ru(rx, rmax)));
    const float t = __fmul_ru(__fmul_ru(root, root), 1.0f + 1.0f / 32768.0f);
    return t >= (float)kExactThrAll ? kExactThrAll : (int)ceilf(t);
}

// Exact kNN mode, per batch: every query row of pair p becomes a "band row" (rows knn_off .. knn_off + qry_rows of the
// candidate scratch) with its own threshold exact_threshold(d1_q, r_x, R_ref).  Grid (pairs, row chunks).
__global__ void __launch_bounds__(256) mark_exact_kernel(const BandParams bp, const float *__restrict__ resid,
                                                         const float *__restrict__ img_rmax) {
    const PairDesc pd = bp.pairs[blockIdx.x];
    if (blockIdx.y == 0 && threadIdx.x == 0) bp.band_counts[blockIdx.x] = pd.qry_rows;
    const float rmax = pd.ref_rows > 0 ? img_rmax[pd.ref_img] : 0.0f;
    for (int q = blockIdx.y * blockDim.x + threadIdx.x; q < pd.qry_rows; q += gridDim.y * blockDim.x) {
        const int4 k = load_knn(bp.knn, pd.knn_off + q);
        const int64_t row = pd.knn_off + q;
        bp.band_q[row] = q;
        bp.band_thr[row] = exact_threshold(k.y >= 0 ? k.w : -1, resid[pd.qry_off + q], rmax);
        bp.band_state[2 * row] = ~0ull;
        bp.band_state[2 * row + 1] = ~0ull;
    }
    // the rows' packed descriptors + column keys into the scratch image the collect pass queries
    const int lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    for (int q = blockIdx.y * nwarps + (threadIdx.x >> 5); q < pd.qry_rows; q += gridDim.y * nwarps) {
        const int64_t src = pd.qry_off + q, dst = pd.knn_off + q;
        reinterpret_cast<uint32_t *>(bp.cand_desc + dst * kDim)[lane] = reinterpret_cast<const uint32_t *>(bp.desc_arena + src * kDim)[lane];
        if (lane == 0) bp.cand_ckeys[dst] = bp.ckeys[src];
    }
}

// Float regime, per batch: lists pair p's band rows (rows knn_off .. knn_off + band_count_p of the candidate scratch),
// each with the threshold exact_threshold(d1_q, r_x, R_ref).
__global__ void __launch_bounds__(1024) mark_band_kernel(const BandParams bp, const float *__restrict__ resid,
                                                         const float *__restrict__ img_rmax) {
    __shared__ int warp_excl[32];
    __shared__ int chunk_total;
    const PairDesc pd = bp.pairs[blockIdx.x];
    int running = 0;
    if (pd.fscale2 > 0.0f) {
        const float rmax = img_rmax[pd.ref_img];
        for (int base = 0; base < pd.qry_rows; base += blockDim.x) {
            const int q = base + threadIdx.x;
            bool in_band = false;
            int d1q = 0;
            if (q < pd.qry_rows) {
                const int4 k = load_knn(bp.knn, pd.knn_off + q);
                d1q = k.w;
                if (k.x >= 0 && k.y >= 0) {
                    const float r = __fdiv_rn((float)k.z, (float)k.w);
                    in_band = fabsf(r - bp.ratio) <= bp.band * bp.ratio;
                    if (bp.ratio_good > 0.0f) in_band = in_band || fabsf(r - bp.ratio_good) <= bp.band * bp.ratio_good;
                }
            }
            const int slot = block_rank(in_band, running, warp_excl, &chunk_total);
            if (in_band) {  // both neighbours exist: d1q >= 0
                bp.band_q[pd.knn_off + slot] = q;
                bp.band_thr[pd.knn_off + slot] = exact_threshold(d1q, resid[pd.qry_off + q], rmax);
                bp.band_state[2 * (pd.knn_off + slot)] = ~0ull;
                bp.band_state[2 * (pd.knn_off + slot) + 1] = ~0ull;
            }
        }
    }
    if (threadIdx.x == 0) bp.band_counts[blockIdx.x] = running;
    if (bp.cand_desc && running > 0) {
        // gather the band rows (packed descriptor + column key) into the scratch image the collect pass queries
        __syncthreads();
        const int lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
        for (int s = threadIdx.x >> 5; s < running; s += nwarps) {
            const int64_t src = pd.qry_off + bp.band_q[pd.knn_off + s], dst = pd.knn_off + s;
            reinterpret_cast<uint32_t *>(bp.cand_desc + dst * kDim)[lane] = reinterpret_cast<const uint32_t *>(bp.desc_arena + src * kDim)[lane];
            if (lane == 0) bp.cand_ckeys[dst] = bp.ckeys[src];
        }
    }
}

__device__ __forceinline__ bool fknn_less(float da, int ia, float db, int ib) { return da < db || (da == db && ia < ib); }

// Decision of one band row from its fp32 nearest (b0, c0i) and second nearest (b1, c1i) reference rows (-1: none).
__device__ __forceinline__ void write_rescored(const BandParams &bp, const PairDesc &pd, int q, float b0, int c0i, float b1, int c1i) {
    if (bp.out_ids) {  // exact kNN mode: FLANN layout, missing neighbour = (-1, +inf)
        const int64_t row = pd.knn_off + q;
        bp.out_ids[2 * row] = c0i;
        bp.out_ids[2 * row + 1] = c1i;
        bp.out_dists[2 * row] = c0i >= 0 ? b0 : INFINITY;
        bp.out_dists[2 * row + 1] = c1i >= 0 ? b1 : INFINITY;
        return;
    }
    int flags = 0;
    if (c0i >= 0 && c1i >= 0) {
        const float r = __fdiv_rn(b0, b1);
        bool keep = bp.reject_gt ? !(r > bp.ratio) : (r < bp.ratio);
        if (bp.max_dist_sq > 0.0f) keep = keep && (b0 * pd.fscale2 < bp.max_dist_sq);
        const bool good = keep && bp.ratio_good > 0.0f && (bp.reject_gt ? !(r > bp.ratio_good) : (r < bp.ratio_good));
        flags = (keep ? 1 : 0) | (good ? 2 : 0);
    }
    // integer distance of the fp32 nearest neighbour (seeds the mutual search of this candidate)
    int di = 0;
    if (c0i >= 0) {
        const uint32_t *qa = reinterpret_cast<const uint32_t *>(bp.desc_arena + (pd.qry_off + q) * kDim);
        const uint32_t *rb = reinterpret_cast<const uint32_t *>(bp.desc_arena + (pd.ref_off + c0i) * kDim);
        uint32_t na = 0, nb = 0, ab = 0;
        for (int k = 0; k < kDim / 4; ++k) { na = __dp4a(qa[k], qa[k], na); nb = __dp4a(rb[k], rb[k], nb); ab = __dp4a(qa[k], rb[k], ab); }
        di = (int)(na + nb - 2u * ab);
    }
    int4 out;
    out.x = (c0i >= 0 ? c0i : 0) | kRescoredFlag;
    out.y = flags;
    out.z = di;
    out.w = __float_as_int(b0);
    bp.knn[pd.knn_off + q] = out;
}

// fp32 squared distance of every collected event; best (distance, reference row) per band row.
__global__ void __launch_bounds__(256) score_events_kernel(const BandParams bp) {
    const unsigned n = *bp.event_count;
    if (n > bp.event_cap) return;  // overflow: rescore_band_kernel takes over
    for (unsigned e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
        const int4 ev = bp.events[e];
        const PairDesc pd = bp.pairs[ev.z];
        const float4 *qf = reinterpret_cast<const float4 *>(bp.fdesc + (pd.qry_off + bp.band_q[ev.x]) * kDim);
        const float4 *rf = reinterpret_cast<const float4 *>(bp.fdesc + (pd.ref_off + ev.y) * kDim);
        float acc = 0.0f;  // index order, separate multiply and add (nanoflann.hpp:376-383 without contraction)
#pragma unroll 4
        for (int k = 0; k < kDim / 4; ++k) {
            const float4 a = __ldg(qf + k), b = __ldg(rf + k);
            float t = __fsub_rn(a.x, b.x); acc = __fadd_rn(acc, __fmul_rn(t, t));
            t = __fsub_rn(a.y, b.y); acc = __fadd_rn(acc, __fmul_rn(t, t));
            t = __fsub_rn(a.z, b.z); acc = __fadd_rn(acc, __fmul_rn(t, t));
            t = __fsub_rn(a.w, b.w); acc = __fadd_rn(acc, __fmul_rn(t, t));
        }
        // distances are >= +0, so their bit patterns order like the values; the low word breaks ties by lowest row
        const unsigned long long key = ((unsigned long long)__float_as_uint(acc) << 32) | (unsigned)ev.y;
        bp.event_keys[e] = key;
        atomicMin(bp.band_state + 2 * (int64_t)ev.x, key);
    }
}

__global__ void __launch_bounds__(256) second_events_kernel(const BandParams bp) {
    const unsigned n = *bp.event_count;
    if (n > bp.event_cap) return;
    for (unsigned e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
        const int64_t row = bp.events[e].x;
        const unsigned long long key = bp.event_keys[e];
        if (key != bp.band_state[2 * row]) atomicMin(bp.band_state + 2 * row + 1, key);
    }
}

__global__ void __launch_bounds__(256) finish_band_kernel(const BandParams bp) {
    if (*bp.event_count > bp.event_cap) return;
    const PairDesc pd = bp.pairs[blockIdx.x];
    const int n_band = bp.band_counts[blockIdx.x];
    for (int s = threadIdx.x; s < n_band; s += blockDim.x) {
        const unsigned long long k0 = bp.band_state[2 * (pd.knn_off + s)], k1 = bp.band_state[2 * (pd.knn_off + s) + 1];
        const int c0i = k0 == ~0ull ? -1 : (int)(unsigned)k0, c1i = k1 == ~0ull ? -1 : (int)(unsigned)k1;
        write_rescored(bp, pd, bp.band_q[pd.knn_off + s], c0i < 0 ? INFINITY : __uint_as_float((unsigned)(k0 >> 32)), c0i,
                       c1i < 0 ? INFINITY : __uint_as_float((unsigned)(k1 >> 32)), c1i);
    }
}

// GATE: a reference row enters a band row's top-2 only if the epipolar or homography gate allows the element, evaluated
// like the matching kernel does (bit for bit: the allowed set is the one the row's threshold came from).  Under the
// homography gate a band row keeps its query keypoint and each reference column is transferred (hom_transfer,
// hom_allowed).  The gate is a separate argument because a longer BandParams would move the parameters after it in
// every kernel that takes one; the other stages of the collect path see gated rows only.
template <GateKind GATE>
__global__ void __launch_bounds__(256) rescore_band_kernel(const BandParams bp, int n_pairs, const EpiGate gate) {
    constexpr bool GUIDED = GATE != GateKind::none, HOMOG = GATE == GateKind::homography;
    __shared__ float sq[kRescoreRows][kDim];                  // band rows, float
    __shared__ __align__(16) uint32_t sq8[kRescoreRows][kDim / 4];  // the same rows, packed u8
    __shared__ int s_na[kRescoreRows], s_thr[kRescoreRows];
    __shared__ float red_d[8][kRescoreRows][2];
    __shared__ int red_i[8][kRescoreRows][2];
    __shared__ EpiLine s_line[GUIDED && !HOMOG ? kRescoreRows : 1];  // epipolar gate: the band rows' query lines
    __shared__ float2 s_kq[HOMOG ? kRescoreRows : 1];                 // homography gate: the band rows' keypoints
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (bp.event_count && *bp.event_count <= bp.event_cap) return;  // the collect path has every event: nothing to do
    for (int p = blockIdx.x; p < n_pairs; p += gridDim.x) {
        const PairDesc pd = bp.pairs[p];
        const int n_band = bp.band_counts[p];
        const float *ref = bp.fdesc + pd.ref_off * kDim;
        const uint8_t *ref8 = bp.desc_arena + pd.ref_off * kDim;
        const int32_t *refk = bp.ckeys + pd.ref_off;
        // chunks of a pair are spread over gridDim.y so that a small batch of pairs still fills the SMs
        for (int c0 = blockIdx.y * kRescoreRows; c0 < n_band; c0 += gridDim.y * kRescoreRows) {
            const int nq = min(kRescoreRows, n_band - c0);
            __syncthreads();  // previous chunk's shared data is no longer read
            for (int i = threadIdx.x; i < kRescoreRows * kDim; i += blockDim.x) {
                const int qi = i / kDim, k = i % kDim;
                sq[qi][k] = qi < nq ? bp.fdesc[(pd.qry_off + bp.band_q[pd.knn_off + c0 + qi]) * kDim + k] : 0.0f;
            }
            for (int i = threadIdx.x; i < kRescoreRows * (kDim / 4); i += blockDim.x) {
                const int qi = i / (kDim / 4), k = i % (kDim / 4);
                sq8[qi][k] = qi < nq ? reinterpret_cast<const uint32_t *>(bp.desc_arena + (pd.qry_off + bp.band_q[pd.knn_off + c0 + qi]) * kDim)[k] : 0u;
            }
            if (threadIdx.x < kRescoreRows) {
                const int qi = threadIdx.x;
                int na = 0, thr = -1;  // rows past the chunk end never pass the prefilter
                if (qi < nq) {
                    const int q = bp.band_q[pd.knn_off + c0 + qi];
                    na = ckey_to_norm(bp.ckeys[pd.qry_off + q]);
                    // Prefilter on the quantised distance: the threshold the collect pass used (exact_threshold)
                    thr = bp.band_thr[pd.knn_off + c0 + qi];
                    if (HOMOG) s_kq[qi] = gate.xy[pd.qry_off + q];
                    else if (GUIDED) s_line[qi] = epi_query_line(gate.fmat + 9 * p, gate.xy[pd.qry_off + q]);
                }
                s_na[qi] = na;
                s_thr[qi] = thr;
            }
            __syncthreads();
            float d0[kRescoreRows], d1[kRescoreRows];
            int i0[kRescoreRows], i1[kRescoreRows];
#pragma unroll
            for (int qi = 0; qi < kRescoreRows; ++qi) { d0[qi] = d1[qi] = INFINITY; i0[qi] = i1[qi] = -1; }
            for (int j = threadIdx.x; j < pd.ref_rows; j += blockDim.x) {
                uint32_t ab[kRescoreRows];
#pragma unroll
                for (int qi = 0; qi < kRescoreRows; ++qi) ab[qi] = 0u;
                const uint4 *r16 = reinterpret_cast<const uint4 *>(ref8 + (int64_t)j * kDim);
#pragma unroll 2
                for (int k4 = 0; k4 < kDim / 16; ++k4) {
                    const uint4 r = __ldg(r16 + k4);
#pragma unroll
                    for (int qi = 0; qi < kRescoreRows; ++qi) {
                        const uint4 a = *reinterpret_cast<const uint4 *>(&sq8[qi][4 * k4]);
                        ab[qi] = __dp4a(a.x, r.x, ab[qi]);
                        ab[qi] = __dp4a(a.y, r.y, ab[qi]);
                        ab[qi] = __dp4a(a.z, r.z, ab[qi]);
                        ab[qi] = __dp4a(a.w, r.w, ab[qi]);
                    }
                }
                const int nb = ckey_to_norm(refk[j]);
                float2 kj{};      // epipolar gate: reference row j's keypoint ...
                float nbj = 0.f;  // ... and |b|^2
                HomPoint hj{};    // homography gate: its transferred keypoint
                if (HOMOG) {
                    hj = hom_transfer(gate.fmat + 9 * p, gate.xy[pd.ref_off + j]);
                } else if (GUIDED) {
                    kj = gate.xy[pd.ref_off + j];
                    nbj = epi_ref_line(gate.fmat + 9 * p, kj).n;
                }
#pragma unroll
                for (int qi = 0; qi < kRescoreRows; ++qi) {
                    const int dint = s_na[qi] + nb - 2 * (int)ab[qi];
                    if (dint <= s_thr[qi] &&
                        (!GUIDED || (HOMOG ? hom_allowed(hj, s_kq[qi], gate.t2) : epi_allowed(s_line[qi], kj, nbj, gate.t2)))) {
                        // rare: exact fp32 distance, accumulated in index order without contraction
                        float acc = 0.0f;
                        const float *rf = ref + (int64_t)j * kDim;
                        for (int k = 0; k < kDim; ++k) {
                            const float t = __fsub_rn(sq[qi][k], __ldg(rf + k));
                            acc = __fadd_rn(acc, __fmul_rn(t, t));
                        }
                        // j ascends per thread: strict '<' keeps the lowest index
                        if (acc < d0[qi]) { d1[qi] = d0[qi]; i1[qi] = i0[qi]; d0[qi] = acc; i0[qi] = j; }
                        else if (acc < d1[qi]) { d1[qi] = acc; i1[qi] = j; }
                    }
                }
            }
            // merge the per-thread top-2 lists: warp shuffles, then across the 8 warps through shared memory
#pragma unroll
            for (int qi = 0; qi < kRescoreRows; ++qi) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const float e0 = __shfl_xor_sync(0xFFFFFFFFu, d0[qi], o), e1 = __shfl_xor_sync(0xFFFFFFFFu, d1[qi], o);
                    const int j0 = __shfl_xor_sync(0xFFFFFFFFu, i0[qi], o), j1 = __shfl_xor_sync(0xFFFFFFFFu, i1[qi], o);
                    const bool mine = i0[qi] >= 0 && (j0 < 0 || fknn_less(d0[qi], i0[qi], e0, j0));
                    // winner w, loser l of the two heads; second = best of {w's second, l's head}
                    const float wd0 = mine ? d0[qi] : e0, wd1 = mine ? d1[qi] : e1, ld0 = mine ? e0 : d0[qi];
                    const int wi0 = mine ? i0[qi] : j0, wi1 = mine ? i1[qi] : j1, li0 = mine ? j0 : i0[qi];
                    const bool second_from_w = wi1 >= 0 && (li0 < 0 || fknn_less(wd1, wi1, ld0, li0));
                    d0[qi] = wd0; i0[qi] = wi0;
                    d1[qi] = second_from_w ? wd1 : ld0;
                    i1[qi] = second_from_w ? wi1 : li0;
                }
                if (lane == 0) { red_d[warp][qi][0] = d0[qi]; red_d[warp][qi][1] = d1[qi]; red_i[warp][qi][0] = i0[qi]; red_i[warp][qi][1] = i1[qi]; }
            }
            __syncthreads();
            if (threadIdx.x < nq) {
                const int qi = threadIdx.x;
                float b0 = INFINITY, b1 = INFINITY;
                int c0i = -1, c1i = -1;
                for (int w = 0; w < 8; ++w)
                    for (int s = 0; s < 2; ++s) {
                        const float d = red_d[w][qi][s];
                        const int i = red_i[w][qi][s];
                        if (i < 0) continue;
                        if (c0i < 0 || fknn_less(d, i, b0, c0i)) { b1 = b0; c1i = c0i; b0 = d; c0i = i; }
                        else if (c1i < 0 || fknn_less(d, i, b1, c1i)) { b1 = d; c1i = i; }
                    }
                write_rescored(bp, pd, bp.band_q[pd.knn_off + c0 + qi], b0, c0i, b1, c1i);
            }
        }
    }
}

// Stage 1 — ratio test (+ the mutual cross-check without a second GEMM pass).  One CTA per pair scans its query rows in
// ascending order (the order of fine_matching_graph.cc:116-133 / feature_matching.cpp:56-64) and writes the one-way
// candidates (query row, nearest reference row, "good" flag) compacted into the pair's scratch region.
//
// Mutual check, exact, from what the forward pass already knows (DESIGN.md §4.4).  Candidate (q, j = nn0(q), d0) survives
// iff no other query row q' has d(q', j) < d0, or == d0 with q' < q (lowest index wins ties, SiftGPU s_col_max).  The
// rivals q' are of two kinds:
//   (A) rows whose own nearest neighbour is j: their distance to j is their d0 — every row does one atomicMin of
//       (d0, q') on a per-pair column table keyed by nn0, which leaves the best of them per reference row;
//   (B) rows for which j is not the nearest: then d(q', j) >= d1(q') (j is at best their second neighbour), so only rows
//       with d1(q') <= d0 can beat or tie the candidate.  A true match has a small d0 and almost no row has a second
//       neighbour that close: the few "dangerous" rows are listed per pair and their distance to j is computed exactly.
// A pair whose dangerous sets are large (repetitive structure, near-duplicate rows: more than kDangerWorkCap candidates
// that have to look at dangerous rows, or more than kDangerEvalBudget exact distances in total), and every pair of the float regime with re-scoring, falls
// back to the tensor twin pass: the candidates' reference rows are gathered into the candidate scratch image, which the
// matching kernel then searches against the query image (twin_counts[pair] > 0 routes the pair there).
constexpr int kDangerWorkCap = 2048;     // candidates per pair that have to look at the dangerous rows (shared memory)
constexpr int kDangerEvalBudget = 65536;  // exact 128-byte distances per pair on CUDA cores
constexpr int kSmemTableRows = 20480;    // reference rows whose column table fits in shared memory (160 KiB)
constexpr int kDangerChunk = 128;        // list rows per work unit of the exact evaluation (= entries of a warp's hit queue)
constexpr int kDangerFlight = 2;         // hits per lane group and round while scoring (8 groups of 4 lanes, 2 row loads per lane and hit)
constexpr size_t kSelectSmemBytes = (size_t)kDangerWorkCap * 16 + 32 * kDangerChunk * 4 + (size_t)kSmemTableRows * 8;  // 208 KiB
constexpr int kCandGood = 1, kCandKilled = 2;  // bits of cand_good[]

struct SelectParams {
    const PairDesc *pairs;
    const int4 *knn;
    float ratio, ratio_good, max_dist_sq;
    int32_t reject_gt;         // ratio rule: 0 accept iff r < ratio; 1 accept iff !(r > ratio) (slam_gps.cc:470-477)
    int32_t *cand_q, *cand_j;  // [forward kNN rows], pair p writes from row knn_off
    int32_t *cand_d0;          // squared distance of the candidate (seeds the mutual search)
    uint8_t *cand_good;        // kCandGood | kCandKilled
    int32_t *counts;           // [n_pairs] one-way candidates
    int32_t mutual;
    unsigned long long *colbest;  // [sum of ref rows of the batch] (d0 << 32 | q), initialised to ~0: column table of the
                                  // pairs with more than smem_table_rows reference rows (the others keep it in shared memory)
    int32_t smem_table_rows;
    int2 *danger;              // [forward kNN rows] per-pair list of (row, d1) of the dangerous rows
    int32_t *twin_counts;      // [n_pairs] candidates routed to the tensor twin pass (0: decided here)
    unsigned int *routed;      // number of pairs routed to the twin pass (the twin launch returns at once when 0)
    const uint8_t *desc_arena;
    const int32_t *ckeys;
    uint8_t *cand_desc;        // [forward kNN rows][128]
    int32_t *cand_ckeys;
    int32_t float_mutual;      // float regime with re-scoring: widen the mutual search by the quantisation slack
    int32_t force_twin;        // test hook: every pair takes the tensor twin pass
};

__device__ __forceinline__ bool ratio_accepts(float r, float th, int reject_gt) { return reject_gt ? !(r > th) : (r < th); }

__device__ __forceinline__ unsigned long long colbest_key(int d0, int q) {
    return ((unsigned long long)(unsigned)d0 << 32) | (unsigned)q;
}

// Exact squared distance of two packed rows (norms from the column keys).
__device__ __forceinline__ int sqdist_u8_rows(const uint8_t *__restrict__ a, const uint8_t *__restrict__ b, int na, int nb) {
    const uint4 *pa = reinterpret_cast<const uint4 *>(a), *pb = reinterpret_cast<const uint4 *>(b);
    uint32_t ab = 0;
#pragma unroll
    for (int k = 0; k < kDim / 16; ++k) {
        const uint4 x = __ldg(pa + k), y = __ldg(pb + k);
        ab = __dp4a(x.x, y.x, ab);
        ab = __dp4a(x.y, y.y, ab);
        ab = __dp4a(x.z, y.z, ab);
        ab = __dp4a(x.w, y.w, ab);
    }
    return na + nb - 2 * (int)ab;
}

// Block-wide exclusive scan of a small per-thread count (threads in index order); adds the block total to `running`.
__device__ __forceinline__ int block_scan_excl(int v, int &running, int *warp_excl, int *chunk_total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int n = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= o) incl += n;
    }
    if (lane == 31) warp_excl[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const int w = (lane < nwarps) ? warp_excl[lane] : 0;
        int wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int n = __shfl_up_sync(0xFFFFFFFFu, wi, o);
            if (lane >= o) wi += n;
        }
        warp_excl[lane] = wi - w;
        if (lane == 31) *chunk_total = wi;
    }
    __syncthreads();
    const int excl = running + warp_excl[warp] + incl - v;
    running += *chunk_total;
    __syncthreads();
    return excl;
}

// Bucket of a dangerous row's bound d in [d1min, d0max]: monotone in d, 0..255.
__device__ __forceinline__ int danger_bucket(int d, int d1min, float inv) { return min(255, max(0, (int)((float)(d - d1min) * inv))); }

constexpr int kSelRows = 8;  // query rows per thread and chunk: their kNN records are loaded together (one L2 round trip)

__global__ void __launch_bounds__(1024) select_candidates_kernel(const SelectParams sp) {
    // dynamic shared memory (mutual launches only): job list, dangerous-row list, column table of pairs with
    // <= smem_table_rows reference rows
    extern __shared__ unsigned long long s_dyn[];
    int4 *s_work = reinterpret_cast<int4 *>(s_dyn);
    int *s_hitq = reinterpret_cast<int *>(s_work + kDangerWorkCap);  // [32 warps][kDangerChunk]
    unsigned long long *s_table = reinterpret_cast<unsigned long long *>(s_hitq + 32 * kDangerChunk);
    __shared__ int warp_excl[32];
    __shared__ int chunk_total;
    __shared__ int s_d0max, s_d1min, s_nd, s_nwork, s_evals, s_unit;
    __shared__ int s_hist[257], s_cursor[256];  // counting sort of the dangerous-row list
    const PairDesc pd = sp.pairs[blockIdx.x];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    int2 *danger = sp.danger + pd.knn_off;  // this pair's dangerous rows (row, d1), unordered; at most one per query row
    // the bound-based check needs integer distances that are final: not in the re-scored float regime
    const bool bounds = sp.mutual && !sp.force_twin && !(sp.float_mutual && pd.fscale2 > 0.0f);
    unsigned long long *table = sp.colbest + pd.col_off;
    if (bounds && pd.ref_rows <= sp.smem_table_rows) {
        table = s_table;
        for (int j = threadIdx.x; j < pd.ref_rows; j += blockDim.x) s_table[j] = ~0ull;
    }
    if (threadIdx.x == 0) { s_d0max = -1; s_d1min = INT_MAX; s_nd = 0; s_nwork = 0; s_evals = 0; s_unit = 0; }
    __syncthreads();
    int running = 0;
    int4 k[kSelRows];  // kNN records of this thread's rows in the current chunk (pass 2 re-uses them when there is only one)
    for (int base = 0; base < pd.qry_rows; base += blockDim.x * kSelRows) {
        const int q0 = base + threadIdx.x * kSelRows;  // this thread's rows are consecutive: thread order = row order
#pragma unroll
        for (int r = 0; r < kSelRows; ++r)
            k[r] = (q0 + r < pd.qry_rows) ? load_knn(sp.knn, pd.knn_off + q0 + r) : make_int4(-1, -1, INT_MAX, INT_MAX);
        unsigned keep = 0, good = 0;
        int d0max = -1;
#pragma unroll
        for (int r = 0; r < kSelRows; ++r) {
            if (k[r].x >= 0 && (k[r].x & kRescoredFlag)) {  // decided on exact fp32 distances by rescore_band_kernel
                if (k[r].y & 1) keep |= 1u << r;
                if (k[r].y & 2) good |= 1u << r;
                k[r].x &= ~kRescoredFlag;
            } else {
                if (k[r].x >= 0 && k[r].y >= 0) {
                    const float d0 = (float)k[r].z, d1 = (float)k[r].w;
                    const float ratio = __fdiv_rn(d0, d1);  // IEEE divide; 0/0 = NaN fails every comparison
                    bool kp = ratio_accepts(ratio, sp.ratio, sp.reject_gt);
                    if (sp.max_dist_sq > 0.0f) kp = kp && (d0 < sp.max_dist_sq);
                    if (kp) keep |= 1u << r;
                    if (kp && sp.ratio_good > 0.0f && ratio_accepts(ratio, sp.ratio_good, sp.reject_gt)) good |= 1u << r;
                }
                // rival kind (A): every row, accepted or not, claims its nearest reference row
                if (bounds && k[r].x >= 0) atomicMin(table + k[r].x, colbest_key(k[r].z, q0 + r));
            }
            if (keep & (1u << r)) d0max = max(d0max, k[r].z);
        }
        int slot = block_scan_excl(__popc(keep), running, warp_excl, &chunk_total);
#pragma unroll
        for (int r = 0; r < kSelRows; ++r)
            if (keep & (1u << r)) {
                sp.cand_q[pd.knn_off + slot] = q0 + r;
                sp.cand_j[pd.knn_off + slot] = k[r].x;
                sp.cand_good[pd.knn_off + slot] = (good >> r) & 1u ? kCandGood : 0;
                // float regime: a query row that is a few 1e-3 farther in quantised units may be the nearer one in fp32,
                // so the mutual search keeps every row within ~3 % of the candidate's distance (see emit_matches_kernel)
                sp.cand_d0[pd.knn_off + slot] = (sp.float_mutual && pd.fscale2 > 0.0f) ? k[r].z + (k[r].z >> 5) + 256 : k[r].z;
                ++slot;
            }
        if (bounds && d0max >= 0) atomicMax(&s_d0max, d0max);
    }
    if (threadIdx.x == 0) sp.counts[blockIdx.x] = running;
    if (!sp.mutual) return;
    __syncthreads();  // candidate list, s_d0max and this pair's column table are complete (only this CTA writes them)
    bool overflow = !bounds;
    if (bounds && running > 0) {
        // ---- rival kind (B): rows whose second neighbour is at least as close as the weakest candidate's match
        //      (unordered list in the pair's scratch region; no block-wide synchronisation inside the loop)
        const int d0max = s_d0max;
        const bool single = pd.qry_rows <= (int)blockDim.x * kSelRows;  // pass 1's records are still in registers
        for (int base = 0; base < pd.qry_rows; base += blockDim.x * kSelRows) {
            const int q0 = base + threadIdx.x * kSelRows;
            if (!single) {
#pragma unroll
                for (int r = 0; r < kSelRows; ++r)
                    k[r] = (q0 + r < pd.qry_rows) ? load_knn(sp.knn, pd.knn_off + q0 + r) : make_int4(-1, -1, INT_MAX, INT_MAX);
            }
#pragma unroll
            for (int r = 0; r < kSelRows; ++r)
                if (k[r].y >= 0 && k[r].w <= d0max) {  // (id1, d1)
                    danger[atomicAdd(&s_nd, 1)] = make_int2(q0 + r, k[r].w);
                    atomicMin(&s_d1min, k[r].w);
                }
        }
        __syncthreads();
        const int nd = s_nd;
        {
            // ---- verdicts.  One thread per candidate: the column table decides kind (A); a candidate whose match is
            //      closer than every dangerous row's second neighbour (the usual case) is done, the others are listed.
            const int d1min = s_d1min;
            for (int i = threadIdx.x; i < running; i += blockDim.x) {
                const int q = sp.cand_q[pd.knn_off + i], j = sp.cand_j[pd.knn_off + i], d0 = sp.cand_d0[pd.knn_off + i];
                const unsigned long long best = (table == s_table) ? s_table[j] : __ldcg(table + j);
                if (best != colbest_key(d0, q)) {  // a kind-(A) rival is closer
                    sp.cand_good[pd.knn_off + i] |= kCandKilled;
                } else if (nd > 0 && d0 >= d1min) {
                    const int slot = atomicAdd(&s_nwork, 1);
                    if (slot < kDangerWorkCap) s_work[slot] = make_int4(i, q, j, d0);
                }
            }
            __syncthreads();
            const int nwork = s_nwork;
            overflow = nwork > kDangerWorkCap;
            bool sorted = false;
            if (!overflow && nwork > 0 && nd <= sp.smem_table_rows) {
                // The column table has done its job (verdicts above): its shared memory now holds the dangerous-row list,
                // counting-sorted into 256 buckets of the bound (d1min .. d0max).  A candidate then only looks at the list
                // prefix up to its own bucket — rows in lower buckets are hits by construction (the bucket function is
                // monotone), rows in higher ones cannot be — instead of testing every listed row.
                int2 *s_danger = reinterpret_cast<int2 *>(s_table);
                const float inv = 256.0f / (float)(s_d0max - d1min + 1);
                for (int b = threadIdx.x; b < 257; b += blockDim.x) s_hist[b] = 0;
                __syncthreads();
                for (int e = threadIdx.x; e < nd; e += blockDim.x) atomicAdd(&s_hist[danger_bucket(danger[e].y, d1min, inv) + 1], 1);
                __syncthreads();
                if (warp == 0) {  // inclusive scan of the 256 counts -> s_hist[b] = first list position of bucket b
                    int v[8], sum = 0;
#pragma unroll
                    for (int i = 0; i < 8; ++i) { v[i] = s_hist[1 + lane * 8 + i]; sum += v[i]; }
                    int incl = sum;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const int t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                        if (lane >= o) incl += t;
                    }
                    int run = incl - sum;
#pragma unroll
                    for (int i = 0; i < 8; ++i) { run += v[i]; s_hist[1 + lane * 8 + i] = run; }
                }
                __syncthreads();
                for (int b = threadIdx.x; b < 256; b += blockDim.x) s_cursor[b] = s_hist[b];
                __syncthreads();
                for (int e = threadIdx.x; e < nd; e += blockDim.x) {
                    const int2 r = danger[e];
                    s_danger[atomicAdd(&s_cursor[danger_bucket(r.y, d1min, inv)], 1)] = r;
                }
                __syncthreads();
                danger = s_danger;
                sorted = true;
            }
            if (!overflow && nwork > 0) {
                // (listed candidate) x (dangerous row).  The bound test is one compare per combination; the few that pass
                // ("hits", ~1e4 per 8192 x 8192 pair) cost an exact 128-byte distance each.  Work unit = (candidate, chunk of
                // kDangerChunk list rows), dealt to the warps on demand: the warp keeps its 32-byte share of the candidate's
                // reference row in registers, queues the chunk's hits in shared memory and scores them 16 at a time —
                // four lanes per distance, four independent row loads in flight per lane.
                const int nchunks = (nd + kDangerChunk - 1) / kDangerChunk;
                int cshift = 0;  // units are numbered candidate * 2^cshift + chunk: no division per unit
                while ((1 << cshift) < nchunks) ++cshift;
                const int units = nwork << cshift;
                const int sub = lane >> 2, part = lane & 3;  // which of the warp's 8 concurrent distances, which 32 bytes
                int *hitq = s_hitq + warp * kDangerChunk;
                const float inv = 256.0f / (float)(s_d0max - d1min + 1);
                for (;;) {
                    int u = 0;
                    if (lane == 0) u = atomicAdd(&s_unit, 1);  // units differ widely in hits
                    u = __shfl_sync(0xFFFFFFFFu, u, 0);
                    if (u >= units || s_evals >= kDangerEvalBudget) break;  // (budget: too ambiguous for CUDA cores)
                    const int w = u >> cshift, e0 = (u & ((1 << cshift) - 1)) * kDangerChunk;
                    const int4 c = s_work[w];  // (candidate, q, j, d0)
                    // list prefix this candidate has to look at (d1min <= c.w <= d0max holds for every listed candidate)
                    const int prefix = sorted ? s_hist[danger_bucket(c.w, d1min, inv) + 1] : nd;
                    if (e0 >= prefix) continue;
                    int n = 0;
                    const int e1 = min(e0 + kDangerChunk, prefix);
                    for (int eb = e0; eb < e1; eb += 32) {  // warp-uniform trip count
                        const int e = eb + lane;
                        bool hit = false;
                        int2 r = make_int2(0, 0);
                        if (e < e1) {
                            r = danger[e];
                            hit = r.y <= c.w && r.x != c.y;
                        }
                        const unsigned hits = __ballot_sync(0xFFFFFFFFu, hit);
                        if (hit) hitq[n + __popc(hits & ((1u << lane) - 1u))] = r.x;
                        n += __popc(hits);
                    }
                    if (n == 0) continue;
                    __syncwarp();
                    if (lane == 0) atomicAdd(&s_evals, n);
                    const uint4 *yp = reinterpret_cast<const uint4 *>(sp.desc_arena + (pd.ref_off + c.z) * kDim) + part * 2;
                    const uint4 y0 = __ldg(yp), y1 = __ldg(yp + 1);
                    const int nb = ckey_to_norm(sp.ckeys[pd.ref_off + c.z]);
                    for (int base = 0; base < n; base += 8 * kDangerFlight) {
                        int row[kDangerFlight];
                        uint4 x0[kDangerFlight], x1[kDangerFlight];
#pragma unroll
                        for (int k2 = 0; k2 < kDangerFlight; ++k2) {
                            const int idx = base + k2 * 8 + sub;
                            row[k2] = idx < n ? hitq[idx] : -1;
                            x0[k2] = x1[k2] = make_uint4(0, 0, 0, 0);
                            if (row[k2] >= 0) {
                                const uint4 *xp = reinterpret_cast<const uint4 *>(sp.desc_arena + (pd.qry_off + row[k2]) * kDim) + part * 2;
                                x0[k2] = __ldg(xp);
                                x1[k2] = __ldg(xp + 1);
                            }
                        }
#pragma unroll
                        for (int k2 = 0; k2 < kDangerFlight; ++k2) {
                            // this lane's share of ||x||^2 - 2 x.y  (the row's norm comes from the row itself)
                            const uint4 a = x0[k2], b = x1[k2];
                            uint32_t ab = __dp4a(a.x, y0.x, 0u), aa = __dp4a(a.x, a.x, 0u);
                            ab = __dp4a(a.y, y0.y, ab); aa = __dp4a(a.y, a.y, aa);
                            ab = __dp4a(a.z, y0.z, ab); aa = __dp4a(a.z, a.z, aa);
                            ab = __dp4a(a.w, y0.w, ab); aa = __dp4a(a.w, a.w, aa);
                            ab = __dp4a(b.x, y1.x, ab); aa = __dp4a(b.x, b.x, aa);
                            ab = __dp4a(b.y, y1.y, ab); aa = __dp4a(b.y, b.y, aa);
                            ab = __dp4a(b.z, y1.z, ab); aa = __dp4a(b.z, b.z, aa);
                            ab = __dp4a(b.w, y1.w, ab); aa = __dp4a(b.w, b.w, aa);
                            int pd2 = (int)aa - 2 * (int)ab;
                            pd2 += __shfl_xor_sync(0xFFFFFFFFu, pd2, 1);  // over the 4 lanes of the group
                            pd2 += __shfl_xor_sync(0xFFFFFFFFu, pd2, 2);
                            if (part == 0 && row[k2] >= 0) {
                                const int d = pd2 + nb;
                                // several rivals may kill the same candidate: they all set the same bit, the other bits are final
                                if (d < c.w || (d == c.w && row[k2] < c.y)) sp.cand_good[pd.knn_off + c.x] |= kCandKilled;
                            }
                        }
                    }
                    __syncwarp();  // the queue is rewritten by the next unit
                }
                __syncthreads();
                overflow = s_evals >= kDangerEvalBudget;
            }
        }
    }
    if (threadIdx.x == 0) {
        sp.twin_counts[blockIdx.x] = overflow ? running : 0;
        if (overflow && running > 0) atomicAdd(sp.routed, 1u);
    }
    if (!overflow) return;
    // ---- tensor twin pass for this pair: gather the candidates' reference rows (+ column keys) into the scratch image
    __syncthreads();
    for (int i = warp; i < running; i += nwarps) {
        const int j = sp.cand_j[pd.knn_off + i];
        const uint32_t w = reinterpret_cast<const uint32_t *>(sp.desc_arena + (pd.ref_off + j) * kDim)[lane];
        reinterpret_cast<uint32_t *>(sp.cand_desc + (pd.knn_off + i) * kDim)[lane] = w;
        if (lane == 0) sp.cand_ckeys[pd.knn_off + i] = sp.ckeys[pd.ref_off + j];
    }
}

// Stage 2 — emission.  Candidate i of pair p survives the mutual check iff select_candidates_kernel did not kill it, or
// (pairs routed to the twin pass) iff the nearest query row of its reference row (row i of the pair's twin kNN region)
// is the candidate's own query row.
struct EmitParams {
    const PairDesc *pairs;
    const int4 *knn;
    int64_t twin_base;        // twin kNN row of candidate i of pair p = twin_base + knn_off + i
    const int32_t *cand_q, *cand_j;
    const uint8_t *cand_good;
    const int32_t *cand_counts;
    const int32_t *twin_counts;
    int2 *matches;             // per-batch scratch; pair p writes its list from row knn_off
    uint8_t *good;
    int32_t *counts;           // [n_pairs] surviving matches
    int32_t mutual, orientation;
    const float *fdesc;        // float regime with re-scoring: retained float rows (else null)
};

// Exact fp32 squared distance, accumulated in index order without contraction (nanoflann.hpp:376-383).
__device__ __forceinline__ float sqdist_f32_rows(const float *__restrict__ a, const float *__restrict__ b) {
    float acc = 0.0f;
    for (int k = 0; k < kDim; ++k) {
        const float t = __fsub_rn(__ldg(a + k), __ldg(b + k));
        acc = __fadd_rn(acc, __fmul_rn(t, t));
    }
    return acc;
}

__global__ void __launch_bounds__(1024) emit_matches_kernel(const EmitParams ep) {
    __shared__ int warp_excl[32];
    __shared__ int chunk_total;
    const PairDesc pd = ep.pairs[blockIdx.x];
    const int n = ep.cand_counts[blockIdx.x];
    const bool twin = ep.mutual && ep.twin_counts[blockIdx.x] > 0;
    int running = 0;
    for (int base = 0; base < n; base += blockDim.x) {
        const int i = base + threadIdx.x;
        bool keep = i < n;
        int q = -1, j = -1;
        uint8_t flags = 0;
        if (keep) {
            q = ep.cand_q[pd.knn_off + i];
            j = ep.cand_j[pd.knn_off + i];
            flags = ep.cand_good[pd.knn_off + i];
            if (ep.mutual && !twin) keep = (flags & kCandKilled) == 0;
            if (twin) {
                const int4 tw = load_knn(ep.knn, ep.twin_base + pd.knn_off + i);
                keep = tw.x == q;
                if (ep.fdesc && pd.fscale2 > 0.0f && tw.x >= 0 && tw.y >= 0 && (tw.x == q || tw.y == q)) {
                    // two query rows within the quantisation slack of reference row j: decide on fp32 distances
                    const float *rj = ep.fdesc + (pd.ref_off + j) * kDim;
                    const float da = sqdist_f32_rows(ep.fdesc + (pd.qry_off + tw.x) * kDim, rj);
                    const float db = sqdist_f32_rows(ep.fdesc + (pd.qry_off + tw.y) * kDim, rj);
                    const int best = (db < da || (db == da && tw.y < tw.x)) ? tw.y : tw.x;
                    keep = best == q;
                }
            }
        }
        const int slot = block_rank(keep, running, warp_excl, &chunk_total);
        if (keep) {
            int2 m;
            if (ep.orientation == 0) { m.x = j; m.y = q; } else { m.x = q; m.y = j; }
            ep.matches[pd.knn_off + slot] = m;
            if (ep.good) ep.good[pd.knn_off + slot] = flags & kCandGood;
        }
    }
    if (threadIdx.x == 0) ep.counts[blockIdx.x] = running;
}

// Exclusive scan of the per-pair counts into int64 offsets[n+1]; single CTA (n is a per-batch pair count).
__global__ void __launch_bounds__(1024) scan_counts_kernel(const int32_t *__restrict__ counts, int n, int64_t *__restrict__ offsets) {
    __shared__ long long warp_excl[32];
    __shared__ long long chunk_total;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long running = 0;
    for (int base = 0; base < n; base += blockDim.x) {
        const int i = base + threadIdx.x;
        const long long v = (i < n) ? counts[i] : 0;
        long long incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) warp_excl[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            const long long w = warp_excl[lane];
            long long wi = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const long long t = __shfl_up_sync(0xFFFFFFFFu, wi, o);
                if (lane >= o) wi += t;
            }
            warp_excl[lane] = wi - w;
            if (lane == 31) chunk_total = wi;
        }
        __syncthreads();
        if (i < n) offsets[i] = running + warp_excl[warp] + incl - v;
        running += chunk_total;
        __syncthreads();
    }
    if (threadIdx.x == 0) offsets[n] = running;
}

// Copy each pair's list from its scratch segment to the tight output.
__global__ void gather_matches_kernel(const PairDesc *__restrict__ pairs, const int32_t *__restrict__ counts,
                                      const int64_t *__restrict__ offsets, const int2 *__restrict__ matches,
                                      const uint8_t *__restrict__ good, int2 *__restrict__ out_matches,
                                      uint8_t *__restrict__ out_good) {
    const PairDesc pd = pairs[blockIdx.x];
    const int n = counts[blockIdx.x];
    const int64_t dst = offsets[blockIdx.x];
    for (int k = threadIdx.x; k < n; k += blockDim.x) {
        out_matches[dst + k] = matches[pd.knn_off + k];
        if (out_good) out_good[dst + k] = good[pd.knn_off + k];
    }
}

// kNN scratch {id0,id1,d0,d1} -> FLANN layout ids[2q..], dists[2q..] (float), one pair.
__global__ void knn_to_flann_kernel(const int4 *__restrict__ knn, int rows, int32_t *__restrict__ ids,
                                    float *__restrict__ dists) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= rows) return;
    const int4 k = load_knn(knn, q);
    ids[2 * q] = k.x;
    ids[2 * q + 1] = k.y;
    dists[2 * q] = k.x >= 0 ? (float)k.z : __int_as_float(0x7f800000);
    dists[2 * q + 1] = k.y >= 0 ? (float)k.w : __int_as_float(0x7f800000);
}

// Nearest neighbour only (used for the "best query of each reference row" query).
__global__ void knn_best_kernel(const int4 *__restrict__ knn, int rows, int32_t *__restrict__ best,
                                float *__restrict__ dist) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= rows) return;
    const int4 k = load_knn(knn, j);
    best[j] = k.x;
    dist[j] = k.x >= 0 ? (float)k.z : __int_as_float(0x7f800000);
}

// ------------------------------------------------------------------------------------------------ cross-check
// CUDA-core brute force (dp4a): thread = query row, loops over all reference rows (warp-uniform broadcast loads).
// Test-only GPU cross-check of the tcgen05 path; exact int32, lowest index on ties.
__global__ void crosscheck_knn2_kernel(const uint8_t *__restrict__ ref, const int32_t *__restrict__ ref_ckeys, int M,
                                       const uint8_t *__restrict__ qry, const int32_t *__restrict__ qry_ckeys, int N,
                                       int4 *__restrict__ knn) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= N) return;
    uint32_t a[32];
    const uint4 *qa = reinterpret_cast<const uint4 *>(qry + (int64_t)q * kDim);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const uint4 v = qa[k];
        a[4 * k] = v.x; a[4 * k + 1] = v.y; a[4 * k + 2] = v.z; a[4 * k + 3] = v.w;
    }
    const int na = ckey_to_norm(qry_ckeys[q]);
    int d0 = INT_MAX, d1 = INT_MAX, i0 = -1, i1 = -1;
    for (int j = 0; j < M; ++j) {
        const uint4 *rb = reinterpret_cast<const uint4 *>(ref + (int64_t)j * kDim);
        uint32_t dot = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const uint4 v = __ldg(rb + k);
            dot = __dp4a(a[4 * k], v.x, dot);
            dot = __dp4a(a[4 * k + 1], v.y, dot);
            dot = __dp4a(a[4 * k + 2], v.z, dot);
            dot = __dp4a(a[4 * k + 3], v.w, dot);
        }
        const int d = na + ckey_to_norm(__ldg(ref_ckeys + j)) - 2 * (int)dot;
        if (d < d1) {
            if (d < d0) { d1 = d0; i1 = i0; d0 = d; i0 = j; }
            else { d1 = d; i1 = j; }
        }
    }
    knn[q] = make_int4(i0, i1, i0 >= 0 ? d0 : INT_MAX, i1 >= 0 ? d1 : INT_MAX);
}

}  // namespace msfm
