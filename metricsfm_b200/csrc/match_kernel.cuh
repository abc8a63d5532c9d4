// match_kernel.cuh — the hot path: persistent, warp-specialised sm_100a kernel that, for a list of
// (pair, query-strip-group) work items, computes the u8 x u8 -> s32 Gram tile on the 5th-gen tensor cores
// (tcgen05.mma.kind::i8, operands TMA-staged in 128B-swizzled shared memory, accumulators in TMEM) and reduces it
// in a fused epilogue to
//   * per query row: exact top-2 of d = ||q||^2 + ||r||^2 - 2 q.r  (lowest reference index on ties),
// so the N x M distance matrix never leaves the SM.  The mutual cross-check ("best query of a reference row") is the
// same reduction with the roles of the two images swapped; the host schedules those items into the same launch.
//
// Replaces the arithmetic of flann_find_nearest_neighbors_index(k=2) at
// /root/reference/SfM/src/graph/fine_matching_graph.cc:99 (and slam_gps.cc:463, feature_matching.cpp:44,336,409)
// with the brute-force/mutual-best semantics of the declared GPU matchers (SiftGPU.h:303-308, cudaSift sift.h:97).
//
// Roles per CTA (4*STRIPS epilogue warps + 1 + STRIPS auxiliary warps padded to whole warpgroups; one CTA per SM,
// persistent over work items):
//   epilogue warps  warp w owns TMEM lanes 32*(w%4).. of query strip w/4 and all TILE_N columns of every tile
//                   (thread = query row)
//   next warp       TMA producer (one elected lane)
//   next STRIPS     MMA issuers, one per query strip (one elected lane each; the first also owns the TMEM allocation):
//                   spreads the issue instructions over the four SM sub-partitions and lets every strip advance as soon
//                   as ITS accumulator buffer is free
//   (padding warps) idle; the auxiliary warpgroups hand their registers to the epilogue warps (setmaxnreg)
//   The service warps share issue slots with the epilogue warps of their sub-partition: their tile loops are unrolled
//   over the B ring (immediate addresses) and they sleep between polls (see the comment at the role dispatch).
// Two template parameters vary the epilogue's exact phase, everything else is shared: COLLECT (float regime) replaces the
// top-2 merge by "append every element under the row's fixed threshold to an event list"; GATE (guided matching) bars
// the elements that fail the epipolar gate (epi_allowed) or the homography gate (hom_allowed) from the row's top-2 or
// event list.
// Work distribution: CTA b takes items b, b + grid, ...; every role walks that list on its own.
// Pipelines (all mbarrier based):
//   A ring (2 deep)     : query strips of a work item, STRIPS x [128 rows x 128 B]
//   B ring (STAGES)     : reference tiles [TILE_N rows x 128 B]
//   column-key ring     : ckey_j = -8*||r_j||^2 + (7 - j%8) of the tile's reference rows + the tile's smallest norm; they
//                         complete the B stage's "full" barrier together with the tile (no barriers of their own: the
//                         epilogue reads them behind the tile's MMAs; for the slot count see MatchKernelCfg::kKeySlots)
//   TMEM                : TBUFS x STRIPS accumulator blocks of TILE_N int32 columns, each with its own full/empty
//                         barrier pair, so the MMA of tile t+1 runs under the epilogue of tile t
#pragma once
#include <cstddef>
#include <cstdint>
#include <climits>
#include <cuda.h>
#include <cuda_runtime.h>

#include "sm100_ptx.cuh"

namespace msfm {

constexpr int kDim = 128;        // bytes per packed descriptor row
constexpr int kStripRows = 128;  // MMA M
constexpr int kAlignRows = 256;  // every image starts on / is padded to a multiple of this many rows
constexpr int kBoxRows = 64;     // rows per TMA box (strips and reference tiles are loaded as 64-row boxes)
constexpr int kKeyTileRows = 64; // granularity of the per-tile minimum-norm table (MatchKernelParams::tilemin) = TILE_N

// Per-row side table ("column keys").  For row j with squared norm nb:  ckey = -8*nb + (7 - j%8).
//   * exact packed score key of element (q, j):  16*acc + ckey = 8*(2*acc - nb) + (7 - j%8)
//     (max key = best score, then lowest column inside a group of 8)
//   * nb = (7 - ckey) >> 3
// Pad rows carry kNormPad so that they lose against every real column.
constexpr uint32_t kNormPad = 0x0FFFFFF0u;
__host__ __device__ constexpr int32_t make_ckey(uint32_t nb, int j) { return -8 * (int32_t)nb + (7 - (j & 7)); }
__host__ __device__ constexpr int32_t ckey_to_norm(int32_t ckey) { return (7 - ckey) >> 3; }

struct PairDesc {
    int32_t ref_img, qry_img;  // tensor-map slots (the slot after the last image maps the candidate scratch)
    int32_t ref_rows, qry_rows;
    int64_t ref_off, qry_off;  // first row in the column-key arena (query side: candidate scratch when cand_idx >= 0)
    int64_t knn_off;           // first row of this pair in the per-batch kNN scratch
    int32_t qry_row_base;      // row coordinate of query row 0 in the query tensor map (0 for whole-image maps)
    int32_t cand_idx;          // >= 0: the query rows are this pair's gathered mutual-check candidates and their
                               // number is counts[cand_idx] (known only on the device); -1: ordinary image rows
    float fscale2;             // float regime: (quantisation scale)^2 when both images keep their float rows, else 0
    int32_t pad_;
    int64_t col_off;           // first entry of this pair in the per-batch column-best table (mutual check, one per ref row)
};

struct WorkItem {
    int32_t pair;  // index into PairDesc[]
    int32_t row0;  // first query row of the item (multiple of STRIPS*128)
};

struct MatchKernelParams {
    const CUtensorMap *maps;      // [max_images] one 2-D map per image: {128 B, rows}, box {128 B, kBoxRows rows}, SW128
    const int32_t *ckeys;         // arena of column keys (see make_ckey)
    const int4 *tilemin;          // [arena rows / kKeyTileRows] {smallest squared norm of the tile's rows, -, -, -}: refreshed per batch
                                  // by tile_min_kernel; images start on multiples of kAlignRows, so tiles never straddle images
    const int32_t *cand_ckeys;    // column keys of the gathered candidate rows (query side of cand_idx >= 0 pairs)
    const int32_t *cand_d0;       // squared distance of each candidate to the query row that proposed it
    const int32_t *counts;        // per-pair candidate counts
    const PairDesc *pairs;
    const WorkItem *items;
    int32_t n_items;
    // A pass writes either top-2 records (and, in the debug build, counters) or events (COLLECT), never both, so those
    // outputs share slots.  COLLECT lists every (row, reference row) whose squared distance is <= cand_d0[row], as
    // {scratch row, reference row, cand_idx, 0}.
    union {
        uint32_t debug_flags;     // timing experiments only (results are wrong): 1 = skip the exact phase,
                                  // 2 = no epilogue work at all, 4 = TMEM loads + hand-back only
        uint32_t event_cap;       // COLLECT
    };
    union {
        unsigned long long *stats;  // optional debug counter (slow-path group visits); null in production
        unsigned int *event_count;  // COLLECT: total events seen (may exceed event_cap: the consumer then falls back)
    };
    union {
        int4 *knn;                // [sum qry_rows] {id0, id1, d0, d1} per query row; id = -1 / d = INT_MAX when absent;
                                  // consumers read it with load_knn()
        int4 *events;             // COLLECT: [event_cap]
    };
    // GATE (msfm_match_pairs_guided / _guided_homography): only elements that pass the gate can enter a row's top-2 or
    // event list.  F (or H) is row p of fmat for a forward item of pair p and for every item with cand_idx = p.  A forward
    // row and a band row (a collect item's row) are query keypoints, so the epipolar gate takes their query line; a twin
    // row is a reference keypoint, and the gate takes the query line of each column instead.  The homography gate
    // transfers the reference keypoint of each element: per column on a forward or band row, once per row on a twin row.
    const float2 *xy;             // keypoints (x, y), indexed like the column-key arena
    const float *fmat;            // [forward pairs of the batch][9] F (epipolar gate) or H (homography gate) rounded to
                                  // fp32, row-major
    const int32_t *src_row;       // [candidate scratch rows] the image row a scratch row came from: a reference row of pair
                                  // cand_idx for a twin row (cand_j), a query row of it for a band row (band_q)
    const unsigned int *routed;   // optional: the whole launch returns at once when *routed == 0 (mutual twin pass with no
                                  // pair routed to the tensor path, see select_candidates_kernel)
    uint32_t prune_q8;            // "dead row" rule of the forward pass (see the epilogue): a row whose two nearest neighbours
                                  // so far satisfy d0 > (prune_q8 / 256) * d1 only follows its NEAREST neighbour exactly.
                                  // kNoPrune = off (exact 2-NN of every row: msfm_knn2, twin and collect passes)
    float t2;                     // GATE: th_epipolar^2 or th_transfer^2, rounded to fp32
};
// The kernel takes the block by value.  Past 128 bytes nvcc addresses it through a pointer and the code of every
// instantiation changes; the top-2 passes, the headline path, read their fields at these offsets.
static_assert(sizeof(MatchKernelParams) == 128, "MatchKernelParams must stay 128 bytes");
static_assert(offsetof(MatchKernelParams, n_items) == 64 && offsetof(MatchKernelParams, debug_flags) == 68 &&
              offsetof(MatchKernelParams, stats) == 72 && offsetof(MatchKernelParams, knn) == 80 &&
              offsetof(MatchKernelParams, xy) == 88 && offsetof(MatchKernelParams, fmat) == 96 &&
              offsetof(MatchKernelParams, src_row) == 104 && offsetof(MatchKernelParams, routed) == 112 &&
              offsetof(MatchKernelParams, prune_q8) == 120 && offsetof(MatchKernelParams, t2) == 124,
              "top-2 passes read the parameter block at fixed offsets");
constexpr uint32_t kNoPrune = 4096;  // ((d1 >> 8) + 1) * 4096 >= 16 * d1 > d0 for every row, and fits in 32 bits (d < 2^25)

template <int STRIPS, int TILE_N, int STAGES, int TBUFS>
struct MatchKernelCfg {
    // One epilogue warp per (strip, 32-row quarter); TBUFS accumulator buffers per strip let the MMA of tile t+1 run
    // under the epilogue of tile t.
    static constexpr int kEpiWarps = 4 * STRIPS;
    static constexpr int kAuxWarps = (1 + STRIPS + 3) / 4 * 4;       // TMA producer + one MMA issuer per strip, padded to warpgroups
    static constexpr int kThreads = (kEpiWarps + kAuxWarps) * 32;
    // Registers: the launch gives every thread 65536 / kThreads (a multiple of 8); the auxiliary warpgroups hand most of
    // their share to the epilogue warps (setmaxnreg), which hold a 64-column accumulator tile each.
    static constexpr int kAuxRegs = 32;
    static constexpr int kLaunchRegs = 65536 / kThreads / 8 * 8;
    static constexpr int kEpiRegs = (kLaunchRegs * kThreads - kAuxWarps * 32 * kAuxRegs) / (kEpiWarps * 32) / 8 * 8;
    // The producer may refill a key slot once the MMAs that share its B stage have completed; those were issued after
    // every epilogue warp released the accumulator buffer TBUFS tiles earlier; a warp releases a buffer before it has
    // finished reading that tile's keys, but it must finish before it can release the next one:
    // tiles <= t-STAGES-TBUFS-1 are done when tile t is loaded.  +1 for margin.
    static constexpr int kKeySlots = 2 * STAGES;  // >= STAGES + TBUFS + 1; two rounds of the B ring, so slot = stage + STAGES * (round & 1)
    static_assert(2 * STAGES >= STAGES + TBUFS + 1 && STAGES % (2 * TBUFS) == 0, "ring position must fix key slot, accumulator buffer and its phase");
    static constexpr int kTmemCols = TBUFS * STRIPS * TILE_N;
    static constexpr int kABytes = STRIPS * kStripRows * kDim;  // one A buffer
    static constexpr int kBBytes = TILE_N * kDim;               // one B stage
    static constexpr int kSmemA = 0;
    static constexpr int kSmemB = kSmemA + 2 * kABytes;
    static constexpr int kSmemKey = kSmemB + STAGES * kBBytes;
    static constexpr int kSmemTmin = kSmemKey + kKeySlots * TILE_N * 4;        // [kKeySlots] int4: the tile's smallest reference norm
    static constexpr int kSmemBar = kSmemTmin + kKeySlots * 16;
    static constexpr int kNumBars = 2 + 2 + STAGES + STAGES + 2 * TBUFS * STRIPS;
    static constexpr int kSmemTmemPtr = kSmemBar + kNumBars * 8;
    static constexpr int kSmemBytes = kSmemTmemPtr + 16;
    static constexpr int kSmemAlloc = kSmemBytes + 1024;  // slack for manual 1024-byte alignment
    static_assert(kTmemCols == 32 || kTmemCols == 64 || kTmemCols == 128 || kTmemCols == 256 || kTmemCols == 512,
                  "TMEM allocation must be a power of two in [32, 512] columns");
    static_assert(TILE_N % kBoxRows == 0 && TILE_N <= 256, "reference tile is loaded as 64-row TMA boxes; UMMA N <= 256");
    static_assert(kAlignRows % TILE_N == 0, "image padding must cover whole reference tiles");
    static_assert(TILE_N == kKeyTileRows, "the minimum-norm table is kept per reference tile");
    static_assert(TILE_N % 16 == 0 && TILE_N / 8 <= 32, "one flag bit per group of 8 columns");
    static_assert(kThreads <= 1024, "too many warps");
    static_assert(kSmemAlloc <= 227 * 1024, "shared memory budget");
};

// Top-2 (largest, second largest) of eight distinct keys: 17 min/max operations, depth 4, no branches.
__device__ __forceinline__ void top2_of8(const int (&k)[8], int &g0, int &g1) {
    const int h0 = max(k[0], k[1]), l0 = min(k[0], k[1]);
    const int h1 = max(k[2], k[3]), l1 = min(k[2], k[3]);
    const int h2 = max(k[4], k[5]), l2 = min(k[4], k[5]);
    const int h3 = max(k[6], k[7]), l3 = min(k[6], k[7]);
    const int H0 = max(h0, h1), L0 = __vimax3_s32(min(h0, h1), l0, l1);
    const int H1 = max(h2, h3), L1 = __vimax3_s32(min(h2, h3), l2, l3);
    g0 = max(H0, H1);
    g1 = __vimax3_s32(min(H0, H1), L0, L1);
}

// Merge a group's two best (score, column) candidates a >= b into the running (S0,J0) >= (S1,J1).  Candidates come
// from higher column indices than anything in the running state, so they must beat it strictly.
__device__ __forceinline__ void merge_top2(int sa, int ja, int sb, int jb, int &S0, int &J0, int &S1, int &J1) {
    const bool t0 = sa > S0, t1 = sa > S1, u = sb > S0;
    const int x1s = u ? sb : S0, x1j = u ? jb : J0;    // second place when a takes first
    const int y1s = t1 ? sa : S1, y1j = t1 ? ja : J1;  // second place when a does not
    S1 = t0 ? x1s : y1s;
    J1 = t0 ? x1j : y1j;
    S0 = t0 ? sa : S0;
    J0 = t0 ? ja : J0;
}

// The score a row prunes against: its second best, or — "dead row" rule, see the epilogue — its best when the running pair
// already violates d0 <= rho * d1 (rho = rho8 / 256, rounded so that the test errs on the live side; d = na - S).
// Placeholder states (nothing or one neighbour seen, pad rows) never count as dead.
__device__ __forceinline__ int prune_score(int S0, int S1, int na, int rho8, int absent) {
    const int d0 = (int)((uint32_t)na - (uint32_t)S0), d1 = (int)((uint32_t)na - (uint32_t)S1);
    const bool dead = (S1 > absent) && (d0 > (d1 >> 8) * rho8 + rho8);
    return dead ? S0 : S1;
}

// Epipolar gate of GUIDED-SPEC (include/msfm_match.h).  Query line a = F^T (xq, yq, 1), reference line b = F (xj, yj, 1),
// s = a . (xj, yj, 1): element (q, j) is allowed iff s^2 <= t2 * min(|a|^2, |b|^2) over the first two components.  Every
// operation is one fp32 rounding (no contraction), and every stage that evaluates the gate (the matching kernel's rows
// and columns in both roles, the brute force rescore_band_kernel) goes through epi_query_line, epi_ref_line and
// epi_allowed below: an element is decided identically everywhere, and a numpy float32 restatement reproduces it bit for bit.
__device__ __forceinline__ float epi_lin(float u, float x, float v, float y, float w) {  // ((u*x) + (v*y)) + w
    return __fadd_rn(__fadd_rn(__fmul_rn(u, x), __fmul_rn(v, y)), w);
}
__device__ __forceinline__ float epi_sq(float u, float v) { return __fadd_rn(__fmul_rn(u, u), __fmul_rn(v, v)); }

struct EpiLine {
    float u, v, w;  // the line u x + v y + w = 0
    float n;        // u^2 + v^2
};
// F is row-major; LDG reads it through the read-only cache (the per-element tests of the matching kernel).
template <bool LDG>
__device__ __forceinline__ float epi_f(const float *F, int i) { return LDG ? __ldg(F + i) : F[i]; }
template <bool LDG = false>
__device__ __forceinline__ EpiLine epi_query_line(const float *F, float2 k) {  // a = F^T (x, y, 1)
    EpiLine a;
    a.u = epi_lin(epi_f<LDG>(F, 0), k.x, epi_f<LDG>(F, 3), k.y, epi_f<LDG>(F, 6));
    a.v = epi_lin(epi_f<LDG>(F, 1), k.x, epi_f<LDG>(F, 4), k.y, epi_f<LDG>(F, 7));
    a.w = epi_lin(epi_f<LDG>(F, 2), k.x, epi_f<LDG>(F, 5), k.y, epi_f<LDG>(F, 8));
    a.n = epi_sq(a.u, a.v);
    return a;
}
template <bool LDG = false>
__device__ __forceinline__ EpiLine epi_ref_line(const float *F, float2 k) {  // b = F (x, y, 1)
    EpiLine b;
    b.u = epi_lin(epi_f<LDG>(F, 0), k.x, epi_f<LDG>(F, 1), k.y, epi_f<LDG>(F, 2));
    b.v = epi_lin(epi_f<LDG>(F, 3), k.x, epi_f<LDG>(F, 4), k.y, epi_f<LDG>(F, 5));
    b.w = epi_lin(epi_f<LDG>(F, 6), k.x, epi_f<LDG>(F, 7), k.y, epi_f<LDG>(F, 8));
    b.n = epi_sq(b.u, b.v);
    return b;
}
// Element (q, j) from q's query line a, j's keypoint kj and |b|^2 of j's reference line.
__device__ __forceinline__ bool epi_allowed(const EpiLine &a, float2 kj, float nb, float t2) {
    const float s = epi_lin(a.u, kj.x, a.v, kj.y, a.w);
    return __fmul_rn(s, s) <= __fmul_rn(t2, nb < a.n ? nb : a.n);
}

// Homography gate of HOMOG-SPEC (include/msfm_match.h).  The reference keypoint kj is transferred once,
// (U, V, W) = H (xj, yj, 1); element (q, j) is allowed iff |(U, V) - (xq, yq) W|^2 <= t2 W^2, the squared transfer
// distance |p_q - pi(H p_j)|^2 <= th^2 without the division (independent of the sign of H; W = 0 bars the element unless
// U = V = 0).  One fp32 rounding per operation, no contraction; every site (the matching kernel's rows and columns in
// every pass, the brute force rescore_band_kernel) goes through hom_transfer and hom_allowed.
struct HomPoint {
    float U, V, W;
};
template <bool LDG = false>
__device__ __forceinline__ HomPoint hom_transfer(const float *H, float2 k) {
    HomPoint t;
    t.U = epi_lin(epi_f<LDG>(H, 0), k.x, epi_f<LDG>(H, 1), k.y, epi_f<LDG>(H, 2));
    t.V = epi_lin(epi_f<LDG>(H, 3), k.x, epi_f<LDG>(H, 4), k.y, epi_f<LDG>(H, 5));
    t.W = epi_lin(epi_f<LDG>(H, 6), k.x, epi_f<LDG>(H, 7), k.y, epi_f<LDG>(H, 8));
    return t;
}
__device__ __forceinline__ bool hom_allowed(const HomPoint &t, float2 kq, float t2) {
    const float du = __fsub_rn(t.U, __fmul_rn(kq.x, t.W)), dv = __fsub_rn(t.V, __fmul_rn(kq.y, t.W));
    return epi_sq(du, dv) <= __fmul_rn(t2, __fmul_rn(t.W, t.W));
}

// Which gate a guided launch applies (the matching kernel's GATE parameter).
enum class GateKind : int { none = 0, epipolar = 1, homography = 2 };

// The gate of a guided batch as the host passes it: keypoints (x, y) indexed like the column-key arena, the
// batch's F (or H) table ([forward pairs][9] rounded to fp32, row-major) and th^2 rounded to fp32.
struct EpiGate {
    const float2 *xy;
    const float *fmat;
    float t2;
};

template <int STRIPS, int TILE_N, int STAGES, int TBUFS, bool DEBUG, bool COLLECT = false, GateKind GATE = GateKind::none>
__global__ void __launch_bounds__(MatchKernelCfg<STRIPS, TILE_N, STAGES, TBUFS>::kThreads, 1)
match_pairs_kernel(const MatchKernelParams p) {
    using Cfg = MatchKernelCfg<STRIPS, TILE_N, STAGES, TBUFS>;
    constexpr bool GATED = GATE != GateKind::none, HOMOG = GATE == GateKind::homography;
    // No static shared memory is declared, so the dynamic window starts at shared offset 0 (1024-byte aligned, as
    // the 128B-swizzled operand tiles require); checked once below.
    extern __shared__ __align__(1024) uint8_t smem[];

    uint8_t *sA = smem + Cfg::kSmemA;
    uint8_t *sB = smem + Cfg::kSmemB;
    int32_t *sKey = reinterpret_cast<int32_t *>(smem + Cfg::kSmemKey);
    int4 *sTmin = reinterpret_cast<int4 *>(smem + Cfg::kSmemTmin);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + Cfg::kSmemBar);
    uint64_t *a_full = bars;                         // [2]
    uint64_t *a_empty = a_full + 2;                  // [2]
    uint64_t *b_full = a_empty + 2;                  // [STAGES]
    uint64_t *b_empty = b_full + STAGES;             // [STAGES]
    uint64_t *t_full = b_empty + STAGES;             // [TBUFS][STRIPS]
    uint64_t *t_empty = t_full + TBUFS * STRIPS;     // [TBUFS][STRIPS]
    uint32_t *tmem_ptr = reinterpret_cast<uint32_t *>(smem + Cfg::kSmemTmemPtr);

    const int warp = __shfl_sync(0xFFFFFFFFu, (int)(threadIdx.x >> 5), 0);  // warp-uniform by construction: lets the compiler keep
                                                                            // everything derived from it in uniform registers
    const int lane = threadIdx.x & 31;
    if (p.routed != nullptr && *p.routed == 0u) return;  // uniform over the grid: nothing was routed to this pass
    if (threadIdx.x == 0 && (ptx::smem_u32(smem) & 1023u) != 0) __trap();

    if (warp == Cfg::kEpiWarps && lane == 0) {
        // A buffers and B stages are released by the commits of all STRIPS MMA issuers
        for (int i = 0; i < 2; ++i) { ptx::mbar_init(&a_full[i], 1); ptx::mbar_init(&a_empty[i], STRIPS); }
        for (int i = 0; i < STAGES; ++i) { ptx::mbar_init(&b_full[i], 1); ptx::mbar_init(&b_empty[i], STRIPS); }
        for (int i = 0; i < TBUFS * STRIPS; ++i) { ptx::mbar_init(&t_full[i], 1); ptx::mbar_init(&t_empty[i], 4); }
        ptx::fence_mbar_init();
    }
    if (warp == Cfg::kEpiWarps + 1) ptx::tmem_alloc<Cfg::kTmemCols>(tmem_ptr);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp >= Cfg::kEpiWarps) {
      ptx::setmaxnreg_dec<Cfg::kAuxRegs>();
      // Aux warp x = warp - kEpiWarps: x = 0 is the TMA loader, x = 1 .. STRIPS are the MMA issuers (one per SM
      // sub-partition), the rest is padding up to whole warpgroups (setmaxnreg) and goes straight to the final barrier.
      // Measured with idle dummy warps: a warp that polls an mbarrier (or merely loops on nanosleep(20)) slows the four
      // epilogue warps of its sub-partition by 7 %, a warp that sleeps 1 us between polls costs nothing, and every
      // instruction a service warp executes per tile costs its sub-partition ~1.4 cycles.  Hence: long sleeps where the
      // latency is hidden anyway (the loader runs STAGES tiles ahead, the issuers have a spare accumulator buffer), and
      // tile loops that walk the B ring unrolled, so that stage / barrier / key-slot addresses are immediates.
      // Spreading the loads over four loader warps was measured too: more total service work, slower.
#ifndef MSFM_LOADER_SLEEP
#define MSFM_LOADER_SLEEP 1000
#endif
#ifndef MSFM_ISSUER_SLEEP
#define MSFM_ISSUER_SLEEP 200
#endif
      constexpr unsigned kLoaderSleepNs = MSFM_LOADER_SLEEP, kIssuerSleepNs = MSFM_ISSUER_SLEEP;
#define LOADER_WAIT(bar, par) ptx::mbar_wait_backoff<kLoaderSleepNs>(bar, par)
#define ISSUER_WAIT(bar, par) ptx::mbar_wait_backoff<kIssuerSleepNs>(bar, par)
      const int x = warp - Cfg::kEpiWarps;
      if (x == 0) {
        // =========================================================== TMA loader
        // The tile loop walks the B ring (unrolled over its STAGES positions, so stage, barrier and key-slot addresses are
        // immediates); items are switched inside it.  Every instruction here is taken from the issue slots of the
        // epilogue warps on the same sub-partition (~1.4 cycles each per tile), hence the lean loop and the long sleeps.
        if (ptx::elect_one()) {
            int cur = (int)blockIdx.x - (int)gridDim.x, left = 0, t = 0;
            uint32_t a = 0, round = 0;  // items started, trips round the B ring
            const CUtensorMap *rmap = nullptr;
            const int32_t *keyp = nullptr;
            const int4 *tminp = nullptr;
            auto next_item = [&]() -> bool {  // next item with work; fetches its query strips
                for (;;) {
                    const int idx = (cur += (int)gridDim.x);
                    if (idx >= p.n_items) return false;
                    const WorkItem wi = p.items[idx];
                    const PairDesc pd = p.pairs[wi.pair];
                    if (pd.cand_idx >= 0 && wi.row0 >= p.counts[pd.cand_idx]) continue;  // item past the candidate list
                    const CUtensorMap *qmap = p.maps + pd.qry_img;
                    const uint32_t abuf = a & 1;
                    LOADER_WAIT(&a_empty[abuf], ((a >> 1) & 1) ^ 1);
                    ptx::mbar_arrive_expect_tx(&a_full[abuf], Cfg::kABytes);
#pragma unroll
                    for (int s = 0; s < STRIPS * kStripRows / kBoxRows; ++s)
                        ptx::tma_load_2d(sA + abuf * Cfg::kABytes + s * kBoxRows * kDim, qmap, &a_full[abuf], 0,
                                         pd.qry_row_base + wi.row0 + s * kBoxRows);
                    rmap = p.maps + pd.ref_img;
                    keyp = p.ckeys + pd.ref_off;
                    tminp = p.tilemin + pd.ref_off / kKeyTileRows;
                    left = (pd.ref_rows + TILE_N - 1) / TILE_N;
                    t = 0;
                    ++a;
                    return true;
                }
            };
            bool more = next_item();
            while (more) {
#pragma unroll
                for (int st = 0; st < STAGES; ++st) {
                    if (!more) break;
                    LOADER_WAIT(&b_empty[st], (round & 1) ^ 1);
                    // one barrier for the tile, its column keys and its minimum norm: the MMAs are issued behind it and the
                    // epilogue reads the keys behind the MMAs, so it needs no barrier of its own for them
                    ptx::mbar_arrive_expect_tx(&b_full[st], Cfg::kBBytes + TILE_N * 4 + 16);
#pragma unroll
                    for (int h = 0; h < TILE_N / kBoxRows; ++h)
                        ptx::tma_load_2d(sB + st * Cfg::kBBytes + h * kBoxRows * kDim, rmap, &b_full[st], 0, t + h * kBoxRows);
                    const uint32_t ks = st + STAGES * (round & 1);
                    ptx::bulk_load_1d(sKey + ks * TILE_N, keyp + t, TILE_N * 4, &b_full[st]);
                    ptx::bulk_load_1d(sTmin + ks, tminp++, 16, &b_full[st]);
                    t += TILE_N;  // first reference row of the next tile
                    if (--left == 0) more = next_item();
                }
                ++round;
            }
        }
      } else if (x >= 1 && x <= STRIPS) {
        // =========================================================== MMA issuers: warp kEpiWarps + 1 + s feeds strip s
        // One issuer per strip (one elected lane each): the strips' MMAs are no longer issued in a fixed round-robin order
        // (a strip whose accumulator buffer is free never queues behind one that is still being drained), and the issuing
        // instructions are spread over the four SM sub-partitions instead of loading one of them.
        const int s = x - 1;
        if (ptx::elect_one()) {
            constexpr uint32_t idesc = ptx::make_idesc_i8(kStripRows, TILE_N, 0, 0);
            // Same loop shape as the loaders: ring position = stage, accumulator buffer (st % TBUFS) and its phase
            // ((st / TBUFS) & 1) are compile-time, descriptors are 32-bit low words (68 -> ~35 instructions per tile).
            const uint32_t b_lo0 = ptx::smem_u32(sB) >> 4;
            const uint32_t a_lo0 = (ptx::smem_u32(sA) + s * kStripRows * kDim) >> 4;
            const uint32_t d_tmem0 = tmem_base + s * TILE_N;
            uint64_t *t_full_s = t_full + s, *t_empty_s = t_empty + s;
            int cur = (int)blockIdx.x - (int)gridDim.x, left = 0;
            uint32_t a = 0, abuf = 0, a_lo = 0, round = 0;
            auto next_item = [&]() -> bool {  // next item with work; waits for its query strips
                for (;;) {
                    const int idx = (cur += (int)gridDim.x);
                    if (idx >= p.n_items) return false;
                    const WorkItem wi = p.items[idx];
                    const PairDesc pd = p.pairs[wi.pair];
                    if (pd.cand_idx >= 0 && wi.row0 >= p.counts[pd.cand_idx]) continue;
                    abuf = a & 1;
                    ISSUER_WAIT(&a_full[abuf], (a >> 1) & 1);
                    a_lo = a_lo0 + abuf * (Cfg::kABytes >> 4);
                    left = (pd.ref_rows + TILE_N - 1) / TILE_N;
                    ++a;
                    return true;
                }
            };
            bool more = next_item();
            while (more) {
#pragma unroll
                for (int st = 0; st < STAGES; ++st) {
                    if (!more) break;
                    constexpr int kBufStride = STRIPS;  // barriers / accumulators are laid out [TBUFS][STRIPS]
                    const int buf = st % TBUFS;
                    long long i0 = 0, i1 = 0, i2 = 0;
                    const bool iprof = DEBUG && (p.debug_flags & 8u) && p.stats != nullptr;
                    if (iprof) i0 = clock64();
                    ISSUER_WAIT(&b_full[st], round & 1);
                    if (iprof) i1 = clock64();
                    ISSUER_WAIT(t_empty_s + buf * kBufStride, ((st / TBUFS) & 1) ^ 1);  // accumulator drained by the epilogue
                    if (iprof) {
                        i2 = clock64();
                        atomicAdd(p.stats + 40 + 2 * s, (unsigned long long)(i1 - i0));  // issuer: waiting for the B tile
                        atomicAdd(p.stats + 41 + 2 * s, (unsigned long long)(i2 - i1));  // issuer: waiting for the accumulator buffer
                    }
                    ptx::tc_fence_after();
                    const uint32_t d_tmem = d_tmem0 + buf * kBufStride * TILE_N;
                    const uint32_t b_lo = b_lo0 + st * (Cfg::kBBytes >> 4);
                    ptx::mma_i8_ss_lo<false>(d_tmem, a_lo, b_lo, idesc);
#pragma unroll
                    for (int k = 1; k < kDim / 32; ++k) ptx::mma_i8_ss_lo<true>(d_tmem, a_lo + k * 2, b_lo + k * 2, idesc);
                    ptx::mma_commit(t_full_s + buf * kBufStride);  // this strip's accumulators are ready
                    ptx::mma_commit(&b_empty[st]);                 // one of STRIPS arrivals that free the B stage
                    if (--left == 0) {
                        ptx::mma_commit(&a_empty[abuf]);           // one of STRIPS arrivals that free the A buffer
                        more = next_item();
                    }
                }
                ++round;
            }
        }
      }
    } else {
        // =========================================================== epilogue (thread = query row)
        ptx::setmaxnreg_inc<(Cfg::kEpiRegs > 232 ? 232 : Cfg::kEpiRegs)>();
        // Scores s = 2*acc - ||r||^2 (maximise; d = ||q||^2 - s).
        // Phase 1 (filter): stream the warp's rows of the strip's accumulator tile through registers once and keep
        //   only the maximum RAW accumulator of every group of 8 columns; a group is flagged when that maximum exceeds
        //   T = floor((theta + min||r||^2 over the tile) / 2) in any lane.  theta is a lower bound of the row's final
        //   second-best score, so an unflagged group cannot enter the row's top-2
        //   (2*acc - nb_j <= 2*acc - nbmin <= theta) and costs ~0.45 instructions per element.
        // Phase 2 (exact): flagged groups (a few per tile) are re-read from TMEM and scored exactly with packed keys
        //   (branch-free top-2-of-8 network + merge), in ascending column order; ties never displace (strict >), hence
        //   lowest-index tie-breaking.  Then the accumulator is handed back to the MMA warp.
        // Each thread holds the row's whole top-2 state and writes the row's one kNN record at the end of the item.
        const int strip = warp >> 2;
        const int quarter = warp & 3;
        const int row_local = strip * kStripRows + quarter * 32 + lane;
        const uint32_t warp_taddr = ptx::opaque(tmem_base + ((uint32_t)(quarter * 32) << 16) + strip * TILE_N);
        constexpr int kAbsent = -0x08000000;  // scores below this are pad columns / "no neighbour"
        // everything the tile loop touches in shared memory, as 32-bit shared addresses
        // (made opaque: otherwise they are re-derived from the shared-window base and the warp index in every tile)
        const uint32_t key_base = ptx::opaque(ptx::smem_u32(sKey));
        const uint32_t tmin_base = ptx::opaque(ptx::smem_u32(sTmin));
        const uint32_t t_full_base = ptx::opaque(ptx::smem_u32(t_full + strip));
        const uint32_t t_empty_base = ptx::opaque(ptx::smem_u32(t_empty + strip));
        const uint32_t lane_pinned = ptx::opaque((uint32_t)lane);  // (not re-read from %tid per tile)
        // Ring positions of the CTA's running tile sequence, carried from tile to tile: the accumulator buffer, its
        // barrier phase and the key slot, as byte offsets (a few ALU operations per tile instead of re-deriving every
        // address from a tile counter and the shared-memory window base).
        static_assert((TBUFS & (TBUFS - 1)) == 0 && (Cfg::kKeySlots & (Cfg::kKeySlots - 1)) == 0, "ring sizes must be powers of two");
        uint32_t buf = 0, t_phase = 0;  // accumulator buffer of the next tile and the parity of its full barrier
        uint32_t koff = 0;              // key slot of the next tile, in bytes of the key ring (TILE_N * 4 per slot)
        constexpr uint32_t kKeyRingBytes = Cfg::kKeySlots * TILE_N * 4, kKeyToTmin = TILE_N * 4 / 16;
        for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
            const WorkItem wi = p.items[item];
            const PairDesc pd = p.pairs[wi.pair];
            const int qry_rows = pd.cand_idx >= 0 ? p.counts[pd.cand_idx] : pd.qry_rows;
            if (wi.row0 >= qry_rows) continue;  // item past the candidate list
            const int q = wi.row0 + row_local;
            const bool valid = q < qry_rows;
            const int na = valid ? ckey_to_norm((pd.cand_idx >= 0 ? p.cand_ckeys : p.ckeys)[pd.qry_off + q]) : 0;
            // rows past the image end hold zeros; park their state where nothing can flag a group
            int S0 = valid ? INT_MIN : 0x20000000, S1 = S0, J0 = -1, J1 = -1;
            // Mutual-check items only need the nearest row, and one row at distance d0 is known to exist (the query
            // row that proposed this candidate): start both slots just below its score so that only rows at least as
            // close are ever scored exactly.  The placeholders carry id -1 and are dropped by the consumers.
            // Collect mode keeps that threshold for the whole row: every reference row at distance <= cand_d0 is listed.
            if (pd.cand_idx >= 0 && valid) S0 = S1 = na - p.cand_d0[pd.qry_off + q] - 1;
            // "Dead row" rule (forward items of msfm_match_pairs only).  The caller keeps a row only if d0/d1 < ratio.  While
            // the running pair violates that with a margin (d0 > rho * d1, rho just above every ratio the caller tests:
            // the row is "dead"), only an element closer than d0 can change the verdict: it becomes the nearest neighbour and
            // the old one — the exact minimum of everything before it, because elements under d0 are never skipped — the
            // second, so the pair is exact again.  Elements between d0 and d1 would only push a dead row further from the
            // threshold, so the pruning threshold of a dead row is its BEST score instead of its second best: about half of
            // the running-top-2 records of such rows (most rows of an image pair) never reach the exact phase.  A row that
            // ends dead reports d1 := d0: "rejected", and still a valid lower bound of its distance to every row but nn0,
            // which is what the mutual check's dangerous-row bound needs (select_candidates_kernel).
            // Under the epipolar gate the rule stays on: it only reasons about elements that can enter the row's top-2,
            // and the gate only removes elements (barred ones never reach the running state).
            const int rho8 = (!COLLECT && pd.cand_idx < 0) ? (int)p.prune_q8 : (int)kNoPrune;
            // Gated items: the row's half of the gate, once per item.  A forward or band row is a query keypoint: its
            // query line.  A band row takes its query row's keypoint and F, so it gets that row's line bit for bit, and
            // its allowed set is the one its gated quantised 2-NN, and hence its threshold T(q), came from.  A twin row is
            // a reference keypoint kr: its reference line, of which the test needs |b|^2 only.
            // Homography gate: a forward row keeps its query keypoint kr, a band row its query row's keypoint (and with
            // that row's H, that row's allowed set bit for bit), a twin row its transferred keypoint ht.
            const bool query_row = COLLECT || pd.cand_idx < 0;
            EpiLine line{};
            float2 kr{};
            HomPoint ht{};
            const float *fm = nullptr;
            if (HOMOG) {
                fm = p.fmat + 9 * (pd.cand_idx >= 0 ? pd.cand_idx : wi.pair);
                if (valid && query_row)
                    kr = p.xy[(!COLLECT || pd.cand_idx < 0) ? pd.qry_off + q : p.pairs[pd.cand_idx].qry_off + p.src_row[pd.qry_off + q]];
                else if (valid) ht = hom_transfer(fm, p.xy[p.pairs[pd.cand_idx].ref_off + p.src_row[pd.qry_off + q]]);
            } else if (GATED) {
                fm = p.fmat + 9 * (pd.cand_idx >= 0 ? pd.cand_idx : wi.pair);
                if (valid && query_row) {
                    line = epi_query_line(fm, p.xy[pd.cand_idx < 0 ? pd.qry_off + q : p.pairs[pd.cand_idx].qry_off + p.src_row[pd.qry_off + q]]);
                } else if (valid) {
                    kr = p.xy[p.pairs[pd.cand_idx].ref_off + p.src_row[pd.qry_off + q]];
                    line = epi_ref_line(fm, kr);
                }
            }
            const int ntiles = (pd.ref_rows + TILE_N - 1) / TILE_N;
            long long acc_wait = 0, acc_load = 0, acc_p1 = 0, acc_p2 = 0, acc_hot = 0, acc_first = 0;
            int theta = prune_score(S0, S1, na, rho8, kAbsent);  // pruning score of the row, refreshed after every hot tile
            int jtile = 0;  // first column of the current tile
            for (int t = 0; t < ntiles; ++t, jtile += TILE_N) {
                // ---- pull the warp's rows of the whole accumulator tile into registers and release TMEM at once
                long long c0 = 0, c1 = 0, c2 = 0, c3 = 0;
                const bool prof = DEBUG && (p.debug_flags & 8u) && p.stats != nullptr;
                if (prof) c0 = clock64();
                ptx::mbar_wait_a(t_full_base + buf * (STRIPS * 8), t_phase);
                ptx::tc_fence_after();
                if (prof) c1 = clock64();
                const uint32_t tile_taddr = warp_taddr + buf * (STRIPS * TILE_N);
                uint32_t acc[TILE_N / 16][16];
#pragma unroll
                for (int c = 0; c < TILE_N / 16; ++c) ptx::tmem_ld_32x32b_x16(tile_taddr + c * 16, acc[c]);
                // ---- while the loads fly: column keys of the tile, smallest reference norm, pruning threshold
                // (the tile's keys and minimum norm landed before its MMAs were issued: they share the B stage's barrier)
                const uint32_t ck = key_base + koff;
                const int nbmin = ptx::lds_s32(tmin_base + koff / kKeyToTmin);  // smallest reference norm of the tile (tile_min_kernel)
                const int T = (theta + nbmin) >> 1;  // dead rows are pruned against their best score, the others against their second best
                ptx::tmem_ld_wait();
                ptx::tc_fence_before();
                __syncwarp();
                if (lane_pinned == 0) ptx::mbar_arrive_a(t_empty_base + buf * (STRIPS * 8));
                if (prof) c2 = clock64();
                if (DEBUG && (p.debug_flags & 6u)) {  // experiments: 2/4 = TMEM loads + hand-back only
                    if (acc[0][0] == 0x7fffffffu) S1 = 0;
                } else {
                    // ---- phase 1: can any column of this tile still matter to some lane?  (maximum of the raw accumulators
                    //      per group of 8 columns, then of the tile: one vote; most tiles late in an item end here)
                    int gm[TILE_N / 8];
#pragma unroll
                    for (int gq = 0; gq < TILE_N / 8; ++gq) {
                        const uint32_t *v = &acc[gq / 2][8 * (gq & 1)];
                        const int m1 = __vimax3_s32((int)v[0], (int)v[1], (int)v[2]);
                        const int m2 = __vimax3_s32((int)v[3], (int)v[4], (int)v[5]);
                        const int m3 = __vimax3_s32((int)v[6], (int)v[7], m1);
                        gm[gq] = max(m2, m3);
                    }
                    int tm = gm[0];
#pragma unroll
                    for (int gq = 1; gq + 1 < TILE_N / 8; gq += 2) tm = __vimax3_s32(tm, gm[gq], gm[gq + 1]);
                    tm = max(tm, gm[TILE_N / 8 - 1]);
                    const bool tile_hot = __any_sync(0xFFFFFFFFu, tm > T);
                    if (prof) c3 = clock64();
                    if (tile_hot) {
                        // ---- which groups?  (one vote and one branch per group: only paid by tiles that have one)
                        bool hot[TILE_N / 8];
#pragma unroll
                        for (int gq = 0; gq < TILE_N / 8; ++gq) hot[gq] = __any_sync(0xFFFFFFFFu, gm[gq] > T);
                        // ---- phase 2: exact scoring of the hot groups straight from the registers
#pragma unroll
                        for (int gq = 0; gq < TILE_N / 8; ++gq) {
                            if (hot[gq] && !(DEBUG && (p.debug_flags & 1u))) {
                                const uint32_t *v = &acc[gq / 2][8 * (gq & 1)];
                                const int4 c0 = ptx::lds_v4(ck + gq * 32);
                                const int4 c1 = ptx::lds_v4(ck + gq * 32 + 16);
                                int key[8] = {16 * (int)v[0] + c0.x, 16 * (int)v[1] + c0.y, 16 * (int)v[2] + c0.z,
                                              16 * (int)v[3] + c0.w, 16 * (int)v[4] + c1.x, 16 * (int)v[5] + c1.y,
                                              16 * (int)v[6] + c1.z, 16 * (int)v[7] + c1.w};
                                const int jb8 = jtile + gq * 8;
                                if (GATED) {
                                    // the group's 8 column keypoints (64 bytes, L2-resident); a barred element gets the
                                    // smallest key, whose score lies below kAbsent: it can only fill an empty slot as
                                    // "no neighbour" and loses against every allowed element (COLLECT: it lies below
                                    // every row's collect threshold and is never listed)
                                    const float4 *kp = reinterpret_cast<const float4 *>(p.xy + pd.ref_off + jb8);
#pragma unroll
                                    for (int h = 0; h < 4; ++h) {
                                        const float4 c = __ldg(kp + h);
                                        const float2 kc[2] = {make_float2(c.x, c.y), make_float2(c.z, c.w)};
#pragma unroll
                                        for (int e = 0; e < 2; ++e) {
                                            bool ok;  // column = reference row j, or query row q
                                            if (HOMOG)
                                                ok = query_row ? hom_allowed(hom_transfer<true>(fm, kc[e]), kr, p.t2)
                                                               : hom_allowed(ht, kc[e], p.t2);
                                            else
                                                ok = query_row
                                                    ? epi_allowed(line, kc[e], epi_ref_line<true>(fm, kc[e]).n, p.t2)
                                                    : epi_allowed(epi_query_line<true>(fm, kc[e]), kr, line.n, p.t2);
                                            if (!ok) key[2 * h + e] = INT_MIN;
                                        }
                                    }
                                }
                                if (COLLECT) {
#pragma unroll
                                    for (int i = 0; i < 8; ++i)
                                        if ((key[i] >> 3) > S1) {
                                            const unsigned slot = atomicAdd(p.event_count, 1u);
                                            if (slot < p.event_cap) p.events[slot] = make_int4((int)(pd.qry_off + q), jb8 + i, pd.cand_idx, 0);
                                        }
                                } else {
                                    int g0, g1;
                                    top2_of8(key, g0, g1);
                                    merge_top2(g0 >> 3, jb8 | (g0 & 7), g1 >> 3, jb8 | (g1 & 7), S0, J0, S1, J1);  // columns stay packed: see the item's end
                                }
                                if (prof) ++acc_hot;
                            }
                        }
                        // the row's pruning score for the next tiles (only a hot tile can change it)
                        theta = prune_score(S0, S1, na, rho8, kAbsent);
                    }
                }
                if (prof) {  // per-warp cycle accounting of the tile loop (debug flag 8)
                    const long long c4 = clock64();
                    acc_wait += c1 - c0;  // waiting for the accumulator
                    if (t == 0) acc_first = c1 - c0;  // ... of the item's first tile (the item-switch bubble)
                    acc_load += c2 - c1;  // TMEM loads + keys + threshold + hand-back
                    acc_p1 += c3 - c2;    // phase 1
                    acc_p2 += c4 - c3;    // phase 2
                }
                koff = (koff + TILE_N * 4) & (kKeyRingBytes - 1);
                buf = (buf + 1) & (TBUFS - 1);
                t_phase ^= (buf == 0);
            }
            if (DEBUG && (p.debug_flags & 8u) && p.stats != nullptr && lane == 0) {
                atomicAdd(p.stats + 0, (unsigned long long)acc_hot);
                atomicAdd(p.stats + 6, (unsigned long long)acc_first);
                atomicAdd(p.stats + 7, 1ull);  // warp-items
                atomicAdd(p.stats + 1, (unsigned long long)acc_wait);
                atomicAdd(p.stats + 2, (unsigned long long)acc_load);
                atomicAdd(p.stats + 3, (unsigned long long)acc_p1);
                atomicAdd(p.stats + 4, (unsigned long long)acc_p2);
                atomicAdd(p.stats + 5, (unsigned long long)ntiles);
                atomicAdd(p.stats + 8 + 2 * quarter, (unsigned long long)acc_wait);  // per SM sub-partition
                atomicAdd(p.stats + 9 + 2 * quarter, (unsigned long long)(acc_load + acc_p1 + acc_p2));
            }
            if (valid && !COLLECT) {
                if (prune_score(S0, S1, na, rho8, kAbsent) != S1) S1 = S0;  // ended dead: d1 := d0 (lower bound)
                int4 out;
                out.x = (S0 > kAbsent && J0 >= 0) ? (J0 ^ 7) : -1;  // low three bits hold 7 - (column mod 8), as in the packed keys;
                                                                   // seeded placeholders (mutual twin items) keep id -1
                out.y = (S1 > kAbsent && J1 >= 0) ? (J1 ^ 7) : -1;
                out.z = (S0 > kAbsent) ? na - S0 : INT_MAX;
                out.w = (S1 > kAbsent) ? na - S1 : INT_MAX;
                p.knn[pd.knn_off + q] = out;
            }
        }
    }

    ptx::tc_fence_before();
    __syncthreads();
    if (warp == Cfg::kEpiWarps + 1) ptx::tmem_dealloc<Cfg::kTmemCols>(tmem_base);
}

}  // namespace msfm
