// geo_kernels.cuh — batched geometric verification of matched pairs (SURVEY.md §8f row 1), the stage right after the
// matching hot path in FineMatchingGraph::BuildMatchGraph (/root/reference/SfM/src/graph/fine_matching_graph.cc:137-153):
//   A  GeoVerification::GeoVerificationFundamental(pt1_good, pt2_good, inliers, F)   utils/geo_verification.cc:30-58
//        >= 30 "good" matches, F by RANSAC with a 3 px epipolar threshold (cv::findFundamentalMat, FM_RANSAC: 7-point
//        minimal solver, error = max of the two squared point-to-epipolar-line distances), >= 30 inliers
//   B  GeoVerification::GeoVerificationFundamental(pt1_all, pt2_all, F, inliers)     utils/geo_verification.cc:60-79
//        keep the "all" matches whose point 2 lies within 3 px of the epipolar line F * p1 (double arithmetic)
// One CTA per image pair; pairs are independent, so the batch is data parallel like the matching itself.  The RANSAC
// draws are counter-based (seed, pair, hypothesis), i.e. reproducible, but they are not OpenCV's RNG stream: parity with
// the reference is statistical for stage A (inlier sets / accept decisions) and exact for stage B given F.
// The same search with a homography model (4-point DLT, one-sided transfer error) is msfm_geo_homography
// (cv::findHomography with RANSAC, without its Levenberg-Marquardt refinement).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace msfm {

constexpr int kGeoThreads = 256;
constexpr int kGeoPointCap = 2048;  // good matches held in shared memory for hypothesis scoring (strided subsample beyond)

struct GeoParams {
    const int64_t *offsets;    // [n_pairs + 1] into matches / good / keep
    const int2 *matches;       // (point id in image 1, point id in image 2), msfm_match_pairs orientation 0
    const uint8_t *good;
    const int32_t *pair_img;   // [n_pairs][2] image ids (ref = image 1, query = image 2)
    const float *xy;           // centred keypoints of all images, concatenated
    const int64_t *xy_off;     // [n_images + 1] keypoint offset of every image in `xy` (in points)
    float th;                  // epipolar threshold in pixels (3.0)
    int32_t min_points, min_inliers, iters;
    unsigned long long seed;
    long long pair_base;       // global index of pair 0 of this call (RANSAC counter)
    int32_t stage_b;           // 1: keep = F-filter of all matches (stage B); 0: keep = RANSAC inlier mask of the good ones
    int32_t *pair_ok;          // [n_pairs]
    int32_t *pair_inliers;     // [n_pairs] stage-A inliers among the good matches
    uint8_t *keep;             // [total matches] stage-B mask
    double *F;                 // [n_pairs][9] row-major, pixel coordinates (F, or H of geo_homography_kernel)
};

__device__ __forceinline__ unsigned long long geo_mix(unsigned long long z) {  // splitmix64
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

__device__ __forceinline__ double det3(const double *m) {
    return m[0] * (m[4] * m[8] - m[5] * m[7]) - m[1] * (m[3] * m[8] - m[5] * m[6]) + m[2] * (m[3] * m[7] - m[4] * m[6]);
}

// Real roots of c3 x^3 + c2 x^2 + c1 x + c0 (degenerate leading coefficients handled); returns their number.
static __device__ int solve_cubic(double c3, double c2, double c1, double c0, double *r) {
    const double eps = 1e-14;
    if (fabs(c3) < eps * (fabs(c2) + fabs(c1) + fabs(c0) + 1e-300)) {
        if (fabs(c2) < eps * (fabs(c1) + fabs(c0) + 1e-300)) {
            if (fabs(c1) < 1e-300) return 0;
            r[0] = -c0 / c1;
            return 1;
        }
        const double d = c1 * c1 - 4.0 * c2 * c0;
        if (d < 0.0) return 0;
        const double s = sqrt(d), q = -0.5 * (c1 + (c1 >= 0.0 ? s : -s));
        r[0] = q / c2;
        int n = 1;
        if (fabs(q) > 1e-300) r[n++] = c0 / q;
        return n;
    }
    const double a = c2 / c3, b = c1 / c3, c = c0 / c3;
    const double Q = (a * a - 3.0 * b) / 9.0, R = (2.0 * a * a * a - 9.0 * a * b + 27.0 * c) / 54.0;
    const double Q3 = Q * Q * Q;
    if (R * R < Q3) {
        const double th = acos(fmax(-1.0, fmin(1.0, R / sqrt(Q3)))), sq = -2.0 * sqrt(Q);
        r[0] = sq * cos(th / 3.0) - a / 3.0;
        r[1] = sq * cos((th + 2.0 * 3.14159265358979323846) / 3.0) - a / 3.0;
        r[2] = sq * cos((th - 2.0 * 3.14159265358979323846) / 3.0) - a / 3.0;
        return 3;
    }
    const double A = -copysign(cbrt(fabs(R) + sqrt(R * R - Q3)), R);
    const double B = (A != 0.0) ? Q / A : 0.0;
    r[0] = (A + B) - a / 3.0;
    return 1;
}

// 7-point algorithm: up to three fundamental matrices (row-major, normalised coordinates) through seven correspondences.
// Null space of the 7 x 9 epipolar system by Gauss-Jordan elimination with full pivoting, then det(F2 + x (F1 - F2)) = 0.
static __device__ int seven_point(const float (&x1)[7], const float (&y1)[7], const float (&x2)[7], const float (&y2)[7], double (*Fout)[9]) {
    double A[7][9];
#pragma unroll
    for (int i = 0; i < 7; ++i) {
        const double a = x1[i], b = y1[i], c = x2[i], d = y2[i];
        A[i][0] = c * a; A[i][1] = c * b; A[i][2] = c;
        A[i][3] = d * a; A[i][4] = d * b; A[i][5] = d;
        A[i][6] = a;     A[i][7] = b;     A[i][8] = 1.0;
    }
    int perm[9];
    for (int j = 0; j < 9; ++j) perm[j] = j;
    for (int k = 0; k < 7; ++k) {
        int pr = k, pc = k;
        double best = 0.0;
        for (int i = k; i < 7; ++i)
            for (int j = k; j < 9; ++j)
                if (fabs(A[i][j]) > best) { best = fabs(A[i][j]); pr = i; pc = j; }
        if (best < 1e-12) return 0;  // degenerate sample
        for (int j = 0; j < 9; ++j) { const double t = A[k][j]; A[k][j] = A[pr][j]; A[pr][j] = t; }
        for (int i = 0; i < 7; ++i) { const double t = A[i][k]; A[i][k] = A[i][pc]; A[i][pc] = t; }
        { const int t = perm[k]; perm[k] = perm[pc]; perm[pc] = t; }
        const double inv = 1.0 / A[k][k];
        for (int j = k; j < 9; ++j) A[k][j] *= inv;
        for (int i = 0; i < 7; ++i) {
            if (i == k) continue;
            const double f = A[i][k];
            if (f != 0.0)
                for (int j = k; j < 9; ++j) A[i][j] -= f * A[k][j];
        }
    }
    // free (permuted) columns 7 and 8: basis vectors v_a (free = (1,0)) and v_b (free = (0,1))
    double f1[9], f2[9];
    for (int k = 0; k < 7; ++k) { f1[perm[k]] = -A[k][7]; f2[perm[k]] = -A[k][8]; }
    f1[perm[7]] = 1.0; f1[perm[8]] = 0.0;
    f2[perm[7]] = 0.0; f2[perm[8]] = 1.0;
    double D[9];
    for (int j = 0; j < 9; ++j) D[j] = f1[j] - f2[j];
    // det(F2 + x D) = c0 + c1 x + c2 x^2 + c3 x^3 by multilinearity in the rows
    double c0 = det3(f2), c3 = det3(D), c1 = 0.0, c2 = 0.0, M[9];
    for (int r = 0; r < 3; ++r) {
        for (int j = 0; j < 9; ++j) M[j] = f2[j];
        for (int j = 0; j < 3; ++j) M[3 * r + j] = D[3 * r + j];
        c1 += det3(M);
        for (int j = 0; j < 9; ++j) M[j] = D[j];
        for (int j = 0; j < 3; ++j) M[3 * r + j] = f2[3 * r + j];
        c2 += det3(M);
    }
    double roots[3];
    const int nr = solve_cubic(c3, c2, c1, c0, roots);
    int n = 0;
    for (int k = 0; k < nr; ++k) {
        double nrm = 0.0;
        for (int j = 0; j < 9; ++j) { Fout[n][j] = f2[j] + roots[k] * D[j]; nrm += Fout[n][j] * Fout[n][j]; }
        if (!(nrm > 1e-300) || !isfinite(nrm)) continue;
        const double inv = rsqrt(nrm);
        for (int j = 0; j < 9; ++j) Fout[n][j] *= inv;
        ++n;
    }
    return n;
}

// cv::findFundamentalMat's RANSAC error (modules/calib3d fundam.cpp computeReprojError): max of the squared distances of
// p2 to the line F p1 and of p1 to the line F^T p2.
template <typename T>
__device__ __forceinline__ T sym_epi_err(const T *F, T ax, T ay, T bx, T by) {
    const T l0 = F[0] * ax + F[1] * ay + F[2], l1 = F[3] * ax + F[4] * ay + F[5], l2 = F[6] * ax + F[7] * ay + F[8];
    const T s = bx * l0 + by * l1 + l2;
    const T m0 = F[0] * bx + F[3] * by + F[6], m1 = F[1] * bx + F[4] * by + F[7];
    const T d2 = s * s / (l0 * l0 + l1 * l1), d1 = s * s / (m0 * m0 + m1 * m1);
    return d1 > d2 ? d1 : d2;
}

// Normalised DLT through four correspondences (x1, y1) -> (x2, y2), p2 ~ H p1 (row-major H, scaled coordinates): the
// 8 x 9 system [x y 1 0 0 0 -u x -u y -u; 0 0 0 x y 1 -v x -v y -v] reduced by Gauss-Jordan elimination with full
// pivoting as in seven_point; h = its null vector (free column 8), unit-normalised.  False: degenerate sample.
static __device__ bool four_point_h(const float (&x1)[4], const float (&y1)[4], const float (&x2)[4], const float (&y2)[4], double (&H)[9]) {
    double A[8][9];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const double x = x1[i], y = y1[i], u = x2[i], v = y2[i];
        A[2 * i][0] = x;   A[2 * i][1] = y;   A[2 * i][2] = 1.0; A[2 * i][3] = 0.0; A[2 * i][4] = 0.0; A[2 * i][5] = 0.0;
        A[2 * i][6] = -u * x; A[2 * i][7] = -u * y; A[2 * i][8] = -u;
        A[2 * i + 1][0] = 0.0; A[2 * i + 1][1] = 0.0; A[2 * i + 1][2] = 0.0; A[2 * i + 1][3] = x; A[2 * i + 1][4] = y; A[2 * i + 1][5] = 1.0;
        A[2 * i + 1][6] = -v * x; A[2 * i + 1][7] = -v * y; A[2 * i + 1][8] = -v;
    }
    int perm[9];
    for (int j = 0; j < 9; ++j) perm[j] = j;
    for (int k = 0; k < 8; ++k) {
        int pr = k, pc = k;
        double best = 0.0;
        for (int i = k; i < 8; ++i)
            for (int j = k; j < 9; ++j)
                if (fabs(A[i][j]) > best) { best = fabs(A[i][j]); pr = i; pc = j; }
        if (best < 1e-12) return false;
        for (int j = 0; j < 9; ++j) { const double t = A[k][j]; A[k][j] = A[pr][j]; A[pr][j] = t; }
        for (int i = 0; i < 8; ++i) { const double t = A[i][k]; A[i][k] = A[i][pc]; A[i][pc] = t; }
        { const int t = perm[k]; perm[k] = perm[pc]; perm[pc] = t; }
        const double inv = 1.0 / A[k][k];
        for (int j = k; j < 9; ++j) A[k][j] *= inv;
        for (int i = 0; i < 8; ++i) {
            if (i == k) continue;
            const double f = A[i][k];
            if (f != 0.0)
                for (int j = k; j < 9; ++j) A[i][j] -= f * A[k][j];
        }
    }
    double nrm = 1.0;
    for (int k = 0; k < 8; ++k) { H[perm[k]] = -A[k][8]; nrm += A[k][8] * A[k][8]; }
    H[perm[8]] = 1.0;
    if (!isfinite(nrm)) return false;
    const double inv = rsqrt(nrm);
    for (int j = 0; j < 9; ++j) H[j] *= inv;
    return true;
}

// Orientation check derived from cv::findHomography's subset check (HomographyEstimatorCallback::checkSubset): every
// triple of the sample must keep its orientation, det[p_a p_b p_c] of image 1 times that of image 2 not negative
// (double, homogeneous points).  Stricter than OpenCV, which also accepts a sample whose four triples all flip (a
// mirror, which no camera motion produces), and without OpenCV's collinearity test (haveCollinearPoints): a sample
// with a collinear triple passes here (det 0) and gives a degenerate model, or none when a DLT pivot falls below 1e-12.
__device__ __forceinline__ bool h_subset_ok(const float (&x1)[4], const float (&y1)[4], const float (&x2)[4], const float (&y2)[4]) {
    const int tt[4][3] = {{0, 1, 2}, {1, 2, 3}, {0, 2, 3}, {0, 1, 3}};
    bool ok = true;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int a = tt[i][0], b = tt[i][1], c = tt[i][2];
        const double A[9] = {x1[a], y1[a], 1.0, x1[b], y1[b], 1.0, x1[c], y1[c], 1.0};
        const double B[9] = {x2[a], y2[a], 1.0, x2[b], y2[b], 1.0, x2[c], y2[c], 1.0};
        ok = ok && !(det3(A) * det3(B) < 0.0);
    }
    return ok;
}

// cv::findHomography's RANSAC error (calib3d fundam.cpp HomographyEstimatorCallback::computeError): the squared
// distance of p2 to H p1 in image 2.  A zero or non-finite w makes the point an outlier (+inf).
template <typename T>
__device__ __forceinline__ T h_transfer_err(const T *H, T ax, T ay, T bx, T by) {
    const T w = H[6] * ax + H[7] * ay + H[8];
    if (w == T(0) || !isfinite(w)) return T(INFINITY);
    const T dx = (H[0] * ax + H[1] * ay + H[2]) / w - bx, dy = (H[3] * ax + H[4] * ay + H[5]) / w - by;
    return dx * dx + dy * dy;
}

enum class GeoModel { fundamental, homography };

// The sample of hypothesis h of the pair with global index `pair`: K distinct indices of the n_pts scaled points, drawn
// from the counter-based state mix(seed ^ mix((pair << 32) | h)) (each slot repeats st = mix(st), idx = (st >> 11) %
// n_pts until the index is new), and their coordinates.  Both models draw through here.
template <int K>
__device__ __forceinline__ void geo_draw(unsigned long long seed, long long pair, int h, int n_pts, const float *sx1,
                                         const float *sy1, const float *sx2, const float *sy2, float (&a)[K], float (&b)[K],
                                         float (&cc)[K], float (&d)[K]) {
    unsigned long long st = geo_mix(seed ^ geo_mix(((unsigned long long)pair << 32) | (unsigned)h));
    int idx[K];
    for (int k = 0; k < K; ++k) {
        bool dup;
        do {
            st = geo_mix(st);
            idx[k] = (int)((st >> 11) % (unsigned long long)n_pts);
            dup = false;
            for (int l = 0; l < k; ++l) dup |= idx[l] == idx[k];
        } while (dup);
    }
    for (int k = 0; k < K; ++k) { a[k] = sx1[idx[k]]; b[k] = sy1[idx[k]]; cc[k] = sx2[idx[k]]; d[k] = sy2[idx[k]]; }
}

// One CTA per pair (msfm_geo_verify / msfm_geo_ransac with the fundamental model, msfm_geo_homography with the
// homography model): used matches into shared memory, hypothesis search, winner, final count over all used matches.
template <GeoModel MODEL>
__device__ __forceinline__ void geo_pairs(const GeoParams gp, int n_pairs) {
    constexpr bool HOMOG = MODEL == GeoModel::homography;
    constexpr int kSample = HOMOG ? 4 : 7;
    __shared__ float sx1[kGeoPointCap], sy1[kGeoPointCap], sx2[kGeoPointCap], sy2[kGeoPointCap];
    __shared__ int s_cnt[kGeoThreads / 32];
    __shared__ int s_red_cnt[kGeoThreads];
    __shared__ int s_red_id[kGeoThreads];
    __shared__ double s_F[9];
    __shared__ int s_ngood, s_best_thread;
    for (int p = blockIdx.x; p < n_pairs; p += gridDim.x) {
        const int64_t m0 = gp.offsets[p];
        const int n_all = (int)(gp.offsets[p + 1] - m0);
        const float *xy1 = gp.xy + 2 * gp.xy_off[gp.pair_img[2 * p]];
        const float *xy2 = gp.xy + 2 * gp.xy_off[gp.pair_img[2 * p + 1]];
        const int2 *mt = gp.matches + m0;
        const uint8_t *gd = gp.good + m0;
        __syncthreads();
        // ---- number of good matches
        int c = 0;
        for (int i = threadIdx.x; i < n_all; i += kGeoThreads) c += gd[i] ? 1 : 0;
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
        if ((threadIdx.x & 31) == 0) s_cnt[threadIdx.x >> 5] = c;
        __syncthreads();
        if (threadIdx.x == 0) {
            int t = 0;
            for (int w = 0; w < kGeoThreads / 32; ++w) t += s_cnt[w];
            s_ngood = t;
        }
        __syncthreads();
        const int n_good = s_ngood;
        bool ok = n_good >= gp.min_points && n_good >= kSample;
        int n_pts = 0;
        float scale = 1.0f;
        if (ok) {
            // ---- good matches (a strided subsample beyond the cap) into shared memory, isotropically scaled:
            //      warp 0 walks the match list 32 entries at a time (ballot + prefix count keeps the list order)
            const int stride = (n_good + kGeoPointCap - 1) / kGeoPointCap;
            if (threadIdx.x < 32) {
                const int lane = threadIdx.x;
                int g = 0, k = 0;  // good matches seen / points stored so far (warp-uniform)
                float mx = 1.0f;
                for (int base = 0; base < n_all; base += 32) {
                    const int i = base + lane;
                    const bool isg = i < n_all && gd[i] != 0;
                    const unsigned bg = __ballot_sync(0xFFFFFFFFu, isg);
                    const int gi = g + __popc(bg & ((1u << lane) - 1u));          // index of this match among the good ones
                    const bool take = isg && (gi % stride == 0);
                    const unsigned bt = __ballot_sync(0xFFFFFFFFu, take);
                    const int ki = k + __popc(bt & ((1u << lane) - 1u));
                    if (take && ki < kGeoPointCap) {
                        const int2 m = mt[i];
                        const float a = xy1[2 * m.x], b = xy1[2 * m.x + 1], c2 = xy2[2 * m.y], d = xy2[2 * m.y + 1];
                        sx1[ki] = a; sy1[ki] = b; sx2[ki] = c2; sy2[ki] = d;
                        mx = fmaxf(mx, fmaxf(fmaxf(fabsf(a), fabsf(b)), fmaxf(fabsf(c2), fabsf(d))));
                    }
                    g += __popc(bg);
                    k += __popc(bt);
                }
                for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, o));
                if (lane == 0) {
                    s_cnt[0] = min(k, kGeoPointCap);
                    s_red_cnt[0] = __float_as_int(1.0f / mx);
                }
            }
            __syncthreads();
            n_pts = s_cnt[0];
            scale = __int_as_float(s_red_cnt[0]);
            __syncthreads();
            for (int i = threadIdx.x; i < n_pts; i += kGeoThreads) { sx1[i] *= scale; sy1[i] *= scale; sx2[i] *= scale; sy2[i] *= scale; }
            __syncthreads();
        }
        // ---- RANSAC: every thread draws hypotheses, solves the 7-point system and scores its candidates on all points
        //      (homography: a 4-point sample that passes the subset check gives one model, id h)
        int best_cnt = -1, best_id = 0x7fffffff;
        float bestF[9];
        for (int j = 0; j < 9; ++j) bestF[j] = 0.0f;
        if constexpr (HOMOG) if (ok && n_pts >= 4) {
            const float th2 = gp.th * scale * gp.th * scale;
            for (int h = threadIdx.x; h < gp.iters; h += kGeoThreads) {
                float a[4], b[4], cc[4], d[4];
                geo_draw(gp.seed, gp.pair_base + p, h, n_pts, sx1, sy1, sx2, sy2, a, b, cc, d);
                double Hc[9];
                if (!h_subset_ok(a, b, cc, d) || !four_point_h(a, b, cc, d, Hc)) continue;
                float Hf[9];
                for (int j = 0; j < 9; ++j) Hf[j] = (float)Hc[j];
                int cnt = 0;
                for (int i = 0; i < n_pts; ++i) cnt += h_transfer_err<float>(Hf, sx1[i], sy1[i], sx2[i], sy2[i]) <= th2 ? 1 : 0;
                if (cnt > best_cnt || (cnt == best_cnt && h < best_id)) {
                    best_cnt = cnt;
                    best_id = h;
                    for (int j = 0; j < 9; ++j) bestF[j] = Hf[j];
                }
            }
        }
        if constexpr (!HOMOG) if (ok && n_pts >= 7) {
            const float th2 = gp.th * scale * gp.th * scale;
            for (int h = threadIdx.x; h < gp.iters; h += kGeoThreads) {
                float a[7], b[7], cc[7], d[7];
                geo_draw(gp.seed, gp.pair_base + p, h, n_pts, sx1, sy1, sx2, sy2, a, b, cc, d);
                double Fc[3][9];
                const int nf = seven_point(a, b, cc, d, Fc);
                for (int f = 0; f < nf; ++f) {
                    float Ff[9];
                    for (int j = 0; j < 9; ++j) Ff[j] = (float)Fc[f][j];
                    int cnt = 0;
                    for (int i = 0; i < n_pts; ++i) cnt += sym_epi_err<float>(Ff, sx1[i], sy1[i], sx2[i], sy2[i]) <= th2 ? 1 : 0;
                    const int id = 3 * h + f;
                    if (cnt > best_cnt || (cnt == best_cnt && id < best_id)) {
                        best_cnt = cnt;
                        best_id = id;
                        for (int j = 0; j < 9; ++j) bestF[j] = Ff[j];
                    }
                }
            }
        }
        s_red_cnt[threadIdx.x] = best_cnt;
        s_red_id[threadIdx.x] = best_id;
        __syncthreads();
        if (threadIdx.x == 0) {
            int bt = 0;
            for (int t = 1; t < kGeoThreads; ++t)
                if (s_red_cnt[t] > s_red_cnt[bt] || (s_red_cnt[t] == s_red_cnt[bt] && s_red_id[t] < s_red_id[bt])) bt = t;
            s_best_thread = s_red_cnt[bt] >= 0 ? bt : -1;
        }
        __syncthreads();
        if (s_best_thread < 0) ok = false;
        if (ok && threadIdx.x == s_best_thread) {
            // back to pixel coordinates: F = T^T F' T with T = diag(s, s, 1); H = T^-1 H' T
            const double s = scale;
            double T[9] = {s * s, s * s, s, s * s, s * s, s, s, s, 1.0};
            if constexpr (HOMOG) { T[0] = T[1] = T[3] = T[4] = 1.0; T[2] = T[5] = 1.0 / s; }
            double nrm = 0.0;
            for (int j = 0; j < 9; ++j) { s_F[j] = (double)bestF[j] * T[j]; nrm += s_F[j] * s_F[j]; }
            // cv::findFundamentalMat scales the result so that F(2,2) = 1 when it is not ~0 (fundam.cpp run7Point);
            // cv::findHomography returns H with H(2,2) = 1
            const double f22 = s_F[8];
            const double k = fabs(f22) > 1e-12 * sqrt(nrm) ? 1.0 / f22 : 1.0 / sqrt(nrm);
            for (int j = 0; j < 9; ++j) s_F[j] *= k;
        }
        __syncthreads();
        // ---- stage A decision: inliers of the best model among ALL good matches (double arithmetic)
        int inl = 0;
        if (ok) {
            const double th2 = (double)gp.th * (double)gp.th;
            for (int i = threadIdx.x; i < n_all; i += kGeoThreads) {
                if (!gd[i]) continue;
                const int2 m = mt[i];
                if constexpr (HOMOG)
                    inl += h_transfer_err<double>(s_F, xy1[2 * m.x], xy1[2 * m.x + 1], xy2[2 * m.y], xy2[2 * m.y + 1]) <= th2 ? 1 : 0;
                else
                    inl += sym_epi_err<double>(s_F, xy1[2 * m.x], xy1[2 * m.x + 1], xy2[2 * m.y], xy2[2 * m.y + 1]) <= th2 ? 1 : 0;
            }
        }
        for (int o = 16; o > 0; o >>= 1) inl += __shfl_xor_sync(0xFFFFFFFFu, inl, o);
        __syncthreads();
        if ((threadIdx.x & 31) == 0) s_cnt[threadIdx.x >> 5] = inl;
        __syncthreads();
        int inliers = 0;
        for (int w = 0; w < kGeoThreads / 32; ++w) inliers += s_cnt[w];
        ok = ok && inliers >= gp.min_inliers;
        // ---- the per-match mask.  Homography: the consensus set, transfer error of the used matches against H <= th^2.
        //      Fundamental, stage B: one-sided distance of p2 to the epipolar line F p1 on every "all" match
        //      (geo_verification.cc:60-79); msfm_geo_ransac: the consensus set of the good matches
        if constexpr (HOMOG) {
            for (int i = threadIdx.x; i < n_all; i += kGeoThreads) {
                uint8_t k = 0;
                if (ok) {
                    const int2 m = mt[i];
                    k = gd[i] && h_transfer_err<double>(s_F, xy1[2 * m.x], xy1[2 * m.x + 1], xy2[2 * m.y], xy2[2 * m.y + 1]) <=
                                     (double)gp.th * (double)gp.th
                            ? 1 : 0;
                }
                gp.keep[m0 + i] = k;
            }
        } else
        for (int i = threadIdx.x; i < n_all; i += kGeoThreads) {
            uint8_t k = 0;
            if (ok && !gp.stage_b) {
                const int2 m = mt[i];
                k = gd[i] && sym_epi_err<double>(s_F, xy1[2 * m.x], xy1[2 * m.x + 1], xy2[2 * m.y], xy2[2 * m.y + 1]) <=
                                 (double)gp.th * (double)gp.th
                        ? 1 : 0;
            } else if (ok) {
                const int2 m = mt[i];
                const double ax = xy1[2 * m.x], ay = xy1[2 * m.x + 1], bx = xy2[2 * m.y], by = xy2[2 * m.y + 1];
                const double l0 = s_F[0] * ax + s_F[1] * ay + s_F[2], l1 = s_F[3] * ax + s_F[4] * ay + s_F[5],
                             l2 = s_F[6] * ax + s_F[7] * ay + s_F[8];
                const double n = sqrt(l0 * l0 + l1 * l1);
                const double dis = (l0 / n) * bx + (l1 / n) * by + (l2 / n);
                k = fabs(dis) < (double)gp.th ? 1 : 0;
            }
            gp.keep[m0 + i] = k;
        }
        if (threadIdx.x == 0) {
            gp.pair_ok[p] = ok ? 1 : 0;
            gp.pair_inliers[p] = inliers;
            if (gp.F)
                for (int j = 0; j < 9; ++j) gp.F[9 * (int64_t)p + j] = ok ? s_F[j] : 0.0;
        }
    }
}

__global__ void __launch_bounds__(kGeoThreads) geo_verify_kernel(const GeoParams gp, int n_pairs) {
    geo_pairs<GeoModel::fundamental>(gp, n_pairs);
}

__global__ void __launch_bounds__(kGeoThreads) geo_homography_kernel(const GeoParams gp, int n_pairs) {
    geo_pairs<GeoModel::homography>(gp, n_pairs);
}

}  // namespace msfm
