// feature_matching_b200.cc — see feature_matching_b200.h.  Pure marshalling over the C ABI.
#include "feature_matching_b200.h"

#include <cmath>

#include <cstring>

namespace objectsfm {

namespace {
bool upload_mat(msfm_ctx *ctx, int slot, cv::Mat &d, float scale, std::string &err) {
    msfm_status st;
    if (d.rows > 0 && d.cols != MSFM_DIM) {
        err = "descriptors must have 128 columns";
        return false;
    }
    if (d.type() == CV_32FC1)
        st = msfm_upload_f32(ctx, slot, d.ptr<float>(0), d.rows, d.rows ? (long long)(d.step / sizeof(float)) : MSFM_DIM, scale);
    else if (d.type() == CV_8UC1)
        st = msfm_upload_u8(ctx, slot, d.ptr<unsigned char>(0), d.rows, d.rows ? (long long)d.step : MSFM_DIM);
    else {
        err = "descriptors must be CV_32FC1 or CV_8UC1";
        return false;
    }
    if (st != MSFM_OK) err = msfm_last_error(ctx);
    return st == MSFM_OK;
}
}  // namespace

FeatureMatchingB200::FeatureMatchingB200(const MatcherB200Options &opt) : opt_(opt) {
    msfm_config cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.device = opt.device;
    cfg.max_images = 2 + (opt.max_indices > 0 ? opt.max_indices : 0);  // slots 0/1: the transient images of a call; 2..: indices
    cfg.arena_rows = opt.arena_rows;
    indices_.assign(opt.max_indices > 0 ? opt.max_indices : 0, nullptr);
    msfm_status st = msfm_create(&cfg, &ctx_);
    if (st != MSFM_OK) {
        ctx_ = nullptr;
        err_ = msfm_status_string(st);
    }
}

FeatureMatchingB200::~FeatureMatchingB200() {
    for (KDIndexB200 *k : indices_) delete k;
    msfm_destroy(ctx_);
}

// A transient image of one call: replaces whatever the slot held (the persistent indices keep their rows).
bool FeatureMatchingB200::Upload(int slot, cv::Mat &d) {
    if (transient_[slot]) msfm_release(ctx_, slot);
    transient_[slot] = upload_mat(ctx_, slot, d, opt_.descriptor_scale, err_);
    return transient_[slot];
}

bool FeatureMatchingB200::Match(cv::Mat &d1, cv::Mat &d2, bool mutual, std::vector<std::pair<int, int>> &matches) {
    if (!ctx_) return false;
    if (!Upload(0, d1) || !Upload(1, d2)) return false;
    // index on image 2, queries = rows of image 1, (i1, i2) ascending i1 (feature_matching.cpp:35-64)
    return MatchSlots(1, 0, d1.rows, mutual, 1, matches);
}

bool FeatureMatchingB200::MatchSlots(int ref_slot, int qry_slot, int qry_rows, bool mutual, int orientation,
                                     std::vector<std::pair<int, int>> &matches) {
    msfm_pair pair = {ref_slot, qry_slot};
    msfm_params prm;
    memset(&prm, 0, sizeof prm);
    prm.ratio = opt_.th_ratio;
    prm.mutual = mutual ? 1 : 0;
    prm.min_keypoints = opt_.th_reject;
    prm.orientation = orientation;
    std::vector<int32_t> buf((size_t)(qry_rows > 0 ? qry_rows : 1) * 2);
    int64_t offsets[2] = {0, 0};
    int32_t okflag = 0;
    msfm_result res;
    res.offsets = offsets;
    res.ok = &okflag;
    res.matches = reinterpret_cast<int32_t(*)[2]>(buf.data());
    res.good = nullptr;
    res.match_capacity = qry_rows;
    msfm_status st = msfm_match_pairs(ctx_, &pair, 1, &prm, &res);
    if (st != MSFM_OK) {
        err_ = msfm_last_error(ctx_);
        return false;
    }
    if (!okflag) return false;  // th_reject gate (feature_matching.cpp:30-33)
    matches.resize((size_t)offsets[1]);  // the reference resizes (feature_matching.cpp:54)
    for (size_t k = 0; k < matches.size(); ++k) matches[k] = std::pair<int, int>(buf[2 * k], buf[2 * k + 1]);
    return true;
}

bool FeatureMatchingB200::KNNMatching(std::vector<cv::KeyPoint> &kp1, cv::Mat &descriptors1, std::vector<cv::KeyPoint> &kp2,
                                      cv::Mat &descriptors2, std::vector<std::pair<int, int>> &matches) {
    if ((int)kp1.size() < opt_.th_reject || (int)kp2.size() < opt_.th_reject) return false;
    return Match(descriptors1, descriptors2, opt_.mutual, matches);
}

bool FeatureMatchingB200::Run(std::vector<cv::KeyPoint> &kp1, cv::Mat &descriptors1, std::vector<cv::KeyPoint> &kp2,
                              cv::Mat &descriptors2, std::vector<std::pair<int, int>> &matches) {
    if ((int)kp1.size() < opt_.th_reject || (int)kp2.size() < opt_.th_reject) return false;
    return Match(descriptors1, descriptors2, true, matches);
}

bool FindHomographyDLT(const std::vector<cv::Point2f> &pt1, const std::vector<cv::Point2f> &pt2, double H[9]) {
    const size_t n = pt1.size();
    if (n < 4 || pt2.size() != n) return false;
    // Hartley normalisation of both point sets
    double c1[2] = {0, 0}, c2[2] = {0, 0};
    for (size_t i = 0; i < n; ++i) { c1[0] += pt1[i].x; c1[1] += pt1[i].y; c2[0] += pt2[i].x; c2[1] += pt2[i].y; }
    for (double *c : {c1, c2}) { c[0] /= n; c[1] /= n; }
    double d1 = 0, d2 = 0;
    for (size_t i = 0; i < n; ++i) {
        d1 += std::hypot(pt1[i].x - c1[0], pt1[i].y - c1[1]);
        d2 += std::hypot(pt2[i].x - c2[0], pt2[i].y - c2[1]);
    }
    if (!(d1 > 0) || !(d2 > 0)) return false;
    const double s1 = std::sqrt(2.0) * n / d1, s2 = std::sqrt(2.0) * n / d2;
    double M[9][9] = {};
    for (size_t i = 0; i < n; ++i) {
        const double x = (pt1[i].x - c1[0]) * s1, y = (pt1[i].y - c1[1]) * s1, u = (pt2[i].x - c2[0]) * s2, v = (pt2[i].y - c2[1]) * s2;
        const double r1[9] = {x, y, 1, 0, 0, 0, -u * x, -u * y, -u}, r2[9] = {0, 0, 0, x, y, 1, -v * x, -v * y, -v};
        for (int a = 0; a < 9; ++a)
            for (int b = 0; b < 9; ++b) M[a][b] += r1[a] * r1[b] + r2[a] * r2[b];
    }
    // cyclic Jacobi: eigenvector of the smallest eigenvalue of the symmetric 9 x 9 matrix
    double V[9][9] = {};
    for (int i = 0; i < 9; ++i) V[i][i] = 1.0;
    for (int sweep = 0; sweep < 60; ++sweep) {
        double off = 0;
        for (int p = 0; p < 9; ++p)
            for (int q = p + 1; q < 9; ++q) off += M[p][q] * M[p][q];
        if (off < 1e-26) break;
        for (int p = 0; p < 9; ++p)
            for (int q = p + 1; q < 9; ++q) {
                if (std::fabs(M[p][q]) < 1e-300) continue;
                const double theta = (M[q][q] - M[p][p]) / (2.0 * M[p][q]);
                const double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
                const double c = 1.0 / std::sqrt(t * t + 1.0), sn = t * c;
                for (int k = 0; k < 9; ++k) { const double a = M[k][p], b = M[k][q]; M[k][p] = c * a - sn * b; M[k][q] = sn * a + c * b; }
                for (int k = 0; k < 9; ++k) { const double a = M[p][k], b = M[q][k]; M[p][k] = c * a - sn * b; M[q][k] = sn * a + c * b; }
                for (int k = 0; k < 9; ++k) { const double a = V[k][p], b = V[k][q]; V[k][p] = c * a - sn * b; V[k][q] = sn * a + c * b; }
            }
    }
    int best = 0;
    for (int i = 1; i < 9; ++i)
        if (M[i][i] < M[best][best]) best = i;
    double h[9];
    for (int i = 0; i < 9; ++i) h[i] = V[i][best];
    // denormalise: H = T2^-1 * Hn * T1 with T = [s 0 -s*cx; 0 s -s*cy; 0 0 1]
    const double T1[9] = {s1, 0, -s1 * c1[0], 0, s1, -s1 * c1[1], 0, 0, 1};
    const double T2i[9] = {1 / s2, 0, c2[0], 0, 1 / s2, c2[1], 0, 0, 1};
    double tmp[9], out[9];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) tmp[3 * r + c] = h[3 * r] * T1[c] + h[3 * r + 1] * T1[3 + c] + h[3 * r + 2] * T1[6 + c];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) out[3 * r + c] = T2i[3 * r] * tmp[c] + T2i[3 * r + 1] * tmp[3 + c] + T2i[3 * r + 2] * tmp[6 + c];
    if (std::fabs(out[8]) < 1e-300) return false;
    for (int i = 0; i < 9; ++i) H[i] = out[i] / out[8];
    return true;
}

bool FeatureMatchingB200::KNNMatchingWithGeoVerify(std::vector<cv::KeyPoint> &kp1, cv::Mat &descriptors1, std::vector<cv::KeyPoint> &kp2,
                                                   cv::Mat &descriptors2, std::vector<std::pair<int, int>> &matches) {
    if ((int)kp1.size() < opt_.th_reject || (int)kp2.size() < opt_.th_reject) return false;  // feature_matching.cpp:74-77
    std::vector<std::pair<int, int>> cur;
    if (!Match(descriptors1, descriptors2, opt_.mutual, cur)) return false;                   // ratio matches (i1, i2)
    return Verify(kp1, kp2, cur, matches);
}

// The verification passes every KNNMatchingWithGeoVerify overload shares (feature_matching.cpp:94-147 and its copies).
bool FeatureMatchingB200::Verify(std::vector<cv::KeyPoint> &kp1, std::vector<cv::KeyPoint> &kp2, std::vector<std::pair<int, int>> &cur,
                                 std::vector<std::pair<int, int>> &matches) {
    std::vector<float> xy1(kp1.size() * 2), xy2(kp2.size() * 2);
    for (size_t i = 0; i < kp1.size(); ++i) { xy1[2 * i] = kp1[i].pt.x; xy1[2 * i + 1] = kp1[i].pt.y; }
    for (size_t i = 0; i < kp2.size(); ++i) { xy2[2 * i] = kp2[i].pt.x; xy2[2 * i + 1] = kp2[i].pt.y; }
    const float th_epipolar[2] = {3.0f, 1.0f};                                                  // feature_matching.cpp:97-99
    for (int iter = 0; iter < 2; ++iter) {
        if ((int)cur.size() < opt_.th_reject) return false;                                     // :114-117
        std::vector<cv::Point2f> p1(cur.size()), p2(cur.size());
        for (size_t k = 0; k < cur.size(); ++k) { p1[k] = kp1[cur[k].first].pt; p2[k] = kp2[cur[k].second].pt; }
        double H[9];
        if (FindHomographyDLT(p1, p2, H) && std::fabs(H[0] - 0.995) < 0.01 && std::fabs(H[4] - 0.995) < 0.01 &&
            std::fabs(H[8] - 0.995) < 0.01)
            return false;                                                                        // :120-127 (no parallax)
        // cv::findFundamentalMat(pt1, pt2, status, FM_RANSAC, th) :129-137 -> msfm_geo_ransac; image 1 plays "ref"
        msfm_pair pair = {0, 1};
        int64_t offsets[2] = {0, (int64_t)cur.size()};
        std::vector<int32_t> m(cur.size() * 2);
        for (size_t k = 0; k < cur.size(); ++k) { m[2 * k] = cur[k].first; m[2 * k + 1] = cur[k].second; }
        std::vector<uint8_t> use(cur.size(), 1), mask(cur.size(), 0);
        const float *xy[2] = {xy1.data(), xy2.data()};
        const int32_t npts[2] = {(int32_t)kp1.size(), (int32_t)kp2.size()};
        msfm_geo_params gp;
        memset(&gp, 0, sizeof gp);
        gp.th_epipolar = th_epipolar[iter];
        gp.min_points = 8;
        gp.min_inliers = 0;
        gp.iters = 1024;
        gp.seed = (uint64_t)iter;
        int32_t ok = 0, inl = 0;
        msfm_status st = msfm_geo_ransac(ctx_, &pair, 1, offsets, reinterpret_cast<const int32_t(*)[2]>(m.data()), use.data(), xy, npts, 2,
                                         &gp, &ok, &inl, mask.data(), nullptr);
        if (st != MSFM_OK) {
            err_ = msfm_last_error(ctx_);
            return false;
        }
        std::vector<std::pair<int, int>> next;
        for (size_t k = 0; k < cur.size(); ++k)
            if (mask[k]) next.push_back(cur[k]);
        cur.swap(next);
    }
    matches.insert(matches.end(), cur.begin(), cur.end());                                       // :141-147 (push_back)
    return true;  // the reference falls off the end here; its callers treat the call as successful
}

// ---------------------------------------------------------------------------------------------------- persistent indices
bool FeatureMatchingB200::GenerateKDIndex(cv::Mat &descriptors, KDIndexB200 **kdindex) {
    if (!ctx_ || !kdindex) return false;
    *kdindex = nullptr;
    for (size_t k = 0; k < indices_.size(); ++k) {
        if (indices_[k]) continue;
        const int slot = 2 + (int)k;
        if (!upload_mat(ctx_, slot, descriptors, opt_.descriptor_scale, err_)) return false;  // packed once; stays in HBM
        KDIndexB200 *idx = new KDIndexB200();
        idx->slot_ = slot;
        idx->rows_ = descriptors.rows;
        indices_[k] = idx;
        *kdindex = idx;
        return true;
    }
    err_ = "no free index slot (MatcherB200Options::max_indices)";
    return false;
}

void FeatureMatchingB200::ReleaseKDIndex(KDIndexB200 *kdindex) {
    if (!ctx_ || !kdindex) return;
    for (size_t k = 0; k < indices_.size(); ++k)
        if (indices_[k] == kdindex) {
            msfm_release(ctx_, kdindex->slot_);
            delete kdindex;
            indices_[k] = nullptr;
        }
}

bool FeatureMatchingB200::MatchAgainstIndex(KDIndexB200 *kdindex, cv::Mat &descriptors_other, bool index_is_image1,
                                            std::vector<std::pair<int, int>> &matches) {
    if (!ctx_ || !kdindex || kdindex->slot_ < 2) return false;
    if (!Upload(0, descriptors_other)) return false;  // only the partner is staged; the index stays where it is
    // index on image 1: pairs (i1, i2) ascending i2 = (ref, query) = orientation 0; index on image 2: (i1, i2) ascending
    // i1 = (query, ref) = orientation 1
    return MatchSlots(kdindex->slot_, 0, descriptors_other.rows, opt_.mutual, index_is_image1 ? 0 : 1, matches);
}

bool FeatureMatchingB200::KNNMatchingWithGeoVerify(std::vector<cv::KeyPoint> &kp1, cv::Mat &descriptors1, std::vector<cv::KeyPoint> &kp2,
                                                   KDIndexB200 *kdindex2, std::vector<std::pair<int, int>> &matches) {
    if ((int)kp1.size() < opt_.th_reject || (int)kp2.size() < opt_.th_reject) return false;  // feature_matching.cpp:157-160
    std::vector<std::pair<int, int>> cur;
    if (!MatchAgainstIndex(kdindex2, descriptors1, false, cur)) return false;
    return Verify(kp1, kp2, cur, matches);
}

bool FeatureMatchingB200::KNNMatchingWithGeoVerify(std::vector<cv::KeyPoint> &kp1, KDIndexB200 *kdindex1, std::vector<cv::KeyPoint> &kp2,
                                                   cv::Mat &descriptors2, std::vector<std::pair<int, int>> &matches) {
    if ((int)kp1.size() < opt_.th_reject || (int)kp2.size() < opt_.th_reject) return false;  // feature_matching.cpp:239-242,325-328
    std::vector<std::pair<int, int>> cur;
    if (!MatchAgainstIndex(kdindex1, descriptors2, true, cur)) return false;
    return Verify(kp1, kp2, cur, matches);
}

bool FeatureMatchingB200::KNNMatchingWithGeoVerify(std::vector<cv::KeyPoint> &kp1, std::vector<cv::KeyPoint> &kp2, int *id, float *dis,
                                                   std::vector<std::pair<int, int>> &matches) {
    if (!ctx_ || !id || !dis) return false;
    if ((int)kp1.size() < opt_.th_reject || (int)kp2.size() < opt_.th_reject) return false;  // feature_matching.cpp:483-486
    std::vector<std::pair<int, int>> cur;
    for (size_t i = 0; i < kp2.size(); ++i) {                                                   // :488-500
        const float ratio = dis[2 * i + 0] / dis[2 * i + 1];
        if (ratio < opt_.th_ratio) cur.push_back(std::pair<int, int>(id[2 * i + 0], (int)i));
    }
    return Verify(kp1, kp2, cur, matches);
}

bool FeatureMatchingB200::KNN2(cv::Mat &descriptors1, cv::Mat &descriptors2, int *id, float *dis) {
    if (!ctx_) return false;
    if (!Upload(0, descriptors1) || !Upload(1, descriptors2)) return false;
    msfm_status st = msfm_knn2(ctx_, 0, 1, id, dis);
    if (st != MSFM_OK) err_ = msfm_last_error(ctx_);
    return st == MSFM_OK;
}

MatchGraphB200::MatchGraphB200(int device, int max_images, long long total_rows, float descriptor_scale) : scale_(descriptor_scale) {
    msfm_config cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.device = device;
    cfg.max_images = max_images;
    cfg.arena_rows = total_rows + 256ll * max_images;  // every image is padded to a multiple of 256 rows
    rows_.assign(max_images, -1);
    msfm_status st = msfm_create(&cfg, &ctx_);
    if (st != MSFM_OK) {
        ctx_ = nullptr;
        err_ = msfm_status_string(st);
    }
}

MatchGraphB200::~MatchGraphB200() { msfm_destroy(ctx_); }

bool MatchGraphB200::AddImage(int idx, cv::Mat &descriptors) {
    if (!ctx_ || idx < 0 || idx >= (int)rows_.size()) return false;
    if (!upload_mat(ctx_, idx, descriptors, scale_, err_)) return false;
    rows_[idx] = descriptors.rows;
    return true;
}

bool MatchGraphB200::ReleaseImage(int idx) {
    if (!ctx_ || idx < 0 || idx >= (int)rows_.size()) return false;
    rows_[idx] = -1;
    return msfm_release(ctx_, idx) == MSFM_OK;
}

bool MatchGraphB200::MatchPairs(const std::vector<std::vector<int>> &match_graph_init, std::vector<std::vector<PairMatches>> &out,
                                float th_good, float th_all, bool mutual, int th_reject) {
    return Match(match_graph_init, nullptr, out, th_good, th_all, mutual, th_reject);
}

bool MatchGraphB200::MatchPairsGuided(const std::vector<std::vector<int>> &match_graph_init, const std::vector<std::array<double, 9>> &F,
                                      const std::vector<std::vector<cv::KeyPoint>> &keypoints, float th_epipolar,
                                      std::vector<std::vector<PairMatches>> &out, float th_good, float th_all, bool mutual, int th_reject) {
    const Guide g = {Guide::epipolar, &F, &keypoints, th_epipolar};
    return Match(match_graph_init, &g, out, th_good, th_all, mutual, th_reject);
}

bool MatchGraphB200::MatchPairsGuidedHomography(const std::vector<std::vector<int>> &match_graph_init,
                                                const std::vector<std::array<double, 9>> &H,
                                                const std::vector<std::vector<cv::KeyPoint>> &keypoints, float th_transfer,
                                                std::vector<std::vector<PairMatches>> &out, float th_good, float th_all, bool mutual,
                                                int th_reject) {
    const Guide g = {Guide::homography, &H, &keypoints, th_transfer};
    return Match(match_graph_init, &g, out, th_good, th_all, mutual, th_reject);
}

bool MatchGraphB200::Match(const std::vector<std::vector<int>> &match_graph_init, const Guide *guide, std::vector<std::vector<PairMatches>> &out,
                           float th_good, float th_all, bool mutual, int th_reject) {
    if (!ctx_) return false;
    std::vector<msfm_pair> pairs;
    long long capacity = 0;
    for (size_t idx1 = 0; idx1 < match_graph_init.size(); ++idx1)
        for (int idx2 : match_graph_init[idx1]) {
            if (idx2 < 0 || idx2 >= (int)rows_.size() || rows_[idx1] < 0 || rows_[idx2] < 0) {
                err_ = "pair list names an image that was not added";
                return false;
            }
            msfm_pair p = {(int32_t)idx1, (int32_t)idx2};  // index on idx1, queries = rows of idx2 (fine_matching_graph.cc:81,99)
            pairs.push_back(p);
            capacity += rows_[idx2];
        }
    std::vector<int64_t> offsets(pairs.size() + 1);
    std::vector<int32_t> okflags(pairs.size());
    std::vector<int32_t> buf((size_t)(capacity > 0 ? capacity : 1) * 2);
    std::vector<uint8_t> good((size_t)(capacity > 0 ? capacity : 1));
    msfm_params prm;
    memset(&prm, 0, sizeof prm);
    prm.ratio = th_all;
    prm.ratio_good = th_good;
    prm.max_dist_sq = 0.f;
    prm.mutual = mutual ? 1 : 0;
    prm.min_keypoints = th_reject;
    prm.orientation = 0;  // (ptid1, ptid2) ascending ptid2 (fine_matching_graph.cc:121,127)
    prm.rescore_band = 0.f;
    msfm_result res;
    res.offsets = offsets.data();
    res.ok = okflags.data();
    res.matches = reinterpret_cast<int32_t(*)[2]>(buf.data());
    res.good = good.data();
    res.match_capacity = capacity;
    msfm_status st;
    if (guide) {
        if (guide->M->size() != pairs.size()) {
            err_ = guide->kind == Guide::homography ? "MatchPairsGuidedHomography needs one H per pair" : "MatchPairsGuided needs one F per pair";
            return false;
        }
        // keypoints as the library takes them: (x, y) per descriptor row, one array per image
        const size_t n_images = rows_.size();
        std::vector<std::vector<float>> xy(n_images);
        std::vector<const float *> xy_ptr(n_images, nullptr);
        std::vector<int32_t> npts(n_images, 0);
        for (size_t i = 0; i < n_images && i < guide->keypoints->size(); ++i) {
            const std::vector<cv::KeyPoint> &kp = (*guide->keypoints)[i];
            for (const cv::KeyPoint &k : kp) {
                xy[i].push_back(k.pt.x);
                xy[i].push_back(k.pt.y);
            }
            xy_ptr[i] = xy[i].data();
            npts[i] = (int32_t)kp.size();
        }
        const double(*M)[9] = reinterpret_cast<const double(*)[9]>(guide->M->data());
        st = guide->kind == Guide::homography
                 ? msfm_match_pairs_guided_homography(ctx_, pairs.data(), (int64_t)pairs.size(), &prm, M, guide->th, xy_ptr.data(),
                                                      npts.data(), (int32_t)n_images, &res)
                 : msfm_match_pairs_guided(ctx_, pairs.data(), (int64_t)pairs.size(), &prm, M, guide->th, xy_ptr.data(), npts.data(),
                                           (int32_t)n_images, &res);
    } else {
        st = msfm_match_pairs(ctx_, pairs.data(), (int64_t)pairs.size(), &prm, &res);
    }
    if (st != MSFM_OK) {
        err_ = msfm_last_error(ctx_);
        return false;
    }
    out.assign(match_graph_init.size(), std::vector<PairMatches>());
    size_t p = 0;
    for (size_t idx1 = 0; idx1 < match_graph_init.size(); ++idx1) {
        out[idx1].resize(match_graph_init[idx1].size());
        for (size_t j = 0; j < match_graph_init[idx1].size(); ++j, ++p) {
            PairMatches &pm = out[idx1][j];
            pm.ok = okflags[p] != 0;
            for (int64_t k = offsets[p]; k < offsets[p + 1]; ++k) {
                pm.matches_all.push_back(std::pair<int, int>(buf[2 * k], buf[2 * k + 1]));
                pm.is_good.push_back(good[k]);
            }
        }
    }
    return true;
}

// ---------------------------------------------------------------------------------------------------- SiftMatchGPU shape
SiftMatchB200::SiftMatchB200(int max_sift, int device) : device_(device), max_sift_(max_sift > 0 ? max_sift : 4096) { SetMaxSift(max_sift_); }

SiftMatchB200::~SiftMatchB200() { msfm_destroy(ctx_); }

void SiftMatchB200::SetMaxSift(int max_sift) {
    if (max_sift <= 0) return;
    if (ctx_ && max_sift <= max_sift_) { max_sift_ = max_sift; return; }  // shrinking keeps the table
    msfm_destroy(ctx_);
    ctx_ = nullptr;
    max_sift_ = max_sift;
    set_[0] = set_[1] = false;
    msfm_config cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.device = device_;
    cfg.max_images = 2;
    cfg.arena_rows = 2ll * ((max_sift + 255) / 256 * 256);
    if (msfm_create(&cfg, &ctx_) != MSFM_OK) ctx_ = nullptr;
}

void SiftMatchB200::SetDescriptors(int index, int num, const float *descriptors, int id) {
    if (!ctx_ || index < 0 || index > 1 || num < 0 || (num > 0 && !descriptors)) return;
    if (id >= 0 && set_[index] && id_[index] == id) return;  // same feature set as last time (SiftGPU.h: "id" caching)
    num = num < max_sift_ ? num : max_sift_;                 // SiftGPU keeps at most max_sift features per set
    if (set_[index]) msfm_release(ctx_, index);
    set_[index] = msfm_upload_f32(ctx_, index, descriptors, num, MSFM_DIM, 512.0f) == MSFM_OK;  // "normalized to 1.0"
    num_[index] = set_[index] ? num : 0;
    id_[index] = id;
}

void SiftMatchB200::SetDescriptors(int index, int num, const unsigned char *descriptors, int id) {
    if (!ctx_ || index < 0 || index > 1 || num < 0 || (num > 0 && !descriptors)) return;
    if (id >= 0 && set_[index] && id_[index] == id) return;
    num = num < max_sift_ ? num : max_sift_;
    if (set_[index]) msfm_release(ctx_, index);
    set_[index] = msfm_upload_u8(ctx_, index, descriptors, num, MSFM_DIM) == MSFM_OK;            // "normalized to 512"
    num_[index] = set_[index] ? num : 0;
    id_[index] = id;
}

int SiftMatchB200::GetSiftMatch(int max_match, int match_buffer[][2], float distmax, float ratiomax, int mutual_best_match) {
    if (!ctx_ || !set_[0] || !set_[1] || max_match <= 0 || !match_buffer || num_[0] == 0 || num_[1] == 0) return 0;
    msfm_pair pair = {1, 0};  // set 1 is searched, the rows of set 0 are the queries
    msfm_params prm;
    memset(&prm, 0, sizeof prm);
    prm.ratio = ratiomax;
    // acos(d1.d2) < distmax  <=>  |d1 - d2|^2 < 2 - 2 cos(distmax) for unit vectors; rows are 512-scaled
    prm.max_dist_sq = distmax > 0.0f ? (float)(512.0 * 512.0 * (2.0 - 2.0 * std::cos((double)distmax))) : 0.0f;
    prm.mutual = mutual_best_match ? 1 : 0;
    prm.min_keypoints = 0;  // SiftMatchGPU has no keypoint gate
    prm.orientation = 1;    // (index in set 0, index in set 1), ascending set-0 index
    std::vector<int32_t> buf((size_t)num_[0] * 2);
    int64_t offsets[2] = {0, 0};
    int32_t okflag = 0;
    msfm_result res;
    res.offsets = offsets;
    res.ok = &okflag;
    res.matches = reinterpret_cast<int32_t(*)[2]>(buf.data());
    res.good = nullptr;
    res.match_capacity = num_[0];
    if (msfm_match_pairs(ctx_, &pair, 1, &prm, &res) != MSFM_OK) return 0;
    const int n = (int)(offsets[1] < max_match ? offsets[1] : max_match);  // "max_match: the length of the match_buffer"
    for (int k = 0; k < n; ++k) { match_buffer[k][0] = buf[2 * k]; match_buffer[k][1] = buf[2 * k + 1]; }
    return n;
}

}  // namespace objectsfm
