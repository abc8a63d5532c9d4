// feature_matching_b200.h — C++ host mirror of MetricSfM's matcher interface on top of the C ABI (include/msfm_match.h).
//
// Same containers in (std::vector<cv::KeyPoint>, cv::Mat CV_32FC1 N x 128), same per-pair match lists out
// (std::vector<std::pair<int,int>>), same bool error convention, so the SfM tracking / triangulation stages
// (sfm_incremental.cc:224-915, slam_gps.cc:557-668) consume the results unchanged:
//
//   reference                                                             here
//   FeatureMatching::KNNMatching(kp1, d1, kp2, d2, matches)               FeatureMatchingB200::KNNMatching
//     SfM/src/feature/feature_matching.h:33-35, .cpp:24-65                  (index on image 2, ratio 0.5, (i1,i2) ascending i1)
//   FeatureMatching::KNNMatchingWithGeoVerify(kp1, kp2, id, dis, matches) FeatureMatchingB200::KNN2 fills id/dis
//     feature_matching.h:57-58, .cpp:477-501                                ([2*N2] FLANN layout, squared L2)
//   FeatureMatchingCudaSift::Run(kp1, d1, kp2, d2, matches)               FeatureMatchingB200::Run
//     feature_matching_cuda_sift.h:34-36, .cpp:21-108 (kNN part)            (mutual best match, ratio as given)
//   FineMatchingGraph::BuildMatchGraph kNN + ratio loops                  MatchGraphB200::{AddImage, MatchPairs}
//     graph/fine_matching_graph.cc:58-133                                    (descriptors staged once, whole pair list batched)
//
// Everything here is a thin marshalling layer: all arithmetic runs in the CUDA library behind msfm_match.h.
#pragma once
#include <array>
#include <string>
#include <utility>
#include <vector>

#include "../../include/msfm_match.h"
#include "cv_standin.h"

namespace objectsfm {

// Float descriptors are quantised q = min(255, max(0, rint(x * scale))): 1 for VLSIFT's 512-scaled rows
// (feature_extractor_vl_sift.cpp:201-203), 512 for unit-norm rows (feature_extractor_cuda_sift.cpp:75-80).
struct MatcherB200Options {
    int device = 0;
    float descriptor_scale = 1.0f;
    float th_ratio = 0.5f;   // feature_matching.cpp:27
    int th_reject = 20;      // feature_matching.cpp:28
    bool mutual = false;     // the CPU paths have none; SiftMatchGPU::GetSiftMatch defaults to 1 (SiftGPU.h:308)
    int max_indices = 14;    // persistent indices (GenerateKDIndex) that can be alive at once
    long long arena_rows = 1ll << 20;  // descriptor rows the matcher's table holds (two transient images + the indices);
                                       // 128 MiB of HBM at the default; idx_max_per_image is 1,000,000 (basic_structs.h:171)
};

class FeatureMatchingB200;

// Stand-in for the reference's persistent kNN indices — cv::flann::Index* (feature_matching.h:41-47, GenerateKDIndex :63),
// my_kd_tree_t* (:49-51), flann_index_t (:53-55): the image's descriptors, packed ONCE into the matcher's table in HBM.
// Build it once per image and match any number of partners against it (fine_matching_graph.cc:72-101 does exactly that
// per idx1); nothing is re-uploaded per pair.
class KDIndexB200 {
public:
    int rows() const { return rows_; }
private:
    friend class FeatureMatchingB200;
    int slot_ = -1, rows_ = 0;
};

class FeatureMatchingB200 {
public:
    explicit FeatureMatchingB200(const MatcherB200Options &opt = MatcherB200Options());
    ~FeatureMatchingB200();
    FeatureMatchingB200(const FeatureMatchingB200 &) = delete;
    FeatureMatchingB200 &operator=(const FeatureMatchingB200 &) = delete;

    bool ok() const { return ctx_ != nullptr; }
    const std::string &last_error() const { return err_; }

    // FeatureMatching::KNNMatching: kd-index on descriptors2, every row of descriptors1 queried, ratio < th_ratio,
    // matches resized to (i1, i2) ascending i1; false when either image has < th_reject keypoints.
    bool KNNMatching(std::vector<cv::KeyPoint> &kp1, cv::Mat &descriptors1, std::vector<cv::KeyPoint> &kp2, cv::Mat &descriptors2,
                     std::vector<std::pair<int, int>> &matches);
    // FeatureMatchingCudaSift::Run kNN part: same as above with the mutual-best-match rule of the declared GPU matchers.
    bool Run(std::vector<cv::KeyPoint> &kp1, cv::Mat &descriptors1, std::vector<cv::KeyPoint> &kp2, cv::Mat &descriptors2,
             std::vector<std::pair<int, int>> &matches);
    // FeatureMatching::KNNMatchingWithGeoVerify(kp1, d1, kp2, d2, matches) (feature_matching.cpp:67-150): ratio matches as in
    // KNNMatching, then two verification passes (epipolar threshold 3 px, then 1 px): fewer than th_reject matches =>
    // false; a least-squares homography close to the identity (diagonal within 0.01 of 0.995) => false (no parallax);
    // RANSAC-F, outliers dropped.  The matches are APPENDED (the reference push_backs).  RANSAC runs on the GPU
    // (msfm_geo_ransac); the homography is a normalised DLT without OpenCV's final Levenberg-Marquardt polish, which the
    // 0.01 test does not resolve.
    bool KNNMatchingWithGeoVerify(std::vector<cv::KeyPoint> &kp1, cv::Mat &descriptors1, std::vector<cv::KeyPoint> &kp2,
                                  cv::Mat &descriptors2, std::vector<std::pair<int, int>> &matches);
    // Index on image 1, 2-NN of every row of image 2 in FLANN layout: id[2*N2], dis[2*N2] (squared L2) — exactly the
    // arrays KNNMatchingWithGeoVerify(kp1, kp2, id, dis, matches) and fine_matching_graph.cc:96-99 consume.
    bool KNN2(cv::Mat &descriptors1, cv::Mat &descriptors2, int *id, float *dis);

    // ---- persistent-index overloads (feature_matching.h:41-55, :63) --------------------------------------------------
    // FeatureMatching::GenerateKDIndex(descriptors, &kdindex): pack the image once.  ReleaseKDIndex frees its table rows.
    bool GenerateKDIndex(cv::Mat &descriptors, KDIndexB200 **kdindex);
    void ReleaseKDIndex(KDIndexB200 *kdindex);
    // KNNMatchingWithGeoVerify(kp1, descriptors1, kp2, kdindex2, matches) (feature_matching.cpp:152-233): index on image 2,
    // every row of image 1 queried, ratio < th_ratio, pairs (i1, i2) ascending i1, then the verification passes.
    bool KNNMatchingWithGeoVerify(std::vector<cv::KeyPoint> &kp1, cv::Mat &descriptors1, std::vector<cv::KeyPoint> &kp2,
                                  KDIndexB200 *kdindex2, std::vector<std::pair<int, int>> &matches);
    // KNNMatchingWithGeoVerify(kp1, kdindex1 | kd_tree1 | flann kd_tree1, kp2, descriptors2, matches)
    // (feature_matching.cpp:235-475): index on image 1, every row of image 2 queried, pairs (i1, i2) ascending i2.
    bool KNNMatchingWithGeoVerify(std::vector<cv::KeyPoint> &kp1, KDIndexB200 *kdindex1, std::vector<cv::KeyPoint> &kp2,
                                  cv::Mat &descriptors2, std::vector<std::pair<int, int>> &matches);
    // The kNN + ratio part of the two overloads above without the verification passes (what FineMatchingGraph's loops do
    // per partner, fine_matching_graph.cc:96-133): index_is_image1 selects the orientation.
    bool MatchAgainstIndex(KDIndexB200 *kdindex, cv::Mat &descriptors_other, bool index_is_image1,
                           std::vector<std::pair<int, int>> &matches);
    // KNNMatchingWithGeoVerify(kp1, kp2, id, dis, matches) (feature_matching.cpp:477-553): the caller supplies the kNN
    // arrays (index on image 1, [2*N2] FLANN layout — e.g. from KNN2 or msfm_knn2); ratio < th_ratio on them, then the
    // verification passes.
    bool KNNMatchingWithGeoVerify(std::vector<cv::KeyPoint> &kp1, std::vector<cv::KeyPoint> &kp2, int *id, float *dis,
                                  std::vector<std::pair<int, int>> &matches);

private:
    bool Match(cv::Mat &d1, cv::Mat &d2, bool mutual, std::vector<std::pair<int, int>> &matches);
    bool MatchSlots(int ref_slot, int qry_slot, int qry_rows, bool mutual, int orientation, std::vector<std::pair<int, int>> &matches);
    bool Verify(std::vector<cv::KeyPoint> &kp1, std::vector<cv::KeyPoint> &kp2, std::vector<std::pair<int, int>> &cur,
                std::vector<std::pair<int, int>> &matches);
    bool Upload(int slot, cv::Mat &d);
    msfm_ctx *ctx_ = nullptr;
    MatcherB200Options opt_;
    std::vector<KDIndexB200 *> indices_;  // slot 2 + k
    bool transient_[2] = {false, false};
    std::string err_;
};

// SiftMatchGPU-shaped front end (thirdparty/siftgpu/include/siftgpu/SiftGPU.h:255-336; declared in the reference, no call
// sites, shipped as a binary): two descriptor sets, then GetSiftMatch.  Set 0 rows are the queries, set 1 the reference
// set; matches come back as (index in set 0, index in set 1), ascending set-0 index, truncated to max_match.
//   * descriptors: unsigned char rows "normalized to 512" (SiftGPU.h:298) are taken as they are; float rows "normalized
//     to 1.0" (:296) are quantised with scale 512
//   * distmax is SiftGPU's angular bound acos(d1.d2) < distmax; it becomes the equivalent squared-L2 gate
//     d^2 < 512^2 * (2 - 2 cos(distmax)) (exact for unit-norm rows)
//   * ratiomax applies to squared L2 distances, strict '<' (north_star fixes the metric; SiftGPU compares angles)
//   * mutual_best_match: lowest index wins ties in both directions, like the recovered s_row_max / s_col_max shaders
class SiftMatchB200 {
public:
    explicit SiftMatchB200(int max_sift = 4096, int device = 0);  // SiftMatchGPU(int max_sift = 4096)
    ~SiftMatchB200();
    SiftMatchB200(const SiftMatchB200 &) = delete;
    SiftMatchB200 &operator=(const SiftMatchB200 &) = delete;
    bool ok() const { return ctx_ != nullptr; }
    void SetMaxSift(int max_sift);
    void SetDescriptors(int index, int num, const float *descriptors, int id = -1);
    void SetDescriptors(int index, int num, const unsigned char *descriptors, int id = -1);
    int GetSiftMatch(int max_match, int match_buffer[][2], float distmax = 0.7f, float ratiomax = 0.8f, int mutual_best_match = 1);

private:
    msfm_ctx *ctx_ = nullptr;
    int device_, max_sift_, num_[2] = {0, 0}, id_[2] = {-1, -1};
    bool set_[2] = {false, false};
};

// Least-squares homography pt2 ~ H pt1 (normalised DLT, smallest eigenvector of A^T A by Jacobi sweeps), scaled so that
// H[8] = 1; false when the system is degenerate.  Stand-in for cv::findHomography(pt1, pt2) with method 0
// (feature_matching.cpp:115).
bool FindHomographyDLT(const std::vector<cv::Point2f> &pt1, const std::vector<cv::Point2f> &pt2, double H[9]);

// Batched form of FineMatchingGraph::BuildMatchGraph's matching loops: stage every image once (replaces the per-idx1
// flann_build_index and the per-pair disk re-reads, fine_matching_graph.cc:69-91), then match the whole candidate pair
// list; per pair the "all" list (ratio < th_all) with a flag for the "good" subset (ratio < th_good), pairs
// (id_in_idx1, id_in_idx2) ascending id_in_idx2 as in fine_matching_graph.cc:116-133.
class MatchGraphB200 {
public:
    MatchGraphB200(int device, int max_images, long long total_rows, float descriptor_scale = 1.0f);
    ~MatchGraphB200();
    MatchGraphB200(const MatchGraphB200 &) = delete;
    MatchGraphB200 &operator=(const MatchGraphB200 &) = delete;

    bool ok() const { return ctx_ != nullptr; }
    const std::string &last_error() const { return err_; }
    bool AddImage(int idx, cv::Mat &descriptors);   // once per image
    bool ReleaseImage(int idx);

    struct PairMatches {
        bool ok = false;                              // false: < 20 keypoints on either side
        std::vector<std::pair<int, int>> matches_all;  // ratio < th_all
        std::vector<unsigned char> is_good;            // 1 iff also ratio < th_good
    };
    // match_graph_init[idx1] = partner list, as produced by InitialMatchingGraph (initial_matching_graph.h:64).
    bool MatchPairs(const std::vector<std::vector<int>> &match_graph_init, std::vector<std::vector<PairMatches>> &out,
                    float th_good = 0.6f, float th_all = 0.85f, bool mutual = false, int th_reject = 20);
    // Guided re-matching of verified pairs (msfm_match_pairs_guided, GUIDED-SPEC in msfm_match.h): MatchPairs with every
    // row's two nearest neighbours searched only among the keypoints within th_epipolar pixels of the pair's epipolar
    // geometry.  F[k] belongs to the k-th pair of match_graph_init in order (row-major, p2^T F p1 = 0 for a keypoint p1 of
    // idx1 and p2 of idx2: what msfm_geo_verify returns); keypoints[idx] holds one keypoint per descriptor row of image
    // idx, in the centred coordinates of the feature files.
    bool MatchPairsGuided(const std::vector<std::vector<int>> &match_graph_init, const std::vector<std::array<double, 9>> &F,
                          const std::vector<std::vector<cv::KeyPoint>> &keypoints, float th_epipolar,
                          std::vector<std::vector<PairMatches>> &out, float th_good = 0.6f, float th_all = 0.85f,
                          bool mutual = false, int th_reject = 20);
    // Homography-guided re-matching (msfm_match_pairs_guided_homography, HOMOG-SPEC in msfm_match.h): MatchPairs with every
    // row's two nearest neighbours searched only among the keypoints of idx1 that H carries to within th_transfer pixels
    // of the row's keypoint.  H[k] belongs to the k-th pair of match_graph_init in order (row-major, p2 ~ H p1 for a
    // keypoint p1 of idx1 and p2 of idx2: what msfm_geo_homography returns); keypoints as in MatchPairsGuided.
    bool MatchPairsGuidedHomography(const std::vector<std::vector<int>> &match_graph_init, const std::vector<std::array<double, 9>> &H,
                                    const std::vector<std::vector<cv::KeyPoint>> &keypoints, float th_transfer,
                                    std::vector<std::vector<PairMatches>> &out, float th_good = 0.6f, float th_all = 0.85f,
                                    bool mutual = false, int th_reject = 20);

private:
    struct Guide {  // the gate of MatchPairsGuided (epipolar, M = F) or MatchPairsGuidedHomography (homography, M = H)
        enum Kind { epipolar, homography } kind;
        const std::vector<std::array<double, 9>> *M;
        const std::vector<std::vector<cv::KeyPoint>> *keypoints;
        float th;
    };
    bool Match(const std::vector<std::vector<int>> &match_graph_init, const Guide *guide, std::vector<std::vector<PairMatches>> &out,
               float th_good, float th_all, bool mutual, int th_reject);
    msfm_ctx *ctx_ = nullptr;
    float scale_;
    std::vector<int> rows_;
    std::string err_;
};

}  // namespace objectsfm
