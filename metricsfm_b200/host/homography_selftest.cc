// homography_selftest.cc — drives MatchGraphB200::MatchPairsGuidedHomography the way the fine matching graph would after
// msfm_geo_homography and prints the match lists so that tests/test_guided_homography.py can check them against the Python binding.
// Input: two float32 descriptor matrices (image 0 then image 1), their keypoints (xy of image 0 then image 1, float32),
// and H of the pair (image 0 -> image 1, index on image 0, queries = rows of image 1) as 9 float64; output: text on stdout.
#include <array>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "feature_matching_b200.h"

template <typename T>
static bool read_all(const char *path, std::vector<T> &v) {
    FILE *f = fopen(path, "rb");
    const bool ok = f && fread(v.data(), sizeof(T), v.size(), f) == v.size();
    if (f) fclose(f);
    if (!ok) fprintf(stderr, "cannot read %s\n", path);
    return ok;
}

int main(int argc, char **argv) {
    if (argc < 7) {
        fprintf(stderr, "usage: %s <desc.f32> <rows0> <rows1> <keypoints.f32> <H.f64> <th_transfer>\n", argv[0]);
        return 2;
    }
    const int n0 = atoi(argv[2]), n1 = atoi(argv[3]);
    const float th = (float)atof(argv[6]);
    std::vector<float> desc((size_t)(n0 + n1) * 128), xy((size_t)(n0 + n1) * 2);
    std::vector<std::array<double, 9>> H(1);
    std::vector<double> f9(9);
    if (!read_all(argv[1], desc) || !read_all(argv[4], xy) || !read_all(argv[5], f9)) return 2;
    for (int k = 0; k < 9; ++k) H[0][k] = f9[k];
    cv::Mat d0(n0, 128, CV_32FC1, desc.data()), d1(n1, 128, CV_32FC1, desc.data() + (size_t)n0 * 128);
    std::vector<std::vector<cv::KeyPoint>> kp(2);
    kp[0].resize(n0);
    kp[1].resize(n1);
    for (int i = 0; i < n0 + n1; ++i) {
        cv::KeyPoint &k = i < n0 ? kp[0][i] : kp[1][i - n0];
        k.pt.x = xy[2 * i];
        k.pt.y = xy[2 * i + 1];
    }

    objectsfm::MatchGraphB200 graph(0, 2, n0 + n1);
    if (!graph.ok() || !graph.AddImage(0, d0) || !graph.AddImage(1, d1)) {
        fprintf(stderr, "matcher: %s\n", graph.last_error().c_str());
        return 3;
    }
    const std::vector<std::vector<int>> init = {{1}, {}};
    for (int mutual = 0; mutual < 2; ++mutual) {
        std::vector<std::vector<objectsfm::MatchGraphB200::PairMatches>> out;
        const bool ok = graph.MatchPairsGuidedHomography(init, H, kp, th, out, 0.6f, 0.85f, mutual != 0);
        printf("MatchPairsGuidedHomography mutual %d ok %d\n", mutual, ok ? 1 : 0);
        if (!ok) {
            fprintf(stderr, "MatchPairsGuidedHomography: %s\n", graph.last_error().c_str());
            return 4;
        }
        const objectsfm::MatchGraphB200::PairMatches &pm = out[0][0];
        printf("pair ok %d n %zu\n", pm.ok ? 1 : 0, pm.matches_all.size());
        for (size_t k = 0; k < pm.matches_all.size(); ++k)
            printf("%d %d %d\n", pm.matches_all[k].first, pm.matches_all[k].second, (int)pm.is_good[k]);
    }
    return 0;
}
