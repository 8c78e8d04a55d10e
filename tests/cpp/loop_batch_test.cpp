// loop_batch_test.cpp — the mirror's sequence extensions of LoopClosureDetector (addFrames, detectBatch) against the
// reference-shaped per-frame use (addFrame + detect() after every query frame, slam_node.cpp:159-167).  Needs a B200;
// built and run by tests/test_loop_batch.py (-m gpu).
#include <cstdio>
#include <cstring>
#include <vector>

#include "slam_viz/core/file_utils.hpp"
#include "slam_viz/core/loop_closure.hpp"

extern "C" {
// synth/libsynth.so
int syn_scene(unsigned long long seed, int n_boxes, float half_extent, int path_kind, float radius, float corridor_half,
              float sensor_height, float* boxes6);
long long syn_scan(int beams, int azimuth_steps, float elev_top_deg, float elev_bot_deg, float max_range,
                   float noise_sigma, float sensor_height, const float* boxes6, int n_boxes, double x, double y,
                   double yaw, unsigned long long noise_seed, double* out_xyz, int n_threads);
}

static int failures = 0;
#define CHECK(cond)                                                        \
    do {                                                                   \
        if (!(cond)) {                                                     \
            std::printf("FAIL %s:%d  %s\n", __FILE__, __LINE__, #cond);    \
            ++failures;                                                    \
        }                                                                  \
    } while (0)

using Matrix = slam::PointCloud::Matrix;

static Matrix scan(const std::vector<float>& boxes, double x, double y, double yaw, unsigned long long seed) {
    const int beams = 16, az = 360;
    std::vector<double> buf((size_t)3 * beams * az);
    long long n = syn_scan(beams, az, 2.0f, -24.8f, 120.0f, 0.02f, 1.73f, boxes.data(), (int)boxes.size() / 6, x, y, yaw,
                           seed, buf.data(), 4);
    Matrix m((long)n, 3);
    for (long long i = 0; i < 3 * n; ++i) m.data()[i] = buf[(size_t)i];
    return slam::voxel_downsample(m, 0.5);
}

int main() {
    std::vector<float> boxes((size_t)6 * 400);
    int nb = syn_scene(1, 400, 90.0f, 0, 0.0f, 6.0f, 1.73f, boxes.data());
    boxes.resize((size_t)6 * nb);
    // a 12 m back-and-forth path: every place is revisited after the frame gap
    std::vector<Matrix> clouds;
    std::vector<int> frames;
    for (int i = 0; i < 40; ++i) {
        const int k = i % 24;
        const double x = k < 12 ? (double)k : (double)(24 - k);
        clouds.push_back(scan(boxes, x, 0.02 * (i % 3), 0.0, 500 + i));
        frames.push_back(i);
    }
    slam::LoopClosureConfig cfg;
    cfg.frame_gap = 8;
    cfg.sc_distance_threshold = 0.5;
    cfg.icp_fitness_threshold = 0.5;
    cfg.max_candidates = 2;
    slam::LoopClosureDetector one(cfg), bulk(cfg);
    std::vector<int> queries;
    std::vector<std::vector<slam::LoopClosureResult>> want;
    for (int i = 0; i < (int)clouds.size(); ++i) {
        one.addFrame(clouds[i], frames[i]);
        if (i > 8 && i % 3 == 0) {
            queries.push_back(i);
            want.push_back(one.detect());
        }
    }
    bulk.addFrames(clouds, frames);
    CHECK(bulk.size() == one.size());
    auto got = bulk.detectBatch(queries);
    CHECK(got.size() == want.size());
    int accepted = 0;
    for (size_t q = 0; q < got.size() && q < want.size(); ++q) {
        CHECK(got[q].size() == want[q].size());
        for (size_t j = 0; j < got[q].size() && j < want[q].size(); ++j) {
            const auto &a = got[q][j], &b = want[q][j];
            CHECK(a.query_frame == b.query_frame && a.query_frame == queries[q]);
            CHECK(a.match_frame == b.match_frame);
            CHECK(a.scan_context_distance == b.scan_context_distance);
            CHECK(a.icp_fitness == b.icp_fitness);
            CHECK(std::memcmp(a.transform.matrix().data(), b.transform.matrix().data(), 16 * sizeof(double)) == 0);
            ++accepted;
        }
    }
    CHECK(accepted > 0);
    // the detector is not modified: the newest entry still answers as before
    auto last = bulk.detect(), last_one = one.detect();
    CHECK(last.size() == last_one.size());
    std::printf("%zu queries, %d accepted loops\n", queries.size(), accepted);
    if (failures) {
        std::printf("%d checks failed\n", failures);
        return 1;
    }
    std::printf("all checks passed\n");
    return 0;
}
