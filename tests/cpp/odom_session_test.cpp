// odom_session_test.cpp — the mirror's streaming session (slam::b200::Odometry, odometry.hpp) against the node's
// per-call use of the mirror (voxel_downsample, icp_point_to_plane, the pose product, LoopClosureDetector::addFrame,
// slam_node.cpp:118-159) over 20 frames: the same rows, ICP results, poses, world-frame float32 clouds and detector.
// Needs a B200; built and run by tests/test_odom_session.py.
#include <cstdio>
#include <cstring>
#include <vector>

#include "slam_viz/core/file_utils.hpp"
#include "slam_viz/core/odometry.hpp"

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

static Matrix raw_scan(const std::vector<float>& boxes, double x, double y, double yaw, unsigned long long seed) {
    const int beams = 16, az = 360;
    std::vector<double> buf((size_t)3 * beams * az);
    long long n = syn_scan(beams, az, 2.0f, -24.8f, 120.0f, 0.02f, 1.73f, boxes.data(), (int)boxes.size() / 6, x, y, yaw,
                           seed, buf.data(), 4);
    Matrix m((long)n, 3);
    for (long long i = 0; i < 3 * n; ++i) m.data()[i] = buf[(size_t)i];
    return m;
}

static bool same(const double* a, const double* b, size_t n) { return std::memcmp(a, b, n * sizeof(double)) == 0; }

int main() {
    std::vector<float> boxes((size_t)6 * 400);
    int nb = syn_scene(1, 400, 90.0f, 0, 0.0f, 6.0f, 1.73f, boxes.data());
    boxes.resize((size_t)6 * nb);
    const int frames = 20;
    slam::LoopClosureConfig lc;
    lc.frame_gap = 8;
    slam::LoopClosureDetector det_session(lc), det_calls(lc);
    slam::b200::OdometryConfig oc;
    oc.min_points = 100;
    slam::b200::Odometry odom(oc, &det_session);
    slam::PointCloud prev;
    slam::Transformation pose;
    int registered = 0;
    for (int i = 0; i < frames; ++i) {
        Matrix raw = raw_scan(boxes, 0.5 * i, 0.01 * (i % 3), 0.01 * i, 700 + i);
        slam::b200::OdometryFrame f = odom.push(slam::PointCloud(raw), i, true, false);
        // the node's per-call path
        slam::PointCloud cur(slam::voxel_downsample(raw, oc.voxel_size));
        CHECK(f.frame_idx == i);
        CHECK((size_t)f.cloud.size() == cur.size());
        CHECK(f.cloud.size() == cur.size() && same(f.cloud.points().data(), cur.points().data(), 3 * cur.size()));
        if (i == 0) {
            CHECK(f.state == slam::b200::OdometryFrame::FIRST);
        } else {
            CHECK(f.state == slam::b200::OdometryFrame::REGISTERED);
            slam::ICPResult r = slam::icp_point_to_plane(cur, prev);
            CHECK(f.icp.converged == r.converged);
            CHECK(f.icp.num_iterations == r.num_iterations);
            CHECK(f.icp.final_error == r.final_error);
            CHECK(f.icp.error_history == r.error_history);
            CHECK(same(f.icp.transformation.matrix().data(), r.transformation.matrix().data(), 16));
            const bool keep = r.converged && !(r.final_error > oc.max_error);   // slam_node.cpp:139-140
            pose = pose * (keep ? r.transformation : slam::Transformation::identity());
            ++registered;
        }
        CHECK(same(f.pose.matrix().data(), pose.matrix().data(), 16));
        slam::PointCloud world = pose.apply(cur);                               // slam_node.cpp:147
        bool wsame = f.world_f32.size() == 3 * world.size();
        for (size_t k = 0; wsame && k < 3 * world.size(); ++k) wsame = f.world_f32[k] == (float)world.points().data()[k];
        CHECK(wsame);
        det_calls.addFrame(cur.points(), i);
        prev = std::move(cur);
    }
    CHECK(det_session.size() == det_calls.size());
    auto a = det_session.detect(), b = det_calls.detect();
    CHECK(a.size() == b.size());
    for (size_t j = 0; j < a.size() && j < b.size(); ++j) {
        CHECK(a[j].match_frame == b[j].match_frame);
        CHECK(a[j].scan_context_distance == b[j].scan_context_distance);
    }
    CHECK(same(odom.pose().matrix().data(), pose.matrix().data(), 16));
    std::printf("%d frames, %d registered, %zu loops\n", frames, registered, a.size());
    if (failures) {
        std::printf("%d checks failed\n", failures);
        return 1;
    }
    std::printf("all checks passed\n");
    return 0;
}
