// odometry.hpp — extension (not a reference name): SlamNode::process_frame (slam_node.cpp:118-175) as one call per
// frame over the streaming session of the C ABI (sb_odom_*).  The previous frame's cloud, index and normals stay on the
// device; the frame is uploaded once.  Results come back as the reference's types (ICPResult, Transformation,
// LoopClosureResult), and frames can go to an existing LoopClosureDetector and an existing Map, which must outlive the
// session.
#pragma once
#include <memory>
#include <vector>

#include "icp.hpp"
#include "loop_closure.hpp"
#include "map.hpp"

namespace slam {
namespace b200 {

struct OdometryConfig {
    double voxel_size = 0.5;     // slam_node voxel_size (<= 0: no voxel grid)
    int min_points = 1000;       // slam_node.hpp:29: frames with fewer rows after the voxel grid are skipped
    double max_error = 1.0;      // slam_node.cpp:139-140
    ICPConfig icp;
    Transformation initial_pose = Transformation::identity();
};

struct OdometryFrame {
    enum State { FIRST = SB_ODOM_FIRST, REGISTERED = SB_ODOM_REGISTERED, SKIPPED = SB_ODOM_SKIPPED };
    int frame_idx = 0;
    State state = FIRST;
    PointCloud cloud;            // the downsampled frame (sensor frame): the node's current_cloud
    Transformation pose;         // the frame's pose after the chain step
    ICPResult icp;               // state == REGISTERED
    std::vector<float> world_f32;                // PointCloud2 payload of publish_current_scan (x, y, z per row)
    std::vector<LoopClosureResult> loops;        // detect = true
};

class Odometry {
public:
    explicit Odometry(const OdometryConfig& config = OdometryConfig(), LoopClosureDetector* loop = nullptr,
                      Map* map = nullptr)
        : loop_(loop), map_(map) {
        sb_odom_config c;
        sb_default_odom_config(&c);
        c.voxel = config.voxel_size;
        c.min_points = config.min_points;
        c.max_error = config.max_error;
        c.icp.max_iterations = config.icp.max_iterations;
        c.icp.tolerance = config.icp.tolerance;
        c.icp.min_error = config.icp.min_error;
        config.icp.initial_transform.to_row_major(c.icp.initial_transform);
        config.initial_pose.to_row_major(c.initial_pose);
        sb_odom* o = nullptr;
        check(sb_odom_create2(context(), &c, loop ? loop->handle() : nullptr, map ? map->handle() : nullptr, &o),
              "Odometry");
        odom_ = std::shared_ptr<sb_odom>(o, [](sb_odom* p) { sb_odom_free(p); });
    }

    void reserve(size_t max_raw_rows) { check(sb_odom_reserve(odom_.get(), (int64_t)max_raw_rows), "Odometry::reserve"); }
    void setPose(const Transformation& pose) {   // slam_node.cpp:177-185: continue from an optimised pose
        double p[16];
        pose.to_row_major(p);
        check(sb_odom_set_pose(odom_.get(), p), "Odometry::setPose");
    }
    Transformation pose() const {
        double p[16];
        check(sb_odom_get_pose(odom_.get(), p), "Odometry::pose");
        return Transformation::from_row_major(p);
    }

    // One scan (raw rows).  add_frame: LoopClosureDetector::addFrame of the downsampled frame (slam_node.cpp:159);
    // detect: its detect() right after (slam_node.cpp:160-167).  Both need the detector given at construction.
    // add_map: the frame goes to the map given at construction (a skipped frame as an entry with no rows).
    OdometryFrame push(const PointCloud& scan, int frame_idx, bool add_frame = true, bool detect = false,
                       bool add_map = true) {
        const int64_t n = (int64_t)scan.size();
        const int flags = (add_frame && loop_ ? SB_ODOM_ADD_FRAME : 0) | (detect ? SB_ODOM_DETECT : 0) |
                          (add_map && map_ ? SB_ODOM_ADD_MAP : 0);
        PointCloud::Matrix cloud(n, 3);
        std::vector<float> world((size_t)(3 * (n > 0 ? n : 1)));
        std::vector<sb_loop_result> raw((size_t)max_loops_);
        sb_odom_frame f;
        check(sb_odom_push(odom_.get(), scan.points().data(), n, frame_idx, flags, &f, cloud.data(), world.data(), nullptr,
                           raw.data(), max_loops_),
              "Odometry::push");
        OdometryFrame out;
        out.frame_idx = f.frame_idx;
        out.state = (OdometryFrame::State)f.state;
        PointCloud::Matrix rows(f.n_points, 3);
        for (int64_t i = 0; i < 3 * f.n_points; ++i) rows.data()[i] = cloud.data()[i];
        out.cloud = PointCloud(std::move(rows));
        out.pose = Transformation::from_row_major(f.pose);
        if (f.state == SB_ODOM_REGISTERED) {
            out.icp.transformation = Transformation::from_row_major(f.icp.transformation);
            out.icp.converged = f.icp.converged != 0;
            out.icp.num_iterations = f.icp.num_iterations;
            out.icp.error_history.assign(f.icp.error_history, f.icp.error_history + f.icp.history_len);
            out.icp.final_error = f.icp.final_error;
        }
        if (f.state != SB_ODOM_SKIPPED) out.world_f32.assign(world.begin(), world.begin() + 3 * f.n_points);
        for (int i = 0; i < f.n_loops && i < max_loops_; ++i) {
            LoopClosureResult r;
            r.query_frame = raw[(size_t)i].query_frame;
            r.match_frame = raw[(size_t)i].match_frame;
            r.transform = Transformation::from_row_major(raw[(size_t)i].transform);
            r.scan_context_distance = raw[(size_t)i].scan_context_distance;
            r.icp_fitness = raw[(size_t)i].icp_fitness;
            out.loops.push_back(r);
        }
        return out;
    }

private:
    LoopClosureDetector* loop_;
    Map* map_;
    std::shared_ptr<sb_odom> odom_;
    static constexpr int max_loops_ = 64;   // accepted loops returned per frame (the node's config accepts 3)
};

}  // namespace b200
}  // namespace slam
