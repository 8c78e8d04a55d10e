// loop_closure.hpp — mirror of slam_viz/include/slam_viz/core/loop_closure.hpp:14-149.
// The descriptor database and the cloud copies live in device memory (csrc/loop.cu).
#pragma once
#include <algorithm>
#include <memory>
#include <vector>

#include "icp.hpp"
#include "scan_context.hpp"

namespace slam {

struct LoopClosureConfig {  // loop_closure.hpp:14-19
    int frame_gap = 50;
    double sc_distance_threshold = 0.25;
    double icp_fitness_threshold = 0.3;
    int max_candidates = 3;
};

struct LoopClosureResult {  // loop_closure.hpp:25-31
    int query_frame;
    int match_frame;
    Transformation transform;
    double scan_context_distance;
    double icp_fitness;
};

class LoopClosureDetector {
public:
    explicit LoopClosureDetector(const LoopClosureConfig& config = LoopClosureConfig()) : config_(config) {
        sb_loop_config c;
        sb_default_loop_config(&c);  // loop ICP: 30 iterations, 1e-6 (loop_closure.hpp:105-107), normals k = 20
        c.frame_gap = config.frame_gap;
        c.sc_distance_threshold = config.sc_distance_threshold;
        c.icp_fitness_threshold = config.icp_fitness_threshold;
        c.max_candidates = config.max_candidates;
        sb_loop* L = nullptr;
        b200::check(sb_loop_create(b200::context(), &c, 0, 1, &L), "LoopClosureDetector");
        loop_ = std::shared_ptr<sb_loop>(L, [](sb_loop* p) { sb_loop_free(p); });
    }

    void addFrame(const PointCloud::Matrix& cloud, int frame_idx) {  // loop_closure.hpp:53-59
        b200::check(sb_loop_add_frame(loop_.get(), cloud.data(), (int64_t)cloud.rows(), frame_idx), "addFrame");
    }

    std::vector<LoopClosureResult> detect() {  // loop_closure.hpp:66-126
        int cap = config_.max_candidates > 0 ? config_.max_candidates : 0;
        std::vector<sb_loop_result> raw((size_t)(cap > 0 ? cap : 1));
        int32_t count = 0;
        b200::check(sb_loop_detect(loop_.get(), raw.data(), cap, &count), "detect");
        std::vector<LoopClosureResult> out;
        for (int i = 0; i < count && i < cap; ++i) out.push_back(result(raw[i]));
        return out;
    }

    size_t size() const { return (size_t)sb_loop_size(loop_.get()); }                // loop_closure.hpp:131
    void clear() { b200::check(sb_loop_clear(loop_.get()), "clear"); }               // loop_closure.hpp:136-141
    // extension: size the device pools for a known sequence (frames, total downsampled rows) before streaming
    void reserve(size_t frames, size_t total_rows) {
        b200::check(sb_loop_reserve(loop_.get(), (int64_t)frames, (int64_t)total_rows), "reserve");
    }
    // extension: addFrame for every cloud of a recorded sequence in one call (same state as one addFrame per cloud)
    void addFrames(const std::vector<PointCloud::Matrix>& clouds, const std::vector<int>& frame_idx) {
        if (clouds.size() != frame_idx.size()) b200::check(SB_ERR_INVALID_ARG, "addFrames: one frame index per cloud");
        std::vector<int64_t> off(1, 0);
        for (const auto& c : clouds) off.push_back(off.back() + (int64_t)c.rows());
        std::vector<double> xyz((size_t)off.back() * 3);
        for (size_t f = 0; f < clouds.size(); ++f)
            std::copy(clouds[f].data(), clouds[f].data() + 3 * clouds[f].rows(), xyz.begin() + 3 * off[f]);
        std::vector<int32_t> fi(frame_idx.begin(), frame_idx.end());
        b200::check(sb_loop_add_frames(loop_.get(), xyz.data(), off.data(), (int32_t)clouds.size(), fi.data(), nullptr),
                    "addFrames");
    }
    // extension: detect() as it would have answered right after each listed entry (strictly ascending) was added
    std::vector<std::vector<LoopClosureResult>> detectBatch(const std::vector<int>& query_entries) {
        const int cap = config_.max_candidates > 0 ? config_.max_candidates : 0;
        const size_t n = query_entries.size();
        std::vector<int32_t> q(query_entries.begin(), query_entries.end()), count(n > 0 ? n : 1, 0);
        std::vector<sb_loop_result> raw(n * (size_t)cap > 0 ? n * (size_t)cap : 1);
        b200::check(sb_loop_detect_batch(loop_.get(), q.data(), (int32_t)n, raw.data(), count.data()), "detectBatch");
        std::vector<std::vector<LoopClosureResult>> out(n);
        for (size_t i = 0; i < n; ++i)
            for (int j = 0; j < count[i]; ++j) out[i].push_back(result(raw[i * (size_t)cap + j]));
        return out;
    }

    // extension: the underlying detector (b200::Odometry adds frames to it and runs its detect())
    sb_loop* handle() const { return loop_.get(); }

private:
    static LoopClosureResult result(const sb_loop_result& raw) {
        LoopClosureResult r;
        r.query_frame = raw.query_frame;
        r.match_frame = raw.match_frame;
        r.transform = Transformation::from_row_major(raw.transform);
        r.scan_context_distance = raw.scan_context_distance;
        r.icp_fitness = raw.icp_fitness;
        return r;
    }

    LoopClosureConfig config_;
    std::shared_ptr<sb_loop> loop_;
};

}  // namespace slam
