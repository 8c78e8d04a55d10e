// map.hpp — extension (not a reference name): the node's map state (slam_node.cpp:147-157, 177-238) over the
// device-resident map of the C ABI (sb_map_*).  The keyframe clouds (sensor frame), their poses and the occupancy cell
// set stay on the device; after a pose-graph optimisation setPoses uploads only the poses and the cells, the global map
// and the world-frame window are rebuilt from the resident clouds.  Every result has the bits of the stateless calls
// (sb_occupancy_cells, sb_global_map[_f32], sb_transform_clouds_f32) on the same clouds and poses.
#pragma once
#include <memory>
#include <utility>
#include <vector>

#include "backend.hpp"
#include "types.hpp"

namespace slam {
namespace b200 {

struct MapConfig {               // slam::OccupancyGridConfig, slam_node.hpp:35-40
    double resolution = 0.2;
    double height_min = 0.3;
    double height_max = 2.0;
    double max_range = 40.0;
};

class Map {
public:
    explicit Map(const MapConfig& config = MapConfig()) {
        sb_grid_config g;
        g.resolution = config.resolution;
        g.height_min = config.height_min;
        g.height_max = config.height_max;
        g.max_range = config.max_range;
        sb_map* m = nullptr;
        check(sb_map_create(context(), &g, &m), "Map");
        map_ = std::shared_ptr<sb_map>(m, [](sb_map* p) { sb_map_free(p); });
    }

    sb_map* handle() const { return map_.get(); }
    void reserve(size_t n_entries, size_t total_rows, size_t n_cells) {
        check(sb_map_reserve(map_.get(), (int64_t)n_entries, (int64_t)total_rows, (int64_t)n_cells), "Map::reserve");
    }
    size_t size() const { return (size_t)sb_map_size(map_.get()); }
    size_t rows() const { return (size_t)sb_map_rows(map_.get()); }
    void clear() { check(sb_map_clear(map_.get()), "Map::clear"); }

    // one keyframe: its downsampled sensor-frame cloud and pose (update_occupancy_grid, slam_node.cpp:152, 211-221)
    void add(const PointCloud::Matrix& cloud, const Transformation& pose) {
        double p[16];
        pose.to_row_major(p);
        check(sb_map_add(map_.get(), cloud.data(), (int64_t)cloud.rows(), p), "Map::add");
    }
    // poses of entries [first, first + poses.size()) (PoseGraph::getAllPoses after optimize, slam_node.cpp:177-185)
    void setPoses(const std::vector<Transformation>& poses, int first = 0) {
        std::vector<double> raw(16 * poses.size());
        for (size_t i = 0; i < poses.size(); ++i) poses[i].to_row_major(raw.data() + 16 * i);
        check(sb_map_set_poses(map_.get(), first, (int32_t)poses.size(), raw.data()), "Map::setPoses");
    }
    std::vector<Transformation> poses() const {
        const int n = (int)size();
        std::vector<double> raw(16 * (size_t)(n > 0 ? n : 1));
        check(sb_map_get_poses(map_.get(), 0, n, raw.data()), "Map::poses");
        std::vector<Transformation> out;
        for (int i = 0; i < n; ++i) out.push_back(Transformation::from_row_major(raw.data() + 16 * (size_t)i));
        return out;
    }

    // the occupancy cells (x, y), ascending
    std::vector<std::pair<int, int>> occupancyCells() const {
        int64_t count = 0;
        check(sb_map_occupancy_cells(map_.get(), nullptr, 0, &count), "Map::occupancyCells");
        std::vector<int32_t> raw(2 * (size_t)(count > 0 ? count : 1));
        check(sb_map_occupancy_cells(map_.get(), raw.data(), count, &count), "Map::occupancyCells");
        std::vector<std::pair<int, int>> out((size_t)count);
        for (int64_t i = 0; i < count; ++i) out[(size_t)i] = {raw[2 * (size_t)i], raw[2 * (size_t)i + 1]};
        return out;
    }
    // entries [first, first + n) in the world frame as PointCloud2 float32 records (x, y, z per row)
    std::vector<float> worldF32(int first, int n) const {
        std::vector<float> out(3 * (rows() > 0 ? rows() : 1));
        int64_t m = 0;
        check(sb_map_world_f32(map_.get(), first, n, out.data(), &m), "Map::worldF32");
        out.resize(3 * (size_t)m);
        return out;
    }
    // all entries in the world frame, voxel grid at `voxel` (the node publishes 2 * voxel_size)
    PointCloud globalMap(double voxel) const {
        PointCloud::Matrix out((long)(rows() > 0 ? rows() : 1), 3);
        int64_t m = 0;
        check(sb_map_global(map_.get(), voxel, out.data(), &m), "Map::globalMap");
        PointCloud::Matrix rows_out((long)m, 3);
        for (int64_t i = 0; i < 3 * m; ++i) rows_out.data()[i] = out.data()[i];
        return PointCloud(std::move(rows_out));
    }
    std::vector<float> globalMapF32(double voxel) const {
        std::vector<float> out(3 * (rows() > 0 ? rows() : 1));
        int64_t m = 0;
        check(sb_map_global_f32(map_.get(), voxel, out.data(), &m), "Map::globalMapF32");
        out.resize(3 * (size_t)m);
        return out;
    }

private:
    std::shared_ptr<sb_map> map_;
};

}  // namespace b200
}  // namespace slam
