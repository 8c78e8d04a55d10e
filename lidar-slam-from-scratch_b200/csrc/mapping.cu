// mapping.cu — the data-parallel steps that follow the registration path in slam_node.cpp (SURVEY.md 8f N2/N3):
//   world-frame clouds      world = cloud * R^T + t           slam_viz/src/ros/slam_node.cpp:147, 189, 201-203
//   occupancy cells         height / range filter + floor(x / resolution) cell set   slam_node.cpp:211-229
//   global map              all clouds in the world frame, voxel grid at 2 * voxel_size     slam_node.cpp:196-209, 235-238
//   PointCloud2 payload     float32 x, y, z records of what is published                      slam_node.cpp:299-322
// The cell set is an unordered_set in the reference; here it comes out sorted by (x, y).  The global map reuses the
// voxel grid of voxel.cu (world coordinates are arbitrary doubles: the sort-based path answers, bit-exact).
#include "common.cuh"

namespace sb {

// out = p * R^T + t with the association of Transformation::apply (types.hpp:110-115)
__global__ void __launch_bounds__(256) k_transform(const double* __restrict__ xyz, const i64* __restrict__ off,
                                                   int n_clouds, const double* __restrict__ poses, i64 n,
                                                   double* __restrict__ out) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double* T = poses + 16 * cloud_of(off, n_clouds, i);
    const double x = xyz[3 * i], y = xyz[3 * i + 1], z = xyz[3 * i + 2];
#pragma unroll
    for (int a = 0; a < 3; ++a) out[3 * i + a] = apply_row(T, a, x, y, z);
}

// update_occupancy_grid (slam_node.cpp:211-221) for world-frame rows: key = biased (x, y) cell, ~0 if filtered out
__global__ void __launch_bounds__(256) k_occ_keys(const double* __restrict__ world, const i64* __restrict__ off,
                                                  int n_clouds, const double* __restrict__ poses, i64 n, double res,
                                                  double hmin, double hmax, double max_range, u64* __restrict__ keys,
                                                  uint32_t* __restrict__ vals, int* __restrict__ flags) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double* T = poses + 16 * cloud_of(off, n_clouds, i);
    bool out_of_range = false;
    keys[i] = occ_key(world[3 * i], world[3 * i + 1], world[3 * i + 2], T[3], T[7], res, hmin, hmax, max_range,
                      &out_of_range);
    if (out_of_range) atomicOr(flags, FLAG_KEY_RANGE);
    vals[i] = (uint32_t)i;
}

__global__ void __launch_bounds__(256) k_occ_flag(const u64* __restrict__ keys, i64 n, uint32_t* __restrict__ flag) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    flag[i] = (keys[i] != ~0ull && (i == 0 || keys[i] != keys[i - 1])) ? 1u : 0u;
}

__global__ void __launch_bounds__(256) k_occ_emit(const u64* __restrict__ keys, const uint32_t* __restrict__ flag,
                                                  const uint32_t* __restrict__ pos, i64 n, i64 capacity,
                                                  int* __restrict__ cells) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !flag[i] || (i64)pos[i] >= capacity) return;
    const u64 k = keys[i];
    cells[2 * (i64)pos[i]] = (int)((uint32_t)(k >> 32) ^ 0x80000000u);
    cells[2 * (i64)pos[i] + 1] = (int)((uint32_t)k ^ 0x80000000u);
}

// eigen_to_pointcloud2 (slam_node.cpp:299-322): the PointCloud2 payload is x, y, z as float32, point_step 12 —
// static_cast<float> of every coordinate (round to nearest even)
__global__ void __launch_bounds__(256) k_pack_f32(const double* __restrict__ in, i64 n3, float* __restrict__ out) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n3) out[i] = __double2float_rn(in[i]);
}

int pack_f32_dev(Ctx* ctx, const double* d_in, i64 n_rows, float* d_out) {
    if (n_rows > 0) SB_LAUNCH(ctx, k_pack_f32, ceil_div(3 * n_rows, 256), 256, 0, d_in, 3 * n_rows, d_out);
    return SB_OK;
}

int transform_clouds_dev(Ctx* ctx, const double* d_xyz, const i64* d_off, int n_clouds, const double* d_poses, i64 n,
                         double* d_out) {
    if (n > 0) SB_LAUNCH(ctx, k_transform, ceil_div(n, 256), 256, 0, d_xyz, d_off, n_clouds, d_poses, n, d_out);
    return SB_OK;
}

// unique occupancy cells of world-frame rows, ascending (x, y); *count = number found (may exceed capacity)
int occupancy_cells_dev(Ctx* ctx, const double* d_world, const i64* d_off, int n_clouds, const double* d_poses, i64 n,
                        const sb_grid_config* cfg, int* d_cells, i64 capacity, i64* count) {
    *count = 0;
    if (n <= 0) return SB_OK;
    if (n >= (i64)0xffffffffLL) return fail(ctx, SB_ERR_RANGE, "occupancy: more than 2^32-1 rows in one call");
    u64 *ka, *kb, *ks;
    uint32_t *va, *vb, *vs, *d_flag, *d_pos, *d_total;
    SB_TRY(arena_get(ctx, (size_t)n, &ka));
    SB_TRY(arena_get(ctx, (size_t)n, &kb));
    SB_TRY(arena_get(ctx, (size_t)n, &va));
    SB_TRY(arena_get(ctx, (size_t)n, &vb));
    SB_TRY(arena_get(ctx, (size_t)n, &d_flag));
    SB_TRY(arena_get(ctx, (size_t)n, &d_pos));
    SB_TRY(arena_get(ctx, 1, &d_total));
    SB_CUDA(ctx, cudaMemsetAsync(ctx->d_flags, 0, sizeof(int), ctx->stream));
    SB_LAUNCH(ctx, k_occ_keys, ceil_div(n, 256), 256, 0, d_world, d_off, n_clouds, d_poses, n, cfg->resolution,
              cfg->height_min, cfg->height_max, cfg->max_range, ka, va, ctx->d_flags);
    i64 seg[2] = {0, n};
    SB_TRY(segmented_sort_pairs(ctx, ka, kb, va, vb, seg, 1, 64, &ks, &vs));
    SB_LAUNCH(ctx, k_occ_flag, ceil_div(n, 256), 256, 0, ks, n, d_flag);
    SB_TRY(exclusive_scan_u32(ctx, d_flag, d_pos, n, d_total));
    SB_LAUNCH(ctx, k_occ_emit, ceil_div(n, 256), 256, 0, ks, d_flag, d_pos, n, capacity, d_cells);
    uint32_t total = 0;
    int flags = 0;
    SB_CUDA(ctx, cudaMemcpyAsync(&total, d_total, sizeof(total), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(ctx, cudaMemcpyAsync(&flags, ctx->d_flags, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (flags & FLAG_KEY_RANGE) return fail(ctx, SB_ERR_RANGE, "occupancy: a cell index does not fit an int");
    *count = (i64)total;
    return SB_OK;
}

}  // namespace sb
