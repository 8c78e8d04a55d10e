// odom.cuh — what the streaming session's two push paths share: the session state, its buffer growth, the output-block
// layout and the epilogue's pose and row expressions.  odom.cu pushes one frame into one session; odom_many.cu pushes
// one frame into each of many sessions with one voxel grid, one index build and one ICP batch, and leaves every
// session exactly where the single push would.
#pragma once
#include <algorithm>

#include "common.cuh"

namespace sb {

// One frame's device state.  d_trees is the two-entry descriptor table of the ICP forest of the frame built in this
// slot: entry 0 = the previous frame's tree (target, copied from its slot), entry 1 = this frame's tree (source, and the
// next frame's target).
struct OdomSlot {
    double* xyz = nullptr;   // voxel-grid output (sized for the raw rows)
    i64 xyz_cap = 0;         // doubles
    TreeStore st;
    TreeDesc* d_trees = nullptr;
    TreeDesc tree;           // host mirror of entry 1 (the seed-grid fields are device-only)
};

// the device-to-host block of a frame: pose | Scan Context | downsampled rows (optional) | world float32 (optional)
static constexpr size_t OUT_DESC = 16 * sizeof(double);
static constexpr size_t OUT_ROWS = OUT_DESC + SB_SC_SIZE * sizeof(double);

#ifdef __CUDACC__
// Entry t (< 16) of the frame's pose: slam_node.cpp:139-147 on the device, the keep rule and the pose product of
// sb_odometry_poses (k ascending from 0.0, every * and + separately rounded).  res == nullptr (first frame): pose_in.
__device__ __forceinline__ double odom_pose_entry(const sb_icp_result* __restrict__ res, double max_error,
                                                  const double* __restrict__ pose_in, int t) {
    double v = pose_in[t];
    if (res) {
        const bool keep = res->status == SB_OK && res->converged && !(res->final_error > max_error);
        const int i = t >> 2, j = t & 3;
        double acc = 0.0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const double d = keep ? res->transformation[4 * k + j] : (k == j ? 1.0 : 0.0);
            acc = __dadd_rn(acc, __dmul_rn(pose_in[4 * i + k], d));
        }
        v = acc;
    }
    return v;
}

// Row r of a frame: the downsampled row copied out, and the row in the world frame with the expression of k_transform
// (apply_row) and static_cast<float> (eigen_to_pointcloud2, slam_node.cpp:299-322).
__device__ __forceinline__ void odom_row(const double* P, const double* __restrict__ xyz, i64 r, double* __restrict__ out_xyz,
                                         float* __restrict__ out_f32) {
    const double x = xyz[3 * r], y = xyz[3 * r + 1], z = xyz[3 * r + 2];
    if (out_xyz) { out_xyz[3 * r] = x; out_xyz[3 * r + 1] = y; out_xyz[3 * r + 2] = z; }
    if (out_f32)
#pragma unroll
        for (int a = 0; a < 3; ++a) out_f32[3 * r + a] = __double2float_rn(apply_row(P, a, x, y, z));
}
#endif

}  // namespace sb

struct sb_odom {
    sb::Ctx* ctx = nullptr;
    sb_odom_config cfg;
    sb_loop* loop = nullptr;
    sb_map* map = nullptr;      // SB_ODOM_ADD_MAP
    sb::OdomSlot slot[2];
    int prev = -1;              // slot of the previous (committed) frame; -1 before the first
    double pose[16];            // host copy of the committed pose
    double* d_pose = nullptr;   // 2 x 16: [pi] the committed pose, [1 - pi] written by the next frame's epilogue
    int pi = 0;
    char* d_raw = nullptr;      // raw rows of the frame as they arrive (fp64 or float32 records)
    sb::i64 raw_cap = 0;
    char* h_in = nullptr;       // pinned staging of pageable input rows
    sb::i64 h_in_cap = 0;
    char* d_out = nullptr;      // device-to-host block (OUT_*)
    sb::i64 d_out_cap = 0;
    char* h_out = nullptr;      // its pinned host copy
    sb::i64 h_out_cap = 0;
    std::vector<void*> retired, retired_host;   // outgrown buffers, freed with the session
};

namespace sb {

template <typename T>
inline int grow_dev(sb_odom* O, T** buf, i64* cap, i64 need) {
    if (need <= *cap) return SB_OK;
    i64 ncap = *cap > 0 ? *cap : need;
    while (ncap < need) ncap *= 2;
    T* nb = nullptr;
    SB_CUDA(O->ctx, cudaMalloc(&nb, sizeof(T) * (size_t)ncap));
    if (*buf) O->retired.push_back(*buf);
    *buf = nb;
    *cap = ncap;
    return SB_OK;
}

inline int grow_host(sb_odom* O, char** buf, i64* cap, i64 need) {
    if (need <= *cap) return SB_OK;
    i64 ncap = *cap > 0 ? *cap : need;
    while (ncap < need) ncap *= 2;
    char* nb = nullptr;
    SB_CUDA(O->ctx, cudaHostAlloc(&nb, (size_t)ncap, cudaHostAllocDefault));
    if (*buf) O->retired_host.push_back(*buf);
    *buf = nb;
    *cap = ncap;
    return SB_OK;
}

// room in slot S for a frame of `raw` input rows of which `pts` survive the voxel grid
inline int slot_reserve(sb_odom* O, OdomSlot& S, i64 raw, i64 pts) {
    SB_TRY(grow_dev(O, &S.xyz, &S.xyz_cap, 3 * std::max<i64>(raw, 1)));
    TreeStore& T = S.st;
    const int k = O->cfg.icp.normals_k;
    if (pts > T.cap_points) {
        i64 c = T.cap_points > 0 ? T.cap_points : pts;
        while (c < pts) c *= 2;
        i64 cap;   // the four per-point arrays share one capacity
        cap = T.cap_points; SB_TRY(grow_dev(O, &T.pts, &cap, c));
        cap = T.cap_points; SB_TRY(grow_dev(O, &T.pts32, &cap, c));
        cap = T.cap_points; SB_TRY(grow_dev(O, &T.normals, &cap, c));
        cap = T.cap_points * k; SB_TRY(grow_dev(O, &T.nbr, &cap, c * k));
        T.cap_points = c;
        T.cap_k = k;
    }
    i64 nb, ns;
    tree_store_need(std::max<i64>(pts, 1), &nb, &ns);
    SB_TRY(grow_dev(O, &T.grid, &T.cap_slots, ns));
    if (nb > T.cap_boxes) {
        i64 c = T.cap_boxes > 0 ? T.cap_boxes : nb;
        while (c < nb) c *= 2;
        i64 cap = 6 * T.cap_boxes;
        SB_TRY(grow_dev(O, &T.boxes, &cap, 6 * c));
        T.cap_boxes = c;
    }
    return SB_OK;
}

inline int out_reserve(sb_odom* O, i64 rows) {
    const i64 need = (i64)OUT_ROWS + 36 * std::max<i64>(rows, 1);
    SB_TRY(grow_dev(O, &O->d_out, &O->d_out_cap, need));
    return grow_host(O, &O->h_out, &O->h_out_cap, need);
}

}  // namespace sb
