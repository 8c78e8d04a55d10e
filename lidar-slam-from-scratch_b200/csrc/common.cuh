// common.cuh — shared host/device plumbing of libslam_b200.so (sm_100a only).
//
// One sb_ctx per (host thread, device): it owns the stream, a grow-only device workspace arena that is reset at
// the start of every C-ABI call, a pinned host staging buffer, the launch counter reported to bench.py and the
// cached ICP while-graph.  Nothing here falls back to the CPU: every failure becomes an sb_status.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdio>
#include <cstring>
#include <functional>
#include <string>
#include <utility>
#include <vector>

#include "../../include/slam_b200.h"

namespace sb {

typedef long long i64;
typedef unsigned long long u64;

struct Ctx;

// ---------------------------------------------------------------------------------------------------------------
// error handling: SB_CUDA(ctx, call) records the message and makes the enclosing function return SB_ERR_CUDA
// ---------------------------------------------------------------------------------------------------------------
int fail(Ctx* ctx, int status, const char* fmt, ...);

#define SB_CUDA(ctx, call)                                                                                    \
    do {                                                                                                      \
        cudaError_t e__ = (call);                                                                             \
        if (e__ != cudaSuccess)                                                                               \
            return sb::fail((ctx), SB_ERR_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #call,                  \
                            cudaGetErrorString(e__));                                                         \
    } while (0)

#define SB_TRY(expr)                  \
    do {                              \
        int s__ = (expr);             \
        if (s__ != SB_OK) return s__; \
    } while (0)

// ---------------------------------------------------------------------------------------------------------------
// Workspace arena: bump allocator over one cudaMalloc'd slab.  If a call needs more than the slab holds the
// overflow goes to individually cudaMalloc'd blocks that are freed at the next reset, and the slab is regrown to
// the high-water mark so that steady-state calls allocate nothing.
// ---------------------------------------------------------------------------------------------------------------
struct Arena {
    char* base = nullptr;
    size_t cap = 0, used = 0;
    size_t req = 0, high = 0;  // bytes currently handed out (slab + overflow) and their peak since the last reset
    std::vector<void*> overflow;
};
struct ArenaMark {
    size_t used, req;
};

struct Ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    // Small host tables (tile lists, offsets, descriptors) reach the device through a mapped pinned buffer and a copy
    // KERNEL, not through the copy engine: while a bulk upload is in flight the engine's queue is minutes of PCIe
    // time deep, and every small cudaMemcpyAsync of the stages running meanwhile would wait behind it.
    char* tbuf = nullptr;        // host address (cudaHostAllocMapped)
    char* tbuf_dev = nullptr;    // device address of the same buffer
    size_t tbuf_cap = 0, tbuf_used = 0;
    cudaStream_t copy_stream = nullptr;   // host-to-device chunks of the pipelined entry points (api.cu)
    cudaEvent_t copy_ev[2] = {nullptr, nullptr};
    Arena arena;
    char* pinned = nullptr;  // pinned host staging
    size_t pinned_cap = 0;
    i64 launches = 0;
    std::string err;
    // device flag word set by kernels on bad input (non-finite coordinates, voxel key overflow)
    int* d_flags = nullptr;
    // cached ICP loop graph (icp.cu)
    void* icp_graph = nullptr;
    // voxel.cu: slots of the per-cloud voxel hash table per input row (raised to 2 after a table overflowed),
    // SB_VOXEL_SORT=1 forces the sort-based path, and which path the last call took (1 hashed, 2 sorted)
    double vox_slots_per_point = 0.25;
    bool vox_force_sort = false;
    int vox_last_path = 0;
    // optional per-stage CUDA-event timing of the last pipeline call (bench.py's roofline figures)
    bool profiling = false;
    cudaEvent_t ev[128];
    int ev_stage[128];
    double ev_host[128];  // host steady_clock milliseconds at the same marks
    int n_ev = 0, ev_created = 0;
    // SB_PIPE_TRACE=1: named device-time marks on the main stream (trace_mark / trace_dump), a debugging aid
    std::vector<std::pair<const char*, cudaEvent_t>> trace;
    // icp.cu: pinned staging of the results of the batches enqueued since the last icp_reserve_results
    static constexpr int ICP_SLOTS = 256;
    sb_icp_result* h_icp_res = nullptr;
    size_t icp_res_cap = 0, icp_res_used = 0;
    int* h_icp_passes = nullptr;
    int icp_slots_used = 0;
    cudaStream_t icp_stream = nullptr;     // api.cu: ICP of the pairs whose scans have arrived, beside the next chunk's stages
    cudaEvent_t icp_ev = nullptr;
    unsigned knn_attr_done = 0;    // forest.cu: k_self_knn instantiations whose shared-memory limit has been raised
    i64 last_icp_iterations = 0;   // max history length of the last icp_batch (launches of k_icp_iter)
    i64 last_counts[4] = {0, 0, 0, 0};  // raw rows, downsampled rows, target rows, sum over pairs of n_src * passes
};

// stage ids for stage_mark / sb_ctx_stage_ms
enum { STAGE_H2D = 0, STAGE_VOXEL = 1, STAGE_SC = 2, STAGE_INDEX = 3, STAGE_NORMALS = 4, STAGE_ICP = 5, STAGE_D2H = 6,
       STAGE_COUNT = 7, STAGE_END = -1 };
void stage_mark(Ctx* ctx, int stage);
void trace_mark(Ctx* ctx, const char* name);
void trace_dump(Ctx* ctx);

int arena_reset(Ctx* ctx);
// Temporaries of one pipeline stage: everything allocated after arena_mark is handed back by arena_release.  Safe
// because all work is ordered on the context's stream (later kernels run after the ones that used the memory).
ArenaMark arena_mark(Ctx* ctx);
void arena_release(Ctx* ctx, ArenaMark m);
int arena_alloc(Ctx* ctx, size_t bytes, void** out);
int pinned_reserve(Ctx* ctx, size_t bytes);
// host table -> device memory (4-byte granularity), ordered on the context's stream; h_src may be reused on return
int table_upload(Ctx* ctx, void* d_dst, const void* h_src, size_t bytes);

template <typename T>
inline int arena_get(Ctx* ctx, size_t count, T** out) {
    void* p = nullptr;
    int s = arena_alloc(ctx, count * sizeof(T), &p);
    *out = static_cast<T*>(p);
    return s;
}

inline int ceil_div(i64 a, i64 b) { return (int)((a + b - 1) / b); }

#define SB_LAUNCH(ctx, kernel, grid, block, smem, ...)                            \
    do {                                                                          \
        kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);          \
        (ctx)->launches++;                                                        \
        SB_CUDA((ctx), cudaGetLastError());                                       \
    } while (0)

// ---------------------------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------------------------
#ifdef __CUDACC__
// d^2 exactly as the oracle defines it: (dx*dx + dy*dy) + dz*dz, round-to-nearest, never contracted to FMA
// (kdtree.hpp:124 squaredNorm; SURVEY.md H2).
__device__ __forceinline__ double dist2_rn(double px, double py, double pz, double qx, double qy, double qz) {
    double dx = __dsub_rn(px, qx), dy = __dsub_rn(py, qy), dz = __dsub_rn(pz, qz);
    return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

// order-preserving map double <-> signed 64-bit so that atomicMin/atomicMax work on doubles exactly
__device__ __forceinline__ long long ordered_from_double(double d) {
    long long b = __double_as_longlong(d);
    return b >= 0 ? b : (b ^ 0x7fffffffffffffffLL);
}
__device__ __forceinline__ double double_from_ordered(long long b) {
    return __longlong_as_double(b >= 0 ? b : (b ^ 0x7fffffffffffffffLL));
}

__device__ __forceinline__ double shfl_d(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }

// Bounds of sqrt(d2) in float32 for the pruning tests: sqrt.approx.f32 is within 2^-23 (relative) of the root, the
// factors leave 8 ulp of slack (also for the rounding of d2 itself).  The IEEE directed-rounding roots these replace
// (__fsqrt_rd / __fsqrt_ru) are ~25-instruction sequences and were 17 % of k_icp_match's instructions.
__device__ __forceinline__ float sqrt_approx(float x) {
    float r;
    asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float sqrt_lower(double d2) { return __fmul_rd(sqrt_approx(__double2float_rd(d2)), 0.999999f); }
__device__ __forceinline__ float sqrt_upper(double d2) { return __fmul_ru(sqrt_approx(__double2float_ru(d2)), 1.000001f); }

__device__ __forceinline__ double shfl_d_xor(double v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }

// Row a of T * p for a row-major 4x4 T: p * R^T + t with the association of Transformation::apply (types.hpp:110-115).
// Every world-frame transform of the library (mapping.cu's k_transform, odom.cu's epilogue) goes through this one
// expression, so their bits cannot drift apart.
__device__ __forceinline__ double apply_row(const double* T, int a, double x, double y, double z) {
    return ((x * T[4 * a] + y * T[4 * a + 1]) + z * T[4 * a + 2]) + T[4 * a + 3];
}

__device__ __forceinline__ unsigned lanemask_lt() {
    unsigned m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}
#endif

// error flag bits written to Ctx::d_flags
enum { FLAG_NONFINITE = 1, FLAG_KEY_RANGE = 2 };

#ifdef __CUDACC__
// cloud of row i of a CSR point set (offsets ascending, offsets[0] <= i; an empty cloud never owns a row)
__device__ __forceinline__ int cloud_of(const i64* __restrict__ off, int n_clouds, i64 i) {
    int lo = 0, hi = n_clouds;
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (off[mid] <= i) lo = mid; else hi = mid;
    }
    return lo;
}

// update_occupancy_grid (slam_node.cpp:211-221) for one world-frame row of a cloud whose pose translation is (tx, ty):
// the biased (x, y) cell key, ascending in (x, y) as an unsigned integer; ~0 if the row is filtered out (*out_of_range
// set if its cell index does not fit an int).  The one expression of mapping.cu's k_occ_keys and map.cu's
// k_map_occ_insert, so both cell sets hold the same keys.
__device__ __forceinline__ u64 occ_key(double x, double y, double z, double tx, double ty, double res, double hmin,
                                       double hmax, double max_range, bool* out_of_range) {
    if (z < hmin || z > hmax) return ~0ull;   // NaN z passes both tests like the reference's comparisons
    const double dx = x - tx, dy = y - ty;
    const double r = sqrt(dx * dx + dy * dy);
    if (r > max_range || r < 0.5) return ~0ull;
    const double cx = floor(__ddiv_rn(x, res)), cy = floor(__ddiv_rn(y, res));
    if (fabs(cx) < 2147483647.0 && fabs(cy) < 2147483647.0)
        return ((u64)(uint32_t)((int)cx ^ 0x80000000) << 32) | (u64)(uint32_t)((int)cy ^ 0x80000000);
    *out_of_range = true;  // static_cast<int> of such a value is undefined in the reference
    return ~0ull;
}
#endif

// ---------------------------------------------------------------------------------------------------------------
// scan_sort.cu
// ---------------------------------------------------------------------------------------------------------------
// exclusive prefix sum of n uint32 values (in may equal out); total (optional device pointer) receives the sum
int exclusive_scan_u32(Ctx* ctx, const uint32_t* d_in, uint32_t* d_out, i64 n, uint32_t* d_total);

// Stable LSD radix sort of (key64, val32) pairs, independently inside each segment [seg_off[s], seg_off[s+1]).
// h_seg_off: host offsets (n_seg + 1).  Sorts on key bits [0, key_bits).  On return *out_keys / *out_vals point to
// whichever of the (a, b) buffers holds the sorted result.
int segmented_sort_pairs(Ctx* ctx, u64* keys_a, u64* keys_b, uint32_t* vals_a, uint32_t* vals_b,
                         const i64* h_seg_off, int n_seg, int key_bits, u64** out_keys, uint32_t** out_vals);

// ---------------------------------------------------------------------------------------------------------------
// voxel.cu
// ---------------------------------------------------------------------------------------------------------------
// Where the raw points of a call live on the device: fp64 rows (the ABI's PointCloud::Matrix layout) or float32 rows
// of `stride` floats with x, y, z first (binary PLY / KITTI .bin records, file_utils.cpp:91-97, 133-136).
struct PointSrc {
    const void* base;
    int f32;
    int stride;
};
int voxel_downsample_src(Ctx* ctx, const PointSrc src, const i64* h_off, int n_clouds, double voxel, double* d_out_xyz,
                         i64* h_out_off, i64* d_out_keys);
// Device-to-device batched voxel grid.  d_out_xyz / d_out_keys (optional) sized for the input row count;
// h_out_off (host, n_clouds + 1) receives the CSR offsets of the output.  Synchronises the stream.
int voxel_downsample_dev(Ctx* ctx, const double* d_xyz, const i64* h_off, int n_clouds, double voxel,
                         double* d_out_xyz, i64* h_out_off, i64* d_out_keys);

// ---------------------------------------------------------------------------------------------------------------
// forest.cu — the spatial index: one implicit 32-ary bounding-box tree per cloud over points sorted along a space-filling curve (Hilbert)
// ---------------------------------------------------------------------------------------------------------------
#define SB_MAX_LEVELS 7

struct TreePoint;
struct TreeNormal;
struct NbrEntry;
struct GridSlot;
struct TreeDesc {      // device-resident, one per indexed cloud
    // The arrays of the batch of trees this tree was built with (forest_append): several batches can live in one
    // forest, e.g. one per uploaded chunk of clouds, so every tree carries its own base pointers.
    const TreePoint* pts;   // points in curve (Hilbert) order
    const float4* pts32;    // the same points as float32 offsets from glo (w unused): candidate PRE-FILTER only
    const float* boxes;     // 6 floats per box: lo xyz (rounded down), hi xyz (up)
    TreeNormal* nrm;        // per sorted point, filled by forest_normals
    NbrEntry* nbr;          // normals_k entries per sorted point, filled by forest_normals
    GridSlot* grid;         // seed-grid slots, filled by forest_normals
    i64 out_off;       // first row of this cloud in forest-wide outputs in ORIGINAL row order
    i64 pt_off;        // first sorted point of this cloud in pts / nrm / nbr
    int n;             // points
    int top;           // top level (boxes at that level <= 32)
    i64 box_off[SB_MAX_LEVELS];  // first box of level l in the forest's box array
    int box_cnt[SB_MAX_LEVELS];  // boxes at level l
    int tab_shift;     // seed grid: 64 - log2(slots of this tree's hash table)
    i64 tab_off;       // seed grid: first slot of this tree in the forest's table
    double glo[3];     // seed grid origin = lower corner of the cloud's bounding box (device copy only)
    double gext;       // largest extent of the bounding box (device copy only)
    double ginv;       // 1 / cell size, set by forest_normals (device copy only)
};

// Seed grid (forest_normals): an open-addressing hash table cell -> one point of that cell per tree.  It only
// provides STARTING points for icp.cu's neighbour-graph walk, never answers.
struct GridSlot {
    unsigned long long key;  // packed cell coordinates, ~0 = empty
    int pos;                 // cloud-local sorted position of a point in the cell
    int pad;
};

// One curve-sorted point: exactly one 32-byte sector, so that a gathered candidate costs one sector and a leaf
// (32 consecutive points) is one coalesced 1 KB load.
struct alignas(32) TreePoint {
    double x, y, z;
    int idx;   // original row of the point, local to its cloud
    int pad;   // float bits: a lower bound of the distance to the nearest OTHER point of the cloud (entry 1 of the point's
               // neighbour list, NbrEntry::r), written with the normals; 0 until then.  It rides in the point's own
               // sector, so icp.cu's walk can prove "this point is the nearest neighbour" from one load.
};
// Unit normal of a sorted point (icp.hpp:23-67), padded to one sector.
struct alignas(32) TreeNormal {
    double x, y, z;
    double pad;
};
// Entry j of a point's k-nearest-neighbour list (ascending by (d2, index), the point itself included): the
// neighbour's cloud-local sorted position and a LOWER bound of its distance to the point.  Every point that is
// not among the first j entries is at least r_j away from the point — the certificate icp.cu's per-thread
// correspondence search rests on.
struct NbrEntry {
    int pos;   // -1: the cloud has fewer than k points
    float r;   // sqrt(d2) rounded down and shrunk by 1e-6 (+inf for padding)
};

struct ForestBatch {    // the arrays of the trees [t0, t0 + n_trees) appended together
    int t0 = 0, n_trees = 0;
    i64 n_points = 0, n_boxes = 0, n_slots = 0;
    TreePoint* pts = nullptr;
    float4* pts32 = nullptr;
    float* boxes = nullptr;
    TreeNormal* normals = nullptr;
    NbrEntry* nbr = nullptr;
    GridSlot* grid = nullptr;
};

// Caller-owned arrays for ONE batch of trees (odom.cu's frame slots): sized up front by the caller, never allocated or
// freed by the forest.  forest_append / forest_normals fail with SB_ERR_CAPACITY if the batch does not fit.
struct TreeStore {
    TreePoint* pts = nullptr;
    float4* pts32 = nullptr;
    float* boxes = nullptr;
    TreeNormal* normals = nullptr;
    NbrEntry* nbr = nullptr;
    GridSlot* grid = nullptr;
    i64 cap_points = 0, cap_boxes = 0, cap_slots = 0;
    int cap_k = 0;
};
// What the arrays of one tree over n points need: boxes of all levels and seed-grid slots (forest_append's layout).
void tree_store_need(i64 n, i64* boxes, i64* slots);

struct Forest {
    Ctx* ctx = nullptr;
    int n_trees = 0, cap_trees = 0;
    i64 n_points = 0;       // over all batches
    std::vector<ForestBatch> batches;
    TreeDesc* d_trees = nullptr;
    std::vector<TreeDesc> h_trees;   // host mirror (the seed-grid fields glo/gext/ginv are device-only)
    int normals_k = 0;      // 0: no normals yet
    bool in_arena = false;  // arrays live in the context arena (valid until the next C-ABI call), not cudaMalloc
    const TreeStore* store = nullptr;  // the next batch's arrays are these (caller-owned); d_trees is the caller's too
};

// Room for `cap_trees` tree descriptors (forest_append fails beyond that).
int forest_reserve(Ctx* ctx, Forest* f, int cap_trees);
// Appends trees over clouds `cloud_ids[0..n_new)` (null: 0..n_new-1) of a device CSR point set as one batch;
// d_xyz rows are row-major fp64.  The new trees are [f->n_trees - n_new, f->n_trees).
int forest_append(Ctx* ctx, Forest* f, const double* d_xyz, const i64* h_off, const int* cloud_ids, int n_new);
// reserve + append: a forest of exactly these trees
int forest_build(Ctx* ctx, const double* d_xyz, const i64* h_off, const int* cloud_ids, int n_trees, Forest* out);
void forest_free(Forest* f);

// Query work item: 32 consecutive queries of one query set against one tree.
struct QueryItem {
    i64 q_off;   // first query row (into the query xyz array)
    int count;   // 1..32
    int tree;    // tree id
};

// kNN over arbitrary query rows.  out_idx/out_d2 (device, optional): k per query, row = query row.
int forest_knn(Ctx* ctx, const Forest* f, const double* d_q, const QueryItem* d_items, i64 n_items, int k,
               int* d_out_idx, double* d_out_d2);
// 1-NN over arbitrary query rows.
int forest_nearest(Ctx* ctx, const Forest* f, const double* d_q, const QueryItem* d_items, i64 n_items,
                   int* d_out_idx, double* d_out_d2, int* d_out_pos);
// Normals, neighbour graph and seed grid of the trees of batch `batch` (-1: the last one) (icp.hpp:23-67); optional
// outputs in the ORIGINAL row order of the clouds: d_out_normals[3*(out_off+orig)] etc.  All batches of a forest
// must use the same k.
int forest_normals(Ctx* ctx, Forest* f, int k, double* d_out_normals, double* d_out_evals, int batch = -1);
// host helper: items covering all points of all trees (queries = the trees' own sorted points)
int make_items_dev(Ctx* ctx, const std::vector<QueryItem>& items, QueryItem** d_items);

// ---------------------------------------------------------------------------------------------------------------
// icp.cu
// ---------------------------------------------------------------------------------------------------------------
struct PairDesc {      // device-resident, one per scan pair
    const TreePoint* src_pts;  // the source cloud in ITS OWN curve order (it is indexed too: forest tree src_tree):
                               // neighbouring lanes then work on neighbouring points, and the order — hence the
                               // summation order — does not depend on what else is in the batch
    int n_src;
    int tree;          // target tree id in the forest (needs normals)
    i64 item_off;      // first 32-point work item of this pair
    int n_items;
    int src_tree;      // source tree id in the forest (no normals needed)
};

// Registers n_pairs pairs of trees of the forest (PairDesc::tree / src_tree; src_pts, item_off and n_items are filled
// in here).  results: host array.
// after_launch (optional) runs on the host right after the loop has been enqueued: host work or copies on another
// stream placed there overlap with the iterations.
int icp_batch(Ctx* ctx, const Forest* f, const std::vector<PairDesc>& pairs, const sb_icp_config* cfg,
              sb_icp_result* results, const std::function<int()>* after_launch = nullptr);
// The same in three steps, for callers that enqueue several batches (on ctx->stream as it is set at the time) before
// waiting: icp_reserve_results(total pairs), icp_enqueue per batch, icp_collect.
struct IcpPending {
    int n_pairs;
    size_t h_off;   // first result of the batch in Ctx::h_icp_res
    int slot;       // index into Ctx::h_icp_passes
    const sb_icp_result* d_res;  // the batch's results in device memory (arena), final once the stream reaches them
};
int icp_reserve_results(Ctx* ctx, size_t n_pairs);
int icp_enqueue(Ctx* ctx, const Forest* f, const std::vector<PairDesc>& pairs, const sb_icp_config* cfg, IcpPending* out);
int icp_collect(Ctx* ctx, cudaStream_t stream, const std::vector<IcpPending>& pending, const std::vector<const int*>& ids,
                sb_icp_result* results);
int ensure_copy_stream(Ctx* ctx);
void icp_graph_free(Ctx* ctx);

// ---------------------------------------------------------------------------------------------------------------
// scancontext.cu
// ---------------------------------------------------------------------------------------------------------------
int sc_compute_dev(Ctx* ctx, const double* d_xyz, const i64* d_off, int n_clouds, double* d_desc);
// one query descriptor against n_db descriptors (all column-major 20x60, device)
int sc_distance_dev(Ctx* ctx, const double* d_query_desc, const double* d_db, int n_db, double* d_out);
int sc_keys_dev(Ctx* ctx, const double* d_desc, double* d_ring, double* d_sector);
// sq[e * 60 + s]: the shifted self sum sum_bb(e, s) of k_sc_distance for n descriptors
int sc_sq_dev(Ctx* ctx, const double* d_desc, int n, double* d_sq);
// Many queries: dist[r * ld + e] = distance of query slot qslot[r] (ascending) to entry slot e, for the entries
// e < n_e of every tile that holds a pair with e < qslot[r] and a frame gap >= frame_gap (d_meta: (frame, entry))
int sc_distance_many_dev(Ctx* ctx, const double* d_desc, const double* d_sq, const int2* d_meta, const int* d_qslot,
                         int n_q, int n_e, int frame_gap, double* d_dist, i64 ld);

// icp.cu
int solve_point_to_plane_dev(Ctx* ctx, const double* d_src, const double* d_tgt, const double* d_nrm, i64 n,
                             double* d_out_T);
// mapping.cu
int transform_clouds_dev(Ctx* ctx, const double* d_xyz, const i64* d_off, int n_clouds, const double* d_poses, i64 n,
                         double* d_out);
int pack_f32_dev(Ctx* ctx, const double* d_in, i64 n_rows, float* d_out);
int occupancy_cells_dev(Ctx* ctx, const double* d_world, const i64* d_off, int n_clouds, const double* d_poses, i64 n,
                        const sb_grid_config* cfg, int* d_cells, i64 capacity, i64* count);
// synth.cu
int synth_scans_dev(Ctx* ctx, int beams, int azimuth_steps, float elev_top_deg, float elev_bot_deg, float max_range,
                    float noise_sigma, float sensor_height, const float* boxes6, int n_boxes, const double* poses,
                    int n_scans, uint64_t noise_seed, double* d_xyz, i64* out_offsets);

}  // namespace sb

struct sb_ctx {
    sb::Ctx c;
};

// loop.cu — state of one loop-closure database (slam::LoopClosureDetector, loop_closure.hpp:143-148)
struct sb_loop {
    sb::Ctx* ctx = nullptr;
    sb_loop_config cfg;
    int rank = 0, world = 1;
    // owned entries (+ possibly the newest one at the end, flagged by last_is_guest)
    std::vector<int> entry_id;       // global entry id of each local slot
    std::vector<int> frame_idx;      // loop_closure.hpp:147
    std::vector<sb::i64> cloud_off;  // CSR into d_clouds (local slots), size = slots + 1
    int n_global = 0;                // entries added so far (all ranks)
    int last_frame = 0;
    bool last_is_guest = false;      // the newest entry sits in the last slot although another rank owns it
    double* d_desc = nullptr;        // slots x 1200
    size_t desc_cap = 0;             // in descriptors
    double* d_clouds = nullptr;      // rows x 3
    size_t cloud_cap = 0;            // in rows
    double* d_meta = nullptr;        // slots x 8 bytes: (frame_idx, entry_id) as two int32 — the device-side search filter
    size_t meta_cap = 0;             // in slots
    std::vector<double*> retired;    // outgrown pools, released with the detector (loop.cu: grow)
};

namespace sb {
int loop_add(sb_loop* L, const double* xyz, i64 n, int frame_idx, const double* desc);
int loop_reserve(sb_loop* L, i64 n_entries, i64 total_rows);
// limit > 0: at most `limit` (<= SB_LOOP_SELECT_MAX) best candidates, selected on the device; limit <= 0: all of them.
// *total: number of candidates under the threshold either way.
// qslot: the query's local slot (entries before it are searched); -1: the newest entry.
int loop_candidates(sb_loop* L, std::vector<std::pair<double, int>>& cand, int limit, int* total, int qslot = -1);
// ICP(query cloud of slot qslots[i] -> cloud of entry entries[i]) for every i.
int loop_verify(sb_loop* L, const int* qslots, const int* entries, const double* dist, int n, sb_loop_result* results,
                int* converged);
// Batch entry points (world == 1 for the two queries; query slots strictly ascending).
int loop_add_many(sb_loop* L, const double* xyz, const i64* offsets, int n_frames, const int* frame_idx, const double* desc);
int loop_candidates_batch(sb_loop* L, const int* qslots, int n_q, std::vector<std::vector<std::pair<double, int>>>& cand,
                          std::vector<int>& total);
int loop_detect_batch(sb_loop* L, const int* qslots, int n_q, sb_loop_result* results, int* count);
// loop_add for a cloud and descriptor already in device memory, in two steps: loop_add_enqueue grows the pools and
// enqueues the device-to-device copies without waiting; loop_add_commit records the entry on the host once the stream
// has run them.  Together they leave the state loop_add(cloud, frame_idx, desc) leaves; without the commit the
// detector is unchanged (the copies land past its last committed entry).
struct LoopAddPending {
    int id, frame_idx;
    i64 end_row;
};
int loop_add_enqueue(sb_loop* L, const double* d_xyz, i64 n, int frame_idx, const double* d_desc, LoopAddPending* out);
void loop_add_commit(sb_loop* L, const LoopAddPending& p);
}  // namespace sb

// map.cu — device-resident keyframe map: every entry's sensor-frame rows and pose, and the occupancy cell set
struct sb_map {
    sb::Ctx* ctx = nullptr;
    sb_grid_config grid;
    std::vector<sb::i64> off{0};     // host CSR of the entries' rows, entries + 1
    std::vector<double> poses;       // host copy of the poses, 16 per entry
    double* d_rows = nullptr;        // rows x 3 (fp64, sensor frame)
    sb::i64 row_cap = 0;             // in rows
    sb::i64* d_off = nullptr;        // device copy of off
    double* d_poses = nullptr;       // 16 per entry
    sb::i64 entry_cap = 0;           // entries d_off / d_poses hold
    unsigned long long* d_table = nullptr;   // open-addressing set of cell keys, ~0 = empty slot
    sb::i64 table_cap = 0;           // slots, a power of two
    sb::i64 n_cells = 0;             // keys in the table
    unsigned long long* d_stat = nullptr;    // [0] keys a launch inserted, [1] flag bits (FLAG_*)
    unsigned long long* h_stat = nullptr;    // pinned copy of d_stat
    bool pending = false;            // an add was enqueued and not finished: the table may hold its cells
    std::vector<void*> retired;      // outgrown buffers, released with the map
};

namespace sb {
// The streaming session's half of sb_map_add (odom.cu): the frame's rows and pose, already in device memory, are copied
// device to device and its cells are inserted, without a synchronise.  After the caller's synchronise, map_add_finish
// records the entry; if the insert failed it restores the cell set from the committed entries and returns the error,
// and the map is as it was.
struct MapAddPending {
    i64 end_row;
};
int map_add_enqueue(sb_map* M, const double* d_xyz, i64 n, const double* d_pose, MapAddPending* out);
int map_add_finish(sb_map* M, const MapAddPending& p, const double* pose16);
// after a failed call that enqueued an add without finishing it: the cell set of the committed entries again
int map_add_abort(sb_map* M);
// sb_map_add: host rows and pose, one synchronise (the session adds a skipped frame this way: no rows, the same pose)
int map_add(sb_map* M, const double* xyz, i64 n, const double* pose16);

// RAII entry guard of every C-ABI call: selects the device and resets the arena
struct Enter {
    Ctx* c;
    explicit Enter(Ctx* ctx) : c(ctx) {
        cudaSetDevice(c->device);
        arena_reset(c);
        c->tbuf_used = 0;  // everything the previous call enqueued has completed
        c->err.clear();
        c->n_ev = 0;
    }
};
}  // namespace sb
