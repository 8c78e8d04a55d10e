// map.cu — the device-resident map (sb_map_*, include/slam_b200.h): the keyframe clouds, their poses and the occupancy
// cell set of slam_node.cpp (update_occupancy_grid :211-221, rebuild after optimize :177-194, global map :196-209)
// kept in device memory, so that a rebuild after a loop closure uploads poses (128 B per entry) instead of every cloud.
//
// Rows: one fp64 pool with a CSR of entries (host and device copies of the offsets), poses on both sides.
// Cells: an open-addressing set of the 64-bit keys k_occ_keys forms (occ_key, common.cuh), linear probing, ~0 = empty.
// A launch inserts at most `limit` new keys, so that the table stays at most half full; a launch that reaches the
// limit flags FLAG_MAP_FULL, the table doubles (k_map_rehash) and the rows go in again (a set: keys already in are
// found, not counted twice).  Extraction compacts the occupied slots and sorts only the distinct keys, whose unsigned
// order is the (x, y) order of mapping.cu's sort over all rows.  World-frame rows come from apply_row as in k_transform.
//
// Failure rule: a call that fails re-derives the cell set from the committed entries and poses (k_map_occ_insert over
// all resident rows), and the host-side entry list changes only after the call's final synchronise.
// Buffers only grow, by doubling; outgrown ones are retired until sb_map_free (cudaMalloc / cudaFree stall the host,
// see loop.cu).
#include <algorithm>
#include <cmath>

#include "common.cuh"

namespace sb {

static constexpr u64 EMPTY_KEY = ~0ull;
enum { FLAG_MAP_FULL = 4 };   // a launch reached its insert limit (beside FLAG_NONFINITE / FLAG_KEY_RANGE)
static const i64 FIRST_ROWS = (i64)1 << 20;        // 24 MB of fp64 rows: ~130 downsampled scans
static const i64 FIRST_ENTRIES = 1024;
static const i64 FIRST_TABLE_SLOTS = (i64)1 << 16;  // 512 KB

__device__ __forceinline__ u64 cell_slot(u64 key, int shift) { return (key * 0x9E3779B97F4A7C15ull) >> shift; }

// One key into the set.  Claims an empty slot only while fewer than `limit` keys were claimed by this launch.
__device__ __forceinline__ void table_insert(u64* table, u64 mask, int shift, u64 key, unsigned long long* count,
                                             u64 limit, unsigned long long* flags) {
    u64 s = cell_slot(key, shift);
    for (u64 step = 0; step <= mask; ++step, s = (s + 1) & mask) {
        const u64 cur = __ldcg(table + s);
        if (cur == key) return;
        if (cur != EMPTY_KEY) continue;
        if (*(volatile unsigned long long*)count >= limit) break;
        const u64 prev = atomicCAS(table + s, EMPTY_KEY, key);
        if (prev == EMPTY_KEY) {
            atomicAdd(count, 1ull);
            return;
        }
        if (prev == key) return;
    }
    atomicOr(flags, (unsigned long long)FLAG_MAP_FULL);
}

// update_occupancy_grid for the resident rows [r0, r1): one thread per row, the row to the world frame with its entry's
// pose (apply_row, as k_transform), the filter and key of k_occ_keys (occ_key), then one probe per distinct key of
// the warp (neighbouring rows of a scan mostly share a cell).
__global__ void __launch_bounds__(256) k_map_occ_insert(const double* __restrict__ rows, const i64* __restrict__ off,
                                                        int n_entries, const double* __restrict__ poses, i64 r0, i64 r1,
                                                        double res, double hmin, double hmax, double max_range,
                                                        u64* table, u64 mask, int shift, unsigned long long* count,
                                                        u64 limit, unsigned long long* flags) {
    const i64 i = r0 + (i64)blockIdx.x * blockDim.x + threadIdx.x;
    u64 key = EMPTY_KEY;
    if (i < r1) {
        const double* T = poses + 16 * cloud_of(off, n_entries, i);
        const double x = rows[3 * i], y = rows[3 * i + 1], z = rows[3 * i + 2];
        if (!(isfinite(x) && isfinite(y) && isfinite(z))) atomicOr(flags, (unsigned long long)FLAG_NONFINITE);
        bool out_of_range = false;
        key = occ_key(apply_row(T, 0, x, y, z), apply_row(T, 1, x, y, z), apply_row(T, 2, x, y, z), T[3], T[7], res,
                      hmin, hmax, max_range, &out_of_range);
        if (out_of_range) atomicOr(flags, (unsigned long long)FLAG_KEY_RANGE);
    }
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    if (key == EMPTY_KEY || (peers & lanemask_lt())) return;
    table_insert(table, mask, shift, key, count, limit, flags);
}

// the keys of an outgrown table into the new one
__global__ void __launch_bounds__(256) k_map_rehash(const u64* __restrict__ old, i64 n_old, u64* table, u64 mask,
                                                    int shift, unsigned long long* count, unsigned long long* flags) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_old) return;
    const u64 key = old[i];
    if (key != EMPTY_KEY) table_insert(table, mask, shift, key, count, EMPTY_KEY, flags);
}

__global__ void __launch_bounds__(256) k_map_occ_flag(const u64* __restrict__ table, i64 n, uint32_t* __restrict__ flag) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flag[i] = table[i] != EMPTY_KEY ? 1u : 0u;
}

// occupied slot i -> keys[pos[i]] (pos: exclusive prefix sum of the occupancy flags; n_keys: the keys the host counted)
__global__ void __launch_bounds__(256) k_map_occ_compact(const u64* __restrict__ table, const uint32_t* __restrict__ pos,
                                                         i64 n, i64 n_keys, u64* __restrict__ keys,
                                                         uint32_t* __restrict__ vals) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u64 k = table[i];
    if (k == EMPTY_KEY || (i64)pos[i] >= n_keys) return;
    keys[pos[i]] = k;
    vals[pos[i]] = pos[i];
}

// sorted distinct keys -> (x, y) cells, unpacked as k_occ_emit does
__global__ void __launch_bounds__(256) k_map_occ_emit(const u64* __restrict__ keys, i64 m, int* __restrict__ cells) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const u64 k = keys[i];
    cells[2 * i] = (int)((uint32_t)(k >> 32) ^ 0x80000000u);
    cells[2 * i + 1] = (int)((uint32_t)k ^ 0x80000000u);
}

__device__ __forceinline__ void store_row(double* p, double v) { *p = v; }
__device__ __forceinline__ void store_row(float* p, double v) { *p = __double2float_rn(v); }   // static_cast<float>

// resident rows [r0, r1) to the world frame, row r at out[3 * (r - r0)]: the expression of k_transform (apply_row)
template <typename Out>
__global__ void __launch_bounds__(256) k_map_transform(const double* __restrict__ rows, const i64* __restrict__ off,
                                                       int n_entries, const double* __restrict__ poses, i64 r0, i64 r1,
                                                       Out* __restrict__ out) {
    const i64 i = r0 + (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= r1) return;
    const double* T = poses + 16 * cloud_of(off, n_entries, i);
    const double x = rows[3 * i], y = rows[3 * i + 1], z = rows[3 * i + 2];
#pragma unroll
    for (int a = 0; a < 3; ++a) store_row(out + 3 * (i - r0) + a, apply_row(T, a, x, y, z));
}

// ------------------------------------------------------------------------------------------------ host side
static int n_entries(const sb_map* M) { return (int)M->off.size() - 1; }

static int log2_slots(i64 slots) {
    int lg = 0;
    while (((i64)1 << lg) < slots) ++lg;
    return lg;
}

// a buffer of `ncap` elements holding the first `used` elements of the old one, which is retired
template <typename T>
static int grow_buf(sb_map* M, T** buf, i64 ncap, i64 used) {
    T* nb = nullptr;
    SB_CUDA(M->ctx, cudaMalloc(&nb, sizeof(T) * (size_t)ncap));
    if (*buf) {
        if (used > 0)
            SB_CUDA(M->ctx, cudaMemcpyAsync(nb, *buf, sizeof(T) * (size_t)used, cudaMemcpyDeviceToDevice, M->ctx->stream));
        M->retired.push_back(*buf);
    }
    *buf = nb;
    return SB_OK;
}

static i64 doubled(i64 cap, i64 need, i64 first) {
    i64 c = cap > 0 ? cap : std::max<i64>(first, 1);
    while (c < need) c *= 2;
    return c;
}

static int grow_rows(sb_map* M, i64 need, i64 first) {
    if (need <= M->row_cap) return SB_OK;
    const i64 ncap = doubled(M->row_cap, need, first);
    SB_TRY(grow_buf(M, &M->d_rows, 3 * ncap, 3 * M->off.back()));
    M->row_cap = ncap;
    return SB_OK;
}

// room for `need` entries in d_off (need + 1 offsets) and d_poses
static int grow_entries(sb_map* M, i64 need, i64 first) {
    if (need <= M->entry_cap) return SB_OK;
    const i64 ncap = doubled(M->entry_cap, need, first);
    const i64 e = n_entries(M);
    SB_TRY(grow_buf(M, &M->d_off, ncap + 1, e + 1));
    SB_TRY(grow_buf(M, &M->d_poses, 16 * ncap, 16 * e));
    M->entry_cap = ncap;
    return SB_OK;
}

// a table of `slots` (a power of two) holding the current keys (rehash = true) or empty
static int table_resize(sb_map* M, i64 slots, bool rehash) {
    Ctx* ctx = M->ctx;
    u64* nt = nullptr;
    SB_CUDA(ctx, cudaMalloc(&nt, sizeof(u64) * (size_t)slots));
    SB_CUDA(ctx, cudaMemsetAsync(nt, 0xff, sizeof(u64) * (size_t)slots, ctx->stream));
    if (rehash && M->d_table && M->table_cap > 0) {
        SB_CUDA(ctx, cudaMemsetAsync(M->d_stat + 2, 0, 2 * sizeof(u64), ctx->stream));
        SB_LAUNCH(ctx, k_map_rehash, ceil_div(M->table_cap, 256), 256, 0, M->d_table, M->table_cap, nt,
                  (u64)(slots - 1), 64 - log2_slots(slots), M->d_stat + 2, M->d_stat + 3);
    }
    if (M->d_table) M->retired.push_back(M->d_table);
    M->d_table = nt;
    M->table_cap = slots;
    return SB_OK;
}

// k_map_occ_insert over rows [r0, r1) of the first `entries` entries, at most `limit` new keys; the launch's count and
// flags go to h_stat at the caller's synchronise
static int launch_insert(sb_map* M, i64 r0, i64 r1, int entries, i64 limit) {
    Ctx* ctx = M->ctx;
    SB_CUDA(ctx, cudaMemsetAsync(M->d_stat, 0, 2 * sizeof(u64), ctx->stream));
    if (r1 > r0)
        SB_LAUNCH(ctx, k_map_occ_insert, ceil_div(r1 - r0, 256), 256, 0, M->d_rows, M->d_off, entries, M->d_poses, r0, r1,
                  M->grid.resolution, M->grid.height_min, M->grid.height_max, M->grid.max_range, M->d_table,
                  (u64)(M->table_cap - 1), 64 - log2_slots(M->table_cap), M->d_stat, (u64)std::max<i64>(limit, 0),
                  M->d_stat + 1);
    SB_CUDA(ctx, cudaMemcpyAsync(M->h_stat, M->d_stat, 2 * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    return SB_OK;
}

// the cell set of the committed entries with the poses in d_poses, into a cleared table that doubles while a launch
// fills it past half; h_stat holds the count and the flags of the last launch
static int rebuild(sb_map* M) {
    Ctx* ctx = M->ctx;
    for (;;) {
        SB_CUDA(ctx, cudaMemsetAsync(M->d_table, 0xff, sizeof(u64) * (size_t)M->table_cap, ctx->stream));
        SB_TRY(launch_insert(M, 0, M->off.back(), n_entries(M), M->table_cap / 2));
        SB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (M->h_stat[1] != FLAG_MAP_FULL) return SB_OK;
        SB_TRY(table_resize(M, 2 * M->table_cap, false));
    }
}

static int fail_flags(Ctx* ctx, u64 flags) {
    if (flags & FLAG_NONFINITE) return fail(ctx, SB_ERR_RANGE, "map: non-finite row");
    return fail(ctx, SB_ERR_RANGE, "map: a cell index does not fit an int");
}

// the committed cell set again (after a failed insert or pose update)
static int restore(sb_map* M) {
    M->pending = false;
    SB_TRY(rebuild(M));
    M->n_cells = (i64)M->h_stat[0];
    return SB_OK;
}

// keeps the load at most one half at the end of every call (a launch can overshoot its limit by the keys in flight)
static int keep_half(sb_map* M) {
    if (2 * M->n_cells <= M->table_cap) return SB_OK;
    return table_resize(M, doubled(M->table_cap, 2 * M->n_cells, FIRST_TABLE_SLOTS), true);
}

static bool finite16(const double* p) {
    for (int i = 0; i < 16; ++i)
        if (!std::isfinite(p[i])) return false;
    return true;
}

// the entry's rows (host or device) and pose into the pools past the committed entries, and its cells into the table
static int add_enqueue(sb_map* M, const double* xyz, bool xyz_dev, i64 n, const double* pose, bool pose_dev,
                       MapAddPending* out) {
    Ctx* ctx = M->ctx;
    const int e = n_entries(M);
    const i64 R = M->off.back();
    SB_TRY(grow_rows(M, R + n, FIRST_ROWS));
    SB_TRY(grow_entries(M, (i64)e + 1, FIRST_ENTRIES));
    M->pending = true;
    if (n > 0)
        SB_CUDA(ctx, cudaMemcpyAsync(M->d_rows + 3 * R, xyz, sizeof(double) * 3 * (size_t)n,
                                     xyz_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, ctx->stream));
    const i64 end = R + n;
    SB_TRY(table_upload(ctx, M->d_off + e + 1, &end, sizeof(end)));
    if (pose_dev)
        SB_CUDA(ctx, cudaMemcpyAsync(M->d_poses + 16 * (size_t)e, pose, sizeof(double) * 16, cudaMemcpyDeviceToDevice,
                                     ctx->stream));
    else
        SB_TRY(table_upload(ctx, M->d_poses + 16 * (size_t)e, pose, sizeof(double) * 16));
    SB_TRY(launch_insert(M, R, end, e + 1, M->table_cap / 2 - M->n_cells));
    out->end_row = end;
    return SB_OK;
}

int map_add_enqueue(sb_map* M, const double* d_xyz, i64 n, const double* d_pose, MapAddPending* out) {
    return add_enqueue(M, d_xyz, true, n, d_pose, true, out);
}

int map_add_finish(sb_map* M, const MapAddPending& p, const double* pose16) {
    Ctx* ctx = M->ctx;
    const int e = n_entries(M);
    const i64 R = M->off.back();
    i64 inserted = (i64)M->h_stat[0];
    u64 flags = M->h_stat[1];
    while (flags == FLAG_MAP_FULL) {   // the launch stopped at half load: double the table and insert the rows again
        SB_TRY(table_resize(M, 2 * M->table_cap, true));
        SB_TRY(launch_insert(M, R, p.end_row, e + 1, M->table_cap / 2 - (M->n_cells + inserted)));
        SB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        inserted += (i64)M->h_stat[0];
        flags = M->h_stat[1];
    }
    if (flags & (FLAG_NONFINITE | FLAG_KEY_RANGE)) {
        SB_TRY(restore(M));
        return fail_flags(ctx, flags);
    }
    M->pending = false;
    M->off.push_back(p.end_row);
    M->poses.insert(M->poses.end(), pose16, pose16 + 16);
    M->n_cells += inserted;
    return keep_half(M);
}

int map_add_abort(sb_map* M) {
    if (!M->pending) return SB_OK;
    cudaStreamSynchronize(M->ctx->stream);
    return restore(M);
}

int map_add(sb_map* M, const double* xyz, i64 n, const double* pose16) {
    MapAddPending p;
    int s = add_enqueue(M, xyz, false, n, pose16, false, &p);
    if (s == SB_OK && cudaStreamSynchronize(M->ctx->stream) != cudaSuccess)
        s = fail(M->ctx, SB_ERR_CUDA, "map: add failed on the device: %s", cudaGetErrorString(cudaGetLastError()));
    if (s != SB_OK) {   // the first failure's message is the one to report
        const std::string msg = M->ctx->err;
        map_add_abort(M);
        M->ctx->err = msg;
        return s;
    }
    return map_add_finish(M, p, pose16);
}

}  // namespace sb

using namespace sb;

namespace {

int map_global(sb_map* M, double voxel, void* out_xyz, bool f32, int64_t* out_m) {
    Ctx* ctx = M->ctx;
    *out_m = 0;
    const i64 n = M->off.back();
    if (n == 0) return SB_OK;
    if (!out_xyz) return fail(ctx, SB_ERR_INVALID_ARG, "map: null output buffer");
    double *d_world, *d_out;
    SB_TRY(arena_get(ctx, (size_t)3 * n, &d_world));
    SB_TRY(arena_get(ctx, (size_t)3 * n, &d_out));
    SB_LAUNCH(ctx, k_map_transform<double>, ceil_div(n, 256), 256, 0, M->d_rows, M->d_off, n_entries(M), M->d_poses,
              (i64)0, n, d_world);
    i64 one[2] = {0, n}, out_off[2] = {0, 0};
    SB_TRY(voxel_downsample_dev(ctx, d_world, one, 1, voxel, d_out, out_off, nullptr));
    const i64 m = out_off[1];
    if (f32) {
        float* d_f32;
        SB_TRY(arena_get(ctx, (size_t)3 * (m > 0 ? m : 1), &d_f32));
        SB_TRY(pack_f32_dev(ctx, d_out, m, d_f32));
        if (m > 0)
            SB_CUDA(ctx, cudaMemcpyAsync(out_xyz, d_f32, sizeof(float) * 3 * (size_t)m, cudaMemcpyDeviceToHost, ctx->stream));
    } else if (m > 0) {
        SB_CUDA(ctx, cudaMemcpyAsync(out_xyz, d_out, sizeof(double) * 3 * (size_t)m, cudaMemcpyDeviceToHost, ctx->stream));
    }
    SB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *out_m = m;
    return SB_OK;
}

}  // namespace

extern "C" {

int sb_map_create(sb_ctx* ctx, const sb_grid_config* grid, sb_map** out) {
    if (!ctx || !out) return SB_ERR_INVALID_ARG;
    *out = nullptr;
    Ctx* c = &ctx->c;
    Enter g(c);
    sb_grid_config cfg;
    if (grid) cfg = *grid;
    else sb_default_grid_config(&cfg);
    if (!(cfg.resolution > 0)) return fail(c, SB_ERR_INVALID_ARG, "map: grid resolution must be positive");
    sb_map* M = new sb_map();
    M->ctx = c;
    M->grid = cfg;
    int s = SB_OK;
    if (cudaMalloc(&M->d_stat, 4 * sizeof(u64)) != cudaSuccess ||
        cudaHostAlloc(&M->h_stat, 4 * sizeof(u64), cudaHostAllocDefault) != cudaSuccess)
        s = fail(c, SB_ERR_CUDA, "map: %s", cudaGetErrorString(cudaGetLastError()));
    if (s == SB_OK) s = grow_entries(M, FIRST_ENTRIES, FIRST_ENTRIES);
    if (s == SB_OK) s = table_resize(M, FIRST_TABLE_SLOTS, false);
    if (s == SB_OK) {
        const i64 zero = 0;
        if (cudaMemcpyAsync(M->d_off, &zero, sizeof(zero), cudaMemcpyHostToDevice, c->stream) != cudaSuccess ||
            cudaStreamSynchronize(c->stream) != cudaSuccess)
            s = fail(c, SB_ERR_CUDA, "map: %s", cudaGetErrorString(cudaGetLastError()));
    }
    if (s != SB_OK) {
        sb_map_free(M);
        return s;
    }
    *out = M;
    return SB_OK;
}

void sb_map_free(sb_map* map) {
    if (!map) return;
    cudaSetDevice(map->ctx->device);
    cudaStreamSynchronize(map->ctx->stream);
    cudaFree(map->d_rows);
    cudaFree(map->d_off);
    cudaFree(map->d_poses);
    cudaFree(map->d_table);
    cudaFree(map->d_stat);
    for (void* p : map->retired) cudaFree(p);
    if (map->h_stat) cudaFreeHost(map->h_stat);
    delete map;
}

int sb_map_reserve(sb_map* map, int64_t n_entries, int64_t total_rows, int64_t n_cells) {
    if (!map || n_entries < 0 || total_rows < 0 || n_cells < 0) return SB_ERR_INVALID_ARG;
    Ctx* c = map->ctx;
    Enter g(c);
    SB_TRY(grow_entries(map, n_entries, n_entries));
    SB_TRY(grow_rows(map, total_rows, total_rows));
    if (2 * n_cells > map->table_cap) SB_TRY(table_resize(map, doubled(map->table_cap, 2 * n_cells, 1), true));
    SB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SB_OK;
}

int64_t sb_map_size(const sb_map* map) { return map ? (int64_t)map->off.size() - 1 : 0; }

int64_t sb_map_rows(const sb_map* map) { return map ? (int64_t)map->off.back() : 0; }

int sb_map_capacity(const sb_map* map, int64_t* caps3) {
    if (!map || !caps3) return SB_ERR_INVALID_ARG;
    caps3[0] = map->entry_cap;
    caps3[1] = map->row_cap;
    caps3[2] = map->table_cap;
    return SB_OK;
}

int sb_map_clear(sb_map* map) {
    if (!map) return SB_ERR_INVALID_ARG;
    Ctx* c = map->ctx;
    Enter g(c);
    SB_CUDA(c, cudaMemsetAsync(map->d_table, 0xff, sizeof(u64) * (size_t)map->table_cap, c->stream));
    SB_CUDA(c, cudaStreamSynchronize(c->stream));
    map->off.assign(1, 0);
    map->poses.clear();
    map->n_cells = 0;
    return SB_OK;
}

int sb_map_add(sb_map* map, const double* xyz, int64_t n, const double* pose16) {
    if (!map) return SB_ERR_INVALID_ARG;
    Ctx* c = map->ctx;
    Enter g(c);
    if (n < 0 || (n > 0 && !xyz) || !pose16) return fail(c, SB_ERR_INVALID_ARG, "map: null buffer or negative row count");
    if (n_entries(map) == 0x7fffffff) return fail(c, SB_ERR_RANGE, "map: 2^31-1 entries");
    if (!finite16(pose16)) return fail(c, SB_ERR_RANGE, "map: non-finite pose");
    return map_add(map, xyz, (i64)n, pose16);
}

int sb_map_set_poses(sb_map* map, int32_t first, int32_t n, const double* poses16) {
    if (!map) return SB_ERR_INVALID_ARG;
    Ctx* c = map->ctx;
    Enter g(c);
    if (first < 0 || n < 0 || (i64)first + n > n_entries(map) || (n > 0 && !poses16))
        return fail(c, SB_ERR_INVALID_ARG, "map: entries [%d, %d + %d) outside [0, %d)", first, first, n, n_entries(map));
    if (n == 0) return SB_OK;
    for (int32_t i = 0; i < n; ++i)
        if (!finite16(poses16 + 16 * (size_t)i)) return fail(c, SB_ERR_RANGE, "map: non-finite pose of entry %d", first + i);
    double* d_dst = map->d_poses + 16 * (size_t)first;
    const size_t bytes = sizeof(double) * 16 * (size_t)n;
    SB_CUDA(c, cudaMemcpyAsync(d_dst, poses16, bytes, cudaMemcpyHostToDevice, c->stream));
    SB_TRY(rebuild(map));
    const u64 flags = map->h_stat[1];
    if (flags) {   // the committed poses again, and their cell set
        SB_CUDA(c, cudaMemcpyAsync(d_dst, map->poses.data() + 16 * (size_t)first, bytes, cudaMemcpyHostToDevice, c->stream));
        SB_TRY(restore(map));
        return fail_flags(c, flags);
    }
    memcpy(map->poses.data() + 16 * (size_t)first, poses16, bytes);
    map->n_cells = (i64)map->h_stat[0];
    return keep_half(map);
}

int sb_map_get_poses(const sb_map* map, int32_t first, int32_t n, double* poses16) {
    if (!map || first < 0 || n < 0 || (i64)first + n > (i64)map->off.size() - 1 || (n > 0 && !poses16))
        return SB_ERR_INVALID_ARG;
    if (n > 0) memcpy(poses16, map->poses.data() + 16 * (size_t)first, sizeof(double) * 16 * (size_t)n);
    return SB_OK;
}

int sb_map_occupancy_cells(sb_map* map, int32_t* out_cells, int64_t capacity, int64_t* out_count) {
    if (!map || !out_count || capacity < 0 || (capacity > 0 && !out_cells)) return SB_ERR_INVALID_ARG;
    Ctx* c = map->ctx;
    Enter g(c);
    const i64 count = map->n_cells;
    *out_count = count;
    const i64 m = std::min<i64>(count, capacity);
    if (m == 0) return SB_OK;
    const i64 slots = map->table_cap;
    uint32_t *d_pos, *va, *vb, *d_total, *vs;
    u64 *ka, *kb, *ks;
    int* d_cells;
    SB_TRY(arena_get(c, (size_t)slots, &d_pos));
    SB_TRY(arena_get(c, 1, &d_total));
    SB_TRY(arena_get(c, (size_t)count, &ka));
    SB_TRY(arena_get(c, (size_t)count, &kb));
    SB_TRY(arena_get(c, (size_t)count, &va));
    SB_TRY(arena_get(c, (size_t)count, &vb));
    SB_TRY(arena_get(c, (size_t)2 * m, &d_cells));
    SB_LAUNCH(c, k_map_occ_flag, ceil_div(slots, 256), 256, 0, map->d_table, slots, d_pos);
    SB_TRY(exclusive_scan_u32(c, d_pos, d_pos, slots, d_total));
    SB_LAUNCH(c, k_map_occ_compact, ceil_div(slots, 256), 256, 0, map->d_table, d_pos, slots, count, ka, va);
    const i64 seg[2] = {0, count};
    SB_TRY(segmented_sort_pairs(c, ka, kb, va, vb, seg, 1, 64, &ks, &vs));
    SB_LAUNCH(c, k_map_occ_emit, ceil_div(m, 256), 256, 0, ks, m, d_cells);
    SB_CUDA(c, cudaMemcpyAsync(out_cells, d_cells, sizeof(int) * 2 * (size_t)m, cudaMemcpyDeviceToHost, c->stream));
    SB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SB_OK;
}

int sb_map_world_f32(sb_map* map, int32_t first, int32_t n, float* out_xyz, int64_t* out_rows) {
    if (!map || !out_rows) return SB_ERR_INVALID_ARG;
    Ctx* c = map->ctx;
    Enter g(c);
    *out_rows = 0;
    if (first < 0 || n < 0 || (i64)first + n > n_entries(map))
        return fail(c, SB_ERR_INVALID_ARG, "map: entries [%d, %d + %d) outside [0, %d)", first, first, n, n_entries(map));
    const i64 r0 = map->off[first], r1 = map->off[first + n];
    if (r1 == r0) return SB_OK;
    if (!out_xyz) return fail(c, SB_ERR_INVALID_ARG, "map: null output buffer");
    float* d_f32;
    SB_TRY(arena_get(c, (size_t)3 * (r1 - r0), &d_f32));
    SB_LAUNCH(c, k_map_transform<float>, ceil_div(r1 - r0, 256), 256, 0, map->d_rows, map->d_off, n_entries(map),
              map->d_poses, r0, r1, d_f32);
    SB_CUDA(c, cudaMemcpyAsync(out_xyz, d_f32, sizeof(float) * 3 * (size_t)(r1 - r0), cudaMemcpyDeviceToHost, c->stream));
    SB_CUDA(c, cudaStreamSynchronize(c->stream));
    *out_rows = r1 - r0;
    return SB_OK;
}

int sb_map_global(sb_map* map, double voxel, double* out_xyz, int64_t* out_m) {
    if (!map || !out_m) return SB_ERR_INVALID_ARG;
    Enter g(map->ctx);
    return map_global(map, voxel, out_xyz, false, out_m);
}

int sb_map_global_f32(sb_map* map, double voxel, float* out_xyz, int64_t* out_m) {
    if (!map || !out_m) return SB_ERR_INVALID_ARG;
    Enter g(map->ctx);
    return map_global(map, voxel, out_xyz, true, out_m);
}

}  // extern "C"
