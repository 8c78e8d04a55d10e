// forest.cu — spatial index build, k-NN / 1-NN query kernels and surface-normal estimation.
//
// Replaces, for a batch of clouds at once:
//   slam::KDTree::KDTree / build          slam_viz/include/slam_viz/core/kdtree.hpp:20-26, 87-110
//   KDTree::nearest / nearest_batch       kdtree.hpp:32-59, 112-142
//   KDTree::k_nearest                     kdtree.hpp:65-78, 144-180
//   slam::estimate_normals                slam_viz/include/slam_viz/core/icp.hpp:23-67
// The index is not a KD-tree: see traverse.cuh.  Build = per-cloud bounding box (exact atomic min/max on ordered
// integers) -> 30-bit Hilbert-curve indices -> segmented radix sort -> gather into SoA + leaf boxes -> upper box levels.
#include "traverse.cuh"

#include <cstdlib>

namespace sb {

static constexpr int CHUNK = 1024;  // points per build work item (32 leaves)

struct Chunk {
    int tree;
    int start;  // cloud-local first point
    int count;
    int pad;
};

// ---------------------------------------------------------------------------------------------------------------
// build kernels
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_bbox(const double* __restrict__ xyz, const i64* __restrict__ src_off,
                                              const Chunk* __restrict__ chunks, long long* __restrict__ bb) {
    Chunk c = chunks[blockIdx.x];
    const double* base = xyz + 3 * (src_off[c.tree] + c.start);
    double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int i = threadIdx.x; i < c.count; i += 256) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            double v = base[3 * i + a];
            lo[a] = fmin(lo[a], v);
            hi[a] = fmax(hi[a], v);
        }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[a] = fmin(lo[a], shfl_d_xor(lo[a], o));
            hi[a] = fmax(hi[a], shfl_d_xor(hi[a], o));
        }
    }
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            if (lo[a] <= hi[a]) {
                atomicMin(&bb[6 * c.tree + a], ordered_from_double(lo[a]));
                atomicMax(&bb[6 * c.tree + 3 + a], ordered_from_double(hi[a]));
            }
        }
    }
}

__device__ __forceinline__ unsigned spread10(unsigned v) {  // 10 bits -> every third bit
    v &= 0x3ffu;
    v = (v | (v << 16)) & 0x030000ffu;
    v = (v | (v << 8)) & 0x0300f00fu;
    v = (v | (v << 4)) & 0x030c30c3u;
    v = (v | (v << 2)) & 0x09249249u;
    return v;
}

// 3 x 10-bit cell coordinates -> their position on the 3-D Hilbert curve, as three "transposed" words whose bit
// interleaving is the 30-bit index (Skilling, "Programming the Hilbert curve", 2004).  Unlike the Z-order curve the
// Hilbert curve has no jumps: points that are consecutive in the sorted order are neighbours in space, so the 32-point
// leaves get tighter boxes and a query's result is a better seed for the next query.
__device__ __forceinline__ void hilbert_transpose10(unsigned (&X)[3]) {
    const unsigned M = 1u << 9;
    for (unsigned Q = M; Q > 1; Q >>= 1) {
        const unsigned P = Q - 1;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            if (X[i] & Q) {
                X[0] ^= P;
            } else {
                const unsigned t = (X[0] ^ X[i]) & P;
                X[0] ^= t;
                X[i] ^= t;
            }
        }
    }
    X[1] ^= X[0];
    X[2] ^= X[1];
    unsigned t = 0;
    for (unsigned Q = M; Q > 1; Q >>= 1)
        if (X[2] & Q) t ^= Q - 1;
    X[0] ^= t; X[1] ^= t; X[2] ^= t;
}

__global__ void __launch_bounds__(256) k_morton(const double* __restrict__ xyz, const i64* __restrict__ src_off,
                                                const Chunk* __restrict__ chunks, const long long* __restrict__ bb,
                                                const TreeDesc* __restrict__ trees, u64* __restrict__ keys,
                                                uint32_t* __restrict__ vals, int hilbert) {
    Chunk c = chunks[blockIdx.x];
    double lo[3], ext = 0.0;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        lo[a] = double_from_ordered(bb[6 * c.tree + a]);
        double e = double_from_ordered(bb[6 * c.tree + 3 + a]) - lo[a];
        ext = fmax(ext, e);
    }
    double inv = ext > 0.0 ? 1024.0 / ext : 0.0;
    if (!(inv < 1.0e300)) inv = 0.0;
    const double* base = xyz + 3 * (src_off[c.tree] + c.start);
    i64 dst = trees[c.tree].pt_off + c.start;
    for (int i = threadIdx.x; i < c.count; i += 256) {
        unsigned q[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            double f = (base[3 * i + a] - lo[a]) * inv;
            int v = (f >= 0.0) ? (f < 1023.0 ? (int)f : 1023) : 0;  // NaN -> 0
            q[a] = (unsigned)v;
        }
        if (hilbert) hilbert_transpose10(q);
        keys[dst + i] = (u64)((spread10(q[0]) << 2) | (spread10(q[1]) << 1) | spread10(q[2]));
        vals[dst + i] = (uint32_t)(c.start + i);
    }
}

// seed-grid origin and extent of every tree (device copy of the descriptors only)
__global__ void k_tree_bounds(TreeDesc* __restrict__ trees, const long long* __restrict__ bb, int n_trees) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_trees) return;
    double ext = 0.0;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        double lo = 0.0, hi = 0.0;
        if (trees[t].n > 0) {
            lo = double_from_ordered(bb[6 * t + a]);
            hi = double_from_ordered(bb[6 * t + 3 + a]);
        }
        trees[t].glo[a] = lo;
        ext = fmax(ext, hi - lo);
    }
    trees[t].gext = ext;
    trees[t].ginv = 1.0;
}

// gathers the sorted points into AoS and builds the level-0 boxes (one warp per leaf)
__global__ void __launch_bounds__(256) k_gather_leaves(const double* __restrict__ xyz, const i64* __restrict__ src_off,
                                                       const Chunk* __restrict__ chunks,
                                                       const TreeDesc* __restrict__ trees,
                                                       const uint32_t* __restrict__ sorted_vals,
                                                       TreePoint* __restrict__ pts, float4* __restrict__ pts32,
                                                       float* __restrict__ boxes) {
    Chunk c = chunks[blockIdx.x];
    const TreeDesc& T = trees[c.tree];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const double* base = xyz + 3 * src_off[c.tree];
    for (int l = warp; l * 32 < c.count; l += 8) {
        int j = c.start + l * 32 + lane;  // cloud-local sorted position
        bool valid = j < T.n;
        double x = 0, y = 0, z = 0;
        if (valid) {
            int o = (int)sorted_vals[T.pt_off + j];
            x = base[3 * (i64)o + 0];
            y = base[3 * (i64)o + 1];
            z = base[3 * (i64)o + 2];
            TreePoint P;
            P.x = x; P.y = y; P.z = z; P.idx = o; P.pad = 0;
            pts[T.pt_off + j] = P;
        }
        double lo[3] = {valid ? x : INFINITY, valid ? y : INFINITY, valid ? z : INFINITY};
        double hi[3] = {valid ? x : -INFINITY, valid ? y : -INFINITY, valid ? z : -INFINITY};
#pragma unroll
        for (int a = 0; a < 3; ++a) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                lo[a] = fmin(lo[a], shfl_d_xor(lo[a], o));
                hi[a] = fmax(hi[a], shfl_d_xor(hi[a], o));
            }
        }
        const float l0 = __double2float_rd(lo[0]), l1 = __double2float_rd(lo[1]), l2 = __double2float_rd(lo[2]);
        // float32 offsets from the leaf box's lower corner (as stored: rounded down to float32), the coordinates of
        // k_self_knn's approximate distances: a value is at most the leaf's extent, so its rounding error is
        // 2^-24 of THAT, not of the coordinate itself
        if (valid)
            pts32[T.pt_off + j] = make_float4((float)(x - (double)l0), (float)(y - (double)l1), (float)(z - (double)l2), 0.f);
        if (lane == 0) {
            float* b = boxes + 6 * (T.box_off[0] + (c.start >> 5) + l);
            b[0] = l0;
            b[1] = l1;
            b[2] = l2;
            b[3] = __double2float_ru(hi[0]);
            b[4] = __double2float_ru(hi[1]);
            b[5] = __double2float_ru(hi[2]);
        }
    }
}

// level >= 1: box b bounds the boxes [32b, 32b+32) of the level below.  One block per tree, warps stride over boxes.
__global__ void __launch_bounds__(256) k_boxes_up(const TreeDesc* __restrict__ trees, int level,
                                                  float* __restrict__ boxes) {
    const TreeDesc& T = trees[blockIdx.x];
    if (level > T.top) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int n_child = T.box_cnt[level - 1];
    for (int b = warp; b < T.box_cnt[level]; b += 8) {
        int ci = b * 32 + lane;
        float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
        if (ci < n_child) {
            const float* cb = boxes + 6 * (T.box_off[level - 1] + ci);
            lo[0] = cb[0]; lo[1] = cb[1]; lo[2] = cb[2];
            hi[0] = cb[3]; hi[1] = cb[4]; hi[2] = cb[5];
        }
#pragma unroll
        for (int a = 0; a < 3; ++a) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
                hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
            }
        }
        if (lane == 0) {
            float* ob = boxes + 6 * (T.box_off[level] + b);
            ob[0] = lo[0]; ob[1] = lo[1]; ob[2] = lo[2];
            ob[3] = hi[0]; ob[4] = hi[1]; ob[5] = hi[2];
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// host: build
// ---------------------------------------------------------------------------------------------------------------
void tree_store_need(i64 n, i64* boxes, i64* slots) {  // the layout loop of forest_append for one tree
    i64 nb = 0, cnt = (n + 31) / 32;
    while (true) {
        nb += cnt;
        if (cnt <= 32) break;
        cnt = (cnt + 31) / 32;
    }
    int lg = 6;
    while (((i64)1 << lg) < 2 * n) ++lg;
    *boxes = nb;
    *slots = (i64)1 << lg;
}

void forest_free(Forest* f) {
    if (!f) return;
    if (!f->in_arena && !f->store) {
        // cudaFree only fails on a context that is already broken (a sticky error of an earlier kernel): it is recorded
        // for sb_last_error, there is nothing else to do with it while tearing down
        cudaError_t e = cudaSuccess;
        auto rel = [&](void* p) { const cudaError_t r = cudaFree(p); if (r != cudaSuccess) e = r; };
        for (ForestBatch& B : f->batches) {
            rel(B.pts); rel(B.pts32); rel(B.boxes); rel(B.normals); rel(B.nbr); rel(B.grid);
        }
        rel(f->d_trees);
        if (e != cudaSuccess && f->ctx) fail(f->ctx, SB_ERR_CUDA, "index: cudaFree failed: %s", cudaGetErrorString(e));
    }
    f->batches.clear();
    f->d_trees = nullptr;
    f->h_trees.clear();
    f->n_trees = 0; f->cap_trees = 0; f->n_points = 0; f->normals_k = 0;
}

int forest_reserve(Ctx* ctx, Forest* f, int cap_trees) {
    f->ctx = ctx;
    if (f->d_trees) return fail(ctx, SB_ERR_INVALID_ARG, "forest: already reserved");
    const size_t cap = (size_t)(cap_trees > 0 ? cap_trees : 1);
    if (f->in_arena) SB_TRY(arena_get(ctx, cap, &f->d_trees));
    else SB_CUDA(ctx, cudaMalloc(&f->d_trees, sizeof(TreeDesc) * cap));
    f->cap_trees = cap_trees;
    f->h_trees.reserve(cap);
    return SB_OK;
}

int forest_build(Ctx* ctx, const double* d_xyz, const i64* h_off, const int* cloud_ids, int n_trees, Forest* f) {
    SB_TRY(forest_reserve(ctx, f, n_trees));
    return forest_append(ctx, f, d_xyz, h_off, cloud_ids, n_trees);
}

int forest_append(Ctx* ctx, Forest* f, const double* d_xyz, const i64* h_off, const int* cloud_ids, int n_new) {
    if (f->n_trees + n_new > f->cap_trees) return fail(ctx, SB_ERR_CAPACITY, "forest: more trees than reserved");
    const int t0 = f->n_trees;
    ForestBatch B;
    B.t0 = t0;
    B.n_trees = n_new;
    f->h_trees.resize((size_t)(t0 + n_new));
    std::vector<i64> src_off((size_t)n_new), seg_off((size_t)n_new + 1);
    std::vector<Chunk> chunks;
    i64 np = 0, nb = 0, n_slots = 0;
    int max_top = 0;
    for (int t = 0; t < n_new; ++t) {
        int c = cloud_ids ? cloud_ids[t] : t;
        i64 n64 = h_off[c + 1] - h_off[c];
        if (n64 < 0 || n64 > 0x7fffffffLL) return fail(ctx, SB_ERR_RANGE, "index: cloud %d has %lld rows", c, n64);
        TreeDesc& T = f->h_trees[(size_t)(t0 + t)];
        memset(&T, 0, sizeof(T));
        T.pt_off = np;
        T.out_off = f->n_points + np;
        T.n = (int)n64;
        src_off[t] = h_off[c];
        seg_off[t] = np;
        int cnt = (T.n + 31) / 32, lev = 0;
        while (true) {
            T.box_off[lev] = nb;
            T.box_cnt[lev] = cnt;
            nb += cnt;
            if (cnt <= 32) break;
            cnt = (cnt + 31) / 32;
            ++lev;
        }
        T.top = lev;
        if (lev > max_top) max_top = lev;
        {  // seed grid: a power-of-two table with at least 2 slots per point
            int lg = 6;
            while (((i64)1 << lg) < 2 * (i64)T.n) ++lg;
            T.tab_off = n_slots;
            T.tab_shift = 64 - lg;
            n_slots += (i64)1 << lg;
        }
        for (int s = 0; s < T.n; s += CHUNK) {
            Chunk ch;
            ch.tree = t; ch.start = s; ch.count = T.n - s < CHUNK ? T.n - s : CHUNK; ch.pad = 0;
            chunks.push_back(ch);
        }
        np += T.n;
    }
    seg_off[n_new] = np;
    B.n_points = np;
    B.n_boxes = nb;
    B.n_slots = n_slots;
    if (np >= (i64)0xffffffffLL) return fail(ctx, SB_ERR_RANGE, "index: more than 2^32-1 points in one batch of trees");
    size_t npa = (size_t)(np > 0 ? np : 1), nba = (size_t)(nb > 0 ? nb : 1);
    if (f->store) {
        const TreeStore& S = *f->store;
        if (!f->batches.empty() || np > S.cap_points || nb > S.cap_boxes || n_slots > S.cap_slots)
            return fail(ctx, SB_ERR_CAPACITY, "forest: batch does not fit the caller's tree store");
        B.pts = S.pts;
        B.pts32 = S.pts32;
        B.boxes = S.boxes;
    } else if (f->in_arena) {
        SB_TRY(arena_get(ctx, npa, &B.pts));
        SB_TRY(arena_get(ctx, npa, &B.pts32));
        SB_TRY(arena_get(ctx, 6 * nba, &B.boxes));
    } else {
        SB_CUDA(ctx, cudaMalloc(&B.pts, sizeof(TreePoint) * npa));
        SB_CUDA(ctx, cudaMalloc(&B.pts32, sizeof(float4) * npa));
        SB_CUDA(ctx, cudaMalloc(&B.boxes, sizeof(float) * 6 * nba));
    }
    for (int t = 0; t < n_new; ++t) {
        f->h_trees[(size_t)(t0 + t)].pts = B.pts;
        f->h_trees[(size_t)(t0 + t)].pts32 = B.pts32;
        f->h_trees[(size_t)(t0 + t)].boxes = B.boxes;
    }
    f->batches.push_back(B);
    f->n_trees = t0 + n_new;
    f->n_points += np;
    TreeDesc* d_new = f->d_trees + t0;
    if (n_new > 0)
        SB_TRY(table_upload(ctx, d_new, f->h_trees.data() + t0, sizeof(TreeDesc) * (size_t)n_new));
    if (np == 0) return SB_OK;

    const ArenaMark mark = arena_mark(ctx);  // everything below is scratch of this build
    i64* d_src_off;
    Chunk* d_chunks;
    long long* d_bb;
    u64 *ka, *kb, *ks;
    uint32_t *va, *vb, *vs;
    SB_TRY(arena_get(ctx, (size_t)n_new, &d_src_off));
    SB_TRY(arena_get(ctx, chunks.size(), &d_chunks));
    SB_TRY(arena_get(ctx, (size_t)6 * n_new, &d_bb));
    SB_TRY(arena_get(ctx, (size_t)np, &ka));
    SB_TRY(arena_get(ctx, (size_t)np, &kb));
    SB_TRY(arena_get(ctx, (size_t)np, &va));
    SB_TRY(arena_get(ctx, (size_t)np, &vb));
    SB_TRY(table_upload(ctx, d_src_off, src_off.data(), sizeof(i64) * (size_t)n_new));
    SB_TRY(table_upload(ctx, d_chunks, chunks.data(), sizeof(Chunk) * chunks.size()));
    {
        std::vector<long long> init((size_t)6 * n_new);
        for (int t = 0; t < n_new; ++t)
            for (int a = 0; a < 3; ++a) { init[6 * t + a] = INT64_MAX; init[6 * t + 3 + a] = INT64_MIN; }
        SB_TRY(table_upload(ctx, d_bb, init.data(), sizeof(long long) * init.size()));
    }
    unsigned nch = (unsigned)chunks.size();
    SB_LAUNCH(ctx, k_bbox, nch, 256, 0, d_xyz, d_src_off, d_chunks, d_bb);
    // Hilbert order by default (SB_INDEX_CURVE=morton for the Z-order curve): measured on 1000 scans, normals 19.7 ->
    // 17.1 ms and the ICP loop 13.7 -> 13.4 ms; results do not depend on the order
    static const int hilbert = getenv("SB_INDEX_CURVE") ? (strcmp(getenv("SB_INDEX_CURVE"), "morton") != 0) : 1;
    SB_LAUNCH(ctx, k_morton, nch, 256, 0, d_xyz, d_src_off, d_chunks, d_bb, d_new, ka, va, hilbert);
    SB_LAUNCH(ctx, k_tree_bounds, ceil_div(n_new, 128), 128, 0, d_new, d_bb, n_new);
    SB_TRY(segmented_sort_pairs(ctx, ka, kb, va, vb, seg_off.data(), n_new, 30, &ks, &vs));
    SB_LAUNCH(ctx, k_gather_leaves, nch, 256, 0, d_xyz, d_src_off, d_chunks, d_new, vs, B.pts, B.pts32, B.boxes);
    for (int l = 1; l <= max_top; ++l) SB_LAUNCH(ctx, k_boxes_up, (unsigned)n_new, 256, 0, d_new, l, B.boxes);
    arena_release(ctx, mark);
    return SB_OK;
}

int make_items_dev(Ctx* ctx, const std::vector<QueryItem>& items, QueryItem** d_items) {
    SB_TRY(arena_get(ctx, items.size() ? items.size() : 1, d_items));
    if (!items.empty()) {
        SB_CUDA(ctx, cudaMemcpyAsync(*d_items, items.data(), sizeof(QueryItem) * items.size(), cudaMemcpyHostToDevice,
                                     ctx->stream));
        SB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return SB_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// query kernels: one warp per 32-query item, persistent grid
// ---------------------------------------------------------------------------------------------------------------
static constexpr int QWARPS = 8;

__device__ __forceinline__ void load_tree(TreeDesc* dst, const TreeDesc* src, int lane) {
    const int* s = reinterpret_cast<const int*>(src);
    int* d = reinterpret_cast<int*>(dst);
    for (int i = lane; i < (int)(sizeof(TreeDesc) / 4); i += 32) d[i] = s[i];
    __syncwarp();
}

// Next work item of a warp: from a device-wide counter (work != nullptr: a grid of resident CTAs whose warps finish
// at different times keeps all of them busy to the end), else a fixed share (item = warp id + r * warps of the grid).
__device__ __forceinline__ i64 next_work(int* __restrict__ work, i64 prev, int lane, int warp, int wpb) {
    if (!work) return prev < 0 ? (i64)blockIdx.x * wpb + warp : prev + (i64)gridDim.x * wpb;
    int v = 0;
    if (lane == 0) v = atomicAdd(work, 1);
    return (i64)__shfl_sync(0xffffffffu, v, 0);
}

__global__ void __launch_bounds__(QWARPS * 32) k_nearest(ForestView F, const double* __restrict__ q,
                                                         const QueryItem* __restrict__ items, i64 n_items,
                                                         int* __restrict__ out_idx, double* __restrict__ out_d2,
                                                         int* __restrict__ out_pos) {
    __shared__ WarpStack stacks[QWARPS];
    __shared__ TreeDesc s_tree[QWARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    WarpStack& S = stacks[warp];
    for (i64 it = (i64)blockIdx.x * QWARPS + warp; it < n_items; it += (i64)gridDim.x * QWARPS) {
        QueryItem I = items[it];
        __syncwarp();
        load_tree(&s_tree[warp], &F.trees[I.tree], lane);
        const TreeDesc& T = s_tree[warp];
        double mx = 0, my = 0, mz = 0;
        if (lane < I.count) {
            const double* p = q + 3 * (I.q_off + lane);
            mx = p[0]; my = p[1]; mz = p[2];
        }
        int r_idx = -1, r_pos = -1;
        double r_d = 1.7976931348623157e308;
        for (int j = 0; j < I.count; ++j) {
            double qx = shfl_d(mx, j), qy = shfl_d(my, j), qz = shfl_d(mz, j);
            NearestVisitor V(F, T, qx, qy, qz, lane);
            traverse(F, T, qx, qy, qz, S, V, lane);
            if (lane == j) { r_idx = V.best_idx; r_pos = V.best_pos; r_d = V.best_d; }
        }
        if (lane < I.count) {
            out_idx[I.q_off + lane] = r_idx;
            if (out_d2) out_d2[I.q_off + lane] = r_d;
            if (out_pos) out_pos[I.q_off + lane] = r_pos;
        }
    }
}

// ----- 3x3 symmetric eigen-decomposition: cyclic Jacobi, the oracle's operation order (oracle/slam_oracle.cpp
// jacobi3; Eigen's SelfAdjointEigenSolver at icp.hpp:55 is an iterative QR — see DESIGN.md "normals").
// This translation unit is compiled with -fmad=false so every * and + below is a separately rounded IEEE op.
template <int P, int Q, int K>
__device__ __forceinline__ void jacobi_rotate(double (&A)[3][3], double (&V)[3][3]) {
    double apq = A[P][Q];
    if (apq == 0.0) return;
    double theta = (A[Q][Q] - A[P][P]) / (2.0 * apq);
    double t = 1.0 / (fabs(theta) + sqrt(theta * theta + 1.0));
    if (theta < 0.0) t = -t;
    double c = 1.0 / sqrt(t * t + 1.0);
    double s = t * c;
    double app = A[P][P], aqq = A[Q][Q];
    A[P][P] = app - t * apq;
    A[Q][Q] = aqq + t * apq;
    A[P][Q] = 0.0; A[Q][P] = 0.0;
    double akp = A[K][P], akq = A[K][Q];
    A[K][P] = c * akp - s * akq; A[P][K] = A[K][P];
    A[K][Q] = s * akp + c * akq; A[Q][K] = A[K][Q];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        double vip = V[i][P], viq = V[i][Q];
        V[i][P] = c * vip - s * viq;
        V[i][Q] = s * vip + c * viq;
    }
}

__device__ __forceinline__ void jacobi3(double (&A)[3][3], double (&w)[3], double (&V)[3][3]) {
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) V[i][j] = (i == j) ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 12; ++sweep) {
        // converged: the rotations left are the identity in fp64 (same test, same expression as the oracle's jacobi3)
        double off = fabs(A[0][1]) + fabs(A[0][2]) + fabs(A[1][2]);
        if (off <= 1.0e-25 * ((fabs(A[0][0]) + fabs(A[1][1])) + fabs(A[2][2]))) break;
        jacobi_rotate<0, 1, 2>(A, V);
        jacobi_rotate<0, 2, 1>(A, V);
        jacobi_rotate<1, 2, 0>(A, V);
    }
    w[0] = A[0][0]; w[1] = A[1][1]; w[2] = A[2][2];
}

// Normal of one sorted point from its m nearest neighbours (cloud-local sorted positions nb[0], nb[stride], ...,
// ascending by (d2, idx), the point itself included): icp.hpp:34-63 in the oracle's operation order.  One thread.
__device__ __forceinline__ void normal_of_point(const TreeDesc& T, const int* nb, int stride, int m, i64 ps,
                                                TreeNormal* __restrict__ nrm_sorted, double* __restrict__ nrm_orig,
                                                double* __restrict__ evals_orig) {
    double n0 = 0.0, n1 = 0.0, n2 = 1.0, e0 = 0.0, e1 = 0.0, e2 = 0.0;
    if (m >= 3) {  // icp.hpp:34-37
        double c0 = 0.0, c1 = 0.0, c2 = 0.0;
        for (int j = 0; j < m; ++j) {  // icp.hpp:40-44, neighbours ascending by (d2, idx)
            TreePoint P = load_point(T.pts + T.pt_off + nb[j * stride]);
            c0 += P.x; c1 += P.y; c2 += P.z;
        }
        double md = (double)m;
        c0 /= md; c1 /= md; c2 /= md;
        double C00 = 0, C01 = 0, C02 = 0, C11 = 0, C12 = 0, C22 = 0;
        for (int j = 0; j < m; ++j) {  // icp.hpp:47-52
            TreePoint P = load_point(T.pts + T.pt_off + nb[j * stride]);
            double d0 = P.x - c0, d1 = P.y - c1, d2 = P.z - c2;
            C00 += d0 * d0; C01 += d0 * d1; C02 += d0 * d2;
            C11 += d1 * d1; C12 += d1 * d2; C22 += d2 * d2;
        }
        double A[3][3], w[3], V[3][3];
        A[0][0] = C00 / md; A[0][1] = C01 / md; A[0][2] = C02 / md;
        A[1][0] = A[0][1];  A[1][1] = C11 / md; A[1][2] = C12 / md;
        A[2][0] = A[0][2];  A[2][1] = A[1][2];  A[2][2] = C22 / md;
        jacobi3(A, w, V);
        // eigenvector of the smallest eigenvalue, first index on ties (icp.hpp:56 col(0))
        double v0 = V[0][0], v1 = V[1][0], v2 = V[2][0], ws = w[0];
        if (w[1] < ws) { ws = w[1]; v0 = V[0][1]; v1 = V[1][1]; v2 = V[2][1]; }
        if (w[2] < ws) { ws = w[2]; v0 = V[0][2]; v1 = V[1][2]; v2 = V[2][2]; }
        if (v2 < 0.0) { v0 = -v0; v1 = -v1; v2 = -v2; }  // icp.hpp:59-61
        double nn = sqrt((v0 * v0 + v1 * v1) + v2 * v2);  // icp.hpp:63
        n0 = v0 / nn; n1 = v1 / nn; n2 = v2 / nn;
        // ascending eigenvalues (diagnostic output)
        e0 = w[0]; e1 = w[1]; e2 = w[2];
        if (e1 < e0) { double t = e0; e0 = e1; e1 = t; }
        if (e2 < e1) { double t = e1; e1 = e2; e2 = t; }
        if (e1 < e0) { double t = e0; e0 = e1; e1 = t; }
    }
    TreeNormal Nn;
    Nn.x = n0; Nn.y = n1; Nn.z = n2; Nn.pad = 0.0;
    nrm_sorted[ps] = Nn;
    i64 po = T.out_off + T.pts[ps].idx;
    if (nrm_orig) { nrm_orig[3 * po + 0] = n0; nrm_orig[3 * po + 1] = n1; nrm_orig[3 * po + 2] = n2; }
    if (evals_orig) { evals_orig[3 * po + 0] = e0; evals_orig[3 * po + 1] = e1; evals_orig[3 * po + 2] = e2; }
}

// largest s in [0, n) with off[s] <= x (off ascending, off[0] <= x), called by the whole (converged) warp with the same
// arguments: every step tests 32 evenly spaced entries at once — three dependent loads for 4096 clouds where the
// binary search took twelve (14 % of k_normals_from_graph's stall samples: every warp starts with this search).
__device__ __forceinline__ int find_segment(const i64* __restrict__ off, int n, i64 x) {
    const int lane = threadIdx.x & 31;
    int lo = 0, len = n;
    while (len > 1) {
        const int step = (len + 31) >> 5;
        const int idx = lo + lane * step;
        const bool le = idx < lo + len && off[idx] <= x;   // true for a prefix of the lanes, lane 0 included
        const int j = 31 - __clz(__ballot_sync(0xffffffffu, le) | 1u);
        const int end = lo + len;
        lo += j * step;
        len = end - lo < step ? end - lo : step;
    }
    return lo;
}

// MODE 0: k-NN of external queries -> out_idx/out_d2 (row-major nq x k)
// MODE 1: normals of the trees' own points (queries are the sorted points; item.q_off is cloud-local sorted start)
template <int MODE>
__global__ void __launch_bounds__(QWARPS * 32, 4) k_knn(ForestView F, const double* __restrict__ q,
                                                     const QueryItem* __restrict__ items, i64 n_items, int k,
                                                     int* __restrict__ out_idx, double* __restrict__ out_d2,
                                                     TreeNormal* __restrict__ nrm_sorted,
                                                     NbrEntry* __restrict__ nbr_sorted, double* __restrict__ nrm_orig,
                                                     double* __restrict__ evals_orig, int n_trees_or_zero,
                                                     unsigned long long* __restrict__ spacing_acc, int qpi,
                                                     int* __restrict__ work) {
    __shared__ WarpStack stacks[QWARPS];
    __shared__ TreeDesc s_tree[QWARPS];
    __shared__ int s_nbr[MODE == 1 ? QWARPS : 1][32][33];  // neighbour positions (cloud-local sorted), padded
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    WarpStack& S = stacks[warp];
    for (i64 it = next_work(work, -1, lane, warp, QWARPS); it < n_items; it = next_work(work, it, lane, warp, QWARPS)) {
        QueryItem I;
        if (MODE == 1) {
            // implicit items: tree_item_off (passed in `items`' place as i64 prefix sums) -> (tree, 32-point chunk)
            const i64* tio = reinterpret_cast<const i64*>(items);
            int t = find_segment(tio, n_trees_or_zero, it);
            I.tree = t;
            // qpi consecutive points per work item: 32 for batches; a single small cloud (the streaming path) is cut
            // finer so that it still fills the chip (see forest_normals)
            I.q_off = (it - tio[t]) * qpi;
            int rem = F.trees[t].n - (int)I.q_off;
            I.count = rem < qpi ? rem : qpi;
        } else {
            I = items[it];
        }
        __syncwarp();
        load_tree(&s_tree[warp], &F.trees[I.tree], lane);
        const TreeDesc& T = s_tree[warp];
        double mx = 0, my = 0, mz = 0;
        if (lane < I.count) {
            if (MODE == 1) {
                TreePoint P = load_point(T.pts + T.pt_off + I.q_off + lane);
                mx = P.x; my = P.y; mz = P.z;
            } else {
                const double* p = q + 3 * (I.q_off + lane);
                mx = p[0]; my = p[1]; mz = p[2];
            }
        }
        int my_m = 0;
        unsigned long long spacing = 0ull;  // lane 1: sum of the nearest-other-point distances, 16.16 fixed point
        int prev_pos = -1;  // this lane's entry of the previous query's list: the seed of the next query
        if (MODE == 1) prev_pos = (int)I.q_off + lane < T.n ? (int)I.q_off + lane : -1;  // own leaf: 32 distinct points
        for (int j = 0; j < I.count; ++j) {
            double qx = shfl_d(mx, j), qy = shfl_d(my, j), qz = shfl_d(mz, j);
            KnnVisitor V(F, T, qx, qy, qz, lane, k);
            if (MODE == 1 || j > 0) V.seed(prev_pos);
            traverse(F, T, qx, qy, qz, S, V, lane);
            prev_pos = V.lpos;
            bool have = lane < k && V.lidx != 0x7fffffff;
            int m = __popc(__ballot_sync(0xffffffffu, have));
            if (MODE == 1) {
                if (lane < k) {
                    s_nbr[warp][j][lane] = V.lpos;
                    // the neighbour graph of icp.cu: position + a lower bound of the distance (padding: -1, +inf)
                    NbrEntry e;
                    e.pos = have ? V.lpos : -1;
                    e.r = have ? sqrt_lower(V.ld) : __int_as_float(0x7f800000);
                    nbr_sorted[(T.pt_off + I.q_off + j) * k + lane] = e;
                    if (lane == 1 && have) spacing += (unsigned long long)(fminf(e.r, 1.0e6f) * 65536.0f);
                    if (lane == 1) const_cast<TreePoint*>(T.pts)[T.pt_off + I.q_off + j].pad = have ? __float_as_int(e.r) : 0;
                }
                if (lane == j) my_m = m;
            } else {
                if (lane < k) {
                    i64 o = (I.q_off + j) * k + lane;
                    out_idx[o] = have ? V.lidx : -1;
                    if (out_d2) out_d2[o] = have ? V.ld : 1.7976931348623157e308;
                }
            }
        }
        if (MODE == 1) {
            if (lane == 1 && spacing) atomicAdd(&spacing_acc[I.tree], spacing);  // integer: order-independent
            __syncwarp();
            if (lane < I.count)
                normal_of_point(T, s_nbr[warp][lane], 1, my_m, T.pt_off + I.q_off + lane, nrm_sorted, nrm_orig, evals_orig);
            __syncwarp();
        }
    }
}


#include "selfknn.cuh"

// ----- seed grid: cell size = 3 x the mean distance to the nearest other point, one representative point per cell
__global__ void k_grid_params(TreeDesc* __restrict__ trees, const unsigned long long* __restrict__ spacing_acc,
                              int n_trees) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_trees) return;
    const int n = trees[t].n;
    double h = n > 0 ? 3.0 * ((double)spacing_acc[t] / 65536.0) / (double)n : 1.0;
    if (!(h > 1.0e-9) || !(h < 1.0e9)) h = 1.0;
    const double ext = trees[t].gext;
    if (ext / h > 1.0e6) h = ext / 1.0e6;  // keep the cell coordinates inside 21 bits
    trees[t].ginv = 1.0 / h;
}

// one warp per leaf (implicit items like k_knn<1>): every point claims the slot of its cell
__global__ void __launch_bounds__(256) k_grid_build(ForestView F, const i64* __restrict__ tio, i64 n_items, int n_trees,
                                                    GridSlot* __restrict__ grid) {
    const int lane = threadIdx.x & 31;
    i64 it = ((i64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (it >= n_items) return;
    const int t = find_segment(tio, n_trees, it);
    const TreeDesc& T = F.trees[t];
    const int pos = (int)(it - tio[t]) * 32 + lane;
    if (pos >= T.n) return;
    TreePoint P = load_point(T.pts + T.pt_off + pos);
    int ix, iy, iz;
    if (!grid_cell(T, P.x, P.y, P.z, ix, iy, iz)) return;  // NaN coordinates: not a seed
    const unsigned long long key = grid_key(ix, iy, iz);
    const unsigned mask = (unsigned)(((i64)1 << (64 - T.tab_shift)) - 1);
    GridSlot* tab = T.grid + T.tab_off;
    unsigned slot = grid_hash(key, T.tab_shift);
    while (true) {
        unsigned long long prev = atomicCAS(&tab[slot].key, SB_GRID_EMPTY, key);
        if (prev == SB_GRID_EMPTY || prev == key) {
            tab[slot].pos = pos;  // any point of the cell will do
            break;
        }
        slot = (slot + 1u) & mask;
    }
}

static ForestView view_of(const Forest* f, int t0 = 0) {
    ForestView v;
    v.trees = f->d_trees + t0;
    return v;
}

// pointers to the arrays forest_normals allocates, into the descriptors of one batch of trees
__global__ void k_tree_attach(TreeDesc* __restrict__ trees, int n_trees, TreeNormal* nrm, NbrEntry* nbr, GridSlot* grid) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_trees) return;
    trees[t].nrm = nrm;
    trees[t].nbr = nbr;
    trees[t].grid = grid;
}

static int query_grid(Ctx* ctx, i64 n_items) {
    i64 blocks = (n_items + QWARPS - 1) / QWARPS;
    static const int per_sm = getenv("SB_KNN_GRID") ? atoi(getenv("SB_KNN_GRID")) : 32;
    i64 cap = (i64)ctx->sm_count * per_sm;  // persistent grid: more CTAs than fit at once evens out uneven items
    return (int)(blocks < cap ? (blocks > 0 ? blocks : 1) : cap);
}

int forest_nearest(Ctx* ctx, const Forest* f, const double* d_q, const QueryItem* d_items, i64 n_items,
                   int* d_out_idx, double* d_out_d2, int* d_out_pos) {
    if (n_items <= 0) return SB_OK;
    SB_LAUNCH(ctx, k_nearest, query_grid(ctx, n_items), QWARPS * 32, 0, view_of(f), d_q, d_items, n_items, d_out_idx,
              d_out_d2, d_out_pos);
    return SB_OK;
}

int forest_knn(Ctx* ctx, const Forest* f, const double* d_q, const QueryItem* d_items, i64 n_items, int k,
               int* d_out_idx, double* d_out_d2) {
    if (n_items <= 0) return SB_OK;
    SB_LAUNCH(ctx, k_knn<0>, query_grid(ctx, n_items), QWARPS * 32, 0, view_of(f), d_q, d_items, n_items, k, d_out_idx,
              d_out_d2, nullptr, nullptr, nullptr, nullptr, 0, nullptr, 32, nullptr);
    return SB_OK;
}

int forest_normals(Ctx* ctx, Forest* f, int k, double* d_out_normals, double* d_out_evals, int batch) {
    if (f->batches.empty()) return SB_OK;
    if (batch < 0) batch = (int)f->batches.size() - 1;
    if (batch >= (int)f->batches.size()) return fail(ctx, SB_ERR_INVALID_ARG, "normals: no such batch of trees");
    ForestBatch& B = f->batches[(size_t)batch];
    if (f->batches.size() > 1 && f->normals_k != 0 && f->normals_k != k)
        return fail(ctx, SB_ERR_INVALID_ARG, "normals: every batch of a forest must use the same k");
    const size_t npa = (size_t)(B.n_points > 0 ? B.n_points : 1);
    const size_t nsa = (size_t)(B.n_slots > 0 ? B.n_slots : 1);
    if (f->store) {
        const TreeStore& S = *f->store;
        if (k > S.cap_k || B.n_slots > S.cap_slots || B.n_points > S.cap_points)
            return fail(ctx, SB_ERR_CAPACITY, "normals: batch does not fit the caller's tree store");
        B.normals = S.normals;
        B.nbr = S.nbr;
        B.grid = S.grid;
    } else if (f->in_arena) {
        SB_TRY(arena_get(ctx, npa, &B.normals));
        SB_TRY(arena_get(ctx, npa * (size_t)k, &B.nbr));
        SB_TRY(arena_get(ctx, nsa, &B.grid));
    } else {
        if (!B.grid) SB_CUDA(ctx, cudaMalloc(&B.grid, sizeof(GridSlot) * nsa));
        if (!B.normals) SB_CUDA(ctx, cudaMalloc(&B.normals, sizeof(TreeNormal) * npa));
        if (B.nbr && f->normals_k != k) {
            SB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            cudaFree(B.nbr);
            B.nbr = nullptr;
        }
        if (!B.nbr) SB_CUDA(ctx, cudaMalloc(&B.nbr, sizeof(NbrEntry) * npa * (size_t)k));
    }
    f->normals_k = k;
    TreeDesc* d_bt = f->d_trees + B.t0;
    for (int t = 0; t < B.n_trees; ++t) {
        TreeDesc& T = f->h_trees[(size_t)(B.t0 + t)];
        T.nrm = B.normals; T.nbr = B.nbr; T.grid = B.grid;
    }
    if (B.n_trees > 0)
        SB_LAUNCH(ctx, k_tree_attach, ceil_div(B.n_trees, 128), 128, 0, d_bt, B.n_trees, B.normals, B.nbr, B.grid);
    // implicit work items: chunk c of tree t is item tree_item_off[t] + c (no per-item table to build or upload)
    std::vector<i64> tio((size_t)B.n_trees + 1, 0);
    for (int t = 0; t < B.n_trees; ++t) tio[t + 1] = tio[t] + (f->h_trees[(size_t)(B.t0 + t)].n + 31) / 32;
    i64 n_items = tio[B.n_trees];
    if (n_items == 0) return SB_OK;
    const ArenaMark mark = arena_mark(ctx);
    i64* d_tio;
    unsigned long long* d_spacing;
    SB_TRY(arena_get(ctx, tio.size(), &d_tio));
    SB_TRY(arena_get(ctx, (size_t)B.n_trees + 1, &d_spacing));   // + the work counter of k_knn<1>
    SB_TRY(table_upload(ctx, d_tio, tio.data(), sizeof(i64) * tio.size()));
    SB_CUDA(ctx, cudaMemsetAsync(d_spacing, 0, sizeof(unsigned long long) * ((size_t)B.n_trees + 1), ctx->stream));
    // work items handed out by a counter to a grid of resident CTAs (SB_KNN_DYN = CTAs per SM, 0: fixed shares)
    static const int dyn = getenv("SB_KNN_DYN") ? atoi(getenv("SB_KNN_DYN")) : 4;
    int* d_work_knn = dyn > 0 ? reinterpret_cast<int*>(d_spacing + B.n_trees) : nullptr;
    auto knn_grid = [&](i64 items) -> int {
        if (!d_work_knn || items >= 0x7fff0000LL) return query_grid(ctx, items);
        const i64 blocks = (items + QWARPS - 1) / QWARPS, cap = (i64)ctx->sm_count * dyn;
        return (int)(blocks < cap ? (blocks > 0 ? blocks : 1) : cap);
    };
    SB_CUDA(ctx, cudaMemsetAsync(B.grid, 0xff, sizeof(GridSlot) * (size_t)B.n_slots, ctx->stream));
    // one lane per query (k_self_knn) for the k the pipelines use; SB_KNN_PACKET=0 or any other k: one warp per query
    static const bool packet = !(getenv("SB_KNN_PACKET") && atoi(getenv("SB_KNN_PACKET")) == 0);
    // k = 10 (config C3: 44 k-point clouds at voxel 0.2) stays with one warp per query unless SB_KNN_PACKET_K10=1: there
    // the packet kernel measured 4.70 ms against 4.37 ms per 47 clouds (4 % of its queries end in the redo list)
    static const bool packet10 = getenv("SB_KNN_PACKET_K10") && atoi(getenv("SB_KNN_PACKET_K10")) != 0;
    // A batch too small to fill the chip with one warp per 32 queries (a single scan: 266 packets on 148 SMs, where a
    // packet's 17 k dependent instructions took 0.44 ms): one warp per `qpi` queries with the warp-per-query kernel
    // instead — it executes 3x the instructions, but 16-32 warps per SM hide each other's latencies.
    int qpi = 32;
    while (qpi > 1 && B.n_points / qpi < (i64)ctx->sm_count * 24) qpi >>= 1;
    static const bool allow_small = !(getenv("SB_KNN_SMALL") && atoi(getenv("SB_KNN_SMALL")) == 0);
    if (qpi < 32 && allow_small) {
        std::vector<i64> tq((size_t)B.n_trees + 1, 0);
        for (int t = 0; t < B.n_trees; ++t) tq[t + 1] = tq[t] + (f->h_trees[(size_t)(B.t0 + t)].n + qpi - 1) / qpi;
        i64* d_tq;
        SB_TRY(arena_get(ctx, tq.size(), &d_tq));
        SB_TRY(table_upload(ctx, d_tq, tq.data(), sizeof(i64) * tq.size()));
        SB_LAUNCH(ctx, k_knn<1>, knn_grid(tq[B.n_trees]), QWARPS * 32, 0, view_of(f, B.t0), nullptr,
                  reinterpret_cast<const QueryItem*>(d_tq), tq[B.n_trees], k, nullptr, nullptr, B.normals, B.nbr,
                  d_out_normals, d_out_evals, B.n_trees, d_spacing, qpi, tq[B.n_trees] < 0x7fff0000LL ? d_work_knn : nullptr);
    } else if (packet && (k == 20 || (k == 10 && packet10))) {
        static const bool want_stats = getenv("SB_KNN_STATS") != nullptr;
        static const int pcap = getenv("SB_KNN_PCAP") ? atoi(getenv("SB_KNN_PCAP")) : 48;
        unsigned long long* d_stats = nullptr;
        if (want_stats) {
            SB_TRY(arena_get(ctx, (size_t)PS_N, &d_stats));
            SB_CUDA(ctx, cudaMemsetAsync(d_stats, 0, sizeof(unsigned long long) * PS_N, ctx->stream));
        }
        static const int per_sm = getenv("SB_KNN_GRID") ? atoi(getenv("SB_KNN_GRID")) : 32;
        i64 blocks = (n_items + PWARPS - 1) / PWARPS, cap = (i64)ctx->sm_count * per_sm;
        const int grid = (int)(blocks < cap ? blocks : cap);
        // queries the packet search leaves open (exact ties, float32 gaps): list + count for k_knn_redo
        RedoEntry* d_redo;
        int* d_redo_count;
        SB_TRY(arena_get(ctx, (size_t)B.n_points, &d_redo));
        SB_TRY(arena_get(ctx, (size_t)4, &d_redo_count));   // [1], [2]: the work counters of k_self_knn and k_knn_redo
        SB_CUDA(ctx, cudaMemsetAsync(d_redo_count, 0, 4 * sizeof(int), ctx->stream));
        int* d_work = (dyn > 0 && n_items < 0x7fff0000LL) ? d_redo_count + 1 : nullptr;
        static const int tot10 = getenv("SB_KNN_TOT10") ? atoi(getenv("SB_KNN_TOT10")) : 16;
        auto launch = [&](auto kern, int cap_entries) -> int {
            const int row = k | 1;
            const size_t entries = (size_t)(32 * row > cap_entries * 32 ? 32 * row : cap_entries * 32);
            const size_t smem = (size_t)PWARPS * entries * sizeof(int2);
            const unsigned bit = 1u << ((k == 20 ? 1 : 0) | (cap_entries >= 64 ? 2 : 0) | (want_stats ? 4 : 0) | (k == 10 && tot10 == 16 ? 8 : 0));
            if (!(ctx->knn_attr_done & bit)) {   // once per kernel instantiation and context (device)
                SB_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                ctx->knn_attr_done |= bit;
            }
            const int g = d_work ? (int)std::min<i64>(blocks, (i64)ctx->sm_count * dyn) : grid;
            SB_LAUNCH(ctx, kern, g, PWARPS * 32, smem, view_of(f, B.t0), d_tio, n_items, B.n_trees, B.nbr, d_redo,
                      d_redo_count, d_stats, d_work);
            return SB_OK;
        };
#define SB_SELF_KNN(KK, TT, CAP) (want_stats ? launch(k_self_knn<KK, TT, CAP, true>, CAP) : launch(k_self_knn<KK, TT, CAP, false>, CAP))
        // list + batch = 32 registers pairs for k = 20 (batches of 11); for k = 10 either 16 (batches of 5) or 32 (21)
        if (k == 20) SB_TRY(pcap >= 64 ? SB_SELF_KNN(20, 32, 64) : SB_SELF_KNN(20, 32, 48));
        else if (tot10 == 16) SB_TRY(SB_SELF_KNN(10, 16, 48));
        else SB_TRY(SB_SELF_KNN(10, 32, 48));
#undef SB_SELF_KNN
        SB_LAUNCH(ctx, k_knn_redo, ctx->sm_count * 8, QWARPS * 32, 0, view_of(f, B.t0), d_redo, d_redo_count, k, B.nbr,
                  d_work ? d_redo_count + 2 : nullptr);
        SB_LAUNCH(ctx, k_normals_from_graph, (unsigned)((n_items * 32 + 255) / 256), 256, 0, view_of(f, B.t0), d_tio,
                  n_items, B.n_trees, k, B.nbr, B.pts, B.normals, d_out_normals, d_out_evals, d_spacing);
        if (d_stats) {
            unsigned long long h[PS_N];
            SB_CUDA(ctx, cudaMemcpyAsync(h, d_stats, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
            SB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            const double np = (double)(h[PS_PACKETS] ? h[PS_PACKETS] : 1);
            fprintf(stderr, "[slam_b200] self-knn k=%d: %llu packets; per packet: leaves offered %.2f, scanned %.2f, candidates "
                    "%.1f, kept/lane %.1f, flushes %.2f, rounds %.2f, merges %.2f, redo queries %.4f\n", k, h[PS_PACKETS],
                    h[PS_LEAVES] / np, h[PS_SCANNED] / np, h[PS_CAND] / np, h[PS_APPENDED] / np / 32.0, h[PS_FLUSHES] / np,
                    h[PS_ROUNDS] / np, h[PS_MERGES] / np, h[PS_REDO] / np);
        }
    } else {
        SB_LAUNCH(ctx, k_knn<1>, knn_grid(n_items), QWARPS * 32, 0, view_of(f, B.t0), nullptr,
                  reinterpret_cast<const QueryItem*>(d_tio), n_items, k, nullptr, nullptr, B.normals, B.nbr, d_out_normals,
                  d_out_evals, B.n_trees, d_spacing, 32, n_items < 0x7fff0000LL ? d_work_knn : nullptr);
    }
    // seed grid for icp.cu (cell size from the measured point spacing)
    SB_LAUNCH(ctx, k_grid_params, ceil_div(B.n_trees, 128), 128, 0, d_bt, d_spacing, B.n_trees);
    SB_LAUNCH(ctx, k_grid_build, (unsigned)((n_items * 32 + 255) / 256), 256, 0, view_of(f, B.t0), d_tio, n_items,
              B.n_trees, B.grid);
    arena_release(ctx, mark);
    return SB_OK;
}

}  // namespace sb
