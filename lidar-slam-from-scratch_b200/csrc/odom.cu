// odom.cu — the streaming odometry session (sb_odom_*, include/slam_b200.h): SlamNode::process_frame
// (slam_viz/src/ros/slam_node.cpp:118-175) one scan per call, with the previous frame's state kept on the device.
//
// The single-call entry points start from host memory and drop their device state on return, so a node built on them
// uploads every frame three times (voxel grid, ICP, addFrame) and indexes it twice (as ICP source, then as the next
// frame's target).  Here a frame is uploaded once and indexed once: its downsampled cloud, tree, normals, neighbour
// graph and seed grid stay in one of two device slots and serve as the next frame's ICP target.  Per registered frame:
//   one host-to-device copy of the raw rows -> voxel grid (voxel.cu) -> one tree + normals (forest.cu, built into the
//   slot's own buffers) -> ICP of the pair (icp.cu) -> Scan Context -> k_odom_epilogue (keep rule, pose, world-frame
//   float32 cloud) -> optional device-to-device addFrame (loop.cu) -> one device-to-host copy of the outputs.
// The host waits for the voxel grid's output count (the tree layout is planned on the host) and at the end of the frame.
//
// A frame is always built into the slot the previous frame does not hold, and the slots swap (and the detector's new
// entry is recorded) only after the frame's final synchronise: a push that fails leaves the session as it was.  Slot
// buffers grow by doubling and outgrown ones are retired until the session is freed, as the detector's pools are
// (loop.cu): cudaMalloc / cudaFree stall the host for up to hundreds of milliseconds.
#include "odom.cuh"

namespace sb {

// slam_node.cpp:139-147 on the device, after the ICP loop, without a host round trip: the keep rule and the pose product
// (odom_pose_entry), then every row to the world frame (odom_row).  res == nullptr (first frame): the pose is pose_in
// itself.  Every block forms the pose; block 0 publishes it.
__global__ void __launch_bounds__(256) k_odom_epilogue(const sb_icp_result* __restrict__ res, double max_error,
                                                       const double* __restrict__ pose_in, double* __restrict__ pose_out,
                                                       const double* __restrict__ xyz, i64 n, double* __restrict__ out_pose,
                                                       double* __restrict__ out_xyz, float* __restrict__ out_f32) {
    __shared__ double P[16];
    if (threadIdx.x < 16) {
        const double v = odom_pose_entry(res, max_error, pose_in, threadIdx.x);
        P[threadIdx.x] = v;
        if (blockIdx.x == 0) {
            pose_out[threadIdx.x] = v;
            out_pose[threadIdx.x] = v;
        }
    }
    __syncthreads();
    for (i64 r = (i64)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (i64)gridDim.x * blockDim.x)
        odom_row(P, xyz, r, out_xyz, out_f32);
}

}  // namespace sb

using namespace sb;

namespace {

int push_impl(sb_odom* O, const void* xyz, int f32, int stride, i64 n, int32_t frame_idx, int32_t flags,
              sb_odom_frame* out, double* out_xyz, float* out_world_f32, double* out_desc, sb_loop_result* loops,
              int32_t loop_capacity) {
    Ctx* ctx = O->ctx;
    if (!out || n < 0 || (n > 0 && !xyz))
        return fail(ctx, SB_ERR_INVALID_ARG, "odom: null frame buffer or negative row count");
    if (stride < 3) return fail(ctx, SB_ERR_INVALID_ARG, "odom: row stride %d < 3", stride);
    if (loop_capacity < 0 || (loop_capacity > 0 && !loops))
        return fail(ctx, SB_ERR_INVALID_ARG, "odom: loops may be NULL only with loop_capacity 0");
    if (flags & ~(SB_ODOM_ADD_FRAME | SB_ODOM_DETECT | SB_ODOM_ADD_MAP))
        return fail(ctx, SB_ERR_INVALID_ARG, "odom: unknown flags %d", flags);
    if ((flags & SB_ODOM_ADD_MAP) && !O->map) return fail(ctx, SB_ERR_INVALID_ARG, "odom: SB_ODOM_ADD_MAP without a map");
    if ((flags & SB_ODOM_ADD_FRAME) && !O->loop)
        return fail(ctx, SB_ERR_INVALID_ARG, "odom: SB_ODOM_ADD_FRAME without a loop-closure detector");
    if ((flags & SB_ODOM_DETECT) && (!O->loop || O->loop->world != 1))
        return fail(ctx, SB_ERR_INVALID_ARG, "odom: SB_ODOM_DETECT needs a loop-closure detector with world == 1");
    // the rows are host memory: pinned rows are copied as they are, anything else goes through pinned staging by
    // memcpy, which a device address would crash
    bool pinned = false;
    if (n > 0) {
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, xyz) == cudaSuccess) {
            if (attr.type == cudaMemoryTypeDevice)
                return fail(ctx, SB_ERR_INVALID_ARG, "odom: xyz is a device pointer; the session takes host rows");
            pinned = attr.type == cudaMemoryTypeHost;
        } else {
            cudaGetLastError();
        }
    }
    memset(out, 0, sizeof(*out));
    out->frame_idx = frame_idx;
    memcpy(out->pose, O->pose, sizeof(O->pose));
    trace_mark(ctx, "odom:begin");

    // 1. the raw rows: one copy, straight from the caller's buffer if it is pinned, else through pinned staging
    const int s = O->prev < 0 ? 0 : 1 - O->prev;   // the slot the previous frame does not hold
    OdomSlot& S = O->slot[s];
    const i64 in_bytes = n * stride * (i64)(f32 ? sizeof(float) : sizeof(double));
    SB_TRY(slot_reserve(O, S, n, 0));
    SB_TRY(grow_dev(O, &O->d_raw, &O->raw_cap, std::max<i64>(in_bytes, 1)));
    if (n > 0) {
        const void* src = xyz;
        if (!pinned) {
            SB_TRY(grow_host(O, &O->h_in, &O->h_in_cap, in_bytes));
            memcpy(O->h_in, xyz, (size_t)in_bytes);
            src = O->h_in;
        }
        SB_CUDA(ctx, cudaMemcpyAsync(O->d_raw, src, (size_t)in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    // 2. voxel grid (slam_node.cpp:122) into the free slot; waits for its output count
    PointSrc ps;
    ps.base = O->d_raw;
    ps.f32 = f32;
    ps.stride = stride;
    i64 in_off[2] = {0, n}, ds_off[2] = {0, 0};
    {
        const ArenaMark mark = arena_mark(ctx);
        SB_TRY(voxel_downsample_src(ctx, ps, in_off, 1, O->cfg.voxel, S.xyz, ds_off, nullptr));
        arena_release(ctx, mark);
    }
    trace_mark(ctx, "odom:voxel");
    const i64 m = ds_off[1];
    out->n_points = m;
    if (m < O->cfg.min_points) {   // slam_node.cpp:125-130: the frame is dropped, nothing else changes
        out->state = SB_ODOM_SKIPPED;
        if (out_xyz && m > 0) {
            SB_CUDA(ctx, cudaMemcpyAsync(out_xyz, S.xyz, sizeof(double) * 3 * m, cudaMemcpyDeviceToHost, ctx->stream));
            SB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        }
        // the map keeps one entry per pose of the node (poses_): no rows, the pose repeated
        if (flags & SB_ODOM_ADD_MAP) SB_TRY(map_add(O->map, nullptr, 0, O->pose));
        return SB_OK;
    }
    if (m == 0) return fail(ctx, SB_ERR_EMPTY, "odom: empty frame (undefined behaviour in the reference, kdtree.hpp:25,119)");
    if (m > 0x7fffffffLL) return fail(ctx, SB_ERR_RANGE, "odom: more than 2^31-1 rows after the voxel grid");

    // 3. one tree + normals over the downsampled rows, in the slot's own buffers: this frame's ICP source and the next
    //    frame's target
    SB_TRY(slot_reserve(O, S, n, m));
    SB_TRY(out_reserve(O, m));
    const bool reg = O->prev >= 0;
    Forest F;
    F.ctx = ctx;
    F.store = &S.st;
    F.d_trees = S.d_trees;
    F.cap_trees = 2;
    F.n_trees = 1;   // entry 0: the target (below), this frame's tree goes to entry 1
    F.h_trees.assign(1, TreeDesc());
    memset(&F.h_trees[0], 0, sizeof(TreeDesc));
    if (reg) F.h_trees[0] = O->slot[O->prev].tree;
    const i64 tree_off[2] = {0, m};
    SB_TRY(forest_append(ctx, &F, S.xyz, tree_off, nullptr, 1));
    SB_TRY(forest_normals(ctx, &F, O->cfg.icp.normals_k, nullptr, nullptr));
    trace_mark(ctx, "odom:index+normals");

    // 4. ICP of this frame onto the previous one (slam_node.cpp:132-138); the results stay on the device for the epilogue
    IcpPending P;
    memset(&P, 0, sizeof(P));
    if (reg) {
        SB_CUDA(ctx, cudaMemcpyAsync(S.d_trees, O->slot[O->prev].d_trees + 1, sizeof(TreeDesc), cudaMemcpyDeviceToDevice,
                                     ctx->stream));
        SB_TRY(icp_reserve_results(ctx, 1));
        std::vector<PairDesc> pairs(1);
        memset(pairs.data(), 0, sizeof(PairDesc));
        pairs[0].tree = 0;
        pairs[0].src_tree = 1;
        pairs[0].n_src = (int)m;
        SB_TRY(icp_enqueue(ctx, &F, pairs, &O->cfg.icp, &P));
        trace_mark(ctx, "odom:icp");
    }
    // 5. Scan Context (loop_closure.hpp:55) straight into the output block; the detector copies it from there
    double* d_desc = reinterpret_cast<double*>(O->d_out + OUT_DESC);
    i64* d_off;
    SB_TRY(arena_get(ctx, 2, &d_off));
    SB_TRY(table_upload(ctx, d_off, tree_off, sizeof(tree_off)));
    SB_TRY(sc_compute_dev(ctx, S.xyz, d_off, 1, d_desc));
    // 6. keep rule, pose chain and the world-frame float32 cloud (slam_node.cpp:139-147)
    const size_t o_f32 = OUT_ROWS + (out_xyz ? sizeof(double) * 3 * (size_t)m : 0);
    const size_t o_end = o_f32 + (out_world_f32 ? sizeof(float) * 3 * (size_t)m : 0);
    {
        const i64 blocks = std::min<i64>((m + 255) / 256, (i64)ctx->sm_count * 4);
        SB_LAUNCH(ctx, k_odom_epilogue, (unsigned)blocks, 256, 0, reg ? P.d_res : nullptr, O->cfg.max_error,
                  O->d_pose + 16 * O->pi, O->d_pose + 16 * (1 - O->pi), S.xyz, m, reinterpret_cast<double*>(O->d_out),
                  out_xyz ? reinterpret_cast<double*>(O->d_out + OUT_ROWS) : nullptr,
                  out_world_f32 ? reinterpret_cast<float*>(O->d_out + o_f32) : nullptr);
    }
    trace_mark(ctx, "odom:sc+epilogue");
    // 7. addFrame (slam_node.cpp:159): device to device, recorded after the final synchronise
    const bool add = (flags & SB_ODOM_ADD_FRAME) != 0;
    LoopAddPending LP;
    if (add) SB_TRY(loop_add_enqueue(O->loop, S.xyz, m, frame_idx, d_desc, &LP));
    // 7b. the map's entry (update_occupancy_grid, slam_node.cpp:152): rows and pose device to device, cells inserted
    const bool add_map = (flags & SB_ODOM_ADD_MAP) != 0;
    MapAddPending MP;
    if (add_map) SB_TRY(map_add_enqueue(O->map, S.xyz, m, O->d_pose + 16 * (1 - O->pi), &MP));
    // 8. one copy of the outputs back, and the frame's final synchronise (icp_collect waits for the stream)
    const size_t d2h = (out_xyz || out_world_f32 || out_desc) ? o_end : OUT_DESC;
    SB_CUDA(ctx, cudaMemcpyAsync(O->h_out, O->d_out, d2h, cudaMemcpyDeviceToHost, ctx->stream));
    if (reg) {
        const std::vector<IcpPending> pending(1, P);
        SB_TRY(icp_collect(ctx, ctx->stream, pending, std::vector<const int*>(1, nullptr), &out->icp));
    } else {
        SB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    trace_mark(ctx, "odom:end");
    trace_dump(ctx);

    // the map's entry first: a map whose insert fails restores itself, and the push fails before anything else commits
    if (add_map) SB_TRY(map_add_finish(O->map, MP, reinterpret_cast<const double*>(O->h_out)));
    // commit: this frame becomes the previous one
    if (add) loop_add_commit(O->loop, LP);
    S.tree = F.h_trees[1];
    O->prev = s;
    O->pi = 1 - O->pi;
    memcpy(O->pose, O->h_out, sizeof(O->pose));
    out->state = reg ? SB_ODOM_REGISTERED : SB_ODOM_FIRST;
    memcpy(out->pose, O->pose, sizeof(O->pose));
    if (out_desc) memcpy(out_desc, O->h_out + OUT_DESC, sizeof(double) * SB_SC_SIZE);
    if (out_xyz) memcpy(out_xyz, O->h_out + OUT_ROWS, sizeof(double) * 3 * (size_t)m);
    if (out_world_f32) memcpy(out_world_f32, O->h_out + o_f32, sizeof(float) * 3 * (size_t)m);

    // 9. detect() (slam_node.cpp:160-167) for the detector's newest entry, with the batch path's candidate walk
    if (flags & SB_ODOM_DETECT) {
        sb_loop* L = O->loop;
        int count = 0;
        if (L->n_global > 0 && L->cfg.max_candidates > 0) {
            const int q = L->n_global - 1;
            std::vector<sb_loop_result> res((size_t)L->cfg.max_candidates);
            SB_TRY(loop_detect_batch(L, &q, 1, res.data(), &count));
            for (int i = 0; i < count && i < loop_capacity; ++i) loops[i] = res[(size_t)i];
        }
        out->n_loops = count;
    }
    return SB_OK;
}

int push_entry(sb_odom* O, const void* xyz, int f32, int stride, int64_t n, int32_t frame_idx, int32_t flags,
               sb_odom_frame* out, double* out_xyz, float* out_world_f32, double* out_desc, sb_loop_result* loops,
               int32_t loop_capacity) {
    if (!O) return SB_ERR_INVALID_ARG;
    Enter g(O->ctx);
    const int s = push_impl(O, xyz, f32, stride, (i64)n, frame_idx, flags, out, out_xyz, out_world_f32, out_desc, loops,
                            loop_capacity);
    // a failed push may leave copies or kernels in flight: the next call reuses the staging buffers and the arena; a map
    // add it enqueued but did not finish is taken back
    if (s != SB_OK) {
        cudaStreamSynchronize(O->ctx->stream);
        if (O->map && O->map->pending) {
            const std::string msg = O->ctx->err;
            map_add_abort(O->map);
            O->ctx->err = msg;
        }
    }
    return s;
}

}  // namespace

extern "C" {

void sb_default_odom_config(sb_odom_config* cfg) {
    if (!cfg) return;
    memset(cfg, 0, sizeof(*cfg));
    cfg->voxel = 0.5;          // slam_node voxel_size
    cfg->min_points = 1000;    // slam_node.hpp:29
    cfg->max_error = 1.0;      // slam_node.cpp:139-140
    sb_default_icp_config(&cfg->icp);
    for (int i = 0; i < 16; ++i) cfg->initial_pose[i] = (i % 5 == 0) ? 1.0 : 0.0;
}

int sb_odom_create(sb_ctx* ctx, const sb_odom_config* cfg, sb_loop* loop, sb_odom** out) {
    return sb_odom_create2(ctx, cfg, loop, nullptr, out);
}

int sb_odom_create2(sb_ctx* ctx, const sb_odom_config* cfg, sb_loop* loop, sb_map* map, sb_odom** out) {
    if (!ctx || !cfg || !out) return SB_ERR_INVALID_ARG;
    *out = nullptr;
    Ctx* c = &ctx->c;
    Enter g(c);
    if (loop && loop->ctx != c) return fail(c, SB_ERR_INVALID_ARG, "odom: the loop-closure detector belongs to another context");
    if (map && map->ctx != c) return fail(c, SB_ERR_INVALID_ARG, "odom: the map belongs to another context");
    if (cfg->icp.normals_k < 1 || cfg->icp.normals_k > SB_MAX_K)
        return fail(c, SB_ERR_INVALID_ARG, "odom: normals_k %d outside [1, %d]", cfg->icp.normals_k, SB_MAX_K);
    if (cfg->icp.max_iterations < 0 || cfg->icp.max_iterations > SB_MAX_ICP_ITERATIONS)
        return fail(c, SB_ERR_INVALID_ARG, "odom: max_iterations %d outside [0, %d]", cfg->icp.max_iterations,
                    SB_MAX_ICP_ITERATIONS);
    sb_odom* O = new sb_odom();
    O->ctx = c;
    O->cfg = *cfg;
    O->loop = loop;
    O->map = map;
    memcpy(O->pose, cfg->initial_pose, sizeof(O->pose));
    int s = SB_OK;
    if (cudaMalloc(&O->d_pose, sizeof(double) * 32) != cudaSuccess ||
        cudaMalloc(&O->slot[0].d_trees, sizeof(TreeDesc) * 2) != cudaSuccess ||
        cudaMalloc(&O->slot[1].d_trees, sizeof(TreeDesc) * 2) != cudaSuccess)
        s = fail(c, SB_ERR_CUDA, "odom: %s", cudaGetErrorString(cudaGetLastError()));
    if (s == SB_OK && (cudaMemcpyAsync(O->d_pose, O->pose, sizeof(O->pose), cudaMemcpyHostToDevice, c->stream) != cudaSuccess ||
                       cudaStreamSynchronize(c->stream) != cudaSuccess))
        s = fail(c, SB_ERR_CUDA, "odom: %s", cudaGetErrorString(cudaGetLastError()));
    if (s != SB_OK) {
        sb_odom_free(O);
        return s;
    }
    *out = O;
    return SB_OK;
}

void sb_odom_free(sb_odom* odom) {
    if (!odom) return;
    cudaSetDevice(odom->ctx->device);
    cudaStreamSynchronize(odom->ctx->stream);
    for (OdomSlot& S : odom->slot) {
        cudaFree(S.xyz);
        cudaFree(S.st.pts); cudaFree(S.st.pts32); cudaFree(S.st.boxes);
        cudaFree(S.st.normals); cudaFree(S.st.nbr); cudaFree(S.st.grid);
        cudaFree(S.d_trees);
    }
    cudaFree(odom->d_pose);
    cudaFree(odom->d_raw);
    cudaFree(odom->d_out);
    for (void* p : odom->retired) cudaFree(p);
    if (odom->h_in) cudaFreeHost(odom->h_in);
    if (odom->h_out) cudaFreeHost(odom->h_out);
    for (void* p : odom->retired_host) cudaFreeHost(p);
    delete odom;
}

int sb_odom_reserve(sb_odom* odom, int64_t max_raw_rows) {
    if (!odom || max_raw_rows < 0) return SB_ERR_INVALID_ARG;
    Enter g(odom->ctx);
    const i64 n = max_raw_rows;
    for (OdomSlot& S : odom->slot) SB_TRY(slot_reserve(odom, S, n, n));
    SB_TRY(grow_dev(odom, &odom->d_raw, &odom->raw_cap, std::max<i64>(n * 4 * (i64)sizeof(float), n * 3 * (i64)sizeof(double))));
    SB_TRY(grow_host(odom, &odom->h_in, &odom->h_in_cap, std::max<i64>(n * 4 * (i64)sizeof(float), n * 3 * (i64)sizeof(double))));
    return out_reserve(odom, n);
}

int sb_odom_set_pose(sb_odom* odom, const double* pose16) {
    if (!odom || !pose16) return SB_ERR_INVALID_ARG;
    Ctx* c = odom->ctx;
    Enter g(c);
    SB_CUDA(c, cudaMemcpyAsync(odom->d_pose + 16 * odom->pi, pose16, sizeof(double) * 16, cudaMemcpyHostToDevice, c->stream));
    SB_CUDA(c, cudaStreamSynchronize(c->stream));
    memcpy(odom->pose, pose16, sizeof(odom->pose));
    return SB_OK;
}

int sb_odom_get_pose(const sb_odom* odom, double* pose16) {
    if (!odom || !pose16) return SB_ERR_INVALID_ARG;
    memcpy(pose16, odom->pose, sizeof(odom->pose));
    return SB_OK;
}

int sb_odom_push(sb_odom* odom, const double* xyz, int64_t n, int32_t frame_idx, int32_t flags, sb_odom_frame* out,
                 double* out_xyz, float* out_world_f32, double* out_desc, sb_loop_result* loops, int32_t loop_capacity) {
    return push_entry(odom, xyz, 0, 3, n, frame_idx, flags, out, out_xyz, out_world_f32, out_desc, loops, loop_capacity);
}

int sb_odom_push_f32(sb_odom* odom, const float* xyz, int32_t stride_floats, int64_t n, int32_t frame_idx,
                     int32_t flags, sb_odom_frame* out, double* out_xyz, float* out_world_f32, double* out_desc,
                     sb_loop_result* loops, int32_t loop_capacity) {
    return push_entry(odom, xyz, 1, stride_floats, n, frame_idx, flags, out, out_xyz, out_world_f32, out_desc, loops,
                      loop_capacity);
}

}  // extern "C"
