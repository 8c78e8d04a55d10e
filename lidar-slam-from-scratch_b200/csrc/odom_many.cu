// odom_many.cu — sb_odom_push_many: one frame into each of n streaming sessions (odom.cu) in one call, for a server
// that runs many live streams on one GPU.  A single push is latency-bound: one scan of ~8 k rows after the voxel grid
// cannot fill the chip, and each push waits on the host twice.  Here every stage runs once for all n frames:
//   one host-to-device copy of all raw rows -> one voxel grid over the n clouds (voxel.cu, one output-count round trip)
//   -> one forest_append + forest_normals over the kept frames into a call-level tree store (forest.cu) -> k_tree_relocate
//   (every new tree into the free slot of its own session, and every previous tree into the ICP batch's table) -> one
//   ICP batch of all registered pairs (icp.cu) -> one Scan Context launch -> k_odom_epilogue_many (keep rule, pose,
//   world-frame float32 of every kept frame) -> per session: addFrame / the map's entry, device to device -> one
//   device-to-host copy of all outputs and one final wait.
// Every stage computes per frame what the single push computes (the voxel grid, the index, the normals, the ICP pairs and
// the Scan Context do not depend on what else is in their batch), so the results are bit for bit those of n calls of
// sb_odom_push in array order, and after the call every session is where those calls would have left it: its newest
// tree lives in its own slot, and single and many pushes mix freely.  Nothing of a session, detector or map changes
// before the final wait; a call that fails for any session leaves all of them as they were.
//
// Layout of the call's device-to-host block: poses (16 doubles per session) | Scan Contexts (SB_SC_SIZE doubles per
// session) | the voxel grid's output rows (CSR over the sessions) | the world-frame float32 rows (the same CSR).
#include <cmath>
#include <string>
#include <unordered_set>

#include "odom.cuh"

namespace sb {

// A new tree built in the call-level store and where it goes: the arrays of the session's free slot and its
// descriptor entry 1; `prev` (null for a first frame): the session's previous tree, copied to `icp_entry`.
struct RelocJob {
    const TreeDesc* prev;
    TreeDesc* icp_entry;
    TreeDesc* dst;
    TreePoint* pts;
    float4* pts32;
    float* boxes;
    TreeNormal* nrm;
    NbrEntry* nbr;
    GridSlot* grid;
    i64 tree;
};

// One CTA row (blockIdx.y) per new tree.  Sorted positions (NbrEntry::pos, GridSlot::pos, TreePoint::idx) and the
// float32 offsets of pts32 are cloud-local; only the descriptor's offsets into the store's arrays (pt_off, box_off[],
// tab_off, out_off) and its base pointers change, to what a tree built alone at the start of the slot's arrays has.
__global__ void __launch_bounds__(256) k_tree_relocate(const TreeDesc* __restrict__ trees, const RelocJob* __restrict__ jobs,
                                                       int k) {
    const RelocJob& J = jobs[blockIdx.y];
    const TreeDesc& T = trees[J.tree];
    const i64 n = T.n, p0 = T.pt_off, b0 = T.box_off[0];
    const i64 nb = T.box_off[T.top] + T.box_cnt[T.top] - b0;
    const i64 ns = (i64)1 << (64 - T.tab_shift);
    const i64 t0 = (i64)blockIdx.x * blockDim.x + threadIdx.x, step = (i64)gridDim.x * blockDim.x;
    for (i64 i = t0; i < n; i += step) {
        J.pts[i] = T.pts[p0 + i];
        J.pts32[i] = T.pts32[p0 + i];
        J.nrm[i] = T.nrm[p0 + i];
    }
    for (i64 i = t0; i < n * k; i += step) J.nbr[i] = T.nbr[p0 * k + i];
    for (i64 i = t0; i < 6 * nb; i += step) J.boxes[i] = T.boxes[6 * b0 + i];
    for (i64 i = t0; i < ns; i += step) J.grid[i] = T.grid[T.tab_off + i];
    if (t0 == 0) {
        TreeDesc* D = J.dst;
        *D = T;
        D->pts = J.pts; D->pts32 = J.pts32; D->boxes = J.boxes; D->nrm = J.nrm; D->nbr = J.nbr; D->grid = J.grid;
        D->out_off = 0;
        D->pt_off = 0;
        for (int l = 0; l <= T.top; ++l) D->box_off[l] = T.box_off[l] - b0;
        D->tab_off = 0;
        if (J.prev) *J.icp_entry = *J.prev;
    }
}

// One kept frame of k_odom_epilogue_many: k_odom_epilogue's arguments (the rows are copied out by the block copy).
struct EpiFrame {
    const sb_icp_result* res;   // null: first frame
    const double* pose_in;
    double* pose_out;
    const double* xyz;
    double* out_pose;
    float* out_f32;             // null: not wanted
    double max_error;
    i64 n;
};

// k_odom_epilogue for many frames in one launch: CTA row blockIdx.y is frame y, with the same pose expression
// (odom_pose_entry) and row expression (odom_row).
__global__ void __launch_bounds__(256) k_odom_epilogue_many(const EpiFrame* __restrict__ frames) {
    const EpiFrame& F = frames[blockIdx.y];
    __shared__ double P[16];
    if (threadIdx.x < 16) {
        const double v = odom_pose_entry(F.res, F.max_error, F.pose_in, threadIdx.x);
        P[threadIdx.x] = v;
        if (blockIdx.x == 0) {
            F.pose_out[threadIdx.x] = v;
            F.out_pose[threadIdx.x] = v;
        }
    }
    __syncthreads();
    for (i64 r = (i64)blockIdx.x * blockDim.x + threadIdx.x; r < F.n; r += (i64)gridDim.x * blockDim.x)
        odom_row(P, F.xyz, r, nullptr, F.out_f32);
}

}  // namespace sb

using namespace sb;

namespace {

// What one call is given, per session (the ABI's arrays; NULL arrays read as NULL entries).
struct ManyArgs {
    sb_odom* const* sessions;
    int n;
    const void* const* xyz;
    int f32, stride;
    const int64_t* n_rows;
    const int32_t* frame_idx;
    const int32_t* flags;
    sb_odom_frame* out;
    double* const* out_xyz;
    float* const* out_world_f32;
    double* const* out_desc;
    sb_loop_result* const* loops;
    const int32_t* loop_capacity;
    double* oxyz(int i) const { return out_xyz ? out_xyz[i] : nullptr; }
    float* of32(int i) const { return out_world_f32 ? out_world_f32[i] : nullptr; }
    double* odesc(int i) const { return out_desc ? out_desc[i] : nullptr; }
    int cap(int i) const { return loop_capacity ? loop_capacity[i] : 0; }
    sb_loop_result* lp(int i) const { return loops ? loops[i] : nullptr; }
    int fl(int i) const { return flags ? flags[i] : 0; }
};

// the context's pinned buffer of this path: the rows on the way in, then the outputs on the way out
int many_host_reserve(Ctx* ctx, size_t bytes) {
    if (bytes <= ctx->h_many_cap) return SB_OK;
    const size_t cap = std::max(bytes, 2 * ctx->h_many_cap);
    SB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->h_many) cudaFreeHost(ctx->h_many);
    ctx->h_many = nullptr;
    ctx->h_many_cap = 0;
    SB_CUDA(ctx, cudaHostAlloc(&ctx->h_many, cap, cudaHostAllocDefault));
    ctx->h_many_cap = cap;
    return SB_OK;
}

// The rules of the call and push_impl's per-session argument checks, before anything is enqueued.
int check_args(Ctx* ctx, const ManyArgs& A, std::vector<char>& pinned) {
    if (A.n > 65535) return fail(ctx, SB_ERR_INVALID_ARG, "odom: %d sessions in one call (at most 65535)", A.n);
    if (!A.n_rows || !A.frame_idx || !A.out || !A.xyz)
        return fail(ctx, SB_ERR_INVALID_ARG, "odom: null xyz, n_rows, frame_idx or out array");
    if (A.stride < 3) return fail(ctx, SB_ERR_INVALID_ARG, "odom: row stride %d < 3", A.stride);
    const sb_odom* O0 = A.sessions[0];
    std::unordered_set<const void*> seen, loops, maps;
    for (int i = 0; i < A.n; ++i) {
        const sb_odom* O = A.sessions[i];
        if (!O) return fail(ctx, SB_ERR_INVALID_ARG, "odom: session %d is NULL", i);
        if (O->ctx != ctx) return fail(ctx, SB_ERR_INVALID_ARG, "odom: session %d belongs to another context", i);
        if (!seen.insert(O).second) return fail(ctx, SB_ERR_INVALID_ARG, "odom: session %d appears twice", i);
        if (O->loop && !loops.insert(O->loop).second)
            return fail(ctx, SB_ERR_INVALID_ARG, "odom: session %d shares its loop-closure detector with another session", i);
        if (O->map && !maps.insert(O->map).second)
            return fail(ctx, SB_ERR_INVALID_ARG, "odom: session %d shares its map with another session", i);
        if (O->cfg.voxel != O0->cfg.voxel || memcmp(&O->cfg.icp, &O0->cfg.icp, sizeof(sb_icp_config)) != 0)
            return fail(ctx, SB_ERR_INVALID_ARG, "odom: session %d has another voxel or icp config than session 0", i);
        const i64 n = A.n_rows[i];
        const int flags = A.fl(i);
        if (n < 0 || (n > 0 && !A.xyz[i]))
            return fail(ctx, SB_ERR_INVALID_ARG, "odom: session %d: null frame buffer or negative row count", i);
        if (A.cap(i) < 0 || (A.cap(i) > 0 && !A.lp(i)))
            return fail(ctx, SB_ERR_INVALID_ARG, "odom: session %d: loops may be NULL only with loop_capacity 0", i);
        if (flags & ~(SB_ODOM_ADD_FRAME | SB_ODOM_DETECT | SB_ODOM_ADD_MAP))
            return fail(ctx, SB_ERR_INVALID_ARG, "odom: session %d: unknown flags %d", i, flags);
        if ((flags & SB_ODOM_ADD_MAP) && !O->map)
            return fail(ctx, SB_ERR_INVALID_ARG, "odom: session %d: SB_ODOM_ADD_MAP without a map", i);
        if ((flags & SB_ODOM_ADD_FRAME) && !O->loop)
            return fail(ctx, SB_ERR_INVALID_ARG, "odom: session %d: SB_ODOM_ADD_FRAME without a loop-closure detector", i);
        if ((flags & SB_ODOM_DETECT) && (!O->loop || O->loop->world != 1))
            return fail(ctx, SB_ERR_INVALID_ARG, "odom: session %d: SB_ODOM_DETECT needs a loop-closure detector with world == 1", i);
        pinned[(size_t)i] = 0;
        if (n > 0) {
            cudaPointerAttributes attr;
            if (cudaPointerGetAttributes(&attr, A.xyz[i]) == cudaSuccess) {
                if (attr.type == cudaMemoryTypeDevice)
                    return fail(ctx, SB_ERR_INVALID_ARG, "odom: session %d: xyz is a device pointer; the session takes host rows", i);
                pinned[(size_t)i] = attr.type == cudaMemoryTypeHost;
            } else {
                cudaGetLastError();
            }
        }
    }
    return SB_OK;
}

// after the voxel grid refused the rows: the first session with a non-finite coordinate
int first_nonfinite(const ManyArgs& A, i64* row) {
    for (int i = 0; i < A.n; ++i)
        for (i64 r = 0; r < A.n_rows[i]; ++r)
            for (int a = 0; a < 3; ++a) {
                const double v = A.f32 ? (double)static_cast<const float*>(A.xyz[i])[r * A.stride + a]
                                       : static_cast<const double*>(A.xyz[i])[r * A.stride + a];
                if (!std::isfinite(v)) { *row = r; return i; }
            }
    return -1;
}

int push_many_impl(Ctx* ctx, const ManyArgs& A) {
    const int N = A.n;
    std::vector<char> pinned((size_t)N);
    SB_TRY(check_args(ctx, A, pinned));
    for (int i = 0; i < N; ++i) {
        memset(&A.out[i], 0, sizeof(sb_odom_frame));
        A.out[i].frame_idx = A.frame_idx[i];
        memcpy(A.out[i].pose, A.sessions[i]->pose, sizeof(A.sessions[i]->pose));
    }
    const sb_odom_config& cfg = A.sessions[0]->cfg;
    const int k = cfg.icp.normals_k;
    trace_mark(ctx, "odom_many:begin");

    // 1. all raw rows in one buffer: pageable rows through the pinned staging (one copy per run of them), pinned rows
    //    straight from the caller's buffer
    const i64 row_bytes = (i64)A.stride * (i64)(A.f32 ? sizeof(float) : sizeof(double));
    std::vector<i64> in_off((size_t)N + 1, 0);
    for (int i = 0; i < N; ++i) in_off[(size_t)i + 1] = in_off[(size_t)i] + A.n_rows[i];
    const i64 n_raw = in_off[(size_t)N];
    char* d_raw;
    SB_TRY(arena_get(ctx, (size_t)std::max<i64>(n_raw * row_bytes, 1), &d_raw));
    SB_TRY(many_host_reserve(ctx, (size_t)std::max<i64>(n_raw * row_bytes, 1)));
    for (int i = 0; i < N;) {
        if (A.n_rows[i] == 0) { ++i; continue; }
        const i64 o = in_off[(size_t)i] * row_bytes;
        if (pinned[(size_t)i]) {
            SB_CUDA(ctx, cudaMemcpyAsync(d_raw + o, A.xyz[i], (size_t)(A.n_rows[i] * row_bytes), cudaMemcpyHostToDevice,
                                         ctx->stream));
            ++i;
            continue;
        }
        int j = i;
        for (; j < N && !pinned[(size_t)j]; ++j)
            if (A.n_rows[j] > 0) memcpy(ctx->h_many + in_off[(size_t)j] * row_bytes, A.xyz[j], (size_t)(A.n_rows[j] * row_bytes));
        const i64 e = in_off[(size_t)j] * row_bytes;
        SB_CUDA(ctx, cudaMemcpyAsync(d_raw + o, ctx->h_many + o, (size_t)(e - o), cudaMemcpyHostToDevice, ctx->stream));
        i = j;
    }

    // 2. one voxel grid over the n clouds, straight into the device-to-host block; waits for the output counts
    const size_t o_desc = sizeof(double) * 16 * (size_t)N;
    const size_t o_rows = o_desc + sizeof(double) * SB_SC_SIZE * (size_t)N;
    char* d_out;
    SB_TRY(arena_get(ctx, o_rows + 36 * (size_t)std::max<i64>(n_raw, 1), &d_out));
    double* d_xyz = reinterpret_cast<double*>(d_out + o_rows);
    PointSrc ps;
    ps.base = d_raw;
    ps.f32 = A.f32;
    ps.stride = A.stride;
    std::vector<i64> ds_off((size_t)N + 1, 0);
    {
        const ArenaMark mark = arena_mark(ctx);
        const int s = voxel_downsample_src(ctx, ps, in_off.data(), N, cfg.voxel, d_xyz, ds_off.data(), nullptr);
        if (s == SB_ERR_RANGE) {
            i64 row = 0;
            const int bad = first_nonfinite(A, &row);
            if (bad >= 0) return fail(ctx, SB_ERR_RANGE, "odom: session %d: non-finite coordinate in row %lld", bad, row);
        }
        SB_TRY(s);
        arena_release(ctx, mark);
    }
    trace_mark(ctx, "odom_many:voxel");
    const i64 n_ds = ds_off[(size_t)N];
    std::vector<int> kept;            // sessions whose frame is registered or first, in array order
    std::vector<int> pair_of((size_t)N, -1);   // ICP pair (= entry of the previous tree) of a registered session
    int n_pairs = 0;
    i64 max_m = 1, store_pts = 0, store_boxes = 0, store_slots = 0;
    for (int i = 0; i < N; ++i) {
        sb_odom* O = A.sessions[i];
        const i64 m = ds_off[(size_t)i + 1] - ds_off[(size_t)i];
        A.out[i].n_points = m;
        if (m < O->cfg.min_points) continue;   // slam_node.cpp:125-130: skipped
        if (m == 0) return fail(ctx, SB_ERR_EMPTY, "odom: session %d: empty frame (undefined behaviour in the reference, kdtree.hpp:25,119)", i);
        if (m > 0x7fffffffLL) return fail(ctx, SB_ERR_RANGE, "odom: session %d: more than 2^31-1 rows after the voxel grid", i);
        kept.push_back(i);
        if (O->prev >= 0) pair_of[(size_t)i] = n_pairs++;
        i64 nb, ns;
        tree_store_need(m, &nb, &ns);
        store_pts += m;
        store_boxes += nb;
        store_slots += ns;
        max_m = std::max(max_m, m);
    }
    const int K = (int)kept.size();
    bool any_xyz = false, any_f32 = false, any_desc = false;
    for (int i = 0; i < N; ++i) {
        any_xyz |= A.oxyz(i) != nullptr;
        any_f32 |= A.of32(i) != nullptr;
        any_desc |= A.odesc(i) != nullptr;
    }
    const size_t o_f32 = o_rows + sizeof(double) * 3 * (size_t)n_ds;
    const size_t d2h = any_f32 ? o_f32 + sizeof(float) * 3 * (size_t)n_ds : any_xyz ? o_f32 : any_desc ? o_rows : o_desc;
    // the staging is free again (the voxel grid's wait came after the upload): it takes the outputs
    SB_TRY(many_host_reserve(ctx, d2h));
    for (int i : kept) {
        sb_odom* O = A.sessions[i];
        SB_TRY(slot_reserve(O, O->slot[O->prev < 0 ? 0 : 1 - O->prev], 0, ds_off[(size_t)i + 1] - ds_off[(size_t)i]));
    }

    // 3. one index + normals over the kept frames in a call-level store.  Entries [0, n_pairs) of the forest's table are
    //    the registered sessions' previous trees (filled by k_tree_relocate), [n_pairs, n_pairs + K) the new ones.
    Forest F;
    TreeStore st;
    IcpPending IP;
    memset(&IP, 0, sizeof(IP));
    std::vector<TreeDesc> moved((size_t)K);   // host mirrors of the relocated trees
    if (K > 0) {
        st.cap_points = store_pts;
        st.cap_boxes = store_boxes;
        st.cap_slots = store_slots;
        st.cap_k = k;
        SB_TRY(arena_get(ctx, (size_t)store_pts, &st.pts));
        SB_TRY(arena_get(ctx, (size_t)store_pts, &st.pts32));
        SB_TRY(arena_get(ctx, (size_t)store_pts, &st.normals));
        SB_TRY(arena_get(ctx, (size_t)(store_pts * k), &st.nbr));
        SB_TRY(arena_get(ctx, (size_t)store_slots, &st.grid));
        SB_TRY(arena_get(ctx, (size_t)(6 * store_boxes), &st.boxes));
        F.ctx = ctx;
        F.store = &st;
        SB_TRY(arena_get(ctx, (size_t)(n_pairs + K), &F.d_trees));
        F.cap_trees = n_pairs + K;
        F.n_trees = n_pairs;
        F.h_trees.assign((size_t)n_pairs, TreeDesc());
        for (int i : kept)
            if (pair_of[(size_t)i] >= 0) F.h_trees[(size_t)pair_of[(size_t)i]] = A.sessions[i]->slot[A.sessions[i]->prev].tree;
        SB_TRY(forest_append(ctx, &F, d_xyz, ds_off.data(), kept.data(), K));
        SB_TRY(forest_normals(ctx, &F, k, nullptr, nullptr));
        trace_mark(ctx, "odom_many:index+normals");

        // 4. every new tree into its session's free slot, every previous tree into the ICP table: one launch
        std::vector<RelocJob> jobs((size_t)K);
        for (int j = 0; j < K; ++j) {
            sb_odom* O = A.sessions[kept[(size_t)j]];
            OdomSlot& S = O->slot[O->prev < 0 ? 0 : 1 - O->prev];
            RelocJob& J = jobs[(size_t)j];
            const int p = pair_of[(size_t)kept[(size_t)j]];
            J.prev = p >= 0 ? O->slot[O->prev].d_trees + 1 : nullptr;
            J.icp_entry = p >= 0 ? F.d_trees + p : nullptr;
            J.dst = S.d_trees + 1;
            J.pts = S.st.pts; J.pts32 = S.st.pts32; J.boxes = S.st.boxes; J.nrm = S.st.normals; J.nbr = S.st.nbr;
            J.grid = S.st.grid;
            J.tree = n_pairs + j;
            TreeDesc& D = moved[(size_t)j];
            D = F.h_trees[(size_t)(n_pairs + j)];
            D.pts = J.pts; D.pts32 = J.pts32; D.boxes = J.boxes; D.nrm = J.nrm; D.nbr = J.nbr; D.grid = J.grid;
            D.out_off = 0;
            D.pt_off = 0;
            const i64 b0 = D.box_off[0];
            for (int l = 0; l <= D.top; ++l) D.box_off[l] -= b0;
            D.tab_off = 0;
        }
        RelocJob* d_jobs;
        SB_TRY(arena_get(ctx, (size_t)K, &d_jobs));
        SB_TRY(table_upload(ctx, d_jobs, jobs.data(), sizeof(RelocJob) * (size_t)K));
        const i64 work = std::max<i64>(max_m * k, 2 * max_m + 64);   // nbr entries / seed-grid slots of the largest tree
        const unsigned gx = (unsigned)std::min<i64>(std::max<i64>((work + 1023) / 1024, 1), 64);
        SB_LAUNCH(ctx, k_tree_relocate, dim3(gx, (unsigned)K), 256, 0, F.d_trees, d_jobs, k);

        // 5. one ICP batch of every registered frame onto its previous frame (slam_node.cpp:132-138)
        if (n_pairs > 0) {
            SB_TRY(icp_reserve_results(ctx, (size_t)n_pairs));
            std::vector<PairDesc> pairs((size_t)n_pairs);
            memset(pairs.data(), 0, sizeof(PairDesc) * (size_t)n_pairs);
            for (int j = 0; j < K; ++j) {
                const int p = pair_of[(size_t)kept[(size_t)j]];
                if (p < 0) continue;
                pairs[(size_t)p].tree = p;
                pairs[(size_t)p].src_tree = n_pairs + j;
            }
            SB_TRY(icp_enqueue(ctx, &F, pairs, &cfg.icp, &IP));
            trace_mark(ctx, "odom_many:icp");
        }
    }
    // 6. Scan Context of every frame (a skipped frame's is not used) straight into the output block
    double* d_desc = reinterpret_cast<double*>(d_out + o_desc);
    i64* d_ds_off;
    SB_TRY(arena_get(ctx, (size_t)N + 1, &d_ds_off));
    SB_TRY(table_upload(ctx, d_ds_off, ds_off.data(), sizeof(i64) * ((size_t)N + 1)));
    if (K > 0) SB_TRY(sc_compute_dev(ctx, d_xyz, d_ds_off, N, d_desc));
    // 7. keep rule, pose chain and world-frame float32 cloud of every kept frame: one launch
    if (K > 0) {
        std::vector<EpiFrame> ef((size_t)K);
        float* d_f32 = reinterpret_cast<float*>(d_out + o_f32);
        for (int j = 0; j < K; ++j) {
            const int i = kept[(size_t)j];
            sb_odom* O = A.sessions[i];
            EpiFrame& E = ef[(size_t)j];
            const int p = pair_of[(size_t)i];
            E.res = p >= 0 ? IP.d_res + p : nullptr;
            E.pose_in = O->d_pose + 16 * O->pi;
            E.pose_out = O->d_pose + 16 * (1 - O->pi);
            E.xyz = d_xyz + 3 * ds_off[(size_t)i];
            E.out_pose = reinterpret_cast<double*>(d_out) + 16 * i;
            E.out_f32 = A.of32(i) ? d_f32 + 3 * ds_off[(size_t)i] : nullptr;
            E.max_error = O->cfg.max_error;
            E.n = ds_off[(size_t)i + 1] - ds_off[(size_t)i];
        }
        EpiFrame* d_ef;
        SB_TRY(arena_get(ctx, (size_t)K, &d_ef));
        SB_TRY(table_upload(ctx, d_ef, ef.data(), sizeof(EpiFrame) * (size_t)K));
        const unsigned gx = (unsigned)std::min<i64>((max_m + 255) / 256, 64);
        SB_LAUNCH(ctx, k_odom_epilogue_many, dim3(gx, (unsigned)K), 256, 0, d_ef);
    }
    trace_mark(ctx, "odom_many:sc+epilogue");
    // 8. addFrame and the map's entry per session (slam_node.cpp:152, 159), device to device
    std::vector<LoopAddPending> LP((size_t)N);
    std::vector<MapAddPending> MP((size_t)N);
    for (int i : kept) {
        sb_odom* O = A.sessions[i];
        const i64 m = ds_off[(size_t)i + 1] - ds_off[(size_t)i];
        const double* rows = d_xyz + 3 * ds_off[(size_t)i];
        if (A.fl(i) & SB_ODOM_ADD_FRAME) SB_TRY(loop_add_enqueue(O->loop, rows, m, A.frame_idx[i], d_desc + (size_t)SB_SC_SIZE * i, &LP[(size_t)i]));
        if (A.fl(i) & SB_ODOM_ADD_MAP) SB_TRY(map_add_enqueue(O->map, rows, m, O->d_pose + 16 * (1 - O->pi), &MP[(size_t)i]));
    }
    // 9. one copy of all outputs back and the call's final wait (icp_collect waits for the stream)
    SB_CUDA(ctx, cudaMemcpyAsync(ctx->h_many, d_out, d2h, cudaMemcpyDeviceToHost, ctx->stream));
    std::vector<sb_icp_result> icp((size_t)std::max(n_pairs, 1));
    if (n_pairs > 0) {
        SB_TRY(icp_collect(ctx, ctx->stream, std::vector<IcpPending>(1, IP), std::vector<const int*>(1, nullptr), icp.data()));
    } else {
        SB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    trace_mark(ctx, "odom_many:end");
    trace_dump(ctx);

    // commit.  The maps first: every insert is checked before any map records its entry, so that a refused insert
    // leaves all maps as they were (the caller takes the pending adds back)
    const char* h = ctx->h_many;
    for (int i : kept)
        if ((A.fl(i) & SB_ODOM_ADD_MAP) && (A.sessions[i]->map->h_stat[1] & (FLAG_NONFINITE | FLAG_KEY_RANGE)))
            return fail(ctx, SB_ERR_RANGE, "odom: session %d: the map refused the frame (a non-finite pose or a cell index "
                        "that does not fit an int)", i);
    for (int i : kept)
        if (A.fl(i) & SB_ODOM_ADD_MAP) {
            const int s = map_add_finish(A.sessions[i]->map, MP[(size_t)i], reinterpret_cast<const double*>(h) + 16 * i);
            if (s != SB_OK) return fail(ctx, s, "odom: session %d: %s", i, std::string(ctx->err).c_str());
        }
    // a skipped frame's map entry: no rows, the pose repeated (the map keeps one entry per pose of the node)
    for (int i = 0; i < N; ++i) {
        sb_odom* O = A.sessions[i];
        if (A.out[i].n_points < O->cfg.min_points && (A.fl(i) & SB_ODOM_ADD_MAP)) SB_TRY(map_add(O->map, nullptr, 0, O->pose));
    }
    for (int j = 0; j < K; ++j) {
        const int i = kept[(size_t)j];
        sb_odom* O = A.sessions[i];
        if (A.fl(i) & SB_ODOM_ADD_FRAME) loop_add_commit(O->loop, LP[(size_t)i]);
        const int s = O->prev < 0 ? 0 : 1 - O->prev;
        const bool reg = O->prev >= 0;
        O->slot[s].tree = moved[(size_t)j];
        O->prev = s;
        O->pi = 1 - O->pi;
        memcpy(O->pose, h + sizeof(double) * 16 * i, sizeof(O->pose));
        sb_odom_frame& f = A.out[i];
        f.state = reg ? SB_ODOM_REGISTERED : SB_ODOM_FIRST;
        memcpy(f.pose, O->pose, sizeof(O->pose));
        if (reg) f.icp = icp[(size_t)pair_of[(size_t)i]];
        if (A.odesc(i)) memcpy(A.odesc(i), h + o_desc + sizeof(double) * SB_SC_SIZE * i, sizeof(double) * SB_SC_SIZE);
        if (A.of32(i))
            memcpy(A.of32(i), h + o_f32 + sizeof(float) * 3 * ds_off[(size_t)i], sizeof(float) * 3 * (size_t)f.n_points);
    }
    for (int i = 0; i < N; ++i) {
        if (A.out[i].n_points < A.sessions[i]->cfg.min_points) A.out[i].state = SB_ODOM_SKIPPED;
        if (A.oxyz(i) && A.out[i].n_points > 0)
            memcpy(A.oxyz(i), h + o_rows + sizeof(double) * 3 * ds_off[(size_t)i], sizeof(double) * 3 * (size_t)A.out[i].n_points);
    }

    // 10. detect() (slam_node.cpp:160-167) per session in array order, for its detector's newest entry
    for (int i : kept) {
        if (!(A.fl(i) & SB_ODOM_DETECT)) continue;
        sb_loop* L = A.sessions[i]->loop;
        int count = 0;
        if (L->n_global > 0 && L->cfg.max_candidates > 0) {
            const int q = L->n_global - 1;
            std::vector<sb_loop_result> res((size_t)L->cfg.max_candidates);
            SB_TRY(loop_detect_batch(L, &q, 1, res.data(), &count));
            for (int c = 0; c < count && c < A.cap(i); ++c) A.lp(i)[c] = res[(size_t)c];
        }
        A.out[i].n_loops = count;
    }
    return SB_OK;
}

int push_many_entry(const ManyArgs& A) {
    if (A.n < 0 || (A.n > 0 && (!A.sessions || !A.sessions[0]))) return SB_ERR_INVALID_ARG;
    if (A.n == 0) return SB_OK;
    Ctx* ctx = A.sessions[0]->ctx;
    Enter g(ctx);
    const int s = push_many_impl(ctx, A);
    // a failed call may leave copies or kernels in flight, and map adds it enqueued but did not finish: those are taken
    // back (only sessions of this context, which check_args ensured before any add was enqueued)
    if (s != SB_OK) {
        cudaStreamSynchronize(ctx->stream);
        const std::string msg = ctx->err;
        for (int i = 0; i < A.n; ++i) {
            sb_odom* O = A.sessions[i];
            if (O && O->ctx == ctx && O->map && O->map->pending) map_add_abort(O->map);
        }
        ctx->err = msg;
    }
    return s;
}

}  // namespace

extern "C" {

int sb_odom_push_many(sb_odom* const* sessions, int32_t n, const double* const* xyz, const int64_t* n_rows,
                      const int32_t* frame_idx, const int32_t* flags, sb_odom_frame* out, double* const* out_xyz,
                      float* const* out_world_f32, double* const* out_desc, sb_loop_result* const* loops,
                      const int32_t* loop_capacity) {
    const ManyArgs A{sessions, n, reinterpret_cast<const void* const*>(xyz), 0, 3, n_rows, frame_idx, flags, out,
                     out_xyz, out_world_f32, out_desc, loops, loop_capacity};
    return push_many_entry(A);
}

int sb_odom_push_many_f32(sb_odom* const* sessions, int32_t n, const float* const* xyz, int32_t stride_floats,
                          const int64_t* n_rows, const int32_t* frame_idx, const int32_t* flags, sb_odom_frame* out,
                          double* const* out_xyz, float* const* out_world_f32, double* const* out_desc,
                          sb_loop_result* const* loops, const int32_t* loop_capacity) {
    const ManyArgs A{sessions, n, reinterpret_cast<const void* const*>(xyz), 1, stride_floats, n_rows, frame_idx, flags,
                     out, out_xyz, out_world_f32, out_desc, loops, loop_capacity};
    return push_many_entry(A);
}

}  // extern "C"
