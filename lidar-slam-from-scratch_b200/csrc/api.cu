// api.cu — the C ABI of include/slam_b200.h: context management, host<->device staging and the glue that turns
// each entry point into calls of the device pipelines (voxel.cu, forest.cu, icp.cu, scancontext.cu, loop.cu).
// There is no CPU implementation of any stage behind these entry points.
#include <chrono>
#include <cstdarg>
#include <limits>
#include <functional>
#include <cstdlib>
#include <algorithm>

#include "common.cuh"

struct sb_index {
    sb::Ctx* ctx = nullptr;
    sb::Forest forest;
    std::vector<double> host_rows;  // the indexed cloud in ORIGINAL row order (find_correspondences), fetched once
};

namespace sb {

int fail(Ctx* ctx, int status, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    return status;
}

int arena_reset(Ctx* ctx) {
    Arena& A = ctx->arena;
    if (!A.overflow.empty()) {
        cudaStreamSynchronize(ctx->stream);
        for (void* p : A.overflow) cudaFree(p);
        A.overflow.clear();
    }
    if (A.high > A.cap) {
        // regrow the slab to the high-water mark (+25 %), never below 64 MB and at least doubling while it is small:
        // cudaMalloc / cudaFree cost up to hundreds of ms on this pool, a streaming caller whose frames vary by a few
        // per cent must stop reaching them after the first frames
        cudaStreamSynchronize(ctx->stream);
        cudaFree(A.base);
        A.base = nullptr;
        size_t ncap = A.high + A.high / 4 + (1u << 20);
        const size_t floor_cap = (size_t)64 << 20, dbl = A.cap < ((size_t)1 << 30) ? 2 * A.cap : 0;
        if (ncap < floor_cap) ncap = floor_cap;
        if (ncap < dbl) ncap = dbl;
        if (cudaMalloc(&A.base, ncap) != cudaSuccess) {
            cudaGetLastError();
            A.cap = 0;
            A.high = 0;
        } else {
            A.cap = ncap;
        }
    }
    A.used = 0;
    A.req = 0;
    A.high = 0;
    return SB_OK;
}

ArenaMark arena_mark(Ctx* ctx) {
    ArenaMark m;
    m.used = ctx->arena.used;
    m.req = ctx->arena.req;
    return m;
}

void arena_release(Ctx* ctx, ArenaMark m) {
    ctx->arena.used = m.used;  // overflow blocks stay allocated until the next reset
    ctx->arena.req = m.req;
}

int arena_alloc(Ctx* ctx, size_t bytes, void** out) {
    Arena& A = ctx->arena;
    size_t sz = (bytes + 255) & ~(size_t)255;
    if (sz == 0) sz = 256;
    A.req += sz;
    if (A.req > A.high) A.high = A.req;
    if (A.used + sz <= A.cap) {
        *out = A.base + A.used;
        A.used += sz;
        return SB_OK;
    }
    void* p = nullptr;
    SB_CUDA(ctx, cudaMalloc(&p, sz));
    A.overflow.push_back(p);
    *out = p;
    return SB_OK;
}

void stage_mark(Ctx* ctx, int stage) {
    if (!ctx->profiling || ctx->n_ev >= 128) return;
    while (ctx->ev_created <= ctx->n_ev) {
        if (cudaEventCreate(&ctx->ev[ctx->ev_created]) != cudaSuccess) return;
        ctx->ev_created++;
    }
    cudaEventRecord(ctx->ev[ctx->n_ev], ctx->stream);
    ctx->ev_host[ctx->n_ev] =
        std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
    ctx->ev_stage[ctx->n_ev] = stage;
    ctx->n_ev++;
}

void trace_mark(Ctx* ctx, const char* name) {
    static const bool on = getenv("SB_PIPE_TRACE") != nullptr;
    if (!on) return;
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    cudaEventRecord(e, ctx->stream);
    ctx->trace.push_back({name, e});
}

void trace_dump(Ctx* ctx) {
    if (ctx->trace.empty()) return;
    cudaStreamSynchronize(ctx->stream);
    for (size_t i = 1; i < ctx->trace.size(); ++i) {
        float ms = 0.f, d = 0.f;
        cudaEventElapsedTime(&ms, ctx->trace[0].second, ctx->trace[i].second);
        cudaEventElapsedTime(&d, ctx->trace[i - 1].second, ctx->trace[i].second);
        fprintf(stderr, "[slam_b200]   %-18s at %8.3f ms (+%.3f)\n", ctx->trace[i].first, ms, d);
    }
    for (auto& t : ctx->trace) cudaEventDestroy(t.second);
    ctx->trace.clear();
}

__global__ void k_copy_words(uint32_t* __restrict__ dst, const uint32_t* __restrict__ src, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) dst[i] = src[i];
}

int table_upload(Ctx* ctx, void* d_dst, const void* h_src, size_t bytes) {
    if (bytes == 0) return SB_OK;
    if (!ctx->tbuf) {
        const size_t cap = (size_t)32 << 20;
        if (cudaHostAlloc(&ctx->tbuf, cap, cudaHostAllocMapped) == cudaSuccess &&
            cudaHostGetDevicePointer((void**)&ctx->tbuf_dev, ctx->tbuf, 0) == cudaSuccess) {
            ctx->tbuf_cap = cap;
        } else {
            cudaGetLastError();
            ctx->tbuf = nullptr;
            ctx->tbuf_cap = 0;
        }
    }
    const size_t need = (bytes + 15) & ~(size_t)15;
    if ((bytes & 3) != 0 || ctx->tbuf_used + need > ctx->tbuf_cap) {  // odd size or buffer full: the copy engine
        SB_CUDA(ctx, cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, ctx->stream));
        return SB_OK;
    }
    memcpy(ctx->tbuf + ctx->tbuf_used, h_src, bytes);
    const size_t words = bytes / 4;
    const int grid = (int)((words + 255) / 256 < 64 ? (words + 255) / 256 : 64);
    SB_LAUNCH(ctx, k_copy_words, grid, 256, 0, static_cast<uint32_t*>(d_dst),
              reinterpret_cast<const uint32_t*>(ctx->tbuf_dev + ctx->tbuf_used), words);
    ctx->tbuf_used += need;
    return SB_OK;
}

int pinned_reserve(Ctx* ctx, size_t bytes) {
    if (bytes <= ctx->pinned_cap) return SB_OK;
    cudaStreamSynchronize(ctx->stream);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    ctx->pinned = nullptr;
    ctx->pinned_cap = 0;
    size_t cap = bytes + bytes / 2 + 4096;
    SB_CUDA(ctx, cudaMallocHost(&ctx->pinned, cap));
    ctx->pinned_cap = cap;
    return SB_OK;
}

static int upload(Ctx* ctx, const void* h, size_t bytes, void** d) {
    SB_TRY(arena_alloc(ctx, bytes, d));
    if (bytes) SB_CUDA(ctx, cudaMemcpyAsync(*d, h, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return SB_OK;
}

static int download(Ctx* ctx, void* h, const void* d, size_t bytes) {
    if (bytes) SB_CUDA(ctx, cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return SB_OK;
}

static std::vector<QueryItem> items_for(i64 nq) {
    std::vector<QueryItem> items;
    items.reserve((size_t)((nq + 31) / 32));
    for (i64 s = 0; s < nq; s += 32) {
        QueryItem I;
        I.q_off = s;
        I.count = (int)(nq - s < 32 ? nq - s : 32);
        I.tree = 0;
        items.push_back(I);
    }
    return items;
}

int ensure_copy_stream(Ctx* ctx) {
    if (!ctx->copy_stream) {
        SB_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i) SB_CUDA(ctx, cudaEventCreateWithFlags(&ctx->copy_ev[i], cudaEventDisableTiming));
    }
    return SB_OK;
}

// Host clouds -> device, voxel grid.  The raw rows are copied in chunks of whole clouds on a second stream and the
// voxel grid of chunk c runs while chunk c+1 is in flight (pinned host memory; pageable memory still works, without
// the overlap).  d_ds receives the downsampled rows of all clouds, off_ds their CSR offsets.
static int upload_voxel_pipelined(Ctx* ctx, const void* h_raw, int f32, int stride, const i64* offsets, int n_clouds,
                                  double voxel, double* d_ds, i64* off_ds,
                                  const std::function<int(int, int)>& after_chunk) {
    const size_t row_bytes = (size_t)stride * (f32 ? sizeof(float) : sizeof(double));
    const i64 n = offsets[n_clouds];
    char* d_raw;
    SB_TRY(arena_get(ctx, (size_t)(n > 0 ? n : 1) * row_bytes, &d_raw));
    SB_TRY(ensure_copy_stream(ctx));
    // chunk boundaries: whole clouds.  The body of the transfer goes in chunks of about 384 MB (SB_CHUNK_MB): smaller
    // chunks pay more per-chunk host round trips than they gain in overlap (measured per C2 step from float32
    // records: 128 MB 57.9 ms, 256 MB 55.5 ms, 384 MB 54.4 ms, 512 MB 55.7 ms).  The first two and the last two chunks
    // are smaller (1/6 and 1/2.4 of that): the device idles while the first chunk arrives and the copy engine idles
    // while the last one is processed, so the pipeline fills and drains on small pieces (SB_CHUNK_RAMP=0: off).
    std::vector<int> cb(1, 0);
    {
        const long chunk_mb = getenv("SB_CHUNK_MB") ? atol(getenv("SB_CHUNK_MB")) : 384;
        const double body = (double)((size_t)(chunk_mb > 0 ? chunk_mb : 384) << 20);
        const double total = (double)n * (double)row_bytes;
        static const bool ramp = !(getenv("SB_CHUNK_RAMP") && atoi(getenv("SB_CHUNK_RAMP")) == 0);
        std::vector<double> sizes;
        const double edge = body / 6.0 + body / 2.4;
        if (ramp && total > 2.0 * edge + 0.5 * body) {
            const int k = (int)ceil((total - 2.0 * edge) / body);
            sizes.push_back(body / 6.0);
            sizes.push_back(body / 2.4);
            for (int i = 0; i < k; ++i) sizes.push_back((total - 2.0 * edge) / k);
            sizes.push_back(body / 2.4);
            sizes.push_back(body / 6.0);
        }
        i64 start = 0;
        size_t si = 0;
        for (int c = 0; c < n_clouds; ++c) {
            const double want = si < sizes.size() ? sizes[si] : body;
            if ((double)(offsets[c + 1] - start) * (double)row_bytes >= want || c == n_clouds - 1) {
                cb.push_back(c + 1);
                start = offsets[c + 1];
                ++si;
            }
        }
        if (cb.back() != n_clouds) cb.push_back(n_clouds);
    }
    const int n_chunks = (int)cb.size() - 1;
    auto enqueue_copy = [&](int k) -> int {
        const i64 r0 = offsets[cb[k]], r1 = offsets[cb[k + 1]];
        if (r1 > r0)
            SB_CUDA(ctx, cudaMemcpyAsync(d_raw + (size_t)r0 * row_bytes, static_cast<const char*>(h_raw) + (size_t)r0 * row_bytes,
                                         (size_t)(r1 - r0) * row_bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
        SB_CUDA(ctx, cudaEventRecord(ctx->copy_ev[k & 1], ctx->copy_stream));
        return SB_OK;
    };
    off_ds[0] = 0;
    // SB_PIPE_TRACE=1: device timeline of the pipeline (copy done / voxel grid / index + normals per chunk) on stderr
    static const bool trace = getenv("SB_PIPE_TRACE") != nullptr;
    std::vector<cudaEvent_t> tev;
    auto tmark = [&](cudaStream_t st) {
        if (!trace) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, st);
        tev.push_back(e);
    };
    tmark(ctx->stream);
    if (n_chunks > 0) SB_TRY(enqueue_copy(0));
    tmark(ctx->copy_stream);
    std::vector<i64> in_off, out_off;
    for (int k = 0; k < n_chunks; ++k) {
        SB_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->copy_ev[k & 1], 0));
        if (k + 1 < n_chunks) SB_TRY(enqueue_copy(k + 1));  // in flight while chunk k is voxelised
        tmark(ctx->copy_stream);
        tmark(ctx->stream);
        const int c0 = cb[k], nc = cb[k + 1] - cb[k];
        in_off.assign((size_t)nc + 1, 0);
        out_off.assign((size_t)nc + 1, 0);
        for (int i = 0; i <= nc; ++i) in_off[i] = offsets[c0 + i] - offsets[c0];
        PointSrc src;
        src.base = d_raw + (size_t)offsets[c0] * row_bytes;
        src.f32 = f32;
        src.stride = stride;
        const ArenaMark mark = arena_mark(ctx);
        stage_mark(ctx, STAGE_VOXEL);
        SB_TRY(voxel_downsample_src(ctx, src, in_off.data(), nc, voxel, d_ds + 3 * off_ds[c0], out_off.data(), nullptr));
        arena_release(ctx, mark);
        tmark(ctx->stream);
        for (int i = 1; i <= nc; ++i) off_ds[c0 + i] = off_ds[c0] + out_off[i];
        if (after_chunk) SB_TRY(after_chunk(c0, c0 + nc));  // more device work on these clouds while the next chunk copies
        tmark(ctx->stream);
    }
    if (trace) {
        cudaStreamSynchronize(ctx->stream);
        cudaStreamSynchronize(ctx->copy_stream);
        auto at = [&](size_t i) { float ms = 0.f; cudaEventElapsedTime(&ms, tev[0], tev[i]); return ms; };
        fprintf(stderr, "[slam_b200] pipeline: first copy done %.2f ms\n", at(1));
        for (int k = 0; k < n_chunks; ++k) {
            const size_t b = 2 + 4 * (size_t)k;
            fprintf(stderr, "[slam_b200]  chunk %d (%d clouds, %.0f MB): next copy done %.2f | compute start %.2f, voxel done %.2f, "
                    "index+normals done %.2f ms\n", k, cb[k + 1] - cb[k],
                    (double)(offsets[cb[k + 1]] - offsets[cb[k]]) * row_bytes / 1048576.0, at(b), at(b + 1), at(b + 2), at(b + 3));
        }
        for (cudaEvent_t e : tev) cudaEventDestroy(e);
        trace_dump(ctx);
    }
    return SB_OK;
}

// shared implementation of sb_register_batch / _dev.  The clouds are either on the device already (src.base) or
// on the host (h_raw != nullptr: uploaded in chunks, overlapped with the voxel grid).
static int register_batch_impl(Ctx* ctx, PointSrc src, const void* h_raw, const i64* offsets, int n_clouds, double voxel,
                               const int32_t* pair_src, const int32_t* pair_tgt, int n_pairs, const sb_icp_config* cfg,
                               sb_icp_result* results, double* sc_desc) {
    for (int p = 0; p < n_pairs; ++p)
        if (pair_src[p] < 0 || pair_src[p] >= n_clouds || pair_tgt[p] < 0 || pair_tgt[p] >= n_clouds)
            return fail(ctx, SB_ERR_INVALID_ARG, "register_batch: pair %d references a cloud outside [0, %d)", p, n_clouds);
    if (cfg->normals_k < 1 || cfg->normals_k > SB_MAX_K)
        return fail(ctx, SB_ERR_INVALID_ARG, "normals_k %d outside [1, %d]", cfg->normals_k, SB_MAX_K);
    // one tree + normals per distinct target cloud (icp.hpp:166-171); clouds that are only sources get a tree too
    // (no normals): the ICP passes read every source in its own curve order (PairDesc::src_pts)
    std::vector<char> is_tgt((size_t)n_clouds, 0), is_src((size_t)n_clouds, 0);
    for (int p = 0; p < n_pairs; ++p) { is_tgt[pair_tgt[p]] = 1; is_src[pair_src[p]] = 1; }
    std::vector<int> tree_of((size_t)n_clouds, -1);
    int n_index = 0;
    for (int c = 0; c < n_clouds; ++c) n_index += (is_tgt[c] || is_src[c]) ? 1 : 0;
    Forest F;
    F.in_arena = true;
    SB_TRY(forest_reserve(ctx, &F, n_index));
    std::vector<i64> off(offsets, offsets + n_clouds + 1);
    const double* d_pts = nullptr;
    // ---- ICP of the pairs whose scans have arrived, while later chunks are still uploading (pipelined host path):
    // a pair is ready once both of its clouds are indexed.  Ready pairs are registered in sub-batches on a stream of
    // their own, so that the few-pairs-left tail of one sub-batch (the GPU is nearly idle then) runs beside the voxel
    // grid / index / normals of the next chunk instead of in front of them.  Results do not depend on how the pairs
    // are grouped (every pair's sums are added in its own fixed order).
    bool pipelined = false;   // set on the chunked host path: index_clouds then also starts the ICP of the ready pairs
    // the pipelined path leaves work on three streams; every return, an error exit included, waits for all of it,
    // because the next call reuses the arena and the staging buffers as soon as it enters
    struct Drain {
        Ctx* c;
        const bool& on;
        ~Drain() {
            if (!on) return;
            if (c->icp_stream) cudaStreamSynchronize(c->icp_stream);
            if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
            cudaStreamSynchronize(c->stream);
        }
    } drain{ctx, pipelined};
    std::vector<char> launched((size_t)n_pairs, 0);
    std::vector<IcpPending> pending;
    std::vector<std::vector<int>> pending_ids;
    static const int sub_min = getenv("SB_ICP_SUB") ? atoi(getenv("SB_ICP_SUB")) : 256;
    auto icp_ready_pairs = [&](int c1, bool last) -> int {
        std::vector<int> ids;
        for (int p = 0; p < n_pairs; ++p)
            if (!launched[p] && pair_src[p] < c1 && pair_tgt[p] < c1) ids.push_back(p);
        if (ids.empty() || (!last && (int)ids.size() < sub_min)) return SB_OK;
        // one staging slot per sub-batch (Ctx::ICP_SLOTS): when only the last one is left, the ready pairs wait for the
        // last chunk and go with its sub-batch
        if (!last && (int)pending.size() >= Ctx::ICP_SLOTS - 1) return SB_OK;
        std::vector<PairDesc> pairs(ids.size());
        for (size_t i = 0; i < ids.size(); ++i) {
            const int p = ids[i];
            memset(&pairs[i], 0, sizeof(PairDesc));
            pairs[i].tree = tree_of[pair_tgt[p]];
            pairs[i].src_tree = tree_of[pair_src[p]];
            pairs[i].n_src = (int)(off[pair_src[p] + 1] - off[pair_src[p]]);
            launched[p] = 1;
        }
        if (!ctx->icp_stream) {
            SB_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->icp_stream, cudaStreamNonBlocking));
            SB_CUDA(ctx, cudaEventCreateWithFlags(&ctx->icp_ev, cudaEventDisableTiming));
        }
        // the ICP stream starts after everything enqueued so far (index + normals of these clouds)
        SB_CUDA(ctx, cudaEventRecord(ctx->icp_ev, ctx->stream));
        SB_CUDA(ctx, cudaStreamWaitEvent(ctx->icp_stream, ctx->icp_ev, 0));
        cudaStream_t main_stream = ctx->stream;
        ctx->stream = ctx->icp_stream;
        IcpPending P;
        const int s = icp_enqueue(ctx, &F, pairs, cfg, &P);
        ctx->stream = main_stream;
        SB_TRY(s);
        pending.push_back(P);
        pending_ids.push_back(std::move(ids));
        return SB_OK;
    };
    // index (+ normals for targets) of the clouds in [c0, c1) (their downsampled rows are final)
    auto index_clouds = [&](int c0, int c1) -> int {
        std::vector<int> ids_t, ids_s;
        for (int c = c0; c < c1; ++c) {
            if (is_tgt[c]) ids_t.push_back(c);
            else if (is_src[c]) ids_s.push_back(c);
        }
        if (!ids_t.empty()) {
            if (!h_raw) stage_mark(ctx, STAGE_INDEX);
            for (size_t i = 0; i < ids_t.size(); ++i) tree_of[ids_t[i]] = F.n_trees + (int)i;
            trace_mark(ctx, "index:begin");
            SB_TRY(forest_append(ctx, &F, d_pts, off.data(), ids_t.data(), (int)ids_t.size()));
            trace_mark(ctx, "index:append");
            if (!h_raw) stage_mark(ctx, STAGE_NORMALS);
            SB_TRY(forest_normals(ctx, &F, cfg->normals_k, nullptr, nullptr));
            trace_mark(ctx, "index:normals");
        }
        if (!ids_s.empty()) {
            for (size_t i = 0; i < ids_s.size(); ++i) tree_of[ids_s[i]] = F.n_trees + (int)i;
            SB_TRY(forest_append(ctx, &F, d_pts, off.data(), ids_s.data(), (int)ids_s.size()));
        }
        if (pipelined && n_pairs > 0) SB_TRY(icp_ready_pairs(c1, c1 == n_clouds));
        return SB_OK;
    };
    // 1. voxel grid (slam_node.cpp:122)
    stage_mark(ctx, STAGE_VOXEL);
    const i64 n_raw = offsets[n_clouds];
    bool indexed = false;
    if (voxel > 0) {
        double* d_ds;
        SB_TRY(arena_get(ctx, (size_t)3 * (n_raw > 0 ? n_raw : 1), &d_ds));
        d_pts = d_ds;
        if (h_raw) {  // upload, voxel grid, index and normals chunk by chunk: the copies overlap all of it
            pipelined = true;
            if (n_pairs > 0) SB_TRY(icp_reserve_results(ctx, (size_t)n_pairs));
            SB_TRY(upload_voxel_pipelined(ctx, h_raw, src.f32, src.stride, offsets, n_clouds, voxel, d_ds, off.data(),
                                          n_pairs > 0 ? std::function<int(int, int)>(index_clouds)
                                                      : std::function<int(int, int)>()));
            indexed = true;
        } else {
            const ArenaMark mark = arena_mark(ctx);
            SB_TRY(voxel_downsample_src(ctx, src, offsets, n_clouds, voxel, d_ds, off.data(), nullptr));
            arena_release(ctx, mark);
        }
    } else {  // no voxel grid: the clouds themselves, as packed fp64 rows on the device
        double* d_all;
        SB_TRY(arena_get(ctx, (size_t)3 * (n_raw > 0 ? n_raw : 1), &d_all));
        if (h_raw && !src.f32 && src.stride == 3) {
            if (n_raw > 0) SB_CUDA(ctx, cudaMemcpyAsync(d_all, h_raw, sizeof(double) * 3 * n_raw, cudaMemcpyHostToDevice, ctx->stream));
        } else {
            PointSrc s2 = src;
            if (h_raw) {
                const size_t bytes = (size_t)n_raw * src.stride * (src.f32 ? sizeof(float) : sizeof(double));
                char* d_raw;
                SB_TRY(arena_get(ctx, bytes ? bytes : 1, &d_raw));
                if (bytes) SB_CUDA(ctx, cudaMemcpyAsync(d_raw, h_raw, bytes, cudaMemcpyHostToDevice, ctx->stream));
                s2.base = d_raw;
            }
            i64 dummy_off[2] = {0, n_raw}, out_off2[2];
            SB_TRY(voxel_downsample_src(ctx, s2, dummy_off, 1, 0.0, d_all, out_off2, nullptr));  // voxel <= 0: copy
        }
        d_pts = d_all;
    }
    // 2. Scan Context of every cloud (loop_closure.hpp:53-59)
    stage_mark(ctx, STAGE_SC);
    ctx->last_counts[0] = n_raw;
    ctx->last_counts[1] = off[n_clouds];
    double* d_desc = nullptr;
    // the descriptors go back to the host on the copy stream while the ICP loop runs (or right away without pairs)
    std::function<int()> fetch_sc = [&]() -> int {
        if (!sc_desc) return SB_OK;
        SB_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->copy_ev[0], 0));
        SB_CUDA(ctx, cudaMemcpyAsync(sc_desc, d_desc, sizeof(double) * SB_SC_SIZE * n_clouds, cudaMemcpyDeviceToHost,
                                     ctx->copy_stream));
        SB_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));
        return SB_OK;
    };
    if (sc_desc) {
        i64* d_off;
        SB_TRY(ensure_copy_stream(ctx));
        SB_TRY(arena_get(ctx, (size_t)n_clouds + 1, &d_off));
        SB_TRY(table_upload(ctx, d_off, off.data(), sizeof(i64) * (n_clouds + 1)));
        SB_TRY(arena_get(ctx, (size_t)n_clouds * SB_SC_SIZE, &d_desc));
        SB_TRY(sc_compute_dev(ctx, d_pts, d_off, n_clouds, d_desc));
        SB_CUDA(ctx, cudaEventRecord(ctx->copy_ev[0], ctx->stream));  // the upload pipeline is done with its events
    }
    if (n_pairs == 0) {
        SB_TRY(fetch_sc());
        stage_mark(ctx, STAGE_END);
        SB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        forest_free(&F);
        return SB_OK;
    }
    // 3. index + normals of the targets (already done chunk by chunk on the pipelined host path)
    int s = SB_OK;
    if (!indexed) s = index_clouds(0, n_clouds);
    stage_mark(ctx, STAGE_ICP);
    ctx->last_counts[2] = F.n_points;
    // 4. the ICP loop for all pairs (icp.hpp:174-255); on the pipelined host path it was enqueued chunk by chunk
    if (s == SB_OK && indexed) {
        s = fetch_sc();
        std::vector<const int*> idp;
        for (const std::vector<int>& v : pending_ids) idp.push_back(v.data());
        if (s == SB_OK) s = icp_collect(ctx, ctx->icp_stream ? ctx->icp_stream : ctx->stream, pending, idp, results);
        if (s == SB_OK) {
            i64 q = 0;
            for (int p = 0; p < n_pairs; ++p) q += (i64)(off[pair_src[p] + 1] - off[pair_src[p]]) * results[p].history_len;
            ctx->last_counts[3] = q;
        }
    } else if (s == SB_OK) {
        std::vector<PairDesc> pairs((size_t)n_pairs);
        for (int p = 0; p < n_pairs; ++p) {
            memset(&pairs[p], 0, sizeof(PairDesc));
            pairs[p].tree = tree_of[pair_tgt[p]];
            pairs[p].src_tree = tree_of[pair_src[p]];
            pairs[p].n_src = (int)(off[pair_src[p] + 1] - off[pair_src[p]]);
        }
        s = icp_batch(ctx, &F, pairs, cfg, results, &fetch_sc);
        if (s == SB_OK) {
            i64 q = 0;
            for (int p = 0; p < n_pairs; ++p) q += (i64)pairs[p].n_src * results[p].history_len;
            ctx->last_counts[3] = q;
        }
    }
    stage_mark(ctx, STAGE_END);
    cudaStreamSynchronize(ctx->stream);
    forest_free(&F);
    return s;
}

}  // namespace sb

using namespace sb;

extern "C" {

const char* sb_version(void) { return "slam_b200 0.1 (sm_100a)"; }

int sb_ctx_create(int device, void* stream, sb_ctx** out) {
    if (!out) return SB_ERR_INVALID_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) {
        cudaGetLastError();
        return SB_ERR_NO_DEVICE;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return SB_ERR_NO_DEVICE;
    if (prop.major != 10 || prop.minor != 0) return SB_ERR_NO_DEVICE;  // the library holds sm_100a SASS only, no PTX
    if (cudaSetDevice(device) != cudaSuccess) return SB_ERR_NO_DEVICE;
    sb_ctx* c = new sb_ctx();
    c->c.device = device;
    c->c.sm_count = prop.multiProcessorCount;
    if (stream) {
        c->c.stream = static_cast<cudaStream_t>(stream);
    } else {
        if (cudaStreamCreateWithFlags(&c->c.stream, cudaStreamNonBlocking) != cudaSuccess) {
            delete c;
            return SB_ERR_CUDA;
        }
        c->c.own_stream = true;
    }
    c->c.vox_force_sort = getenv("SB_VOXEL_SORT") != nullptr;
    if (cudaMalloc(&c->c.d_flags, sizeof(int)) != cudaSuccess) {
        if (c->c.own_stream) cudaStreamDestroy(c->c.stream);
        delete c;
        return SB_ERR_CUDA;
    }
    *out = c;
    return SB_OK;
}

void sb_ctx_destroy(sb_ctx* ctx) {
    if (!ctx) return;
    Ctx* c = &ctx->c;
    cudaSetDevice(c->device);
    if (c->icp_stream) cudaStreamSynchronize(c->icp_stream);
    if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    cudaStreamSynchronize(c->stream);
    icp_graph_free(c);
    for (void* p : c->arena.overflow) cudaFree(p);
    cudaFree(c->arena.base);
    cudaFree(c->d_flags);
    for (int i = 0; i < c->ev_created; ++i) cudaEventDestroy(c->ev[i]);
    if (c->pinned) cudaFreeHost(c->pinned);
    if (c->h_many) cudaFreeHost(c->h_many);
    if (c->h_icp_res) cudaFreeHost(c->h_icp_res);
    if (c->h_icp_passes) cudaFreeHost(c->h_icp_passes);
    if (c->icp_stream) cudaStreamDestroy(c->icp_stream);
    if (c->icp_ev) cudaEventDestroy(c->icp_ev);
    if (c->tbuf) cudaFreeHost(c->tbuf);
    for (int i = 0; i < 2; ++i)
        if (c->copy_ev[i]) cudaEventDestroy(c->copy_ev[i]);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->own_stream) cudaStreamDestroy(c->stream);
    delete ctx;
}

const char* sb_last_error(const sb_ctx* ctx) { return ctx ? ctx->c.err.c_str() : "null context"; }

int sb_ctx_synchronize(sb_ctx* ctx) {
    if (!ctx) return SB_ERR_INVALID_ARG;
    SB_CUDA(&ctx->c, cudaStreamSynchronize(ctx->c.stream));
    return SB_OK;
}

int64_t sb_ctx_launch_count(const sb_ctx* ctx) { return ctx ? ctx->c.launches : 0; }

int sb_ctx_set_profiling(sb_ctx* ctx, int enable) {
    if (!ctx) return SB_ERR_INVALID_ARG;
    ctx->c.profiling = enable != 0;
    ctx->c.n_ev = 0;
    return SB_OK;
}

int sb_ctx_stage_ms(sb_ctx* ctx, double* ms7) {
    if (!ctx || !ms7) return SB_ERR_INVALID_ARG;
    Ctx* c = &ctx->c;
    for (int i = 0; i < STAGE_COUNT; ++i) ms7[i] = 0.0;
    SB_CUDA(c, cudaStreamSynchronize(c->stream));
    for (int i = 0; i + 1 < c->n_ev; ++i) {
        int st = c->ev_stage[i];
        if (st < 0 || st >= STAGE_COUNT) continue;
        float ms = 0.f;
        SB_CUDA(c, cudaEventElapsedTime(&ms, c->ev[i], c->ev[i + 1]));
        ms7[st] += (double)ms;
    }
    return SB_OK;
}

int sb_ctx_stage_host_ms(sb_ctx* ctx, double* ms7) {
    if (!ctx || !ms7) return SB_ERR_INVALID_ARG;
    Ctx* c = &ctx->c;
    for (int i = 0; i < STAGE_COUNT; ++i) ms7[i] = 0.0;
    for (int i = 0; i + 1 < c->n_ev; ++i) {
        int st = c->ev_stage[i];
        if (st >= 0 && st < STAGE_COUNT) ms7[st] += c->ev_host[i + 1] - c->ev_host[i];
    }
    return SB_OK;
}

int sb_ctx_last_counts(sb_ctx* ctx, int64_t* counts5) {
    if (!ctx || !counts5) return SB_ERR_INVALID_ARG;
    for (int i = 0; i < 4; ++i) counts5[i] = ctx->c.last_counts[i];
    counts5[4] = ctx->c.last_icp_iterations;
    return SB_OK;
}

int sb_ctx_last_voxel_path(const sb_ctx* ctx) { return ctx ? ctx->c.vox_last_path : 0; }

void sb_default_icp_config(sb_icp_config* cfg) {  // types.hpp:143-148, icp.hpp:170
    cfg->max_iterations = 50;
    cfg->normals_k = 20;
    cfg->tolerance = 1e-6;
    cfg->min_error = 1e-9;
    for (int i = 0; i < 16; ++i) cfg->initial_transform[i] = (i % 5 == 0) ? 1.0 : 0.0;
}

void sb_default_loop_config(sb_loop_config* cfg) {  // loop_closure.hpp:14-19, 105-107
    cfg->frame_gap = 50;
    cfg->max_candidates = 3;
    cfg->sc_distance_threshold = 0.25;
    cfg->icp_fitness_threshold = 0.3;
    cfg->icp_max_iterations = 30;
    cfg->normals_k = 20;
    cfg->icp_tolerance = 1e-6;
    cfg->verify_chunk = 0;
    cfg->reserved = 0;
}

// ---------------------------------------------------------------- voxel grid
int sb_voxel_downsample_batch_dev(sb_ctx* ctx, const double* d_xyz, const int64_t* offsets, int32_t n_clouds,
                                  double voxel, double* d_out_xyz, int64_t* out_offsets, int64_t* d_out_keys) {
    if (!ctx || !offsets || !out_offsets || n_clouds < 0) return SB_ERR_INVALID_ARG;
    Ctx* c = &ctx->c;
    Enter g(c);
    for (int i = 0; i < n_clouds; ++i)
        if (offsets[i + 1] < offsets[i]) return fail(c, SB_ERR_INVALID_ARG, "offsets must be non-decreasing");
    if (offsets[n_clouds] > 0 && (!d_xyz || !d_out_xyz)) return fail(c, SB_ERR_INVALID_ARG, "null point buffer");
    return voxel_downsample_dev(c, d_xyz, (const i64*)offsets, n_clouds, voxel, d_out_xyz, (i64*)out_offsets,
                                (i64*)d_out_keys);
}

int sb_voxel_downsample_batch(sb_ctx* ctx, const double* xyz, const int64_t* offsets, int32_t n_clouds, double voxel,
                              double* out_xyz, int64_t* out_offsets, int64_t* out_keys) {
    if (!ctx || !offsets || !out_offsets || n_clouds < 0) return SB_ERR_INVALID_ARG;
    Ctx* c = &ctx->c;
    Enter g(c);
    for (int i = 0; i < n_clouds; ++i)
        if (offsets[i + 1] < offsets[i]) return fail(c, SB_ERR_INVALID_ARG, "offsets must be non-decreasing");
    i64 n = offsets[n_clouds];
    if (n > 0 && (!xyz || !out_xyz)) return fail(c, SB_ERR_INVALID_ARG, "null point buffer");
    double *d_in, *d_out;
    i64* d_keys = nullptr;
    SB_TRY(upload(c, xyz, sizeof(double) * 3 * n, (void**)&d_in));
    SB_TRY(arena_get(c, (size_t)3 * (n > 0 ? n : 1), &d_out));
    if (out_keys) SB_TRY(arena_get(c, (size_t)3 * (n > 0 ? n : 1), &d_keys));
    SB_TRY(voxel_downsample_dev(c, d_in, (const i64*)offsets, n_clouds, voxel, d_out, (i64*)out_offsets, d_keys));
    i64 m = out_offsets[n_clouds];
    SB_TRY(download(c, out_xyz, d_out, sizeof(double) * 3 * m));
    if (out_keys) SB_TRY(download(c, out_keys, d_keys, sizeof(i64) * 3 * m));
    SB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SB_OK;
}

int sb_voxel_downsample_batch_f32(sb_ctx* ctx, const float* xyz, int32_t stride_floats, const int64_t* offsets,
                                  int32_t n_clouds, double voxel, double* out_xyz, int64_t* out_offsets,
                                  int64_t* out_keys) {
    if (!ctx || !offsets || !out_offsets || n_clouds < 0) return SB_ERR_INVALID_ARG;
    Ctx* c = &ctx->c;
    Enter g(c);
    if (stride_floats < 3) return fail(c, SB_ERR_INVALID_ARG, "row stride %d < 3", stride_floats);
    if (offsets[0] != 0) return fail(c, SB_ERR_INVALID_ARG, "offsets must start at 0");
    for (int i = 0; i < n_clouds; ++i)
        if (offsets[i + 1] < offsets[i]) return fail(c, SB_ERR_INVALID_ARG, "offsets must be non-decreasing");
    i64 n = offsets[n_clouds];
    if (n > 0 && (!xyz || !out_xyz)) return fail(c, SB_ERR_INVALID_ARG, "null point buffer");
    float* d_in;
    double* d_out;
    i64* d_keys = nullptr;
    SB_TRY(upload(c, xyz, sizeof(float) * (size_t)stride_floats * n, (void**)&d_in));
    SB_TRY(arena_get(c, (size_t)3 * (n > 0 ? n : 1), &d_out));
    if (out_keys) SB_TRY(arena_get(c, (size_t)3 * (n > 0 ? n : 1), &d_keys));
    PointSrc src;
    src.base = d_in; src.f32 = 1; src.stride = stride_floats;
    SB_TRY(voxel_downsample_src(c, src, (const i64*)offsets, n_clouds, voxel, d_out, (i64*)out_offsets, d_keys));
    i64 m = out_offsets[n_clouds];
    SB_TRY(download(c, out_xyz, d_out, sizeof(double) * 3 * m));
    if (out_keys) SB_TRY(download(c, out_keys, d_keys, sizeof(i64) * 3 * m));
    SB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SB_OK;
}

int sb_voxel_downsample(sb_ctx* ctx, const double* xyz, int64_t n, double voxel, double* out_xyz, int64_t* out_m,
                        int64_t* out_keys) {
    if (!ctx || !out_m || n < 0) return SB_ERR_INVALID_ARG;
    int64_t off[2] = {0, n}, out_off[2] = {0, 0};
    int s = sb_voxel_downsample_batch(ctx, xyz, off, 1, voxel, out_xyz, out_off, out_keys);
    *out_m = out_off[1];
    return s;
}

// ---------------------------------------------------------------- spatial index
int sb_index_build(sb_ctx* ctx, const double* xyz, int64_t n, sb_index** out) {
    if (!ctx || !out || n < 0 || (n > 0 && !xyz)) return SB_ERR_INVALID_ARG;
    Ctx* c = &ctx->c;
    Enter g(c);
    *out = nullptr;
    if (n > 0x7fffffffLL) return fail(c, SB_ERR_RANGE, "index: more than 2^31-1 points");
    double* d_xyz;
    SB_TRY(upload(c, xyz, sizeof(double) * 3 * n, (void**)&d_xyz));
    sb_index* ix = new sb_index();
    ix->ctx = c;
    i64 off[2] = {0, n};
    int s = forest_build(c, d_xyz, off, nullptr, 1, &ix->forest);
    if (s == SB_OK && cudaStreamSynchronize(c->stream) != cudaSuccess)
        s = fail(c, SB_ERR_CUDA, "index build: %s", cudaGetErrorString(cudaGetLastError()));
    if (s != SB_OK) {
        forest_free(&ix->forest);
        delete ix;
        return s;
    }
    *out = ix;
    return SB_OK;
}

void sb_index_free(sb_index* index) {
    if (!index) return;
    cudaSetDevice(index->ctx->device);
    cudaStreamSynchronize(index->ctx->stream);
    forest_free(&index->forest);
    delete index;
}

int64_t sb_index_size(const sb_index* index) { return index ? index->forest.n_points : 0; }

int sb_index_nearest_batch(sb_index* index, const double* queries, int64_t nq, int32_t* out_idx, double* out_d2) {
    if (!index || nq < 0 || (nq > 0 && (!queries || !out_idx))) return SB_ERR_INVALID_ARG;
    Ctx* c = index->ctx;
    Enter g(c);
    if (nq == 0) return SB_OK;
    double* d_q;
    int* d_idx;
    double* d_d2 = nullptr;
    QueryItem* d_items;
    SB_TRY(upload(c, queries, sizeof(double) * 3 * nq, (void**)&d_q));
    SB_TRY(arena_get(c, (size_t)nq, &d_idx));
    if (out_d2) SB_TRY(arena_get(c, (size_t)nq, &d_d2));
    std::vector<QueryItem> items = items_for(nq);
    SB_TRY(make_items_dev(c, items, &d_items));
    SB_TRY(forest_nearest(c, &index->forest, d_q, d_items, (i64)items.size(), d_idx, d_d2, nullptr));
    SB_TRY(download(c, out_idx, d_idx, sizeof(int) * nq));
    if (out_d2) SB_TRY(download(c, out_d2, d_d2, sizeof(double) * nq));
    SB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SB_OK;
}

int sb_index_knn(sb_index* index, const double* queries, int64_t nq, int32_t k, int32_t* out_idx, double* out_d2) {
    if (!index || nq < 0 || (nq > 0 && (!queries || !out_idx))) return SB_ERR_INVALID_ARG;
    Ctx* c = index->ctx;
    Enter g(c);
    if (k < 1 || k > SB_MAX_K) return fail(c, SB_ERR_INVALID_ARG, "k %d outside [1, %d]", k, SB_MAX_K);
    if (nq == 0) return SB_OK;
    double* d_q;
    int* d_idx;
    double* d_d2 = nullptr;
    QueryItem* d_items;
    SB_TRY(upload(c, queries, sizeof(double) * 3 * nq, (void**)&d_q));
    SB_TRY(arena_get(c, (size_t)nq * k, &d_idx));
    if (out_d2) SB_TRY(arena_get(c, (size_t)nq * k, &d_d2));
    std::vector<QueryItem> items = items_for(nq);
    SB_TRY(make_items_dev(c, items, &d_items));
    if (index->forest.n_points == 0) {  // empty tree: every slot is padding
        SB_CUDA(c, cudaMemsetAsync(d_idx, 0xff, sizeof(int) * nq * k, c->stream));
        SB_TRY(download(c, out_idx, d_idx, sizeof(int) * nq * k));
        SB_CUDA(c, cudaStreamSynchronize(c->stream));
        if (out_d2) for (i64 i = 0; i < nq * k; ++i) out_d2[i] = 1.7976931348623157e308;
        return SB_OK;
    }
    SB_TRY(forest_knn(c, &index->forest, d_q, d_items, (i64)items.size(), k, d_idx, d_d2));
    SB_TRY(download(c, out_idx, d_idx, sizeof(int) * nq * k));
    if (out_d2) SB_TRY(download(c, out_d2, d_d2, sizeof(double) * nq * k));
    SB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SB_OK;
}

int sb_index_find_correspondences(sb_index* index, const double* source, int64_t ns, double* matched_xyz,
                                  double* distances) {
    if (!index || ns < 0 || (ns > 0 && (!source || !matched_xyz))) return SB_ERR_INVALID_ARG;
    Ctx* c = index->ctx;
    if (ns > 0 && index->forest.n_points == 0) {
        Enter g(c);
        return fail(c, SB_ERR_EMPTY, "find_correspondences on an empty index (kdtree.hpp:211 is undefined there)");
    }
    std::vector<int32_t> idx((size_t)ns);
    std::vector<double> d2((size_t)ns);
    SB_TRY(sb_index_nearest_batch(index, source, ns, idx.data(), d2.data()));
    // matched rows (kdtree.hpp:208-212): from a host copy of the indexed cloud in original row order, fetched from the
    // device tree on the first call only — callers of the mirror's NearestNeighborSearch make this call once per
    // ICP iteration
    Enter g(c);
    const Forest& F = index->forest;
    const i64 n = F.n_points;
    if ((i64)index->host_rows.size() != 3 * n) {
        std::vector<TreePoint> pts((size_t)n);
        SB_TRY(download(c, pts.data(), F.batches[0].pts, sizeof(TreePoint) * n));
        SB_CUDA(c, cudaStreamSynchronize(c->stream));
        index->host_rows.assign((size_t)(3 * n), 0.0);
        for (i64 p = 0; p < n; ++p) {
            double* r = index->host_rows.data() + 3 * (size_t)pts[p].idx;
            r[0] = pts[p].x; r[1] = pts[p].y; r[2] = pts[p].z;
        }
    }
    const double nan = std::numeric_limits<double>::quiet_NaN();
    for (i64 i = 0; i < ns; ++i) {
        // a NaN query has no nearest neighbour (index -1, kdtree.hpp:125 never updates): NaN row, NaN distance
        const bool hit = idx[i] >= 0 && idx[i] < n;
        const double* r = hit ? index->host_rows.data() + 3 * (size_t)idx[i] : nullptr;
        matched_xyz[3 * i] = hit ? r[0] : nan; matched_xyz[3 * i + 1] = hit ? r[1] : nan; matched_xyz[3 * i + 2] = hit ? r[2] : nan;
        if (distances) distances[i] = hit ? sqrt(d2[i]) : nan;
    }
    return SB_OK;
}

int sb_estimate_normals(sb_index* index, int32_t k, double* out_normals, double* out_evals) {
    if (!index || !out_normals) return SB_ERR_INVALID_ARG;
    Ctx* c = index->ctx;
    Enter g(c);
    if (k < 1 || k > SB_MAX_K) return fail(c, SB_ERR_INVALID_ARG, "k %d outside [1, %d]", k, SB_MAX_K);
    i64 n = index->forest.n_points;
    if (n == 0) return SB_OK;
    double *d_n, *d_e = nullptr;
    SB_TRY(arena_get(c, (size_t)3 * n, &d_n));
    if (out_evals) SB_TRY(arena_get(c, (size_t)3 * n, &d_e));
    SB_TRY(forest_normals(c, &index->forest, k, d_n, d_e));
    SB_TRY(download(c, out_normals, d_n, sizeof(double) * 3 * n));
    if (out_evals) SB_TRY(download(c, out_evals, d_e, sizeof(double) * 3 * n));
    SB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SB_OK;
}

// ---------------------------------------------------------------- ICP
int sb_solve_point_to_plane(sb_ctx* ctx, const double* source, const double* target, const double* normals, int64_t n,
                            double* out_T16) {
    if (!ctx || !out_T16 || n < 0 || (n > 0 && (!source || !target || !normals))) return SB_ERR_INVALID_ARG;
    Ctx* c = &ctx->c;
    Enter g(c);
    double *d_s, *d_t, *d_n, *d_T;
    SB_TRY(upload(c, source, sizeof(double) * 3 * n, (void**)&d_s));
    SB_TRY(upload(c, target, sizeof(double) * 3 * n, (void**)&d_t));
    SB_TRY(upload(c, normals, sizeof(double) * 3 * n, (void**)&d_n));
    SB_TRY(arena_get(c, 16, &d_T));
    SB_TRY(solve_point_to_plane_dev(c, d_s, d_t, d_n, n, d_T));
    SB_TRY(download(c, out_T16, d_T, sizeof(double) * 16));
    SB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SB_OK;
}

static int register_batch_entry(sb_ctx* ctx, const void* xyz, int on_host, int f32, int stride, const int64_t* offsets,
                                int32_t n_clouds, double voxel, const int32_t* pair_src, const int32_t* pair_tgt,
                                int32_t n_pairs, const sb_icp_config* cfg, sb_icp_result* results, double* sc_desc) {
    if (!ctx || !offsets || n_clouds < 0 || n_pairs < 0 || !cfg) return SB_ERR_INVALID_ARG;
    if (n_pairs > 0 && (!pair_src || !pair_tgt || !results)) return SB_ERR_INVALID_ARG;
    Ctx* c = &ctx->c;
    Enter g(c);
    if (stride < 3) return fail(c, SB_ERR_INVALID_ARG, "row stride %d < 3", stride);
    if (offsets[0] != 0) return fail(c, SB_ERR_INVALID_ARG, "offsets must start at 0");
    for (int i = 0; i < n_clouds; ++i)
        if (offsets[i + 1] < offsets[i]) return fail(c, SB_ERR_INVALID_ARG, "offsets must be non-decreasing");
    if (offsets[n_clouds] > 0 && !xyz) return fail(c, SB_ERR_INVALID_ARG, "null point buffer");
    PointSrc src;
    src.base = on_host ? nullptr : xyz;
    src.f32 = f32;
    src.stride = stride;
    return register_batch_impl(c, src, on_host ? xyz : nullptr, (const i64*)offsets, n_clouds, voxel, pair_src, pair_tgt,
                               n_pairs, cfg, results, sc_desc);
}

int sb_register_batch_dev(sb_ctx* ctx, const double* d_xyz, const int64_t* offsets, int32_t n_clouds, double voxel,
                          const int32_t* pair_src, const int32_t* pair_tgt, int32_t n_pairs, const sb_icp_config* cfg,
                          sb_icp_result* results, double* sc_desc) {
    return register_batch_entry(ctx, d_xyz, 0, 0, 3, offsets, n_clouds, voxel, pair_src, pair_tgt, n_pairs, cfg, results,
                                sc_desc);
}

int sb_register_batch(sb_ctx* ctx, const double* xyz, const int64_t* offsets, int32_t n_clouds, double voxel,
                      const int32_t* pair_src, const int32_t* pair_tgt, int32_t n_pairs, const sb_icp_config* cfg,
                      sb_icp_result* results, double* sc_desc) {
    return register_batch_entry(ctx, xyz, 1, 0, 3, offsets, n_clouds, voxel, pair_src, pair_tgt, n_pairs, cfg, results,
                                sc_desc);
}

int sb_register_batch_f32(sb_ctx* ctx, const float* xyz, int32_t stride_floats, const int64_t* offsets, int32_t n_clouds,
                          double voxel, const int32_t* pair_src, const int32_t* pair_tgt, int32_t n_pairs,
                          const sb_icp_config* cfg, sb_icp_result* results, double* sc_desc) {
    return register_batch_entry(ctx, xyz, 1, 1, stride_floats, offsets, n_clouds, voxel, pair_src, pair_tgt, n_pairs, cfg,
                                results, sc_desc);
}

int sb_register_batch_f32_dev(sb_ctx* ctx, const float* d_xyz, int32_t stride_floats, const int64_t* offsets,
                              int32_t n_clouds, double voxel, const int32_t* pair_src, const int32_t* pair_tgt,
                              int32_t n_pairs, const sb_icp_config* cfg, sb_icp_result* results, double* sc_desc) {
    return register_batch_entry(ctx, d_xyz, 0, 1, stride_floats, offsets, n_clouds, voxel, pair_src, pair_tgt, n_pairs, cfg,
                                results, sc_desc);
}

int sb_icp_point_to_plane(sb_ctx* ctx, const double* source, int64_t ns, const double* target, int64_t nt,
                          const sb_icp_config* cfg, sb_icp_result* out) {
    if (!ctx || !cfg || !out || ns < 0 || nt < 0) return SB_ERR_INVALID_ARG;
    if (ns == 0 || nt == 0) {
        Enter g(&ctx->c);
        return fail(&ctx->c, SB_ERR_EMPTY, "icp: empty %s cloud (undefined behaviour in the reference, kdtree.hpp:25,119)",
                    ns == 0 ? "source" : "target");
    }
    std::vector<double> both((size_t)3 * (ns + nt));
    memcpy(both.data(), source, sizeof(double) * 3 * ns);
    memcpy(both.data() + 3 * ns, target, sizeof(double) * 3 * nt);
    int64_t off[3] = {0, ns, ns + nt};
    int32_t ps = 0, pt = 1;
    int s = sb_register_batch(ctx, both.data(), off, 2, 0.0, &ps, &pt, 1, cfg, out, nullptr);
    if (s == SB_OK && out->status != SB_OK) s = out->status;
    return s;
}

// ---------------------------------------------------------------- Scan Context
int sb_sc_compute(sb_ctx* ctx, const double* xyz, int64_t n, double* desc) {
    if (!ctx || !desc || n < 0 || (n > 0 && !xyz)) return SB_ERR_INVALID_ARG;
    Ctx* c = &ctx->c;
    Enter g(c);
    double *d_xyz, *d_desc;
    i64* d_off;
    i64 off[2] = {0, n};
    SB_TRY(upload(c, xyz, sizeof(double) * 3 * n, (void**)&d_xyz));
    SB_TRY(upload(c, off, sizeof(off), (void**)&d_off));
    SB_TRY(arena_get(c, SB_SC_SIZE, &d_desc));
    SB_TRY(sc_compute_dev(c, d_xyz, d_off, 1, d_desc));
    SB_TRY(download(c, desc, d_desc, sizeof(double) * SB_SC_SIZE));
    SB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SB_OK;
}

int sb_sc_distance_batch(sb_ctx* ctx, const double* query, const double* db, int32_t n_db, double* out_dist) {
    if (!ctx || !query || n_db < 0 || (n_db > 0 && (!db || !out_dist))) return SB_ERR_INVALID_ARG;
    Ctx* c = &ctx->c;
    Enter g(c);
    if (n_db == 0) return SB_OK;
    double *d_q, *d_db, *d_out;
    SB_TRY(upload(c, query, sizeof(double) * SB_SC_SIZE, (void**)&d_q));
    SB_TRY(upload(c, db, sizeof(double) * SB_SC_SIZE * n_db, (void**)&d_db));
    SB_TRY(arena_get(c, (size_t)n_db, &d_out));
    SB_TRY(sc_distance_dev(c, d_q, d_db, n_db, d_out));
    SB_TRY(download(c, out_dist, d_out, sizeof(double) * n_db));
    SB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SB_OK;
}

int sb_sc_distance(sb_ctx* ctx, const double* desc_a, const double* desc_b, double* out) {
    return sb_sc_distance_batch(ctx, desc_a, desc_b, 1, out);
}

int sb_sc_keys(sb_ctx* ctx, const double* desc, double* ring_key20, double* sector_key60) {
    if (!ctx || !desc || !ring_key20 || !sector_key60) return SB_ERR_INVALID_ARG;
    Ctx* c = &ctx->c;
    Enter g(c);
    double *d_desc, *d_r, *d_s;
    SB_TRY(upload(c, desc, sizeof(double) * SB_SC_SIZE, (void**)&d_desc));
    SB_TRY(arena_get(c, SB_SC_RINGS, &d_r));
    SB_TRY(arena_get(c, SB_SC_SECTORS, &d_s));
    SB_TRY(sc_keys_dev(c, d_desc, d_r, d_s));
    SB_TRY(download(c, ring_key20, d_r, sizeof(double) * SB_SC_RINGS));
    SB_TRY(download(c, sector_key60, d_s, sizeof(double) * SB_SC_SECTORS));
    SB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SB_OK;
}

// ---------------------------------------------------------------- loop closure
int sb_loop_create(sb_ctx* ctx, const sb_loop_config* cfg, int32_t rank, int32_t world, sb_loop** out) {
    if (!ctx || !cfg || !out || world < 1 || rank < 0 || rank >= world) return SB_ERR_INVALID_ARG;
    if (cfg->normals_k < 1 || cfg->normals_k > SB_MAX_K || cfg->icp_max_iterations < 0 ||
        cfg->icp_max_iterations > SB_MAX_ICP_ITERATIONS)
        return fail(&ctx->c, SB_ERR_INVALID_ARG, "loop config out of range");
    sb_loop* L = new sb_loop();
    L->ctx = &ctx->c;
    L->cfg = *cfg;
    L->rank = rank;
    L->world = world;
    *out = L;
    return SB_OK;
}

void sb_loop_free(sb_loop* loop) {
    if (!loop) return;
    cudaSetDevice(loop->ctx->device);
    cudaStreamSynchronize(loop->ctx->stream);
    cudaFree(loop->d_desc);
    cudaFree(loop->d_clouds);
    cudaFree(loop->d_meta);
    for (double* p : loop->retired) cudaFree(p);
    delete loop;
}

int sb_loop_reserve(sb_loop* loop, int64_t n_entries, int64_t total_rows) {
    if (!loop || n_entries < 0 || total_rows < 0) return SB_ERR_INVALID_ARG;
    Enter g(loop->ctx);
    return loop_reserve(loop, n_entries, total_rows);
}

int sb_loop_add_frame_desc(sb_loop* loop, const double* xyz, int64_t n, int32_t frame_idx, const double* desc) {
    if (!loop || n < 0 || (n > 0 && !xyz)) return SB_ERR_INVALID_ARG;
    Enter g(loop->ctx);
    return loop_add(loop, xyz, n, frame_idx, desc);
}

int sb_loop_add_frame(sb_loop* loop, const double* xyz, int64_t n, int32_t frame_idx) {
    return sb_loop_add_frame_desc(loop, xyz, n, frame_idx, nullptr);
}

int64_t sb_loop_size(const sb_loop* loop) { return loop ? loop->n_global : 0; }

int sb_loop_clear(sb_loop* loop) {  // loop_closure.hpp:136-141
    if (!loop) return SB_ERR_INVALID_ARG;
    loop->entry_id.clear();
    loop->frame_idx.clear();
    loop->cloud_off.clear();
    loop->n_global = 0;
    loop->last_is_guest = false;
    return SB_OK;
}

int sb_loop_candidates_local(sb_loop* loop, double* dist, int32_t* entry, int32_t capacity, int32_t* count) {
    if (!loop || !count || capacity < 0 || (capacity > 0 && (!dist || !entry))) return SB_ERR_INVALID_ARG;
    Enter g(loop->ctx);
    std::vector<std::pair<double, int>> cand;
    int total = 0;
    // a short list is selected on the device (k x 12 bytes come back instead of one distance per entry)
    SB_TRY(loop_candidates(loop, cand, capacity > 0 && capacity <= SB_LOOP_SELECT_MAX ? capacity : 0, &total));
    *count = (int32_t)total;
    for (int i = 0; i < capacity && i < (int)cand.size(); ++i) {
        dist[i] = cand[i].first;
        entry[i] = cand[i].second;
    }
    return SB_OK;
}

int sb_loop_verify_entries(sb_loop* loop, const int32_t* entry, const double* dist, int32_t n, sb_loop_result* results,
                           int32_t* converged) {
    if (!loop || n < 0 || (n > 0 && (!entry || !results || !converged))) return SB_ERR_INVALID_ARG;
    Enter g(loop->ctx);
    const std::vector<int> qslots((size_t)n, (int)loop->entry_id.size() - 1);   // the newest entry is the query
    return loop_verify(loop, qslots.data(), entry, dist, n, results, converged);
}

int sb_loop_detect(sb_loop* loop, sb_loop_result* results, int32_t capacity, int32_t* count) {
    if (!loop || !count || capacity < 0 || (capacity > 0 && !results)) return SB_ERR_INVALID_ARG;
    Ctx* c = loop->ctx;
    Enter g(c);
    *count = 0;
    if (loop->world != 1) return fail(c, SB_ERR_INVALID_ARG, "sb_loop_detect needs world == 1; use candidates_local + verify_entries");
    std::vector<std::pair<double, int>> cand;
    int total = 0;
    // the best SB_LOOP_SELECT_MAX candidates, selected on the device; the full sorted list only if the walk below
    // gets through all of them without max_candidates acceptances (verified counts successes only)
    SB_TRY(loop_candidates(loop, cand, SB_LOOP_SELECT_MAX, &total));
    if (cand.empty()) return SB_OK;  // loop_closure.hpp:91
    int chunk = loop->cfg.verify_chunk > 0 ? loop->cfg.verify_chunk : loop->cfg.max_candidates;
    if (chunk < 1) chunk = 1;
    int verified = 0;  // counts acceptances only (loop_closure.hpp:95-97, 121)
    bool have_all = (int)cand.size() >= total;
    for (size_t b = 0; verified < loop->cfg.max_candidates; b += (size_t)chunk) {
        if (b >= cand.size()) {
            if (have_all) break;
            arena_reset(c);
            SB_TRY(loop_candidates(loop, cand, 0, &total));   // same order, now complete: continue where the short list ended
            have_all = true;
            if (b >= cand.size()) break;
        }
        int m = (int)std::min(cand.size() - b, (size_t)chunk);
        std::vector<int> ent((size_t)m), conv((size_t)m);
        std::vector<double> dist((size_t)m);
        std::vector<sb_loop_result> res((size_t)m);
        for (int i = 0; i < m; ++i) { ent[i] = cand[b + i].second; dist[i] = cand[b + i].first; }
        const std::vector<int> qslots((size_t)m, (int)loop->entry_id.size() - 1);
        arena_reset(c);
        SB_TRY(loop_verify(loop, qslots.data(), ent.data(), dist.data(), m, res.data(), conv.data()));
        for (int i = 0; i < m && verified < loop->cfg.max_candidates; ++i) {
            if (conv[i] && res[i].icp_fitness < loop->cfg.icp_fitness_threshold) {  // loop_closure.hpp:112
                if (*count < capacity) results[*count] = res[i];
                ++*count;
                ++verified;
            }
        }
    }
    return SB_OK;
}

int sb_loop_add_frames(sb_loop* loop, const double* xyz, const int64_t* offsets, int32_t n_frames,
                       const int32_t* frame_idx, const double* desc) {
    if (!loop || n_frames < 0 || (n_frames > 0 && (!offsets || !frame_idx))) return SB_ERR_INVALID_ARG;
    Ctx* c = loop->ctx;
    Enter g(c);
    if (n_frames == 0) return SB_OK;
    if (offsets[0] != 0) return fail(c, SB_ERR_INVALID_ARG, "offsets must start at 0");
    for (int i = 0; i < n_frames; ++i)
        if (offsets[i + 1] < offsets[i]) return fail(c, SB_ERR_INVALID_ARG, "offsets must be non-decreasing");
    if (offsets[n_frames] > 0 && !xyz) return fail(c, SB_ERR_INVALID_ARG, "null buffer");
    return loop_add_many(loop, xyz, reinterpret_cast<const i64*>(offsets), n_frames, frame_idx, desc);
}

// query entry ids of the batch entry points: world == 1 (entry id = slot), strictly ascending, below size()
static int check_queries(sb_loop* loop, const int32_t* q, int32_t n) {
    Ctx* c = loop->ctx;
    if (loop->world != 1) return fail(c, SB_ERR_INVALID_ARG, "batch loop detection needs world == 1");
    for (int i = 0; i < n; ++i) {
        if (q[i] < 0 || q[i] >= loop->n_global)
            return fail(c, SB_ERR_INVALID_ARG, "query entry %d out of range [0, %d)", q[i], loop->n_global);
        if (i > 0 && q[i] <= q[i - 1]) return fail(c, SB_ERR_INVALID_ARG, "query entries must be strictly ascending");
    }
    return SB_OK;
}

int sb_loop_candidates_batch(sb_loop* loop, const int32_t* query_entries, int32_t n_queries, int32_t k, double* dist,
                             int32_t* entry, int32_t* count) {
    if (!loop || n_queries < 0 || k < 1 || k > SB_LOOP_SELECT_MAX ||
        (n_queries > 0 && (!query_entries || !dist || !entry || !count)))
        return SB_ERR_INVALID_ARG;
    Enter g(loop->ctx);
    SB_TRY(check_queries(loop, query_entries, n_queries));
    std::vector<std::vector<std::pair<double, int>>> cand;
    std::vector<int> total;
    SB_TRY(loop_candidates_batch(loop, query_entries, n_queries, cand, total));
    for (int i = 0; i < n_queries; ++i) {
        count[i] = total[i];
        for (int j = 0; j < k && j < (int)cand[i].size(); ++j) {
            dist[(size_t)i * k + j] = cand[i][j].first;
            entry[(size_t)i * k + j] = cand[i][j].second;
        }
    }
    return SB_OK;
}

int sb_loop_detect_batch(sb_loop* loop, const int32_t* query_entries, int32_t n_queries, sb_loop_result* results,
                         int32_t* count) {
    if (!loop || n_queries < 0 || (n_queries > 0 && (!query_entries || !count)) ||
        (n_queries > 0 && loop->cfg.max_candidates > 0 && !results))
        return SB_ERR_INVALID_ARG;
    Enter g(loop->ctx);
    SB_TRY(check_queries(loop, query_entries, n_queries));
    return loop_detect_batch(loop, query_entries, n_queries, results, count);
}

// rules of the cross-detector calls; the message names the offending detector or query index
static int check_across(sb_loop* const* dbs, int32_t n_dbs, const int32_t* qdb, const int32_t* qe, int32_t n_q,
                        std::vector<sb_loop*>& out) {
    Ctx* c = dbs[0]->ctx;
    const sb_loop_config& a = dbs[0]->cfg;
    for (int d = 0; d < n_dbs; ++d) {
        const sb_loop* L = dbs[d];
        if (L->ctx != c) return fail(c, SB_ERR_INVALID_ARG, "detector %d is on another context than detector 0", d);
        for (int o = 0; o < d; ++o)
            if (dbs[o] == L) return fail(c, SB_ERR_INVALID_ARG, "detector %d appears twice (also detector %d)", d, o);
        if (L->world != 1) return fail(c, SB_ERR_INVALID_ARG, "detector %d has world %d; search across detectors needs world == 1", d, L->world);
        const sb_loop_config& b = L->cfg;
        const char* diff = b.sc_distance_threshold != a.sc_distance_threshold ? "sc_distance_threshold"
                         : b.icp_fitness_threshold != a.icp_fitness_threshold ? "icp_fitness_threshold"
                         : b.max_candidates != a.max_candidates ? "max_candidates"
                         : b.icp_max_iterations != a.icp_max_iterations ? "icp_max_iterations"
                         : b.normals_k != a.normals_k ? "normals_k"
                         : b.icp_tolerance != a.icp_tolerance ? "icp_tolerance"
                         : b.verify_chunk != a.verify_chunk ? "verify_chunk" : nullptr;
        if (diff) return fail(c, SB_ERR_INVALID_ARG, "detector %d: %s differs from detector 0's", d, diff);
    }
    for (int i = 0; i < n_q; ++i) {
        if (qdb[i] < 0 || qdb[i] >= n_dbs)
            return fail(c, SB_ERR_INVALID_ARG, "query %d: detector %d out of range [0, %d)", i, qdb[i], n_dbs);
        const int n = dbs[qdb[i]]->n_global;
        if (qe[i] < 0 || qe[i] >= n)
            return fail(c, SB_ERR_INVALID_ARG, "query %d: entry %d out of range [0, %d) of detector %d", i, qe[i], n, qdb[i]);
    }
    out.assign(dbs, dbs + n_dbs);
    return SB_OK;
}

static bool null_db(sb_loop* const* dbs, int32_t n_dbs) {
    if (!dbs) return true;
    for (int d = 0; d < n_dbs; ++d)
        if (!dbs[d]) return true;
    return false;
}

int sb_loop_candidates_across(sb_loop* const* dbs, int32_t n_dbs, const int32_t* query_db, const int32_t* query_entry,
                              int32_t n_queries, int32_t k, double* dist, int32_t* db, int32_t* entry, int32_t* count) {
    if (n_dbs < 0 || n_queries < 0 || k < 1 || k > SB_LOOP_SELECT_MAX) return SB_ERR_INVALID_ARG;
    if (n_queries == 0) return SB_OK;
    if (n_dbs == 0 || null_db(dbs, n_dbs) || !query_db || !query_entry || !dist || !db || !entry || !count)
        return SB_ERR_INVALID_ARG;
    Enter g(dbs[0]->ctx);
    std::vector<sb_loop*> L;
    SB_TRY(check_across(dbs, n_dbs, query_db, query_entry, n_queries, L));
    std::vector<std::vector<std::pair<double, int>>> cand;
    std::vector<int> total;
    SB_TRY(loop_candidates_across(L, query_db, query_entry, n_queries, cand, total));
    std::vector<ScDbRow> tab;
    loop_across_table(L, tab);
    for (int i = 0; i < n_queries; ++i) {
        count[i] = total[i];
        for (int j = 0; j < k && j < (int)cand[i].size(); ++j) {
            const size_t o = (size_t)i * k + j;
            dist[o] = cand[i][j].first;
            loop_across_decode(tab, cand[i][j].second, &db[o], &entry[o]);
        }
    }
    return SB_OK;
}

int sb_loop_detect_across(sb_loop* const* dbs, int32_t n_dbs, const int32_t* query_db, const int32_t* query_entry,
                          int32_t n_queries, sb_loop_result* results, int32_t* match_db, int32_t* count) {
    if (n_dbs < 0 || n_queries < 0) return SB_ERR_INVALID_ARG;
    if (n_queries == 0) return SB_OK;
    if (n_dbs == 0 || null_db(dbs, n_dbs) || !query_db || !query_entry || !count) return SB_ERR_INVALID_ARG;
    if (dbs[0]->cfg.max_candidates > 0 && (!results || !match_db)) return SB_ERR_INVALID_ARG;
    Enter g(dbs[0]->ctx);
    std::vector<sb_loop*> L;
    SB_TRY(check_across(dbs, n_dbs, query_db, query_entry, n_queries, L));
    return loop_detect_across(L, query_db, query_entry, n_queries, results, match_db, count);
}

// ---------------------------------------------------------------- after the path: world frame, map
void sb_default_grid_config(sb_grid_config* cfg) {  // slam_node.hpp:35-40
    cfg->resolution = 0.2;
    cfg->height_min = 0.3;
    cfg->height_max = 2.0;
    cfg->max_range = 40.0;
}

static int check_clouds(Ctx* c, const double* xyz, const int64_t* offsets, int32_t n_clouds, const double* poses16) {
    if (offsets[0] != 0) return fail(c, SB_ERR_INVALID_ARG, "offsets must start at 0");
    for (int i = 0; i < n_clouds; ++i)
        if (offsets[i + 1] < offsets[i]) return fail(c, SB_ERR_INVALID_ARG, "offsets must be non-decreasing");
    if (offsets[n_clouds] > 0 && (!xyz || !poses16)) return fail(c, SB_ERR_INVALID_ARG, "null buffer");
    return SB_OK;
}

// uploads clouds, offsets and poses and transforms the clouds into the world frame
static int world_clouds(Ctx* c, const double* xyz, const int64_t* offsets, int32_t n_clouds, const double* poses16,
                        double** d_world, i64** d_off, double** d_poses) {
    const i64 n = offsets[n_clouds];
    double* d_in;
    SB_TRY(upload(c, xyz, sizeof(double) * 3 * n, (void**)&d_in));
    SB_TRY(upload(c, offsets, sizeof(i64) * (n_clouds + 1), (void**)d_off));
    SB_TRY(upload(c, poses16, sizeof(double) * 16 * (size_t)(n_clouds > 0 ? n_clouds : 0), (void**)d_poses));
    SB_TRY(arena_get(c, (size_t)3 * (n > 0 ? n : 1), d_world));
    return transform_clouds_dev(c, d_in, *d_off, n_clouds, *d_poses, n, *d_world);
}

int sb_transform_clouds(sb_ctx* ctx, const double* xyz, const int64_t* offsets, int32_t n_clouds, const double* poses16,
                        double* out_xyz) {
    if (!ctx || !offsets || n_clouds < 0) return SB_ERR_INVALID_ARG;
    Ctx* c = &ctx->c;
    Enter g(c);
    SB_TRY(check_clouds(c, xyz, offsets, n_clouds, poses16));
    const i64 n = offsets[n_clouds];
    if (n == 0) return SB_OK;
    if (!out_xyz) return fail(c, SB_ERR_INVALID_ARG, "null output buffer");
    double *d_world, *d_poses;
    i64* d_off;
    SB_TRY(world_clouds(c, xyz, offsets, n_clouds, poses16, &d_world, &d_off, &d_poses));
    SB_TRY(download(c, out_xyz, d_world, sizeof(double) * 3 * n));
    SB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SB_OK;
}

// publish_current_scan (slam_node.cpp:147, 231-233, 299-322): the world-frame cloud as the float32 records of a
// PointCloud2 message — converted on the device, so half the bytes come back
int sb_transform_clouds_f32(sb_ctx* ctx, const double* xyz, const int64_t* offsets, int32_t n_clouds,
                            const double* poses16, float* out_xyz) {
    if (!ctx || !offsets || n_clouds < 0) return SB_ERR_INVALID_ARG;
    Ctx* c = &ctx->c;
    Enter g(c);
    SB_TRY(check_clouds(c, xyz, offsets, n_clouds, poses16));
    const i64 n = offsets[n_clouds];
    if (n == 0) return SB_OK;
    if (!out_xyz) return fail(c, SB_ERR_INVALID_ARG, "null output buffer");
    double *d_world, *d_poses;
    i64* d_off;
    float* d_f32;
    SB_TRY(world_clouds(c, xyz, offsets, n_clouds, poses16, &d_world, &d_off, &d_poses));
    SB_TRY(arena_get(c, (size_t)3 * n, &d_f32));
    SB_TRY(pack_f32_dev(c, d_world, n, d_f32));
    SB_TRY(download(c, out_xyz, d_f32, sizeof(float) * 3 * n));
    SB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SB_OK;
}

int sb_occupancy_cells(sb_ctx* ctx, const double* xyz, const int64_t* offsets, int32_t n_clouds, const double* poses16,
                       const sb_grid_config* cfg, int32_t* out_cells, int64_t capacity, int64_t* out_count) {
    if (!ctx || !offsets || n_clouds < 0 || !cfg || !out_count || capacity < 0 || (capacity > 0 && !out_cells))
        return SB_ERR_INVALID_ARG;
    Ctx* c = &ctx->c;
    Enter g(c);
    *out_count = 0;
    SB_TRY(check_clouds(c, xyz, offsets, n_clouds, poses16));
    if (!(cfg->resolution > 0)) return fail(c, SB_ERR_INVALID_ARG, "grid resolution must be positive");
    const i64 n = offsets[n_clouds];
    if (n == 0) return SB_OK;
    double *d_world, *d_poses;
    i64* d_off;
    int* d_cells;
    SB_TRY(world_clouds(c, xyz, offsets, n_clouds, poses16, &d_world, &d_off, &d_poses));
    SB_TRY(arena_get(c, (size_t)2 * (capacity > 0 ? capacity : 1), &d_cells));
    i64 count = 0;
    SB_TRY(occupancy_cells_dev(c, d_world, d_off, n_clouds, d_poses, n, cfg, d_cells, capacity, &count));
    *out_count = count;
    const i64 m = count < capacity ? count : capacity;
    SB_TRY(download(c, out_cells, d_cells, sizeof(int) * 2 * (size_t)m));
    SB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SB_OK;
}

// slam_node.cpp:139-145: delta = identity unless the registration converged with final_error <= max_error;
// new_pose = poses_.back() * delta (Transformation::operator*, types.hpp:118-125: plain 4x4 product, k ascending)
int sb_odometry_poses(sb_ctx*, const sb_icp_result* results, int32_t n, double max_error, const double* initial_pose16,
                      double* poses16_out) {
    if (n < 0 || !poses16_out || (n > 0 && !results)) return SB_ERR_INVALID_ARG;
    static const double I16[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
    memcpy(poses16_out, initial_pose16 ? initial_pose16 : I16, sizeof(I16));
    for (int32_t f = 0; f < n; ++f) {
        const sb_icp_result& R = results[f];
        const bool keep = R.status == SB_OK && R.converged && !(R.final_error > max_error);
        const double* D = keep ? R.transformation : I16;
        const double* P = poses16_out + 16 * (size_t)f;
        double* O = poses16_out + 16 * ((size_t)f + 1);
        for (int i = 0; i < 4; ++i)
            for (int j = 0; j < 4; ++j) {
                double acc = 0.0;
                for (int k = 0; k < 4; ++k) acc += P[4 * i + k] * D[4 * k + j];
                O[4 * i + j] = acc;
            }
    }
    return SB_OK;
}

// slam_node.cpp:139-145 for a batch: delta selection + the arguments of PoseGraph::addOdometryFactor
int sb_odometry_factors(sb_ctx*, const sb_icp_result* results, int32_t n, int32_t first_frame, double max_error,
                        sb_pose_factor* out) {
    if (n < 0 || (n > 0 && (!results || !out))) return SB_ERR_INVALID_ARG;
    static const double I16[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
    for (int32_t i = 0; i < n; ++i) {
        const sb_icp_result& R = results[i];
        const bool keep = R.status == SB_OK && R.converged && !(R.final_error > max_error);
        sb_pose_factor& f = out[i];
        f.kind = SB_FACTOR_ODOMETRY;
        f.from = first_frame + i;
        f.to = first_frame + i + 1;
        f.pad = 0;
        memcpy(f.relative, keep ? R.transformation : I16, sizeof(I16));
        f.fitness = R.final_error;
        f.noise_scale = 1.0 + R.final_error * 10.0;  // pose_graph.cpp:88
    }
    return SB_OK;
}

// slam_node.cpp:163-167: addLoopClosure(lc.match_frame, lc.query_frame, lc.transform)
int sb_loop_factors(sb_ctx*, const sb_loop_result* results, int32_t n, sb_pose_factor* out) {
    if (n < 0 || (n > 0 && (!results || !out))) return SB_ERR_INVALID_ARG;
    for (int32_t i = 0; i < n; ++i) {
        sb_pose_factor& f = out[i];
        f.kind = SB_FACTOR_LOOP;
        f.from = results[i].match_frame;
        f.to = results[i].query_frame;
        f.pad = 0;
        memcpy(f.relative, results[i].transform, sizeof(f.relative));
        f.fitness = results[i].icp_fitness;
        f.noise_scale = 1.0;
    }
    return SB_OK;
}

int sb_global_map(sb_ctx* ctx, const double* xyz, const int64_t* offsets, int32_t n_clouds, const double* poses16,
                  double voxel, double* out_xyz, int64_t* out_m) {
    if (!ctx || !offsets || n_clouds < 0 || !out_m) return SB_ERR_INVALID_ARG;
    Ctx* c = &ctx->c;
    Enter g(c);
    *out_m = 0;
    SB_TRY(check_clouds(c, xyz, offsets, n_clouds, poses16));
    const i64 n = offsets[n_clouds];
    if (n == 0) return SB_OK;
    if (!out_xyz) return fail(c, SB_ERR_INVALID_ARG, "null output buffer");
    double *d_world, *d_poses, *d_out;
    i64* d_off;
    SB_TRY(world_clouds(c, xyz, offsets, n_clouds, poses16, &d_world, &d_off, &d_poses));
    SB_TRY(arena_get(c, (size_t)3 * n, &d_out));
    i64 one[2] = {0, n}, out_off[2] = {0, 0};
    SB_TRY(voxel_downsample_dev(c, d_world, one, 1, voxel, d_out, out_off, nullptr));
    *out_m = out_off[1];
    SB_TRY(download(c, out_xyz, d_out, sizeof(double) * 3 * (size_t)out_off[1]));
    SB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SB_OK;
}

// publish_global_map (slam_node.cpp:235-238, 299-322): the downsampled global map as PointCloud2 float32 records
int sb_global_map_f32(sb_ctx* ctx, const double* xyz, const int64_t* offsets, int32_t n_clouds, const double* poses16,
                      double voxel, float* out_xyz, int64_t* out_m) {
    if (!ctx || !offsets || n_clouds < 0 || !out_m) return SB_ERR_INVALID_ARG;
    Ctx* c = &ctx->c;
    Enter g(c);
    *out_m = 0;
    SB_TRY(check_clouds(c, xyz, offsets, n_clouds, poses16));
    const i64 n = offsets[n_clouds];
    if (n == 0) return SB_OK;
    if (!out_xyz) return fail(c, SB_ERR_INVALID_ARG, "null output buffer");
    double *d_world, *d_poses, *d_out;
    i64* d_off;
    float* d_f32;
    SB_TRY(world_clouds(c, xyz, offsets, n_clouds, poses16, &d_world, &d_off, &d_poses));
    SB_TRY(arena_get(c, (size_t)3 * n, &d_out));
    SB_TRY(arena_get(c, (size_t)3 * n, &d_f32));
    i64 one[2] = {0, n}, out_off[2] = {0, 0};
    SB_TRY(voxel_downsample_dev(c, d_world, one, 1, voxel, d_out, out_off, nullptr));
    *out_m = out_off[1];
    SB_TRY(pack_f32_dev(c, d_out, out_off[1], d_f32));
    SB_TRY(download(c, out_xyz, d_f32, sizeof(float) * 3 * (size_t)out_off[1]));
    SB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SB_OK;
}

// ---------------------------------------------------------------- synthetic input generator
int sb_synth_scans_dev(sb_ctx* ctx, int32_t beams, int32_t azimuth_steps, float elev_top_deg, float elev_bot_deg,
                       float max_range, float noise_sigma, float sensor_height, const float* boxes, int32_t n_boxes,
                       const double* poses, int32_t n_scans, uint64_t noise_seed, double* d_xyz, int64_t* out_offsets) {
    if (!ctx || !poses || !out_offsets || n_scans < 0 || n_boxes < 0 || (n_boxes > 0 && !boxes)) return SB_ERR_INVALID_ARG;
    Ctx* c = &ctx->c;
    Enter g(c);
    return synth_scans_dev(c, beams, azimuth_steps, elev_top_deg, elev_bot_deg, max_range, noise_sigma, sensor_height,
                           boxes, n_boxes, poses, n_scans, noise_seed, d_xyz, (i64*)out_offsets);
}

}  // extern "C"
