// loop.cu — device-resident loop-closure database; replaces slam::LoopClosureDetector
// (slam_viz/include/slam_viz/core/loop_closure.hpp:41-149).
//
// The reference keeps a vector of Eigen descriptors plus a full copy of every cloud on the host and scans it
// linearly (loop_closure.hpp:78-89), then verifies candidates one by one with ICP (:95-122).  Here descriptors
// and clouds live in two growing device pools; the Scan Context search is one kernel over the whole database and
// the ICP verifications of a chunk of candidates run as ONE batch (they are independent); acceptance then walks the
// candidates in the reference's (distance, entry) order so the accepted set is the same as the sequential loop's.
// With world > 1, entry i is owned by rank i % world; every rank also keeps the newest entry (the query).
#include "common.cuh"

#include <algorithm>
#include <functional>
#include <map>

namespace sb {

// Pools only ever grow, by doubling, and the outgrown buffer is retired (freed with the detector) rather than
// released: cudaMalloc / cudaFree stall the calling thread for up to hundreds of milliseconds (measured on the B200
// pool: 100 ms / 580 ms worst case) while a frame takes 1.7 ms, so the streaming path must not reach them in steady
// state.  The first allocation holds ~1300 voxel-downsampled scans / 4096 descriptors; sb_loop_reserve sizes the
// pools for a known sequence length up front.
static const size_t FIRST_CLOUD_ROWS = (size_t)11 << 20;   // 264 MB of fp64 xyz rows
static const size_t FIRST_DESC_SLOTS = 4096;               // 39 MB

static int grow(sb_loop* L, double** buf, size_t* cap, size_t need, size_t used, size_t unit, size_t first) {
    if (need <= *cap) return SB_OK;
    Ctx* ctx = L->ctx;
    size_t ncap = *cap ? *cap : first;
    while (ncap < need) ncap *= 2;
    double* nb;
    SB_CUDA(ctx, cudaMalloc(&nb, ncap * unit * sizeof(double)));
    if (used) SB_CUDA(ctx, cudaMemcpyAsync(nb, *buf, used * unit * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    if (*buf) L->retired.push_back(*buf);
    *buf = nb;
    *cap = ncap;
    return SB_OK;
}

int loop_reserve(sb_loop* L, i64 n_entries, i64 total_rows) {
    size_t slots = L->entry_id.size();
    i64 rows = L->cloud_off.empty() ? 0 : L->cloud_off.back();
    if (n_entries > 0) SB_TRY(grow(L, &L->d_desc, &L->desc_cap, (size_t)n_entries, slots, SB_SC_SIZE, (size_t)n_entries));
    if (n_entries > 0) SB_TRY(grow(L, &L->d_meta, &L->meta_cap, (size_t)n_entries, slots, 1, (size_t)n_entries));
    if (total_rows > 0) SB_TRY(grow(L, &L->d_clouds, &L->cloud_cap, (size_t)total_rows, (size_t)rows, 3, (size_t)total_rows));
    SB_CUDA(L->ctx, cudaStreamSynchronize(L->ctx->stream));
    return SB_OK;
}

int loop_add(sb_loop* L, const double* xyz, i64 n, int frame_idx, const double* desc) {
    Ctx* ctx = L->ctx;
    // drop a guest (non-owned former query) before appending
    if (L->last_is_guest) {
        L->entry_id.pop_back();
        L->frame_idx.pop_back();
        L->cloud_off.pop_back();
        L->last_is_guest = false;
    }
    int id = L->n_global++;
    size_t slots = L->entry_id.size();
    i64 rows = L->cloud_off.empty() ? 0 : L->cloud_off.back();
    if (L->cloud_off.empty()) L->cloud_off.push_back(0);
    SB_TRY(grow(L, &L->d_desc, &L->desc_cap, slots + 1, slots, SB_SC_SIZE, FIRST_DESC_SLOTS));
    SB_TRY(grow(L, &L->d_meta, &L->meta_cap, slots + 1, slots, 1, FIRST_DESC_SLOTS));
    {
        const int meta[2] = {frame_idx, id};
        SB_CUDA(ctx, cudaMemcpyAsync(L->d_meta + slots, meta, sizeof(meta), cudaMemcpyHostToDevice, ctx->stream));
    }
    SB_TRY(grow(L, &L->d_clouds, &L->cloud_cap, (size_t)(rows + n), (size_t)rows, 3, FIRST_CLOUD_ROWS));
    if (n > 0)
        SB_CUDA(ctx, cudaMemcpyAsync(L->d_clouds + 3 * rows, xyz, sizeof(double) * 3 * n, cudaMemcpyHostToDevice, ctx->stream));
    double* d_slot = L->d_desc + slots * SB_SC_SIZE;
    if (desc) {
        SB_CUDA(ctx, cudaMemcpyAsync(d_slot, desc, sizeof(double) * SB_SC_SIZE, cudaMemcpyHostToDevice, ctx->stream));
    } else {  // ScanContext sc(points), loop_closure.hpp:55
        i64* d_off;
        SB_TRY(arena_get(ctx, 2, &d_off));
        i64 h[2] = {rows, rows + n};
        SB_CUDA(ctx, cudaMemcpyAsync(d_off, h, sizeof(h), cudaMemcpyHostToDevice, ctx->stream));
        SB_TRY(sc_compute_dev(ctx, L->d_clouds, d_off, 1, d_slot));
    }
    SB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    L->entry_id.push_back(id);
    L->frame_idx.push_back(frame_idx);
    L->cloud_off.push_back(rows + n);
    L->last_frame = frame_idx;
    L->last_is_guest = (id % L->world) != L->rank;
    return SB_OK;
}

// The streaming session's addFrame (odom.cu): the same pool layout as loop_add, with the cloud and the descriptor copied
// device to device and no synchronise.  The host-side vectors change only in loop_add_commit.
int loop_add_enqueue(sb_loop* L, const double* d_xyz, i64 n, int frame_idx, const double* d_desc, LoopAddPending* out) {
    Ctx* ctx = L->ctx;
    // the slot loop_add would use: a guest (non-owned former query) gives way
    const size_t held = L->entry_id.size();
    const size_t slots = held - (L->last_is_guest ? 1 : 0);
    const i64 rows = L->cloud_off.empty() ? 0 : L->cloud_off[slots];
    const int id = L->n_global;
    SB_TRY(grow(L, &L->d_desc, &L->desc_cap, slots + 1, held, SB_SC_SIZE, FIRST_DESC_SLOTS));
    SB_TRY(grow(L, &L->d_meta, &L->meta_cap, slots + 1, held, 1, FIRST_DESC_SLOTS));
    const i64 held_rows = L->cloud_off.empty() ? 0 : L->cloud_off.back();
    SB_TRY(grow(L, &L->d_clouds, &L->cloud_cap, (size_t)(rows + n), (size_t)held_rows, 3, FIRST_CLOUD_ROWS));
    const int meta[2] = {frame_idx, id};
    SB_TRY(table_upload(ctx, L->d_meta + slots, meta, sizeof(meta)));
    if (n > 0)
        SB_CUDA(ctx, cudaMemcpyAsync(L->d_clouds + 3 * rows, d_xyz, sizeof(double) * 3 * n, cudaMemcpyDeviceToDevice,
                                     ctx->stream));
    SB_CUDA(ctx, cudaMemcpyAsync(L->d_desc + slots * SB_SC_SIZE, d_desc, sizeof(double) * SB_SC_SIZE,
                                 cudaMemcpyDeviceToDevice, ctx->stream));
    out->id = id;
    out->frame_idx = frame_idx;
    out->end_row = rows + n;
    return SB_OK;
}

void loop_add_commit(sb_loop* L, const LoopAddPending& p) {
    if (L->last_is_guest) {
        L->entry_id.pop_back();
        L->frame_idx.pop_back();
        L->cloud_off.pop_back();
        L->last_is_guest = false;
    }
    if (L->cloud_off.empty()) L->cloud_off.push_back(0);
    L->n_global = p.id + 1;
    L->entry_id.push_back(p.id);
    L->frame_idx.push_back(p.frame_idx);
    L->cloud_off.push_back(p.end_row);
    L->last_frame = p.frame_idx;
    L->last_is_guest = (p.id % L->world) != L->rank;
}

// -------------------------------------------------------------------------------------------------------------
// Candidate selection on the device (loop_closure.hpp:78-92: frame-gap filter, threshold, sort by (distance, entry)):
// one block.  Every warp keeps the KSEL best (distance, entry) pairs of its share of the database in registers, entry
// j in lane j, ascending; warp 0 then merges the 32 lists.  The host receives KSEL x 12 bytes and the number of
// entries under the threshold instead of one distance per database entry.
// -------------------------------------------------------------------------------------------------------------
static constexpr int KSEL = SB_LOOP_SELECT_MAX;

struct SelList {   // lane j of a warp holds the j-th best pair
    unsigned long long d;   // order-preserving image of the distance; ~0: empty
    int e;
    __device__ __forceinline__ bool less_than(unsigned long long od, int oe) const { return d < od || (d == od && e < oe); }
    // inserts the candidates of the lanes in `m` (warp-uniform mask), each lane's own (cd, ce)
    __device__ __forceinline__ void insert(unsigned m, unsigned long long cd, int ce, int lane) {
        while (m) {
            const int b = __ffs(m) - 1;
            m &= m - 1u;
            const unsigned long long bd = __shfl_sync(0xffffffffu, cd, b);
            const int be = __shfl_sync(0xffffffffu, ce, b);
            const int pos = __popc(__ballot_sync(0xffffffffu, less_than(bd, be)));   // sorted: a prefix
            if (pos >= 32) continue;
            const unsigned long long ud = __shfl_up_sync(0xffffffffu, d, 1);
            const int ue = __shfl_up_sync(0xffffffffu, e, 1);
            if (lane > pos) { d = ud; e = ue; }
            else if (lane == pos) { d = bd; e = be; }
        }
    }
};

// Which entries of a row a query may match: keep(i, id) says whether entry i passes and sets the id it is ordered and
// reported by.  detect() of one detector: the frame gap (loop_closure.hpp:79-81), id = entry.
struct GapFilter {
    const int2* __restrict__ meta;
    int query_frame, frame_gap;
    __device__ __forceinline__ bool operator()(int i, int& id) const {
        const int2 mt = meta[i];
        id = mt.y;
        return query_frame - mt.x >= frame_gap;
    }
};

// One row: the entries [0, n_db) that pass `keep`.  Shared by the single-query launch, the one-CTA-per-query batch
// launch (k_loop_select_many) and the cross-detector launch (k_loop_select_across), so all select with the same code.
template <class Keep>
__device__ __forceinline__ void loop_select_row(const double* __restrict__ dist, int n_db, const Keep& keep,
                                                double threshold, unsigned long long* __restrict__ out_d,
                                                int* __restrict__ out_e, int* __restrict__ out_total) {
    __shared__ unsigned long long s_d[32][KSEL];
    __shared__ int s_e[32][KSEL];
    __shared__ int s_total;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_total = 0;
    __syncthreads();
    SelList L;
    L.d = ~0ull; L.e = 0x7fffffff;
    int mine = 0;
    for (int base = warp * 32; base < n_db; base += 1024) {
        const int i = base + lane;
        unsigned long long cd = ~0ull;
        int ce = 0x7fffffff;
        bool ok = false;
        if (i < n_db) {
            int id;
            const double dv = dist[i];
            ok = keep(i, id) && (dv < threshold);   // loop_closure.hpp:79-81, 86-88 (NaN: false)
            if (ok) {   // order-preserving image of the double (a cosine distance can round to -1e-16)
                const unsigned long long b = (unsigned long long)__double_as_longlong(dv);
                cd = (b >> 63) ? ~b : (b | 0x8000000000000000ull);
                if (cd == ~0ull) cd = ~0ull - 1ull;
                ce = id;
                ++mine;
            }
        }
        // only candidates better than the list's last entry can enter it
        const unsigned long long ld = __shfl_sync(0xffffffffu, L.d, 31);
        const int le = __shfl_sync(0xffffffffu, L.e, 31);
        const unsigned m = __ballot_sync(0xffffffffu, ok && (cd < ld || (cd == ld && ce < le)));
        L.insert(m, cd, ce, lane);
    }
    mine = __reduce_add_sync(0xffffffffu, mine);
    if (lane == 0 && mine) atomicAdd(&s_total, mine);
    s_d[warp][lane] = L.d;
    s_e[warp][lane] = L.e;
    __syncthreads();
    if (warp != 0) return;
    SelList M;
    M.d = ~0ull; M.e = 0x7fffffff;
    for (int w = 0; w < 32; ++w) {
        const unsigned long long cd = s_d[w][lane];
        const int ce = s_e[w][lane];
        const unsigned long long ld = __shfl_sync(0xffffffffu, M.d, 31);
        const int le = __shfl_sync(0xffffffffu, M.e, 31);
        const unsigned m = __ballot_sync(0xffffffffu, cd != ~0ull && (cd < ld || (cd == ld && ce < le)));
        M.insert(m, cd, ce, lane);
    }
    out_d[lane] = M.d;
    out_e[lane] = M.e;
    if (lane == 0) *out_total = s_total;
}

__global__ void __launch_bounds__(1024) k_loop_select(const double* __restrict__ dist, const int2* __restrict__ meta,
                                                      int n_db, int last_frame, int frame_gap, double threshold,
                                                      unsigned long long* __restrict__ out_d, int* __restrict__ out_e,
                                                      int* __restrict__ out_total) {
    loop_select_row(dist, n_db, GapFilter{meta, last_frame, frame_gap}, threshold, out_d, out_e, out_total);
}

// row r: query slot qslot[r] against the entries below it, distances at dist + r * ld (k_sc_distance_many)
__global__ void __launch_bounds__(1024) k_loop_select_many(const double* __restrict__ dist, i64 ld,
                                                           const int2* __restrict__ meta, const int* __restrict__ qslot,
                                                           int frame_gap, double threshold,
                                                           unsigned long long* __restrict__ out_d,
                                                           int* __restrict__ out_e, int* __restrict__ out_total) {
    const int r = blockIdx.x, q = qslot[r];
    loop_select_row(dist + (i64)r * ld, q, GapFilter{meta, meta[q].x, frame_gap}, threshold, out_d + (i64)r * KSEL,
                    out_e + (i64)r * KSEL, out_total + r);
}

// Across detectors: column i passes iff it is an entry (not padding) of a detector other than the query's.  The id is
// the column, so (distance, id) order is (distance, detector, entry).
struct OtherDbFilter {
    const int* __restrict__ col_db;
    int query_db;
    __device__ __forceinline__ bool operator()(int i, int& id) const {
        const int d = col_db[i];
        id = i;
        return d >= 0 && d != query_db;
    }
};

// row r: query r of the group (detector qdb[r]) against every column, distances at dist + r * ld (k_sc_distance_across)
__global__ void __launch_bounds__(1024) k_loop_select_across(const double* __restrict__ dist, i64 ld,
                                                             const int* __restrict__ col_db, const int* __restrict__ qdb,
                                                             double threshold, unsigned long long* __restrict__ out_d,
                                                             int* __restrict__ out_e, int* __restrict__ out_total) {
    const int r = blockIdx.x;
    loop_select_row(dist + (i64)r * ld, (int)ld, OtherDbFilter{col_db, qdb[r]}, threshold, out_d + (i64)r * KSEL,
                    out_e + (i64)r * KSEL, out_total + r);
}

static void decode_selection(const unsigned long long* h_d, const int* h_e, int limit,
                             std::vector<std::pair<double, int>>& cand) {
    for (int i = 0; i < KSEL && i < limit && h_d[i] != ~0ull; ++i) {
        const unsigned long long b = (h_d[i] >> 63) ? (h_d[i] & 0x7fffffffffffffffull) : ~h_d[i];
        double d;
        memcpy(&d, &b, sizeof(d));
        cand.push_back({d, h_e[i]});
    }
}

// loop_closure.hpp:75-92 restricted to the entries this rank owns; qslot < 0: the newest entry is the query
int loop_candidates(sb_loop* L, std::vector<std::pair<double, int>>& cand, int limit, int* total, int qslot) {
    Ctx* ctx = L->ctx;
    cand.clear();
    if (total) *total = 0;
    if (L->n_global < 2) return SB_OK;  // loop_closure.hpp:69
    int slots = (int)L->entry_id.size();
    if (qslot < 0) qslot = slots - 1;  // the newest entry (the query) is always the last slot
    const int n_db = qslot;            // the query sees the entries before it
    const int qframe = L->frame_idx[qslot];
    if (n_db <= 0) return SB_OK;
    double* d_out;
    SB_TRY(arena_get(ctx, (size_t)n_db, &d_out));
    SB_TRY(sc_distance_dev(ctx, L->d_desc + (size_t)qslot * SB_SC_SIZE, L->d_desc, n_db, d_out));
    if (limit > 0 && limit <= KSEL) {
        unsigned long long* d_sel_d;
        int* d_sel_e;
        SB_TRY(arena_get(ctx, (size_t)KSEL, &d_sel_d));
        SB_TRY(arena_get(ctx, (size_t)KSEL + 1, &d_sel_e));
        SB_LAUNCH(ctx, k_loop_select, 1, 1024, 0, d_out, reinterpret_cast<const int2*>(L->d_meta), n_db, qframe,
                  L->cfg.frame_gap, L->cfg.sc_distance_threshold, d_sel_d, d_sel_e, d_sel_e + KSEL);
        SB_TRY(pinned_reserve(ctx, KSEL * 12 + 16));
        unsigned long long* h_d = reinterpret_cast<unsigned long long*>(ctx->pinned);
        int* h_e = reinterpret_cast<int*>(ctx->pinned + KSEL * 8);
        SB_CUDA(ctx, cudaMemcpyAsync(h_d, d_sel_d, KSEL * 8, cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(ctx, cudaMemcpyAsync(h_e, d_sel_e, (KSEL + 1) * 4, cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (total) *total = h_e[KSEL];
        decode_selection(h_d, h_e, limit, cand);
        return SB_OK;
    }
    std::vector<double> dist((size_t)n_db);
    SB_CUDA(ctx, cudaMemcpyAsync(dist.data(), d_out, sizeof(double) * n_db, cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < n_db; ++i) {
        if (qframe - L->frame_idx[i] < L->cfg.frame_gap) continue;                    // loop_closure.hpp:79-81
        if (dist[i] < L->cfg.sc_distance_threshold) cand.push_back({dist[i], L->entry_id[i]});  // :86-88
    }
    std::sort(cand.begin(), cand.end());  // loop_closure.hpp:92: (distance, entry) ascending
    if (total) *total = (int)cand.size();
    return SB_OK;
}

// The Q x D distance matrix of one group of queries stays under this many bytes; groups run one after the other.
static constexpr size_t LOOP_DIST_BYTES = (size_t)32 << 20;

// loop_candidates for many query slots (world == 1, ascending): the best KSEL per query, selected on the device, and
// the number under the threshold.  One squared-sum pre-pass, then per group of queries one search and one selection
// launch; the selections of all groups come back in one copy.
int loop_candidates_batch(sb_loop* L, const int* qslots, int n_q, std::vector<std::vector<std::pair<double, int>>>& cand,
                          std::vector<int>& total) {
    Ctx* ctx = L->ctx;
    cand.assign((size_t)n_q, {});
    total.assign((size_t)n_q, 0);
    if (n_q <= 0) return SB_OK;
    const int ld = qslots[n_q - 1];   // the widest row: entries below the last query
    if (ld <= 0) return SB_OK;        // only query 0: nothing before it
    const i64 rows = std::max<i64>(8, (i64)(LOOP_DIST_BYTES / (sizeof(double) * (size_t)ld)) / 8 * 8);
    const int2* d_meta = reinterpret_cast<const int2*>(L->d_meta);
    double *d_sq, *d_dist;
    int* d_q;
    char* d_sel;
    const size_t sel_bytes = (size_t)n_q * (KSEL * 12 + 4);
    SB_TRY(arena_get(ctx, (size_t)(ld + 1) * SB_SC_SECTORS, &d_sq));
    SB_TRY(arena_get(ctx, (size_t)std::min<i64>(rows, n_q) * ld, &d_dist));
    SB_TRY(arena_get(ctx, (size_t)n_q, &d_q));
    SB_TRY(arena_get(ctx, sel_bytes, &d_sel));
    unsigned long long* d_sel_d = reinterpret_cast<unsigned long long*>(d_sel);
    int* d_sel_e = reinterpret_cast<int*>(d_sel + (size_t)n_q * KSEL * 8);
    int* d_tot = d_sel_e + (size_t)n_q * KSEL;
    SB_CUDA(ctx, cudaMemcpyAsync(d_q, qslots, sizeof(int) * n_q, cudaMemcpyHostToDevice, ctx->stream));
    SB_TRY(sc_sq_dev(ctx, L->d_desc, ld + 1, d_sq));
    for (i64 g0 = 0; g0 < n_q; g0 += rows) {
        const int ng = (int)std::min<i64>(rows, n_q - g0);
        SB_TRY(sc_distance_many_dev(ctx, L->d_desc, d_sq, d_meta, d_q + g0, ng, qslots[g0 + ng - 1], L->cfg.frame_gap,
                                    d_dist, ld));
        SB_LAUNCH(ctx, k_loop_select_many, (unsigned)ng, 1024, 0, d_dist, (i64)ld, d_meta, d_q + g0, L->cfg.frame_gap,
                  L->cfg.sc_distance_threshold, d_sel_d + g0 * KSEL, d_sel_e + g0 * KSEL, d_tot + g0);
    }
    SB_TRY(pinned_reserve(ctx, sel_bytes));
    SB_CUDA(ctx, cudaMemcpyAsync(ctx->pinned, d_sel, sel_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const unsigned long long* h_d = reinterpret_cast<const unsigned long long*>(ctx->pinned);
    const int* h_e = reinterpret_cast<const int*>(ctx->pinned + (size_t)n_q * KSEL * 8);
    for (int r = 0; r < n_q; ++r) {
        total[r] = h_e[(size_t)n_q * KSEL + r];
        decode_selection(h_d + (size_t)r * KSEL, h_e + (size_t)r * KSEL, KSEL, cand[r]);
    }
    return SB_OK;
}

static int slot_of(const sb_loop* L, int entry) {
    // owned entries are stored in ascending id order: entry = rank + slot * world
    int slot = (entry - L->rank) / L->world;
    if (entry % L->world != L->rank || slot < 0 || slot >= (int)L->entry_id.size() || L->entry_id[slot] != entry) return -1;
    return slot;
}

// ICP batches of loop verification: at most this many pairs per icp_batch call
static constexpr int VERIFY_BATCH = 4096;

struct CloudRef {   // a cloud of the loop-closure database: slot `slot` of detector L
    const sb_loop* L;
    int slot;
};

// loop_closure.hpp:99-109 for n (source cloud, target cloud) pairs, each cloud a slot of some detector, with the loop
// ICP settings of cfg.  The forest indexes every distinct target cloud once (with normals) and every distinct source
// cloud once (as a source): one forest_append per detector, targets first, in order of first appearance.
static int verify_pairs(Ctx* ctx, const sb_loop_config& cfg, const CloudRef* src, const CloudRef* tgt, int n,
                        sb_icp_result* res) {
    // distinct clouds grouped by detector: trees[k] = (detector, its slots); index[i] = tree of pair i within its group
    struct Group {
        const sb_loop* L;
        std::vector<int> slots;
    };
    auto group = [](const CloudRef* refs, int n, std::vector<Group>& groups, std::vector<int>& tree_of) {
        std::map<std::pair<const sb_loop*, int>, std::pair<int, int>> seen;   // -> (group, index in group)
        std::map<const sb_loop*, int> group_of;
        std::vector<std::pair<int, int>> at((size_t)n);
        for (int i = 0; i < n; ++i) {
            auto it = seen.find({refs[i].L, refs[i].slot});
            if (it == seen.end()) {
                auto g = group_of.find(refs[i].L);
                if (g == group_of.end()) {
                    g = group_of.emplace(refs[i].L, (int)groups.size()).first;
                    groups.push_back({refs[i].L, {}});
                }
                std::vector<int>& sl = groups[(size_t)g->second].slots;
                it = seen.emplace(std::make_pair(refs[i].L, refs[i].slot), std::make_pair(g->second, (int)sl.size())).first;
                sl.push_back(refs[i].slot);
            }
            at[i] = it->second;
        }
        std::vector<int> first((size_t)groups.size() + 1, 0);
        for (size_t g = 0; g < groups.size(); ++g) first[g + 1] = first[g] + (int)groups[g].slots.size();
        tree_of.resize((size_t)n);
        for (int i = 0; i < n; ++i) tree_of[i] = first[(size_t)at[i].first] + at[i].second;
        return first.back();
    };
    std::vector<Group> tgt_groups, src_groups;
    std::vector<int> tgt_of, src_of;
    const int n_tgt = group(tgt, n, tgt_groups, tgt_of);
    const int n_src = group(src, n, src_groups, src_of);
    Forest F;
    F.in_arena = true;
    int s = forest_reserve(ctx, &F, n_tgt + n_src);
    for (const Group& g : tgt_groups) {   // candidates
        if (s == SB_OK) s = forest_append(ctx, &F, g.L->d_clouds, g.L->cloud_off.data(), g.slots.data(), (int)g.slots.size());
        if (s == SB_OK) s = forest_normals(ctx, &F, cfg.normals_k, nullptr, nullptr);
    }
    for (const Group& g : src_groups)     // queries
        if (s == SB_OK) s = forest_append(ctx, &F, g.L->d_clouds, g.L->cloud_off.data(), g.slots.data(), (int)g.slots.size());
    if (s == SB_OK) {
        sb_icp_config icfg;
        sb_default_icp_config(&icfg);
        icfg.max_iterations = cfg.icp_max_iterations;  // loop_closure.hpp:106
        icfg.tolerance = cfg.icp_tolerance;            // loop_closure.hpp:107
        icfg.normals_k = cfg.normals_k;
        for (int b = 0; b < n && s == SB_OK; b += VERIFY_BATCH) {
            const int m = std::min(VERIFY_BATCH, n - b);
            std::vector<PairDesc> pairs((size_t)m);
            for (int i = 0; i < m; ++i) {
                const CloudRef& q = src[b + i];
                memset(&pairs[i], 0, sizeof(PairDesc));
                pairs[i].src_tree = n_tgt + src_of[b + i];   // source = query cloud (loop_closure.hpp:102)
                pairs[i].n_src = (int)(q.L->cloud_off[q.slot + 1] - q.L->cloud_off[q.slot]);
                pairs[i].tree = tgt_of[b + i];               // target = candidate cloud (loop_closure.hpp:103)
            }
            s = icp_batch(ctx, &F, pairs, &icfg, res + b);
        }
    }
    const cudaError_t sync_err = cudaStreamSynchronize(ctx->stream);
    forest_free(&F);
    if (s != SB_OK) return s;
    if (sync_err != cudaSuccess) return fail(ctx, SB_ERR_CUDA, "loop: verification failed on the device: %s", cudaGetErrorString(sync_err));
    return SB_OK;
}

static void fill_result(const CloudRef& q, const CloudRef& t, double dist, const sb_icp_result& r, sb_loop_result* R,
                        int* converged) {
    R->query_frame = q.L->frame_idx[q.slot];
    R->match_frame = t.L->frame_idx[t.slot];
    memcpy(R->transform, r.transformation, sizeof(R->transform));
    R->scan_context_distance = dist;
    R->icp_fitness = r.final_error;
    *converged = r.converged && r.status == SB_OK;
}

// loop_closure.hpp:99-109 for a set of (query slot, entry) pairs of one detector at once.
int loop_verify(sb_loop* L, const int* qslots, const int* entries, const double* dist, int n, sb_loop_result* results,
                int* converged) {
    Ctx* ctx = L->ctx;
    if (n <= 0) return SB_OK;
    const int n_slots = (int)L->entry_id.size();
    if (n_slots == 0) return fail(ctx, SB_ERR_EMPTY, "loop: empty database");
    std::vector<CloudRef> src((size_t)n), tgt((size_t)n);
    for (int i = 0; i < n; ++i) {
        const int qs = qslots[i];
        if (qs < 0 || qs >= n_slots) return fail(ctx, SB_ERR_INVALID_ARG, "loop: query slot %d out of range", qs);
        const int slot = slot_of(L, entries[i]);
        if (slot < 0 || slot == qs)
            return fail(ctx, SB_ERR_INVALID_ARG, "loop: entry %d is not owned by rank %d", entries[i], L->rank);
        src[i] = {L, qs};
        tgt[i] = {L, slot};
    }
    std::vector<sb_icp_result> res((size_t)n);
    SB_TRY(verify_pairs(ctx, L->cfg, src.data(), tgt.data(), n, res.data()));
    for (int i = 0; i < n; ++i) fill_result(src[i], tgt[i], dist ? dist[i] : 0.0, res[i], &results[i], &converged[i]);
    return SB_OK;
}

// addFrame for n_frames clouds (host CSR rows): the state n_frames calls of loop_add leave, with one upload per run of
// kept frames (world == 1: one), one descriptor launch and one synchronise.  Kept: the frames this rank owns and the
// newest one (a guest when another rank owns it).
int loop_add_many(sb_loop* L, const double* xyz, const i64* offsets, int n_frames, const int* frame_idx,
                  const double* desc) {
    Ctx* ctx = L->ctx;
    if (n_frames <= 0) return SB_OK;
    if (L->last_is_guest) {   // as loop_add: the former guest gives way
        L->entry_id.pop_back();
        L->frame_idx.pop_back();
        L->cloud_off.pop_back();
        L->last_is_guest = false;
    }
    std::vector<int> keep;
    for (int f = 0; f < n_frames; ++f)
        if ((L->n_global + f) % L->world == L->rank || f == n_frames - 1) keep.push_back(f);
    const int n_keep = (int)keep.size();
    const size_t slots = L->entry_id.size();
    const i64 rows = L->cloud_off.empty() ? 0 : L->cloud_off.back();
    if (L->cloud_off.empty()) L->cloud_off.push_back(0);
    std::vector<i64> off((size_t)n_keep + 1, rows);   // pool rows of the kept clouds
    std::vector<int> meta((size_t)n_keep * 2);
    for (int k = 0; k < n_keep; ++k) {
        const int f = keep[k];
        off[k + 1] = off[k] + (offsets[f + 1] - offsets[f]);
        meta[2 * k] = frame_idx[f];
        meta[2 * k + 1] = L->n_global + f;
    }
    SB_TRY(grow(L, &L->d_desc, &L->desc_cap, slots + n_keep, slots, SB_SC_SIZE, FIRST_DESC_SLOTS));
    SB_TRY(grow(L, &L->d_meta, &L->meta_cap, slots + n_keep, slots, 1, FIRST_DESC_SLOTS));
    SB_TRY(grow(L, &L->d_clouds, &L->cloud_cap, (size_t)off[n_keep], (size_t)rows, 3, FIRST_CLOUD_ROWS));
    SB_CUDA(ctx, cudaMemcpyAsync(L->d_meta + slots, meta.data(), sizeof(int) * meta.size(), cudaMemcpyHostToDevice, ctx->stream));
    double* d_slot = L->d_desc + slots * SB_SC_SIZE;
    for (int k0 = 0, k1; k0 < n_keep; k0 = k1) {   // runs of consecutive kept frames are contiguous in the input
        for (k1 = k0 + 1; k1 < n_keep && keep[k1] == keep[k1 - 1] + 1; ++k1) {}
        const i64 r0 = offsets[keep[k0]], r1 = offsets[keep[k1 - 1] + 1];
        if (r1 > r0)
            SB_CUDA(ctx, cudaMemcpyAsync(L->d_clouds + 3 * off[k0], xyz + 3 * r0, sizeof(double) * 3 * (r1 - r0),
                                         cudaMemcpyHostToDevice, ctx->stream));
        if (desc)
            SB_CUDA(ctx, cudaMemcpyAsync(d_slot + (size_t)k0 * SB_SC_SIZE, desc + (size_t)keep[k0] * SB_SC_SIZE,
                                         sizeof(double) * SB_SC_SIZE * (k1 - k0), cudaMemcpyHostToDevice, ctx->stream));
    }
    if (!desc) {   // ScanContext sc(points), loop_closure.hpp:55
        i64* d_off;
        SB_TRY(arena_get(ctx, off.size(), &d_off));
        SB_CUDA(ctx, cudaMemcpyAsync(d_off, off.data(), sizeof(i64) * off.size(), cudaMemcpyHostToDevice, ctx->stream));
        SB_TRY(sc_compute_dev(ctx, L->d_clouds, d_off, n_keep, d_slot));
    }
    SB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int k = 0; k < n_keep; ++k) {
        L->entry_id.push_back(meta[2 * k + 1]);
        L->frame_idx.push_back(meta[2 * k]);
        L->cloud_off.push_back(off[k + 1]);
    }
    const int last_id = L->n_global + n_frames - 1;
    L->n_global += n_frames;
    L->last_frame = frame_idx[n_frames - 1];
    L->last_is_guest = (last_id % L->world) != L->rank;
    return SB_OK;
}

// The walk of detect() (loop_closure.hpp:95-122) for many queries at once.  Every round verifies, for each query that
// still needs acceptances, its next `chunk` candidates; all pairs of a round go through one verify call.  Each query's
// walk then takes its results in list order and advances by the number of candidates verified, so none is skipped.  A
// query that exhausts its short list (fewer entries than total[i]) gets its full sorted list from full_list and
// continues where the short list ended.  The candidate id of every acceptance goes to accepted_id (if not null).
using Cands = std::vector<std::pair<double, int>>;
using WalkVerify = std::function<int(const std::vector<int>& query, const std::vector<int>& id,
                                     const std::vector<double>& dist, sb_loop_result* res, int* conv)>;
static int detect_walk(Ctx* ctx, const sb_loop_config& cfg, int n_q, std::vector<Cands>& cand, const std::vector<int>& total,
                       const std::function<int(int, Cands&)>& full_list, const WalkVerify& verify,
                       sb_loop_result* results, int* accepted_id, int* count) {
    const int maxc = cfg.max_candidates;
    int chunk = cfg.verify_chunk > 0 ? cfg.verify_chunk : maxc;
    if (chunk < 1) chunk = 1;
    std::vector<size_t> pos((size_t)n_q, 0);
    std::vector<char> have_all((size_t)n_q);
    for (int i = 0; i < n_q; ++i) have_all[i] = (int)cand[i].size() >= total[i];
    for (;;) {
        std::vector<int> rq, re, owner, take;
        std::vector<double> rd;
        for (int i = 0; i < n_q; ++i) {
            if (count[i] >= maxc) continue;
            if (pos[i] >= cand[i].size()) {
                if (have_all[i]) continue;
                arena_reset(ctx);
                SB_TRY(full_list(i, cand[i]));   // same order, now complete
                have_all[i] = 1;
                if (pos[i] >= cand[i].size()) continue;
            }
            const int m = (int)std::min(cand[i].size() - pos[i], (size_t)chunk);
            for (int t = 0; t < m; ++t) {
                rq.push_back(i);
                re.push_back(cand[i][pos[i] + t].second);
                rd.push_back(cand[i][pos[i] + t].first);
            }
            owner.push_back(i);
            take.push_back(m);
        }
        if (owner.empty()) break;
        const int n = (int)rq.size();
        std::vector<sb_loop_result> res((size_t)n);
        std::vector<int> conv((size_t)n);
        arena_reset(ctx);
        SB_TRY(verify(rq, re, rd, res.data(), conv.data()));
        for (size_t k = 0, p = 0; k < owner.size(); p += (size_t)take[k], ++k) {
            const int i = owner[k];
            for (int t = 0; t < take[k] && count[i] < maxc; ++t)
                if (conv[p + t] && res[p + t].icp_fitness < cfg.icp_fitness_threshold) {   // loop_closure.hpp:112
                    if (accepted_id) accepted_id[(size_t)i * maxc + count[i]] = re[p + t];
                    results[(size_t)i * maxc + count[i]++] = res[p + t];
                }
            pos[i] += (size_t)take[k];
        }
    }
    return SB_OK;
}

// detect() for many query slots (world == 1, ascending).
int loop_detect_batch(sb_loop* L, const int* qslots, int n_q, sb_loop_result* results, int* count) {
    Ctx* ctx = L->ctx;
    for (int i = 0; i < n_q; ++i) count[i] = 0;
    if (L->cfg.max_candidates <= 0 || n_q <= 0) return SB_OK;
    std::vector<Cands> cand;
    std::vector<int> total;
    SB_TRY(loop_candidates_batch(L, qslots, n_q, cand, total));
    auto full_list = [&](int i, Cands& c) -> int {
        int t = 0;
        return loop_candidates(L, c, 0, &t, qslots[i]);
    };
    WalkVerify verify = [&](const std::vector<int>& q, const std::vector<int>& e, const std::vector<double>& d,
                            sb_loop_result* res, int* conv) -> int {
        std::vector<int> qs(q.size());
        for (size_t k = 0; k < q.size(); ++k) qs[k] = qslots[q[k]];
        return loop_verify(L, qs.data(), e.data(), d.data(), (int)q.size(), res, conv);
    };
    return detect_walk(ctx, L->cfg, n_q, cand, total, full_list, verify, results, nullptr, count);
}

// ---------------------------------------------------------------------------------------------------------------
// Across detectors (sb_loop_candidates_across / sb_loop_detect_across): query i is entry qe[i] of dbs[qdb[i]], and its
// candidates are the entries of every other detector under the threshold, ordered by (distance, detector, entry) —
// detect()'s rule without the frame gap.  Candidate ids are columns of the padded column space of ScDbRow.
// ---------------------------------------------------------------------------------------------------------------
int loop_across_table(const std::vector<sb_loop*>& dbs, std::vector<ScDbRow>& tab) {
    tab.resize(dbs.size());
    int ld = 0;
    for (size_t d = 0; d < dbs.size(); ++d) {
        const int n = (int)dbs[d]->entry_id.size();
        tab[d] = {dbs[d]->d_desc, n, ld};
        ld += (n + 7) / 8 * 8;   // whole tiles (SC_TE = 8): a tile never straddles two detectors
    }
    return ld;
}

void loop_across_decode(const std::vector<ScDbRow>& tab, int col, int* db, int* entry) {
    // the first detector whose padded columns end after col (padded ends never decrease; an empty detector has none)
    int lo = 0, hi = (int)tab.size() - 1;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (tab[mid].base + (tab[mid].count + 7) / 8 * 8 > col) hi = mid;
        else lo = mid + 1;
    }
    *db = lo;
    *entry = col - tab[lo].base;
}

int loop_candidates_across(const std::vector<sb_loop*>& dbs, const int* qdb, const int* qe, int n_q,
                           std::vector<Cands>& cand, std::vector<int>& total) {
    Ctx* ctx = dbs[0]->ctx;
    cand.assign((size_t)n_q, {});
    total.assign((size_t)n_q, 0);
    if (n_q <= 0) return SB_OK;
    std::vector<ScDbRow> tab;
    const int ld = loop_across_table(dbs, tab);
    if (ld <= 0) return SB_OK;   // every detector is empty
    const int n_dbs = (int)dbs.size();
    const i64 rows = std::max<i64>(8, (i64)(LOOP_DIST_BYTES / (sizeof(double) * (size_t)ld)) / 8 * 8);
    ScDbRow* d_tab;
    int *d_q, *d_col_db;
    double *d_sq, *d_qdesc, *d_dist;
    char* d_sel;
    const size_t sel_bytes = (size_t)n_q * (KSEL * 12 + 4);
    SB_TRY(arena_get(ctx, (size_t)n_dbs, &d_tab));
    SB_TRY(arena_get(ctx, (size_t)2 * n_q, &d_q));
    SB_TRY(arena_get(ctx, (size_t)ld, &d_col_db));
    SB_TRY(arena_get(ctx, (size_t)(ld + n_q) * SB_SC_SECTORS, &d_sq));
    SB_TRY(arena_get(ctx, (size_t)n_q * SB_SC_SIZE, &d_qdesc));
    SB_TRY(arena_get(ctx, (size_t)std::min<i64>(rows, n_q) * ld, &d_dist));
    SB_TRY(arena_get(ctx, sel_bytes, &d_sel));
    unsigned long long* d_sel_d = reinterpret_cast<unsigned long long*>(d_sel);
    int* d_sel_e = reinterpret_cast<int*>(d_sel + (size_t)n_q * KSEL * 8);
    int* d_tot = d_sel_e + (size_t)n_q * KSEL;
    std::vector<int> q((size_t)2 * n_q);
    std::copy(qdb, qdb + n_q, q.begin());
    std::copy(qe, qe + n_q, q.begin() + n_q);
    SB_TRY(table_upload(ctx, d_tab, tab.data(), sizeof(ScDbRow) * tab.size()));
    SB_TRY(table_upload(ctx, d_q, q.data(), sizeof(int) * q.size()));
    const double thr = dbs[0]->cfg.sc_distance_threshold;
    SB_TRY(sc_sq_across_dev(ctx, d_tab, n_dbs, ld, d_q, d_q + n_q, n_q, d_col_db, d_sq, d_qdesc));
    for (i64 g0 = 0; g0 < n_q; g0 += rows) {
        const int ng = (int)std::min<i64>(rows, n_q - g0);
        SB_TRY(sc_distance_across_dev(ctx, d_tab, d_col_db, d_qdesc + g0 * SB_SC_SIZE, d_sq + (ld + g0) * SB_SC_SECTORS,
                                      d_q + g0, ng, d_sq, d_dist, ld));
        SB_LAUNCH(ctx, k_loop_select_across, (unsigned)ng, 1024, 0, d_dist, (i64)ld, d_col_db, d_q + g0, thr,
                  d_sel_d + g0 * KSEL, d_sel_e + g0 * KSEL, d_tot + g0);
    }
    SB_TRY(pinned_reserve(ctx, sel_bytes));
    SB_CUDA(ctx, cudaMemcpyAsync(ctx->pinned, d_sel, sel_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const unsigned long long* h_d = reinterpret_cast<const unsigned long long*>(ctx->pinned);
    const int* h_e = reinterpret_cast<const int*>(ctx->pinned + (size_t)n_q * KSEL * 8);
    for (int r = 0; r < n_q; ++r) {
        total[r] = h_e[(size_t)n_q * KSEL + r];
        decode_selection(h_d + (size_t)r * KSEL, h_e + (size_t)r * KSEL, KSEL, cand[r]);
    }
    return SB_OK;
}

// Query i's complete list (distance, column), sorted: the one-query search against each other detector's pool.
static int across_full_list(const std::vector<sb_loop*>& dbs, const std::vector<ScDbRow>& tab, int qdb, int qe, Cands& cand) {
    Ctx* ctx = dbs[0]->ctx;
    cand.clear();
    int n = 0;
    for (const ScDbRow& t : tab) n += t.count;
    if (n == 0) return SB_OK;
    double* d_out;
    SB_TRY(arena_get(ctx, (size_t)n, &d_out));
    const double* q = dbs[qdb]->d_desc + (size_t)qe * SB_SC_SIZE;
    for (size_t d = 0, off = 0; d < tab.size(); off += (size_t)tab[d].count, ++d)
        if ((int)d != qdb) SB_TRY(sc_distance_dev(ctx, q, tab[d].desc, tab[d].count, d_out + off));
    std::vector<double> dist((size_t)n);
    SB_CUDA(ctx, cudaMemcpyAsync(dist.data(), d_out, sizeof(double) * n, cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const double thr = dbs[0]->cfg.sc_distance_threshold;
    for (size_t d = 0, off = 0; d < tab.size(); off += (size_t)tab[d].count, ++d) {
        if ((int)d == qdb) continue;
        for (int e = 0; e < tab[d].count; ++e)
            if (dist[off + e] < thr) cand.push_back({dist[off + e], tab[d].base + e});   // loop_closure.hpp:86-88
    }
    std::sort(cand.begin(), cand.end());   // (distance, column) = (distance, detector, entry)
    return SB_OK;
}

int loop_detect_across(const std::vector<sb_loop*>& dbs, const int* qdb, const int* qe, int n_q, sb_loop_result* results,
                       int* match_db, int* count) {
    Ctx* ctx = dbs[0]->ctx;
    const sb_loop_config& cfg = dbs[0]->cfg;
    const int maxc = cfg.max_candidates;
    for (int i = 0; i < n_q; ++i) count[i] = 0;
    if (maxc <= 0 || n_q <= 0) return SB_OK;
    std::vector<Cands> cand;
    std::vector<int> total;
    SB_TRY(loop_candidates_across(dbs, qdb, qe, n_q, cand, total));
    std::vector<ScDbRow> tab;
    loop_across_table(dbs, tab);
    auto full_list = [&](int i, Cands& c) -> int { return across_full_list(dbs, tab, qdb[i], qe[i], c); };
    WalkVerify verify = [&](const std::vector<int>& q, const std::vector<int>& col, const std::vector<double>& d,
                            sb_loop_result* res, int* conv) -> int {
        const int n = (int)q.size();
        std::vector<CloudRef> src((size_t)n), tgt((size_t)n);
        for (int k = 0; k < n; ++k) {
            int db, e;
            loop_across_decode(tab, col[k], &db, &e);
            src[k] = {dbs[qdb[q[k]]], qe[q[k]]};
            tgt[k] = {dbs[db], e};
        }
        std::vector<sb_icp_result> icp((size_t)n);
        SB_TRY(verify_pairs(ctx, cfg, src.data(), tgt.data(), n, icp.data()));
        for (int k = 0; k < n; ++k) fill_result(src[k], tgt[k], d[k], icp[k], &res[k], &conv[k]);
        return SB_OK;
    };
    std::vector<int> cols((size_t)n_q * maxc);
    SB_TRY(detect_walk(ctx, cfg, n_q, cand, total, full_list, verify, results, cols.data(), count));
    for (int i = 0; i < n_q; ++i)
        for (int j = 0; j < count[i]; ++j) {
            int e;
            loop_across_decode(tab, cols[(size_t)i * maxc + j], &match_db[(size_t)i * maxc + j], &e);
        }
    return SB_OK;
}

}  // namespace sb
