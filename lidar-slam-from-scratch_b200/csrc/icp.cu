// icp.cu — batched point-to-plane ICP; replaces slam::solve_point_to_plane and slam::icp_point_to_plane
// (slam_viz/include/slam_viz/core/icp.hpp:89-144 and :157-258).
//
// The reference runs, per pair and per iteration: a KD-tree 1-NN pass over the source (twice, icp.hpp:185,190),
// an RMS pass, an n x 6 Jacobian build, J^T J, an LDLT solve, a Rodrigues update and a full rewrite of the
// source cloud.  Here one iteration of ALL pairs of a batch is four kernels:
//   k_icp_match     one warp per 32 consecutive source points (in the source's own curve order), one point per lane:
//                   cur = T * src (never stored); a walk over the target's k-nearest-neighbour graph from the previous
//                   correspondence that ends with a PROOF that the best point seen is the exact nearest neighbour.
//                   Lanes left without a proof go to a device-wide queue: one entry per point, or — when an item has
//                   many of them (the first pass: no previous correspondences) — ONE entry for the item;
//   k_icp_fallback  one WARP per queue entry: a point by the exact warp-cooperative tree traversal of traverse.cuh, an
//                   item's open points together by ONE packet traversal (NearestPacketVisitor, traverse.cuh);
//   k_icp_accum     one warp per 32 source points: residual + the 29 sums (21 of J^T J, 6 of J^T r, sum r^2, matched
//                   points), fixed-order shuffle tree, one 232-byte partial per work item (items whose points were
//                   all settled in k_icp_match are finished there, same device function, same bits; the others are
//                   listed in IcpJob::open_items, which is what this kernel works off);
//   k_icp_solve     one block per pair: adds the pair's partials in item order (run-to-run deterministic), RMS error,
//                   convergence test (icp.hpp:210-217), 6x6 pivoted LDL^T, Rodrigues (icp.hpp:127-142), T <- delta * T.
// The three per-item kernels run as grids of resident CTAs whose warps take their work from device-wide counters
// (WorkIter).  The loop is a CUDA-graph WHILE node whose condition k_icp_solve's last block sets from the device-side
// count of still-active pairs: no host round trip per iteration.  All kernels read their arguments from one device-resident
// IcpJob, so the instantiated graph is reused by every call on the context.
#include "traverse.cuh"

#include <cstdlib>

namespace sb {

enum { ST_ACTIVE = 0, ST_CONVERGED = 1, ST_EXHAUSTED = 2, ST_DONE = 3 };

struct PairState {
    double prev_error;
    int state;
    int iter;
};

struct FallbackEntry {   // a source point whose walk did not end with a proof
    i64 q;               // item * ITEM_Q + lane
    int seed;            // best target position the walk found (-1: none); item entries: mask of the open lanes
    int pad;             // pair << 1 | (1: item entry)
};

struct IcpJob {
    ForestView F;
    int* match;                 // n_items x ITEM_Q: correspondence of every source point (seed of the next pass)
    i64 n_items;
    const PairDesc* pairs;
    sb_icp_result* results;
    PairState* state;
    double* partials;           // n_items x 28
    int* act_pair;              // pairs the next pass works on (ascending), rebuilt after every solve
    i64* act_off;               // n_act + 1 prefix sums of their work items
    int2* open_items;           // (work item, pair) of the items k_icp_match could not finish in this pass: k_icp_accum's list
    FallbackEntry* queue;       // capacity n_items x ITEM_Q
    unsigned long long* stats;  // optional (SB_ICP_STATS): per iteration bucket [queries, answered by the tree]
    double T0[16];
    double tol, min_err;
    int n_pairs;
    int max_it;
    int n_active;
    int ticket;
    int nbr_k;
    int q_count;                // entries in `queue` (reset by k_icp_solve / k_icp_init)
    int n_act;                  // entries of act_pair
    int packet_min;             // open lanes of a work item from which the packet traversal takes over (SB_ICP_PACKET_MIN)
    int passes;                 // batch passes run so far (launch accounting)
    int n_open;                 // entries of open_items (reset with q_count)
    int work[4];                // next work item of k_icp_match / k_icp_fallback / k_icp_accum in this pass (reset with q_count)
    i64 n_act_items;            // = act_off[n_act]
};

static constexpr int IWARPS = 8;
static constexpr int NSUM = 29;      // 21 of J^T J, 6 of J^T r, sum r^2, and the number of points with a correspondence
static constexpr int ITEM_Q = 32;   // source points per warp work item: one per lane
static constexpr int PACKET_MIN_ITEMS = 32768;  // work items of a pass (32 source points each) from which packets are used
#ifndef SB_MAX_HOPS
#define SB_MAX_HOPS 6
#endif
static constexpr int MAX_HOPS = SB_MAX_HOPS;  // re-centrings of the neighbour-graph walk before the tree takes over

// -------------------------------------------------------------------------------------------------------------
// Block-wide (256 threads): the list of pairs in state `want` and the prefix sums of their work items.  The passes
// iterate over this list only, so an iteration costs what its ACTIVE pairs cost — the batch keeps running until
// the slowest pair stops (icp.hpp:181, max_iterations), long after most pairs have converged.
__device__ void build_active(IcpJob* __restrict__ job, int want, bool from_list) {
    __shared__ int s_wc[8];
    __shared__ i64 s_wi[8];
    __shared__ int s_bc;
    __shared__ i64 s_bi;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) { s_bc = 0; s_bi = 0; }
    __syncthreads();
    // from_list: a pair only ever leaves ST_ACTIVE, so the next active list is a filter of the current one — compacted
    // in place (round r reads entries [256 r, 256 r + 256) before its first barrier and writes below 256 r + 256 after
    // it).  With 4096 pairs the scan over all of them was 16 rounds of three barriers in EVERY pass, run by one block
    // while the rest of the chip waits.
    const int n = from_list ? job->n_act : job->n_pairs;
    for (int base = 0; base < n; base += 256) {
        const int e = base + tid;
        int p = e;
        if (from_list && e < n) p = job->act_pair[e];
        const bool flag = e < n && __ldcg(&job->state[p].state) == want;
        const i64 items = flag ? (i64)job->pairs[p].n_items : 0;
        const unsigned bal = __ballot_sync(0xffffffffu, flag);
        i64 inc = items;  // inclusive warp scan of the item counts
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            i64 v = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += v;
        }
        if (lane == 31) { s_wc[warp] = __popc(bal); s_wi[warp] = inc; }
        __syncthreads();
        int c0 = s_bc;
        i64 i0 = s_bi;
        for (int w = 0; w < warp; ++w) { c0 += s_wc[w]; i0 += s_wi[w]; }
        if (flag) {
            const int a = c0 + __popc(bal & lanemask_lt());
            job->act_pair[a] = p;
            job->act_off[a] = i0 + inc - items;
        }
        __syncthreads();
        if (tid == 255) { s_bc = c0 + __popc(bal); s_bi = i0 + inc; }
        __syncthreads();
    }
    if (tid == 0) {
        job->act_off[s_bc] = s_bi;
        job->n_act = s_bc;
        job->n_act_items = s_bi;
    }
}

// one block
__global__ void __launch_bounds__(256) k_icp_init(IcpJob* __restrict__ job, cudaGraphConditionalHandle cond,
                                                  int use_cond) {
    const int n = job->n_pairs;
    for (int p = threadIdx.x; p < n; p += blockDim.x) {
        sb_icp_result& R = job->results[p];
        PairDesc P = job->pairs[p];
#pragma unroll
        for (int i = 0; i < 16; ++i) R.transformation[i] = job->T0[i];
        R.final_error = 0.0;
        R.converged = 0;
        R.num_iterations = 0;
        R.history_len = 0;
        bool empty = P.n_src <= 0 || job->F.trees[P.tree].n <= 0;
        R.status = empty ? SB_ERR_EMPTY : SB_OK;
        PairState s;
        s.prev_error = 1.7976931348623157e308;  // icp.hpp:178
        s.iter = 0;
        s.state = empty ? ST_DONE : (job->max_it > 0 ? ST_ACTIVE : ST_EXHAUSTED);
        job->state[p] = s;
    }
    __syncthreads();
    const bool loop = job->n_active > 0 && job->max_it > 0;
    build_active(job, loop ? ST_ACTIVE : ST_EXHAUSTED, false);
    if (threadIdx.x == 0) {
        job->q_count = 0;
        job->n_open = 0;
        job->work[0] = job->work[1] = job->work[2] = 0;
        if (use_cond) cudaGraphSetConditional(cond, loop ? 1u : 0u);
    }
}

// largest a in [0, n) with off[a] <= x (off[0] = 0 <= x), called by the whole (converged) warp.  These loads head the
// dependency chain of every work item, and a pass with few pairs left costs what its longest chain costs: up to 256
// active pairs the warp tests 32 evenly spaced entries per step — two dependent loads instead of eight.  Above that
// (a pass that is throughput-bound anyway) the plain binary search: one broadcast load per step.
__device__ __forceinline__ int find_active(const i64* __restrict__ off, int n, i64 x, int lane) {
    int lo = 0, len = n;
    if (n > 256) {
        int hi = n;
        while (hi - lo > 1) {
            int mid = (lo + hi) >> 1;
            if (off[mid] <= x) lo = mid; else hi = mid;
        }
        return lo;
    }
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

// Work distribution of the three per-pass kernels: the warps of a grid of resident CTAs take their work items from a
// device-wide counter, `chunk` consecutive items per fetch.  With fixed shares (item = warp id + r * warps of the
// grid, until round 2) the CTA slots of the early finishers idled while one warp of the CTA still walked its last
// items — a work item costs anything between 32 one-load proofs and a packet traversal of the tree.  A pass with no
// more items than the grid has warps (few pairs left, a single pair) costs what its longest chain costs: there warp w
// takes item w, without the round trip to the counter.
struct WorkIter {   // (item counts are below 2^31 / 32: icp_enqueue checks)
    int* counter;
    int n, cur, end, chunk, lane;
    __device__ __forceinline__ WorkIter(int* c, i64 n_, int lane_, int gwarp, int gwarps, int chunk_)
        : counter(c), n((int)n_), cur(-1), end(0), chunk(chunk_), lane(lane_) {
        if (n <= gwarps) { chunk = 0; cur = gwarp; }
    }
    __device__ __forceinline__ bool next(i64& it) {
        if (chunk == 0) {            // one item per warp
            it = cur;
            const bool have = cur < n;
            cur = n;
            return have;
        }
        if (cur + 1 >= end) {        // cur: the item handed out last; end: the end of the chunk in hand
            int v = 0;
            if (lane == 0) v = atomicAdd(counter, chunk);
            cur = __shfl_sync(0xffffffffu, v, 0);
            end = cur + chunk;
        } else {
            ++cur;
        }
        it = cur;
        return cur < n;
    }
};

// upper bound of sqrt(d2), with 1e-6 of slack for the rounding of d2 itself
__device__ __forceinline__ float sqrt_up(double d2) {
    return sqrt_upper(d2);
}

// cur = src * R^T + t with the oracle's association (types.hpp:110-115)
__device__ __forceinline__ void transform_point(const double* __restrict__ Tm, const double* __restrict__ p,
                                                double& cx, double& cy, double& cz) {
    double x = p[0], y = p[1], z = p[2];
    cx = ((x * Tm[0] + y * Tm[1]) + z * Tm[2]) + Tm[3];
    cy = ((x * Tm[4] + y * Tm[5]) + z * Tm[6]) + Tm[7];
    cz = ((x * Tm[8] + y * Tm[9]) + z * Tm[10]) + Tm[11];
}

__device__ __forceinline__ int grid_find(const GridSlot* __restrict__ tab, unsigned mask, int shift, int ix, int iy,
                                         int iz) {
    if ((unsigned)ix > 0x1fffffu || (unsigned)iy > 0x1fffffu || (unsigned)iz > 0x1fffffu) return -1;
    const unsigned long long key = grid_key(ix, iy, iz);
    unsigned slot = grid_hash(key, shift);
    while (true) {
        const ulonglong2 e = __ldg(reinterpret_cast<const ulonglong2*>(tab + slot));
        if (e.x == key) return (int)(unsigned)e.y;
        if (e.x == SB_GRID_EMPTY) return -1;
        slot = (slot + 1u) & mask;
    }
}

// A target point near the query: the representative of the query's grid cell, else the nearest representative of
// the 26 surrounding cells (fp32: a starting point, never an answer).  -1 if all 27 cells are empty.
__device__ __forceinline__ int grid_seed(const TreeDesc& T, double qx, double qy, double qz) {
    int ix, iy, iz;
    if (!grid_cell(T, qx, qy, qz, ix, iy, iz)) return -1;
    const GridSlot* tab = T.grid + T.tab_off;
    const unsigned mask = (unsigned)(((i64)1 << (64 - T.tab_shift)) - 1);
    int pos = grid_find(tab, mask, T.tab_shift, ix, iy, iz);
    if (pos >= 0) return pos;
    float best = __int_as_float(0x7f800000);
    const float fx = (float)qx, fy = (float)qy, fz = (float)qz;
    for (int c = 0; c < 27; ++c) {
        if (c == 13) continue;
        int p = grid_find(tab, mask, T.tab_shift, ix + c % 3 - 1, iy + (c / 3) % 3 - 1, iz + c / 9 - 1);
        if (p < 0) continue;
        const double* P = reinterpret_cast<const double*>(T.pts + T.pt_off + p);
        const double2 xy = __ldg(reinterpret_cast<const double2*>(P));
        const double z = __ldg(P + 2);
        float dx = (float)xy.x - fx, dy = (float)xy.y - fy, dz = (float)z - fz;
        float d = dx * dx + dy * dy + dz * dz;
        if (d < best) { best = d; pos = p; }
    }
    return pos;
}

// Correspondence search (replaces KDTree::nearest_batch, kdtree.hpp:43-59, exact): start from the previous
// iteration's match (or the seed grid) and walk the target's k-nearest-neighbour graph.  With c the current centre,
// entries of c's list are evaluated in ascending distance from c; every point not yet evaluated is at least r_j
// from c, hence at least r_j - |q c| from the query q.  As soon as that bound exceeds the best distance found, the
// best point IS the nearest neighbour (all bounds rounded conservatively in fp32, the candidates themselves compared
// in the oracle's fp64 (d2, index) order).  If the list runs out first, re-centre on the best point and repeat.
// Points whose walk ends without that proof are answered by packet_nearest (many per item) or k_icp_fallback (few).
// The walk of one source point (one lane): cur = Tm * src, then the neighbour-graph walk from `center` (the previous
// correspondence; < 0 or stale: the seed grid).  Returns the best target position found (-1: none) and whether it is
// PROVEN to be the nearest neighbour.
__device__ __forceinline__ void walk_lane(const TreeDesc& T, int K, const double* __restrict__ Tm,
                                          const TreePoint* __restrict__ src_pt, int center, int& bpos, bool& cert,
                                          double& cx, double& cy, double& cz) {
    bpos = -1;
    cert = false;
    transform_point(Tm, reinterpret_cast<const double*>(src_pt), cx, cy, cz);
    if (center < 0 || center >= T.n) center = grid_seed(T, cx, cy, cz);
    if (center < 0) return;
    const TreePoint* TP = T.pts + T.pt_off;
    const NbrEntry* TN = T.nbr + T.pt_off * (i64)K;
    TreePoint c = load_point(TP + center);
    double bd = dist2_rn(c.x, c.y, c.z, cx, cy, cz);
    int bidx = c.idx;
    bpos = center;
    if (!(bd == bd)) {  // NaN query: never matches (kdtree.hpp:125 strict <); the traversal returns -1 for it
        bpos = -1;
        return;
    }
    {   // One-load proof: every other point is at least r1 from the centre (TreePoint::pad), hence at least r1 - |q c|
        // from the query; if that exceeds |q c| the centre IS the nearest neighbour — no list, no candidates.
        const float dc = sqrt_up(bd);
        if (__fsub_rd(__int_as_float(c.pad), dc) > dc) { cert = true; return; }
    }
    for (int hop = 0; hop < MAX_HOPS; ++hop) {
        const float dc = sqrt_up(bd);  // |q centre|: the centre is the best point so far
        float sb = dc;
        const int2* L = reinterpret_cast<const int2*>(TN + (i64)center * K);
        float rlast = 0.f;
        for (int j = 0; j < K && !cert; ++j) {
            const int2 e = __ldg(L + j);
            rlast = __int_as_float(e.y);
            if (e.x < 0 || __fsub_rd(rlast, dc) > sb) { cert = true; break; }
            if (e.x == center) continue;
            const TreePoint t = load_point(TP + e.x);
            const double d = dist2_rn(t.x, t.y, t.z, cx, cy, cz);
            if (d < bd || (d == bd && t.idx < bidx)) {
                bd = d; bidx = t.idx; bpos = e.x;
                sb = sqrt_up(bd);
            }
        }
        if (!cert && __fsub_rd(rlast, dc) > sb) cert = true;  // list exhausted: the rest is >= r_{K-1}
        if (cert || bpos == center) break;
        center = bpos;
    }
}

// ordered image of a float for warp-wide min / max reductions
__device__ __forceinline__ unsigned ordered_u32(float f) {
    const unsigned b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float float_from_ordered_u32(unsigned u) {
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// Exact nearest neighbours of the lanes in `todo` (queries (cx, cy, cz), starting points bpos): one packet traversal
// for all of them (NearestPacketVisitor, traverse.cuh).  The caller checks T.gext < 1e15 (float32 bounds).
__device__ __forceinline__ void packet_nearest(const ForestView& F, const TreeDesc& T, WarpStack& S, int lane,
                                               unsigned todo, double cx, double cy, double cz, int& bpos, unsigned stage) {
    const bool mine = (todo >> lane) & 1u;
    NearestPacketVisitor V(T, lane, stage);
    V.init(mine, cx, cy, cz, bpos);
    // bounding box of the packet's queries (float32, rounded outwards)
    const float inf = __int_as_float(0x7f800000);
    const bool in = V.need;
    const float lx = float_from_ordered_u32(__reduce_min_sync(0xffffffffu, ordered_u32(in ? __double2float_rd(cx) : inf)));
    const float ly = float_from_ordered_u32(__reduce_min_sync(0xffffffffu, ordered_u32(in ? __double2float_rd(cy) : inf)));
    const float lz = float_from_ordered_u32(__reduce_min_sync(0xffffffffu, ordered_u32(in ? __double2float_rd(cz) : inf)));
    const float hx = float_from_ordered_u32(__reduce_max_sync(0xffffffffu, ordered_u32(in ? __double2float_ru(cx) : -inf)));
    const float hy = float_from_ordered_u32(__reduce_max_sync(0xffffffffu, ordered_u32(in ? __double2float_ru(cy) : -inf)));
    const float hz = float_from_ordered_u32(__reduce_max_sync(0xffffffffu, ordered_u32(in ? __double2float_ru(cz) : -inf)));
    if (lx <= hx) {   // at least one searchable query
        BoxQuery Q;
        Q.lox = lx; Q.loy = ly; Q.loz = lz; Q.hix = hx; Q.hiy = hy; Q.hiz = hz;
        traverse(F, T, Q, S, V, lane);
    }
    if (mine) bpos = V.bpos;
}

__device__ __forceinline__ void accumulate_item(const IcpJob* __restrict__ job, const TreeDesc& T, i64 it, int lane,
                                                int my_pos, double cx, double cy, double cz);

// Term T of a source point's contribution to its work item's 29 sums: 0..20 the upper triangle of J^T J row by row,
// 21..26 J^T r, 27 r^2, 28 the point counts; 29..31 unused.
template <int T>
__device__ __forceinline__ double item_term(const double (&J)[6], double b, double cnt) {
    if constexpr (T < 21) {
        constexpr int A = T < 6 ? 0 : T < 11 ? 1 : T < 15 ? 2 : T < 18 ? 3 : T < 20 ? 4 : 5;
        constexpr int first = A == 0 ? 0 : A == 1 ? 6 : A == 2 ? 11 : A == 3 ? 15 : A == 4 ? 18 : 20;
        return J[A] * J[A + (T - first)];
    } else if constexpr (T < 27) {
        return J[T - 21] * b;
    } else if constexpr (T == 27) {
        return b * b;
    } else if constexpr (T == 28) {
        return cnt;
    } else {
        return 0.0;
    }
}
// Slot T (0 <= T < M) after the reduction step with partner lane ^ M: the lane's own bit M decides which of the two
// slots T, T + M of the step before it keeps; the other goes to the partner.  item_sum<1, 0> = sum `lane` over the warp.
template <int M, int T>
__device__ __forceinline__ double item_sum(const double (&J)[6], double b, double cnt, int lane) {
    if constexpr (M == 32) {
        return item_term<T>(J, b, cnt);
    } else {
        const double lo = item_sum<2 * M, T>(J, b, cnt, lane);
        const double hi = item_sum<2 * M, T + M>(J, b, cnt, lane);
        const bool up = (lane & M) != 0;
        const double keep = up ? hi : lo, send = up ? lo : hi;
        return keep + shfl_d_xor(send, M);
    }
}

// Works on the pairs listed in job->act_pair: the ST_ACTIVE ones inside the loop, the ST_EXHAUSTED ones in the final
// error pass (icp.hpp:235-252).  Work item = ITEM_Q consecutive source points of one pair (implicit: binary search
// over the prefix sums act_off), one source point per lane.  Replaces KDTree::nearest_batch (kdtree.hpp:43-59), exact.
__global__ void __launch_bounds__(IWARPS * 32, 5) k_icp_match(IcpJob* __restrict__ job) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const ForestView F = job->F;
    const i64 n_act_items = job->n_act_items;
    const int n_act = job->n_act;
    const int K = job->nbr_k;
    const int packet_min = job->packet_min;
    WorkIter W(&job->work[0], n_act_items, lane, (int)(blockIdx.x * IWARPS + warp), (int)(gridDim.x * IWARPS), n_act_items >= 262144 ? 4 : 1);
    i64 ai;
    while (W.next(ai)) {
        const int a = find_active(job->act_off, n_act, ai, lane);
        const int pair = job->act_pair[a];
        const PairDesc P = job->pairs[pair];
        const i64 it = P.item_off + (ai - job->act_off[a]);
        const int s0 = (int)(it - P.item_off) * ITEM_Q;
        const int count = P.n_src - s0 < ITEM_Q ? P.n_src - s0 : ITEM_Q;
        const TreeDesc& T = F.trees[P.tree];
        const double* Tm = job->results[pair].transformation;
        int bpos = -1;
        bool cert = false;
        double cx = 0, cy = 0, cz = 0;
        if (lane < count) {
            walk_lane(T, K, Tm, P.src_pts + s0 + lane, job->match[it * ITEM_Q + lane], bpos, cert, cx, cy, cz);
            job->match[it * ITEM_Q + lane] = bpos;   // proven, or the starting point of the tree search
        }
        // The points without a proof go to the device-wide queue of k_icp_fallback: one entry per point, or — when the
        // item has many of them (the first pass: no previous correspondences) — ONE entry for the item, whose open
        // points are then answered together by a packet traversal.
        const unsigned todo = __ballot_sync(0xffffffffu, lane < count && !cert);
        if (todo) {
            // (only while the pass is busy enough to be bound by instruction throughput: the packet visits a leaf's 32
            // points one after the other, the warp-cooperative search all at once, and with few pairs left a pass costs
            // what its longest dependency chain costs — measured: 149 vs 79 us per pass with 34 pairs iterating)
            const bool as_item = __popc(todo) >= packet_min && n_act_items >= PACKET_MIN_ITEMS;
            int base = 0;
            if (lane == 0) {
                base = atomicAdd(&job->q_count, as_item ? 1 : __popc(todo));
                // ... and the item itself goes on k_icp_accum's list (it scanned a done-flag per item before: with three
                // quarters of the items finished here, most of that kernel was waiting for flags and its work counter)
                job->open_items[atomicAdd(&job->n_open, 1)] = make_int2((int)it, pair);
            }
            base = __shfl_sync(0xffffffffu, base, 0);
            FallbackEntry e;
            if (as_item) {
                e.q = it * ITEM_Q; e.seed = (int)todo; e.pad = (pair << 1) | 1;
                if (lane == 0) job->queue[base] = e;
            } else if ((todo >> lane) & 1u) {
                e.q = it * ITEM_Q + lane; e.seed = bpos; e.pad = pair << 1;
                job->queue[base + __popc(todo & lanemask_lt())] = e;
            }
        }
        // every point of the item has its proven correspondence: finish the item here (k_icp_accum skips it)
        if (!todo) accumulate_item(job, T, it, lane, lane < count ? bpos : -1, cx, cy, cz);
        if (job->stats && lane == 0) {  // SB_ICP_STATS: buckets by iteration: 0, 1, 2..11, >= 12
            int bkt = job->state[pair].iter;
            bkt = bkt >= 12 ? 3 : (bkt >= 2 ? 2 : bkt);
            atomicAdd(&job->stats[2 * bkt], (unsigned long long)count);
            if (todo) atomicAdd(&job->stats[2 * bkt + 1], (unsigned long long)__popc(todo));
        }
    }
}

// One warp per queue entry.  A point entry: the exact warp-cooperative tree traversal, started from the best point of
// the walk.  An item entry (pad == 1, seed = mask of the item's open lanes): one packet traversal for all of them.
__global__ void __launch_bounds__(IWARPS * 32, 5) k_icp_fallback(IcpJob* __restrict__ job) {
    __shared__ WarpStack stacks[IWARPS];
    __shared__ TreeDesc s_tree[IWARPS];
    __shared__ __align__(16) float4 s_stage[IWARPS][32];   // NearestPacketVisitor's staging rows
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    WarpStack& S = stacks[warp];
    const ForestView F = job->F;
    const int n = job->q_count;
    // (one entry per fetch: a point and a whole item by packet traversal differ too much to be taken in groups)
    WorkIter W(&job->work[1], (i64)n, lane, (int)(blockIdx.x * IWARPS + warp), (int)(gridDim.x * IWARPS), 1);
    i64 e64;
    while (W.next(e64)) {
        const int e = (int)e64;
        const FallbackEntry E = job->queue[e];
        const i64 it = E.q / ITEM_Q;
        const int pair = E.pad >> 1;   // (a binary search over all pairs' item offsets — ten dependent loads — until round 2)
        const bool item_entry = (E.pad & 1) != 0;
        const PairDesc P = job->pairs[pair];
        __syncwarp();
        {
            const int* s = reinterpret_cast<const int*>(&F.trees[P.tree]);
            int* d = reinterpret_cast<int*>(&s_tree[warp]);
            for (int i = lane; i < (int)(sizeof(TreeDesc) / 4); i += 32) d[i] = s[i];
            __syncwarp();
        }
        const TreeDesc& T = s_tree[warp];
        const double* Tm = job->results[pair].transformation;
        if (item_entry && T.gext < 1.0e15) {
            const int s0 = (int)(it - P.item_off) * ITEM_Q;
            const int count = P.n_src - s0 < ITEM_Q ? P.n_src - s0 : ITEM_Q;
            const unsigned todo = (unsigned)E.seed;
            double cx = 0, cy = 0, cz = 0;
            int bpos = -1;
            if (lane < count) {
                transform_point(Tm, reinterpret_cast<const double*>(P.src_pts + s0 + lane), cx, cy, cz);
                bpos = job->match[E.q + lane];
            }
            packet_nearest(F, T, S, lane, todo, cx, cy, cz, bpos, (unsigned)__cvta_generic_to_shared(&s_stage[warp][0]));
            if ((todo >> lane) & 1u) job->match[E.q + lane] = bpos;
        } else {
            unsigned todo = item_entry ? (unsigned)E.seed : 1u;   // (an item entry of a tree of extreme extent: lane by lane)
            while (todo) {
                const int j = __ffs(todo) - 1;
                todo &= todo - 1u;
                const i64 q = item_entry ? E.q + j : E.q;
                double qx, qy, qz;
                transform_point(Tm, reinterpret_cast<const double*>(P.src_pts + (q - P.item_off * ITEM_Q)), qx, qy, qz);
                NearestVisitor V(F, T, qx, qy, qz, lane);
                V.seed(item_entry ? job->match[q] : E.seed);
                traverse(F, T, qx, qy, qz, S, V, lane);
                if (lane == 0) job->match[q] = V.best_pos;
            }
        }
    }
}

// Residual and the 28 sums of one work item (32 source points, one per lane; my_pos < 0: no correspondence, the lane
// adds zeros): fixed-order butterfly, one 224-byte partial per item.  (cx, cy, cz) = the lane's transformed source
// point.
__device__ __forceinline__ void accumulate_item(const IcpJob* __restrict__ job, const TreeDesc& T, i64 it, int lane,
                                                int my_pos, double cx, double cy, double cz) {
    double tx = 0, ty = 0, tz = 0, nx = 0, ny = 0, nz = 0;
    if (my_pos >= 0) {
        TreePoint q = load_point(T.pts + T.pt_off + my_pos);
        tx = q.x; ty = q.y; tz = q.z;
        const double2* np = reinterpret_cast<const double2*>(T.nrm + T.pt_off + my_pos);
        double2 n01 = __ldg(np), n2 = __ldg(np + 1);
        nx = n01.x; ny = n01.y; nz = n2.x;
    } else {
        cx = cy = cz = 0.0;
    }
    double J[6];
    J[0] = cy * nz - cz * ny;  // p x n, icp.hpp:105
    J[1] = cz * nx - cx * nz;
    J[2] = cx * ny - cy * nx;
    J[3] = nx; J[4] = ny; J[5] = nz;
    const double b = ((tx - cx) * nx + (ty - cy) * ny) + (tz - cz) * nz;  // icp.hpp:116
    // 29 sums over the item's 32 points, sum t ending in lane t.  Every sum is the butterfly tree ((v_i + v_{i^16}) +
    // (v_{i^8} + v_{i^24})) + ..., but instead of 29 separate butterflies (145 shuffle steps) the lanes split the sums
    // between them as they go: at the step with partner lane ^ m a lane keeps the sums whose index has its own bit m and
    // sends the others — 16 + 8 + 4 + 2 + 1 = 31 shuffle steps, the same additions on the same operands, the same bits
    // (item_sum below, evaluated depth first so that five partial sums are live at a time, not thirty-two).
    const double mine = item_sum<1, 0>(J, b, my_pos >= 0 ? 1.0 : 0.0, lane);
    if (lane < NSUM) job->partials[it * NSUM + lane] = mine;
}

// Residuals and sums of the work items that k_icp_match could not finish itself (some point was queued): the items of
// job->open_items, one warp each.
__global__ void __launch_bounds__(IWARPS * 32, 5) k_icp_accum(const IcpJob* __restrict__ job) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const ForestView F = job->F;
    WorkIter W(const_cast<int*>(&job->work[2]), (i64)job->n_open, lane, (int)(blockIdx.x * IWARPS + warp),
               (int)(gridDim.x * IWARPS), 1);
    i64 e;
    while (W.next(e)) {
        const int2 E = job->open_items[e];
        const i64 it = E.x;
        const int pair = E.y;
        const PairDesc P = job->pairs[pair];
        const int s0 = (int)(it - P.item_off) * ITEM_Q;
        const int count = P.n_src - s0 < ITEM_Q ? P.n_src - s0 : ITEM_Q;
        const TreeDesc& T = F.trees[P.tree];
        double cx = 0, cy = 0, cz = 0;
        int my_pos = -1;
        if (lane < count) {
            my_pos = job->match[it * ITEM_Q + lane];
            if (my_pos >= 0)
                transform_point(job->results[pair].transformation, reinterpret_cast<const double*>(P.src_pts + s0 + lane), cx, cy, cz);
        }
        accumulate_item(job, T, it, lane, my_pos, cx, cy, cz);
    }
}

// 6x6 symmetric solve by LDL^T with diagonal pivoting (Eigen's (J^T J).ldlt().solve, icp.hpp:120; the oracle's
// ldlt6_solve, same operation order): largest remaining diagonal entry first (first one on ties), symmetric swaps, and
// a pivot that is exactly zero leaves its component at zero, so a rank-deficient J^T J (planar target, fewer than
// six points) gives a finite step instead of 0/0.  Every index is a compile-time constant — the pivot row is swapped
// in by predicated exchanges — so the matrix stays in registers: one thread per pair and iteration runs this, and
// with dynamically indexed (local-memory) arrays the first touch of every line cost that thread ~14 us per pass.
__device__ __forceinline__ void cswap(bool c, double& x, double& y) {
    const double t = x;
    x = c ? y : x;
    y = c ? t : y;
}
// (one step of the elimination per template instance: written as one `for k` loop, the compiler left the swap loop of
// some k rolled — `.pragma "nounroll"` in the PTX — which made every index of it dynamic, put the matrix in local
// memory after all and cost k_icp_solve 683 local loads/stores on its one solving thread)
template <int K, int R>
__device__ __forceinline__ void ldlt_swap(int p, double (&a)[6][6], double (&y)[6], int (&perm)[6]) {
    if constexpr (R < 6) {
        const bool c = p == R;   // swap rows and columns K <-> R
#pragma unroll
        for (int j = 0; j < 6; ++j) cswap(c, a[K][j], a[R][j]);
#pragma unroll
        for (int i = 0; i < 6; ++i) cswap(c, a[i][K], a[i][R]);
        cswap(c, y[K], y[R]);
        const int t = perm[K];
        perm[K] = c ? perm[R] : perm[K];
        perm[R] = c ? t : perm[R];
        ldlt_swap<K, R + 1>(p, a, y, perm);
    }
}
template <int K>
__device__ __forceinline__ void ldlt_step(double (&a)[6][6], double (&y)[6], int (&perm)[6]) {
    if constexpr (K < 6) {
        int p = K;
        double best = fabs(a[K][K]);
#pragma unroll
        for (int i = K + 1; i < 6; ++i)
            if (fabs(a[i][i]) > best) { best = fabs(a[i][i]); p = i; }
        ldlt_swap<K, K + 1>(p, a, y, perm);
        const double d = a[K][K];
        if (d != 0.0) {
#pragma unroll
            for (int i = K + 1; i < 6; ++i) a[i][K] /= d;  // column K of L
#pragma unroll
            for (int i = K + 1; i < 6; ++i)
#pragma unroll
                for (int j = K + 1; j <= i; ++j) {
                    a[i][j] -= a[i][K] * d * a[j][K];
                    a[j][i] = a[i][j];
                }
        }
        ldlt_step<K + 1>(a, y, perm);
    }
}
__device__ __forceinline__ void ldlt6_solve(const double (&Ain)[6][6], const double (&bin)[6], double (&x)[6]) {
    double a[6][6], y[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        y[i] = bin[i];   // permuted along with the rows: y = P b
#pragma unroll
        for (int j = 0; j < 6; ++j) a[i][j] = Ain[i][j];
    }
    int perm[6] = {0, 1, 2, 3, 4, 5};
    ldlt_step<0>(a, y, perm);
#pragma unroll
    for (int i = 0; i < 6; ++i)  // L y' = P b
#pragma unroll
        for (int j = 0; j < i; ++j) y[i] -= a[i][j] * y[j];
#pragma unroll
    for (int i = 0; i < 6; ++i) y[i] = a[i][i] == 0.0 ? 0.0 : y[i] / a[i][i];  // D z = y'
#pragma unroll
    for (int i = 5; i >= 0; --i)  // L^T w = z
#pragma unroll
        for (int j = i + 1; j < 6; ++j) y[i] -= a[j][i] * y[j];
#pragma unroll
    for (int o = 0; o < 6; ++o) {   // x = P^T w: x[perm[i]] = y[i], as selects (a scatter would put x in local memory)
        double v = y[0];
#pragma unroll
        for (int i = 1; i < 6; ++i) v = perm[i] == o ? y[i] : v;
        x[o] = v;
    }
}

// x -> 4x4 row-major delta (icp.hpp:123-144)
__device__ __forceinline__ void delta_from_x(const double (&x)[6], double (&Dm)[16]) {
    double angle = sqrt((x[0] * x[0] + x[1] * x[1]) + x[2] * x[2]);  // icp.hpp:127
    double R[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
    if (!(angle < 1e-10)) {
        double ax = x[0] / angle, ay = x[1] / angle, az = x[2] / angle;
        double K[3][3] = {{0, -az, ay}, {az, 0, -ax}, {-ay, ax, 0}};
        double K2[3][3];
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                double s = 0;
#pragma unroll
                for (int k = 0; k < 3; ++k) s += K[i][k] * K[k][j];
                K2[i][j] = s;
            }
        double sn = sin(angle), cs = 1 - cos(angle);
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) R[i][j] = (R[i][j] + sn * K[i][j]) + cs * K2[i][j];
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) Dm[i] = (i % 5 == 0) ? 1.0 : 0.0;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = 0; j < 3; ++j) Dm[4 * i + j] = R[i][j];
        Dm[4 * i + 3] = x[3 + i];
    }
}

__device__ __forceinline__ void mat4_mul(const double (&A)[16], const double* B, double (&C)[16]) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            double s = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) s += A[4 * i + k] * B[4 * k + j];
            C[4 * i + j] = s;
        }
}

// One pair, one block of 256 threads.  mode 0: the end of a loop iteration (icp.hpp:198-232: error, convergence test,
// Gauss-Newton step); mode 1: the final error (icp.hpp:235-255).  Warp w adds the partials of the items w, w+8,
// w+16, ... in that order, warp 0 adds the eight warp sums in warp order — a fixed association, so the result is
// run-to-run, batch-composition and code-path independent (k_icp_solve and k_icp_tail both call this).
// The partials are read past L1 (__ldcg): in k_icp_tail other CTAs of the cluster rewrote them since the last pass.
__device__ __forceinline__ void solve_pair(IcpJob* __restrict__ job, int p, int mode, double (&s_part)[8][32]) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    PairState st;
    st.prev_error = __ldcg(&job->state[p].prev_error);
    st.state = __ldcg(&job->state[p].state);
    st.iter = __ldcg(&job->state[p].iter);
    sb_icp_result& R = job->results[p];
    if (mode == 1) {
        if (st.state == ST_CONVERGED) {
            if (threadIdx.x == 0) {  // broke out of the loop: the final pass repeats the last error (Appendix A.5)
                double e = R.error_history[R.history_len - 1];
                R.final_error = e;
                R.error_history[R.history_len] = e;
                R.history_len += 1;
                R.num_iterations = R.history_len - 1;  // icp.hpp:255
                job->state[p].state = ST_DONE;
            }
            return;
        }
        if (st.state != ST_EXHAUSTED) return;
    } else if (st.state != ST_ACTIVE) {
        return;
    }
    const PairDesc P = job->pairs[p];
    {
        double s = 0.0;
        if (lane < NSUM) {
            const double* base = job->partials + P.item_off * NSUM + lane;
            int i = warp;
            for (; i + 56 < P.n_items; i += 64) {  // eight loads in flight, additions in item order
                double v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = __ldcg(base + (i64)(i + 8 * u) * NSUM);
#pragma unroll
                for (int u = 0; u < 8; ++u) s += v[u];
            }
            for (; i + 24 < P.n_items; i += 32) {  // four
                const double v0 = __ldcg(base + (i64)i * NSUM), v1 = __ldcg(base + (i64)(i + 8) * NSUM),
                             v2 = __ldcg(base + (i64)(i + 16) * NSUM), v3 = __ldcg(base + (i64)(i + 24) * NSUM);
                s += v0; s += v1; s += v2; s += v3;
            }
            for (; i < P.n_items; i += 8) s += __ldcg(base + (i64)i * NSUM);
        }
        __syncthreads();  // the previous pair's sums have been consumed
        s_part[warp][lane] = s;
        __syncthreads();
    }
    if (warp != 0) return;
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += s_part[w][lane];
    double sr2 = shfl_d(s, 27);
    const double n_match = shfl_d(s, 28);
    double e = sqrt(sr2 / (double)P.n_src);  // icp.hpp:198-207
    if (mode == 1) {
        if (lane == 0) {
            if (n_match == 0.0) { R.status = SB_ERR_RANGE; R.converged = 0; }  // see the loop pass below
            R.final_error = e;
            R.error_history[R.history_len] = e;
            R.history_len += 1;
            R.num_iterations = R.history_len - 1;
            job->state[p].state = ST_DONE;
        }
        return;
    }
    double A[6][6], g[6];
    {
        int t = 0;
#pragma unroll
        for (int a2 = 0; a2 < 6; ++a2)
#pragma unroll
            for (int c = a2; c < 6; ++c) {
                double v = shfl_d(s, t);
                A[a2][c] = v;
                A[c][a2] = v;
                ++t;
            }
#pragma unroll
        for (int a2 = 0; a2 < 6; ++a2) g[a2] = shfl_d(s, 21 + a2);
    }
    if (lane == 0) {
        int hl = R.history_len;
        R.error_history[hl] = e;  // icp.hpp:207
        R.history_len = hl + 1;
        if (n_match == 0.0) {
            // not one source point has a nearest neighbour (every query or every target coordinate is NaN:
            // kdtree.hpp:125 never updates): the sums are empty and e = 0 would pass for convergence
            R.status = SB_ERR_RANGE;
            R.converged = 0;
            R.final_error = e;
            R.num_iterations = R.history_len - 1;
            job->state[p].state = ST_DONE;
            atomicSub(&job->n_active, 1);
        } else if (e < job->min_err || fabs(st.prev_error - e) < job->tol) {  // icp.hpp:210-217
            R.converged = 1;
            job->state[p].state = ST_CONVERGED;
            atomicSub(&job->n_active, 1);
        } else {
            double x[6], Dm[16], Tn[16];
            ldlt6_solve(A, g, x);
            delta_from_x(x, Dm);
            mat4_mul(Dm, R.transformation, Tn);  // total = delta * total, icp.hpp:229
            bool finite = true;
#pragma unroll
            for (int i = 0; i < 12; ++i) finite = finite && (fabs(Tn[i]) <= 1.7976931348623157e308);
            PairState ns;
            ns.prev_error = e;
            ns.iter = st.iter + 1;
            ns.state = ST_ACTIVE;
            if (!finite) {
                // NaN / Inf in the sums (non-finite input coordinates): the reference would carry the NaN on and
                // compare it against the tolerances; here the pair stops, unconverged, with a status to say why
                R.status = SB_ERR_RANGE;
                R.converged = 0;
                R.final_error = e;
                R.num_iterations = R.history_len - 1;
                ns.state = ST_DONE;
                atomicSub(&job->n_active, 1);
            } else {
#pragma unroll
                for (int i = 0; i < 16; ++i) R.transformation[i] = Tn[i];
                if (ns.iter >= job->max_it) {
                    ns.state = ST_EXHAUSTED;
                    atomicSub(&job->n_active, 1);
                }
            }
            job->state[p] = ns;
        }
    }
}

// mode 0: loop body for the pairs of the active list; mode 1: final error of every pair.  One block per pair.
__global__ void __launch_bounds__(256) k_icp_solve(IcpJob* __restrict__ job, int mode, cudaGraphConditionalHandle cond,
                                                   int use_cond) {
    __shared__ double s_part[8][32];
    const int n_loop = mode == 0 ? job->n_act : job->n_pairs;
    for (int a = blockIdx.x; a < n_loop; a += gridDim.x) {
        const int p = mode == 0 ? job->act_pair[a] : a;
        solve_pair(job, p, mode, s_part);
    }
    if (mode == 0) {
        // last block to finish decides whether the WHILE node runs another iteration
        __shared__ int s_last;
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) {
            int t = atomicAdd(&job->ticket, 1);
            s_last = (t == (int)gridDim.x - 1);
        }
        __syncthreads();
        if (s_last) {  // every other block's state updates are visible now
            __threadfence();
            const int active = *reinterpret_cast<volatile int*>(&job->n_active);
            // next pass: the pairs still iterating, or — once none is left — the final error pass of the pairs that
            // ran out of iterations (icp.hpp:235-252)
            build_active(job, active > 0 ? ST_ACTIVE : ST_EXHAUSTED, active > 0);
            if (threadIdx.x == 0) {
                job->ticket = 0;
                job->q_count = 0;
                job->n_open = 0;
                job->work[0] = job->work[1] = job->work[2] = 0;
                job->passes += 1;
                if (use_cond) cudaGraphSetConditional(cond, active > 0 ? 1u : 0u);
            }
        }
    }
}

// solve_point_to_plane on explicit correspondences (icp.hpp:89-144): one block, fixed-order reduction
__global__ void __launch_bounds__(256) k_solve_p2p(const double* __restrict__ src, const double* __restrict__ tgt,
                                                   const double* __restrict__ nrm, i64 n, double* __restrict__ out_T) {
    __shared__ double sm[8][NSUM];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double acc[NSUM];
#pragma unroll
    for (int i = 0; i < NSUM; ++i) acc[i] = 0.0;
    for (i64 i = threadIdx.x; i < n; i += 256) {
        double cx = src[3 * i], cy = src[3 * i + 1], cz = src[3 * i + 2];
        double tx = tgt[3 * i], ty = tgt[3 * i + 1], tz = tgt[3 * i + 2];
        double nx = nrm[3 * i], ny = nrm[3 * i + 1], nz = nrm[3 * i + 2];
        double J[6];
        J[0] = cy * nz - cz * ny; J[1] = cz * nx - cx * nz; J[2] = cx * ny - cy * nx;
        J[3] = nx; J[4] = ny; J[5] = nz;
        double b = ((tx - cx) * nx + (ty - cy) * ny) + (tz - cz) * nz;
        int t = 0;
#pragma unroll
        for (int a = 0; a < 6; ++a)
#pragma unroll
            for (int c = a; c < 6; ++c) acc[t++] += J[a] * J[c];
#pragma unroll
        for (int a = 0; a < 6; ++a) acc[21 + a] += J[a] * b;
        acc[27] += b * b;
    }
#pragma unroll
    for (int i = 0; i < NSUM; ++i) {
        double v = acc[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += shfl_d_xor(v, o);
        if (lane == 0) sm[warp][i] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double s[NSUM];
#pragma unroll
        for (int i = 0; i < NSUM; ++i) {
            double v = 0;
#pragma unroll
            for (int w = 0; w < 8; ++w) v += sm[w][i];
            s[i] = v;
        }
        double A[6][6], g[6], x[6], Dm[16];
        int t = 0;
#pragma unroll
        for (int a = 0; a < 6; ++a)
#pragma unroll
            for (int c = a; c < 6; ++c) { A[a][c] = s[t]; A[c][a] = s[t]; ++t; }
#pragma unroll
        for (int a = 0; a < 6; ++a) g[a] = s[21 + a];
        ldlt6_solve(A, g, x);
        delta_from_x(x, Dm);
#pragma unroll
        for (int i = 0; i < 16; ++i) out_T[i] = Dm[i];
    }
}

int solve_point_to_plane_dev(Ctx* ctx, const double* d_src, const double* d_tgt, const double* d_nrm, i64 n,
                             double* d_out_T) {
    SB_LAUNCH(ctx, k_solve_p2p, 1, 256, 0, d_src, d_tgt, d_nrm, n, d_out_T);
    return SB_OK;
}

// -------------------------------------------------------------------------------------------------------------
// host: graph construction + batch driver
// -------------------------------------------------------------------------------------------------------------
struct IcpGraph {
    IcpJob* d_job = nullptr;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    int iter_grid = 0, solve_grid = 0;
    unsigned long long* d_stats = nullptr;  // SB_ICP_STATS=1: per iteration bucket [queries, queued for the tree]
};

void icp_graph_free(Ctx* ctx) {
    IcpGraph* G = static_cast<IcpGraph*>(ctx->icp_graph);
    if (!G) return;
    if (G->exec) cudaGraphExecDestroy(G->exec);
    if (G->graph) cudaGraphDestroy(G->graph);
    if (G->d_stats) {
        unsigned long long h[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        cudaMemcpy(h, G->d_stats, sizeof(h), cudaMemcpyDeviceToHost);
        for (int b = 0; b < 4; ++b)
            fprintf(stderr, "[slam_b200] icp iterations %s: nearest-neighbour queries %llu, tree fallbacks %llu (%.3f %%)\n",
                    b == 0 ? "0" : b == 1 ? "1" : b == 2 ? "2-11" : ">=12", h[2 * b], h[2 * b + 1],
                    h[2 * b] ? 100.0 * (double)h[2 * b + 1] / (double)h[2 * b] : 0.0);
        cudaFree(G->d_stats);
    }
    cudaFree(G->d_job);
    delete G;
    ctx->icp_graph = nullptr;
}

static int add_kernel(Ctx* ctx, cudaGraph_t g, cudaGraphNode_t* node, const cudaGraphNode_t* dep, void* fn, int grid,
                      int block, void** args) {
    cudaKernelNodeParams kp = {};
    kp.func = fn;
    kp.gridDim = dim3((unsigned)grid, 1, 1);
    kp.blockDim = dim3((unsigned)block, 1, 1);
    kp.sharedMemBytes = 0;
    kp.kernelParams = args;
    kp.extra = nullptr;
    SB_CUDA(ctx, cudaGraphAddKernelNode(node, g, dep, dep ? 1 : 0, &kp));
    return SB_OK;
}

// match -> fallback -> accum -> solve(mode) appended to graph g after `dep` (may be null); *last = the solve node
static int add_pass(Ctx* ctx, IcpGraph* G, cudaGraph_t g, const cudaGraphNode_t* dep, int phase,
                    cudaGraphConditionalHandle cond, int use_cond, cudaGraphNode_t* last) {
    IcpJob* job = G->d_job;
    cudaGraphNode_t n_match, n_fb, n_acc;
    {
        void* args[] = {&job};
        SB_TRY(add_kernel(ctx, g, &n_match, dep, (void*)k_icp_match, G->iter_grid, IWARPS * 32, args));
    }
    {
        void* args[] = {&job};
        SB_TRY(add_kernel(ctx, g, &n_fb, &n_match, (void*)k_icp_fallback, G->iter_grid, IWARPS * 32, args));
    }
    {
        void* args[] = {&job};
        SB_TRY(add_kernel(ctx, g, &n_acc, &n_fb, (void*)k_icp_accum, G->iter_grid, IWARPS * 32, args));
    }
    {
        void* args[] = {&job, &phase, &cond, &use_cond};
        SB_TRY(add_kernel(ctx, g, last, &n_acc, (void*)k_icp_solve, G->solve_grid, 256, args));
    }
    return SB_OK;
}

static void icp_graph_destroy(IcpGraph* G) {
    if (G->exec) cudaGraphExecDestroy(G->exec);
    if (G->graph) cudaGraphDestroy(G->graph);
    cudaFree(G->d_stats);
    cudaFree(G->d_job);
    delete G;
}

static int icp_graph_build(Ctx* ctx, IcpGraph* G) {
    SB_CUDA(ctx, cudaMalloc(&G->d_job, sizeof(IcpJob)));
    // resident CTAs that take their work items from a counter (WorkIter): 8 per SM (SB_ICP_GRID; measured: 5 or 8
    // alike, 4 and 16 slower)
    G->iter_grid = ctx->sm_count * (getenv("SB_ICP_GRID") ? atoi(getenv("SB_ICP_GRID")) : 8);
    G->solve_grid = ctx->sm_count * 4;
    if (getenv("SB_ICP_STATS")) {
        SB_CUDA(ctx, cudaMalloc(&G->d_stats, 8 * sizeof(unsigned long long)));
        SB_CUDA(ctx, cudaMemset(G->d_stats, 0, 8 * sizeof(unsigned long long)));
    }
    if (getenv("SB_ICP_NOGRAPH")) return SB_OK;
    SB_CUDA(ctx, cudaGraphCreate(&G->graph, 0));
    cudaGraphConditionalHandle cond;
    SB_CUDA(ctx, cudaGraphConditionalHandleCreate(&cond, G->graph, 1, cudaGraphCondAssignDefault));
    IcpJob* job = G->d_job;
    int one = 1;
    cudaGraphNode_t n_init, n_while, n_body_last, n_final;
    {
        void* args[] = {&job, &cond, &one};
        SB_TRY(add_kernel(ctx, G->graph, &n_init, nullptr, (void*)k_icp_init, 1, 256, args));
    }
    cudaGraphNodeParams wp = {};
    wp.type = cudaGraphNodeTypeConditional;
    wp.conditional.handle = cond;
    wp.conditional.type = cudaGraphCondTypeWhile;
    wp.conditional.size = 1;
    SB_CUDA(ctx, cudaGraphAddNode(&n_while, G->graph, &n_init, 1, &wp));
    cudaGraph_t body = wp.conditional.phGraph_out[0];
    SB_TRY(add_pass(ctx, G, body, nullptr, 0, cond, 1, &n_body_last));       // icp.hpp:181-232
    SB_TRY(add_pass(ctx, G, G->graph, &n_while, 1, cond, 0, &n_final));      // icp.hpp:235-255
    SB_CUDA(ctx, cudaGraphInstantiate(&G->exec, G->graph, 0));
    return SB_OK;
}

// The loop graph of the context, built on first use.  It is cached only once it is complete: a failure on the way
// (no conditional-node support in the driver, out of memory) is reported and leaves nothing half-built behind.
static int icp_graph_get(Ctx* ctx, IcpGraph** out) {
    if (ctx->icp_graph) {
        *out = static_cast<IcpGraph*>(ctx->icp_graph);
        return SB_OK;
    }
    IcpGraph* G = new IcpGraph();
    const int s = icp_graph_build(ctx, G);
    if (s != SB_OK) {
        icp_graph_destroy(G);
        return s;
    }
    ctx->icp_graph = G;
    *out = G;
    return SB_OK;
}

// Enqueues the registration of `pairs_in` on ctx->stream and the copy of its results into the context's pinned result
// buffer; returns without waiting.  Several batches may be enqueued back to back (they share one device-resident
// IcpJob: stream order keeps them apart); icp_collect waits for all of them.
int icp_enqueue(Ctx* ctx, const Forest* f, const std::vector<PairDesc>& pairs_in, const sb_icp_config* cfg,
                IcpPending* out) {
    const int n_pairs = (int)pairs_in.size();
    out->n_pairs = n_pairs;
    out->h_off = ctx->icp_res_used;
    out->slot = -1;
    out->d_res = nullptr;
    if (n_pairs == 0) return SB_OK;
    if (cfg->max_iterations < 0 || cfg->max_iterations > SB_MAX_ICP_ITERATIONS)
        return fail(ctx, SB_ERR_INVALID_ARG, "icp: max_iterations %d outside [0, %d]", cfg->max_iterations,
                    SB_MAX_ICP_ITERATIONS);
    if (f->normals_k <= 0) return fail(ctx, SB_ERR_INVALID_ARG, "icp: forest has no normals");
    // staging for the results and the pass count: checked before anything is enqueued, so that a batch that cannot be
    // staged launches nothing
    if (ctx->icp_res_used + (size_t)n_pairs > ctx->icp_res_cap || ctx->icp_slots_used >= Ctx::ICP_SLOTS)
        return fail(ctx, SB_ERR_CAPACITY, "icp: result staging full (icp_reserve_results sizes it per call)");
    IcpGraph* G;
    SB_TRY(icp_graph_get(ctx, &G));
    std::vector<PairDesc> pairs(pairs_in);
    int n_valid = 0;
    i64 n_items = 0;
    for (int p = 0; p < n_pairs; ++p) {
        PairDesc& P = pairs[p];
        if (P.tree < 0 || P.tree >= f->n_trees || P.src_tree < 0 || P.src_tree >= f->n_trees)
            return fail(ctx, SB_ERR_INVALID_ARG, "icp: pair %d names a tree outside the forest", p);
        const TreeDesc& Tt = f->h_trees[(size_t)P.tree];
        const TreeDesc& Ts = f->h_trees[(size_t)P.src_tree];
        if (Tt.n > 0 && (!Tt.nrm || !Tt.nbr || !Tt.grid))
            return fail(ctx, SB_ERR_INVALID_ARG, "icp: target tree %d has no normals", P.tree);
        P.src_pts = Ts.pts + Ts.pt_off;
        P.n_src = Ts.n;
        P.item_off = n_items;
        P.n_items = P.n_src > 0 ? (P.n_src + ITEM_Q - 1) / ITEM_Q : 0;
        n_items += P.n_items;
        if (P.n_src > 0 && f->h_trees[P.tree].n > 0) ++n_valid;
    }
    if (n_items * ITEM_Q >= 0x7fffffffLL) return fail(ctx, SB_ERR_RANGE, "icp: more than 2^31 source points in one batch");
    PairDesc* d_pairs;
    int* d_match;
    sb_icp_result* d_res;
    PairState* d_state;
    double* d_part;
    int* d_act_pair;
    i64* d_act_off;
    size_t ni = (size_t)(n_items > 0 ? n_items : 1);
    SB_TRY(arena_get(ctx, (size_t)n_pairs, &d_pairs));
    SB_TRY(arena_get(ctx, ni * ITEM_Q, &d_match));
    SB_TRY(arena_get(ctx, (size_t)n_pairs, &d_res));
    SB_TRY(arena_get(ctx, (size_t)n_pairs, &d_state));
    SB_TRY(arena_get(ctx, ni * NSUM, &d_part));
    FallbackEntry* d_queue;
    int2* d_open;
    SB_TRY(arena_get(ctx, ni * ITEM_Q, &d_queue));
    SB_TRY(arena_get(ctx, ni, &d_open));
    SB_TRY(arena_get(ctx, (size_t)n_pairs, &d_act_pair));
    SB_TRY(arena_get(ctx, (size_t)n_pairs + 1, &d_act_off));
    SB_CUDA(ctx, cudaMemcpyAsync(d_pairs, pairs.data(), sizeof(PairDesc) * n_pairs, cudaMemcpyHostToDevice, ctx->stream));
    SB_CUDA(ctx, cudaMemsetAsync(d_match, 0xff, sizeof(int) * ni * ITEM_Q, ctx->stream));  // -1: no correspondence yet
    IcpJob job;
    memset(&job, 0, sizeof(job));
    job.F.trees = f->d_trees;
    job.nbr_k = f->normals_k;
    job.stats = G->d_stats;
    job.match = d_match;
    job.n_items = n_items;
    job.pairs = d_pairs;
    job.results = d_res;
    out->d_res = d_res;
    job.state = d_state;
    job.partials = d_part;
    job.queue = d_queue;
    job.open_items = d_open;
    job.n_open = 0;
    job.q_count = 0;
    job.act_pair = d_act_pair;
    job.act_off = d_act_off;
    memcpy(job.T0, cfg->initial_transform, sizeof(job.T0));
    job.tol = cfg->tolerance;
    job.min_err = cfg->min_error;
    job.n_pairs = n_pairs;
    job.max_it = cfg->max_iterations;
    job.n_active = cfg->max_iterations > 0 ? n_valid : 0;
    job.ticket = 0;
    static const int packet_min = getenv("SB_ICP_PACKET_MIN") ? atoi(getenv("SB_ICP_PACKET_MIN")) : 6;
    job.packet_min = packet_min;
    SB_CUDA(ctx, cudaMemcpyAsync(G->d_job, &job, sizeof(job), cudaMemcpyHostToDevice, ctx->stream));
    if (G->exec) {
        SB_CUDA(ctx, cudaGraphLaunch(G->exec, ctx->stream));
    } else {  // debugging / profiling path (SB_ICP_NOGRAPH=1): same kernels, host-driven loop
        cudaGraphConditionalHandle none = 0;
        SB_LAUNCH(ctx, k_icp_init, 1, 256, 0, G->d_job, none, 0);
        for (int it = 0; it < cfg->max_iterations; ++it) {
            if ((it & 3) == 0) {  // the graph decides after every pass; looking every fourth pass gives the same results
                int active = 0;
                SB_CUDA(ctx, cudaMemcpyAsync(&active, &G->d_job->n_active, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
                SB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
                if (active <= 0) break;
            }
            SB_LAUNCH(ctx, k_icp_match, G->iter_grid, IWARPS * 32, 0, G->d_job);
            SB_LAUNCH(ctx, k_icp_fallback, G->iter_grid, IWARPS * 32, 0, G->d_job);
            SB_LAUNCH(ctx, k_icp_accum, G->iter_grid, IWARPS * 32, 0, G->d_job);
            SB_LAUNCH(ctx, k_icp_solve, G->solve_grid, 256, 0, G->d_job, 0, none, 0);
        }
        SB_LAUNCH(ctx, k_icp_match, G->iter_grid, IWARPS * 32, 0, G->d_job);
        SB_LAUNCH(ctx, k_icp_fallback, G->iter_grid, IWARPS * 32, 0, G->d_job);
        SB_LAUNCH(ctx, k_icp_accum, G->iter_grid, IWARPS * 32, 0, G->d_job);
        SB_LAUNCH(ctx, k_icp_solve, G->solve_grid, 256, 0, G->d_job, 1, none, 0);
    }
    // results and the pass count: into pinned host memory, asynchronously
    out->slot = ctx->icp_slots_used++;
    ctx->icp_res_used += (size_t)n_pairs;
    SB_CUDA(ctx, cudaMemcpyAsync(ctx->h_icp_res + out->h_off, d_res, sizeof(sb_icp_result) * n_pairs, cudaMemcpyDeviceToHost,
                                 ctx->stream));
    SB_CUDA(ctx, cudaMemcpyAsync(ctx->h_icp_passes + out->slot, &G->d_job->passes, sizeof(int), cudaMemcpyDeviceToHost,
                                 ctx->stream));
    return SB_OK;
}

// Pinned staging for the results of all batches enqueued until the next icp_collect (n_pairs in total).
int icp_reserve_results(Ctx* ctx, size_t n_pairs) {
    ctx->icp_res_used = 0;
    ctx->icp_slots_used = 0;
    if (!ctx->h_icp_passes) SB_CUDA(ctx, cudaHostAlloc(&ctx->h_icp_passes, sizeof(int) * Ctx::ICP_SLOTS, cudaHostAllocDefault));
    if (n_pairs > ctx->icp_res_cap) {
        if (ctx->h_icp_res) cudaFreeHost(ctx->h_icp_res);
        ctx->h_icp_res = nullptr;
        ctx->icp_res_cap = 0;
        size_t cap = n_pairs < 64 ? 64 : n_pairs;
        SB_CUDA(ctx, cudaHostAlloc(&ctx->h_icp_res, sizeof(sb_icp_result) * cap, cudaHostAllocDefault));
        ctx->icp_res_cap = cap;
    }
    return SB_OK;
}

// Waits for the stream the batches were enqueued on and hands their results out: pending[i]'s pair j goes to
// results[ids[i][j]] (ids[i] == nullptr: results[offset so far + j]).
int icp_collect(Ctx* ctx, cudaStream_t stream, const std::vector<IcpPending>& pending, const std::vector<const int*>& ids,
                sb_icp_result* results) {
    SB_CUDA(ctx, cudaStreamSynchronize(stream));
    IcpGraph* G = static_cast<IcpGraph*>(ctx->icp_graph);
    int max_hist = 1;
    size_t seq = 0;
    for (size_t b = 0; b < pending.size(); ++b) {
        const IcpPending& P = pending[b];
        for (int j = 0; j < P.n_pairs; ++j) {
            const sb_icp_result& r = ctx->h_icp_res[P.h_off + (size_t)j];
            results[ids[b] ? (size_t)ids[b][j] : seq + (size_t)j] = r;
            if (r.history_len > max_hist) max_hist = r.history_len;
        }
        seq += (size_t)P.n_pairs;
        if (P.slot >= 0 && G && G->exec) ctx->launches += 5 + 4 * (i64)ctx->h_icp_passes[P.slot];  // init + 4 per pass + 4 final
    }
    ctx->last_icp_iterations = max_hist;
    return SB_OK;
}

int icp_batch(Ctx* ctx, const Forest* f, const std::vector<PairDesc>& pairs_in, const sb_icp_config* cfg,
              sb_icp_result* results, const std::function<int()>* after_launch) {
    if (pairs_in.empty()) return SB_OK;
    SB_TRY(icp_reserve_results(ctx, pairs_in.size()));
    std::vector<IcpPending> pending(1);
    SB_TRY(icp_enqueue(ctx, f, pairs_in, cfg, &pending[0]));
    if (after_launch && *after_launch) SB_TRY((*after_launch)());
    return icp_collect(ctx, ctx->stream, pending, std::vector<const int*>(1, nullptr), results);
}

}  // namespace sb
