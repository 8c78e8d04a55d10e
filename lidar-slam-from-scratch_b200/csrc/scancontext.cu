// scancontext.cu — Scan Context descriptor build and column-shift distance search; replaces
// slam::ScanContext::compute / distance / column_shifted_distance / ring_key / sector_key
// (slam_viz/include/slam_viz/core/scan_context.hpp:44-82, 90-102, 121-142, 107-118).
//
// Build: one CTA per cloud, 1200 shared-memory bins, atomicMax on the order-preserving integer image of z, so the
// result is exact and independent of the order in which points arrive.  Range/sector use the reference's fp64
// expressions (sqrt, atan2 + pi, division by the bin size, truncation, clamp).
// Search: one (database entry, shift) pair per thread.  Each thread walks the 1200 cells in the reference's order
// (ring outer, sector inner) with separately rounded multiply and add (this file is compiled with -fmad=false), so
// sum_ab, sum_aa and sum_bb — and therefore the distance — are bit-identical to the scalar reference; the minimum
// over the 60 shifts is an exact reduction.  The query and the entry are staged ring-major in shared memory, so a
// warp's 32 shifts read 32 consecutive doubles (no bank conflicts) and the query cell is a broadcast.
#include "common.cuh"

namespace sb {

static constexpr int RINGS = SB_SC_RINGS, SECTORS = SB_SC_SECTORS, CELLS = SB_SC_SIZE;

__global__ void __launch_bounds__(256) k_sc_compute(const double* __restrict__ xyz, const i64* __restrict__ off,
                                                    double* __restrict__ desc) {
    __shared__ long long bins[CELLS];
    const int c = blockIdx.x;
    const long long empty = ordered_from_double(-1.7976931348623157e308);  // scan_context.hpp:46
    for (int t = threadIdx.x; t < CELLS; t += blockDim.x) bins[t] = empty;
    __syncthreads();
    const double ring_size = 80.0 / RINGS;                            // scan_context.hpp:47
    const double sector_size = 2.0 * 3.14159265358979323846 / SECTORS;  // scan_context.hpp:48
    const i64 b = off[c], e = off[c + 1];
    for (i64 i = b + threadIdx.x; i < e; i += blockDim.x) {
        double x = xyz[3 * i], y = xyz[3 * i + 1], z = xyz[3 * i + 2];
        double range = sqrt(x * x + y * y);                       // scan_context.hpp:56
        double angle = atan2(y, x) + 3.14159265358979323846;      // scan_context.hpp:57
        if (range > 80.0 || range < 0.1) continue;                // scan_context.hpp:59
        int ring = (int)(range / ring_size);                      // scan_context.hpp:62
        int sector = (int)(angle / sector_size);                  // scan_context.hpp:63
        ring = min(max(ring, 0), RINGS - 1);                      // scan_context.hpp:65-66
        sector = min(max(sector, 0), SECTORS - 1);
        if (z == z) atomicMax(&bins[sector * RINGS + ring], ordered_from_double(z));  // scan_context.hpp:69-71
    }
    __syncthreads();
    for (int t = threadIdx.x; t < CELLS; t += blockDim.x) {
        double v = double_from_ordered(bins[t]);
        if (v < -1000.0) v = 0.0;  // scan_context.hpp:77-81
        desc[(i64)c * CELLS + t] = v;  // column-major 20x60: (ring i, sector j) at j*20 + i
    }
}

int sc_compute_dev(Ctx* ctx, const double* d_xyz, const i64* d_off, int n_clouds, double* d_desc) {
    if (n_clouds <= 0) return SB_OK;
    SB_LAUNCH(ctx, k_sc_compute, (unsigned)n_clouds, 256, 0, d_xyz, d_off, d_desc);
    return SB_OK;
}

// ---------------------------------------------------------------------------------------------------------------
static constexpr int ENTRIES_PER_CTA = 2;

__global__ void __launch_bounds__(64 * ENTRIES_PER_CTA) k_sc_distance(const double* __restrict__ query,
                                                                      const double* __restrict__ db, int n_db,
                                                                      double* __restrict__ out) {
    __shared__ double sa[CELLS];                      // query, ring-major: (i, j) at i*60 + j
    __shared__ double sb_[ENTRIES_PER_CTA][CELLS];    // entries, ring-major
    __shared__ double smin[ENTRIES_PER_CTA][2];
    const int sub = threadIdx.x >> 6;       // entry within the CTA
    const int s = threadIdx.x & 63;         // shift handled by this thread (60..63 idle)
    const int entry = blockIdx.x * ENTRIES_PER_CTA + sub;
    for (int t = threadIdx.x; t < CELLS; t += blockDim.x) {
        int j = t / RINGS, i = t - j * RINGS;
        sa[i * SECTORS + j] = query[t];
    }
    if (entry < n_db) {
        const double* g = db + (i64)entry * CELLS;
        for (int t = s; t < CELLS; t += 64) {
            int j = t / RINGS, i = t - j * RINGS;
            sb_[sub][i * SECTORS + j] = g[t];
        }
    }
    __syncthreads();
    double d = 1.7976931348623157e308;
    if (entry < n_db && s < SECTORS) {
        double sum_ab = 0.0, sum_aa = 0.0, sum_bb = 0.0;
        const double* B = sb_[sub];
        for (int i = 0; i < RINGS; ++i) {           // scan_context.hpp:126-135, same order
            const double* ar = sa + i * SECTORS;
            const double* br = B + i * SECTORS;
            int jj = s;
#pragma unroll 4
            for (int j = 0; j < SECTORS; ++j) {
                double a = ar[j];
                double b = br[jj];
                sum_ab += a * b;
                sum_aa += a * a;
                sum_bb += b * b;
                jj = jj + 1 == SECTORS ? 0 : jj + 1;
            }
        }
        double norm = sqrt(sum_aa) * sqrt(sum_bb);                 // scan_context.hpp:137
        d = norm < 1e-10 ? 1.0 : 1.0 - sum_ab / norm;             // scan_context.hpp:138-141
        if (!(d == d)) d = 1.7976931348623157e308;                 // NaN never wins `dist < min_dist` (:96)
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) d = fmin(d, shfl_d_xor(d, o));
    if ((threadIdx.x & 31) == 0) smin[sub][(threadIdx.x >> 5) & 1] = d;
    __syncthreads();
    if (entry < n_db && s == 0) out[entry] = fmin(smin[sub][0], smin[sub][1]);  // scan_context.hpp:93-99
}

int sc_distance_dev(Ctx* ctx, const double* d_query_desc, const double* d_db, int n_db, double* d_out) {
    if (n_db <= 0) return SB_OK;
    SB_LAUNCH(ctx, k_sc_distance, (unsigned)ceil_div(n_db, ENTRIES_PER_CTA), 64 * ENTRIES_PER_CTA, 0, d_query_desc,
              d_db, n_db, d_out);
    return SB_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Many queries against one database (sb_loop_candidates_batch / sb_loop_detect_batch).
//
// k_sc_distance's three sums per (query, entry, shift) are not all pair sums: sum_bb(e, s) = sum of b(i, (j+s) % 60)^2
// in ring-outer, sector-inner order depends on the entry and the shift only, and sum_aa(q) is that same sum for the
// query descriptor at shift 0.  k_sc_sq computes them once per descriptor with the very loop of k_sc_distance (same
// operands, same order, separately rounded), so the batch kernel below needs only sum_ab and its distances are the
// same bits.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(64) k_sc_sq(const double* __restrict__ desc, double* __restrict__ sq) {
    __shared__ double sb_[CELLS];   // ring-major
    const int e = blockIdx.x, s = threadIdx.x;
    const double* g = desc + (i64)e * CELLS;
    for (int t = s; t < CELLS; t += 64) {
        int j = t / RINGS, i = t - j * RINGS;
        sb_[i * SECTORS + j] = g[t];
    }
    __syncthreads();
    if (s >= SECTORS) return;
    double sum_bb = 0.0;
    for (int i = 0; i < RINGS; ++i) {
        const double* br = sb_ + i * SECTORS;
        int jj = s;
#pragma unroll 4
        for (int j = 0; j < SECTORS; ++j) {
            double b = br[jj];
            sum_bb += b * b;
            jj = jj + 1 == SECTORS ? 0 : jj + 1;
        }
    }
    sq[(i64)e * SECTORS + s] = sum_bb;
}

int sc_sq_dev(Ctx* ctx, const double* d_desc, int n, double* d_sq) {
    if (n <= 0) return SB_OK;
    SB_LAUNCH(ctx, k_sc_sq, (unsigned)n, 64, 0, d_desc, d_sq);
    return SB_OK;
}

// Tile: SC_TQ queries x SC_TE entries per CTA, both staged ring-major in shared memory (9.6 KB per descriptor).
// Thread (query half h, entry e, shift group g) accumulates sum_ab for its SC_QT = SC_TQ / 2 queries and the four
// shifts g, g + 15, g + 30, g + 45 of entry e: 16 independent accumulators, per cell 4 query loads (the same address
// for the lanes of a warp: broadcasts) and 4 entry loads (15 consecutive doubles per entry: no bank conflicts) feed
// 16 DMUL + 16 DADD.  The cell order is the reference's (ring outer, sector inner), one accumulator per
// (query, shift), so every sum_ab is the same sequence of roundings as in k_sc_distance.
static constexpr int SC_TQ = 8, SC_TE = 8, SC_QT = SC_TQ / 2, SC_SG = SECTORS / 4;
static constexpr int SC_MANY_THREADS = 2 * SC_TE * SC_SG;   // 240
static constexpr size_t SC_MANY_SMEM = sizeof(double) * CELLS * (SC_TQ + SC_TE) + sizeof(double) * 64;

// dist[r * ld + e] for query r of the group (slot qslot[r]) and every entry e < qslot[r] whose tile survives: a tile is
// skipped when none of its (query, entry) pairs is causal (e < q) and passes the frame gap (the same int expression as
// the selection, k_loop_select); distances of pairs the selection filters out are never read.
__global__ void __launch_bounds__(SC_MANY_THREADS, 1) k_sc_distance_many(const double* __restrict__ desc,
                                                                     const double* __restrict__ sq,
                                                                     const int2* __restrict__ meta,
                                                                     const int* __restrict__ qslot, int n_q, int frame_gap,
                                                                     double* __restrict__ dist, i64 ld) {
    extern __shared__ double smem[];
    double* sa = smem;                    // [SC_TQ][RINGS][SECTORS]
    double* sb_ = smem + SC_TQ * CELLS;   // [SC_TE][RINGS][SECTORS]
    // [SC_TQ][SC_TE] minima over the shifts, as order-preserving unsigned images (atomicMin)
    unsigned long long* smin_u = reinterpret_cast<unsigned long long*>(sb_ + SC_TE * CELLS);
    __shared__ int s_q[SC_TQ];
    const int q0 = blockIdx.y * SC_TQ, e0 = blockIdx.x * SC_TE;
    const int tid = threadIdx.x;
    if (tid < SC_TQ) s_q[tid] = q0 + tid < n_q ? qslot[q0 + tid] : -1;
    __syncthreads();
    bool live = false;
    if (tid < SC_TQ * SC_TE) {
        const int q = s_q[tid / SC_TE], e = e0 + tid % SC_TE;
        live = q >= 0 && e < q && meta[q].x - meta[e].x >= frame_gap;   // loop_closure.hpp:79-81
    }
    if (!__syncthreads_or(live)) return;
    int q_hi = 0;
#pragma unroll
    for (int r = 0; r < SC_TQ; ++r) q_hi = max(q_hi, s_q[r]);
    const int n_e = min(SC_TE, q_hi - e0);   // entries of the tile below the last query (>= 1: the tile is live)
    for (int t = tid; t < SC_TQ * CELLS; t += SC_MANY_THREADS) {
        const int r = t / CELLS, c = t - r * CELLS;
        const int j = c / RINGS, i = c - j * RINGS;
        sa[r * CELLS + i * SECTORS + j] = s_q[r] >= 0 ? desc[(i64)s_q[r] * CELLS + c] : 0.0;
    }
    for (int t = tid; t < SC_TE * CELLS; t += SC_MANY_THREADS) {
        const int r = t / CELLS, c = t - r * CELLS;
        const int j = c / RINGS, i = c - j * RINGS;
        sb_[r * CELLS + i * SECTORS + j] = r < n_e ? desc[(i64)(e0 + r) * CELLS + c] : 0.0;
    }
    if (tid < SC_TQ * SC_TE) smin_u[tid] = ~0ull;
    __syncthreads();
    const int g = tid % SC_SG, el = (tid / SC_SG) % SC_TE, h = tid / (SC_SG * SC_TE);
    if (el < n_e) {
        double acc[SC_QT][4];
#pragma unroll
        for (int r = 0; r < SC_QT; ++r)
#pragma unroll
            for (int k = 0; k < 4; ++k) acc[r][k] = 0.0;
        const double* A = sa + h * SC_QT * CELLS;
        const double* B = sb_ + el * CELLS;
        for (int i = 0; i < RINGS; ++i) {           // scan_context.hpp:126-135, same order
            const double* ar = A + i * SECTORS;
            const double* br = B + i * SECTORS;
            int jj = g;                              // column of shift g; shift g + 15k reads column jj + 15k (mod 60)
#pragma unroll 2
            for (int j = 0; j < SECTORS; ++j) {
                double b[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    int c = jj + 15 * k;
                    b[k] = br[c >= SECTORS ? c - SECTORS : c];
                }
#pragma unroll
                for (int r = 0; r < SC_QT; ++r) {
                    const double a = ar[r * CELLS + j];
#pragma unroll
                    for (int k = 0; k < 4; ++k) acc[r][k] += a * b[k];
                }
                jj = jj + 1 == SECTORS ? 0 : jj + 1;
            }
        }
        const int e = e0 + el;
#pragma unroll
        for (int r = 0; r < SC_QT; ++r) {
            const int qr = h * SC_QT + r;
            const int q = s_q[qr];
            if (q < 0) continue;
            const double sum_aa = sq[(i64)q * SECTORS];
            double d = 1.7976931348623157e308;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const double sum_bb = sq[(i64)e * SECTORS + g + 15 * k];
                double norm = sqrt(sum_aa) * sqrt(sum_bb);                     // scan_context.hpp:137
                double dk = norm < 1e-10 ? 1.0 : 1.0 - acc[r][k] / norm;       // scan_context.hpp:138-141
                if (!(dk == dk)) dk = 1.7976931348623157e308;                  // NaN never wins (:96)
                d = fmin(d, dk);
            }
            // the min over the 60 shifts (scan_context.hpp:93-99): 15 lanes of this (query, entry) — an exact reduction
            atomicMin(smin_u + qr * SC_TE + el, (unsigned long long)ordered_from_double(d) ^ 0x8000000000000000ull);
        }
    }
    __syncthreads();
    if (tid < SC_TQ * SC_TE) {
        const int qr = tid / SC_TE, e = tid % SC_TE;
        if (s_q[qr] >= 0 && e < n_e) {
            const unsigned long long u = smin_u[tid];
            dist[(i64)(q0 + qr) * ld + e0 + e] = double_from_ordered((long long)(u ^ 0x8000000000000000ull));
        }
    }
}

int sc_distance_many_dev(Ctx* ctx, const double* d_desc, const double* d_sq, const int2* d_meta, const int* d_qslot,
                         int n_q, int n_e, int frame_gap, double* d_dist, i64 ld) {
    if (n_q <= 0 || n_e <= 0) return SB_OK;
    SB_CUDA(ctx, cudaFuncSetAttribute(k_sc_distance_many, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SC_MANY_SMEM));
    dim3 grid((unsigned)ceil_div(n_e, SC_TE), (unsigned)ceil_div(n_q, SC_TQ));
    SB_LAUNCH(ctx, k_sc_distance_many, grid, SC_MANY_THREADS, SC_MANY_SMEM, d_desc, d_sq, d_meta, d_qslot, n_q,
              frame_gap, d_dist, ld);
    return SB_OK;
}

// ring_key: row means over the 60 sectors; sector_key: column means over the 20 rings (scan_context.hpp:107-118)
__global__ void k_sc_keys(const double* __restrict__ desc, double* __restrict__ ring_key, double* __restrict__ sector_key) {
    int t = threadIdx.x;
    if (t < RINGS) {
        double s = 0.0;
        for (int j = 0; j < SECTORS; ++j) s += desc[j * RINGS + t];
        ring_key[t] = s / (double)SECTORS;
    } else if (t < RINGS + SECTORS) {
        int j = t - RINGS;
        double s = 0.0;
        for (int i = 0; i < RINGS; ++i) s += desc[j * RINGS + i];
        sector_key[j] = s / (double)RINGS;
    }
}

int sc_keys_dev(Ctx* ctx, const double* d_desc, double* d_ring, double* d_sector) {
    SB_LAUNCH(ctx, k_sc_keys, 1, 96, 0, d_desc, d_ring, d_sector);
    return SB_OK;
}

}  // namespace sb
