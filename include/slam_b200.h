/* slam_b200.h — C ABI of the B200 (sm_100a) scan-registration engine.
 *
 * This is the drop-in boundary for the data-parallel front end of kaushik884/LiDAR-SLAM-from-scratch.  The
 * reference has no FFI: its hot path is the header-only C++ API in namespace slam (slam_viz/include/slam_viz/core/)
 * called from slam_viz/src/ros/slam_node.cpp.  Every entry point below names the reference interface it replaces
 * (paths relative to the reference root).  The C++17 header mirror that keeps the reference's class and function
 * names on top of this ABI lives in lidar-slam-from-scratch_b200/host/slam_viz/core/.
 *
 * Conventions
 *   - extern "C", POD only, no exceptions cross the ABI.  Every function returns an sb_status (0 = SB_OK);
 *     sb_last_error(ctx) gives the message of the last failure on that context.
 *   - Point clouds are row-major contiguous fp64 xyz (exactly PointCloud::Matrix::data(), types.hpp:17).
 *   - Functions without a _dev suffix take HOST pointers and return to HOST buffers owned by the caller (value
 *     semantics like the reference).  *_dev functions take DEVICE pointers on the context's device and enqueue on the
 *     context's stream without synchronising unless stated.
 *   - A context (one per host thread and device) owns the stream, the workspace arena and all index/database
 *     objects created from it.  There is NO CPU fallback: if no sm_100-class device is usable, sb_ctx_create fails.
 */
#ifndef SLAM_B200_H
#define SLAM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum sb_status {
    SB_OK = 0,
    SB_ERR_INVALID_ARG = 1,   /* null pointer, negative size, k out of range ...                                  */
    SB_ERR_EMPTY = 2,         /* empty cloud where the reference would be undefined behaviour (kdtree.hpp:25,119) */
    SB_ERR_CUDA = 3,          /* a CUDA runtime call failed; message in sb_last_error                              */
    SB_ERR_NO_DEVICE = 4,     /* no usable CUDA device                                                             */
    SB_ERR_RANGE = 5,         /* voxel keys of one call span more than 2^63 packed cells, or non-finite input      */
    SB_ERR_CAPACITY = 6       /* caller-provided output capacity too small                                         */
} sb_status;

typedef struct sb_ctx sb_ctx;
typedef struct sb_index sb_index;   /* replaces slam::KDTree / NearestNeighborSearch (kdtree.hpp:18-221)          */
typedef struct sb_loop sb_loop;     /* replaces slam::LoopClosureDetector (loop_closure.hpp:41-149)               */

#define SB_SC_RINGS 20              /* scan_context.hpp:27 */
#define SB_SC_SECTORS 60            /* scan_context.hpp:28 */
#define SB_SC_SIZE 1200
#define SB_MAX_K 32                 /* largest k of sb_index_knn / sb_estimate_normals                            */
#define SB_MAX_ICP_ITERATIONS 128   /* largest ICPConfig::max_iterations; history holds max_iterations + 1 values */

/* slam::ICPConfig (types.hpp:143-148) + the normals k that icp.hpp:170 hard-codes to 20. */
typedef struct sb_icp_config {
    int32_t max_iterations;       /* 50   */
    int32_t normals_k;            /* 20   */
    double tolerance;             /* 1e-6 */
    double min_error;             /* 1e-9 */
    double initial_transform[16]; /* row-major 4x4, identity */
} sb_icp_config;

/* slam::ICPResult (types.hpp:155-164). */
typedef struct sb_icp_result {
    double transformation[16];    /* row-major 4x4 */
    double final_error;
    int32_t converged;
    int32_t num_iterations;       /* = history_len - 1 (icp.hpp:255) */
    int32_t history_len;
    int32_t status;               /* per-pair sb_status in batch calls */
    double error_history[SB_MAX_ICP_ITERATIONS + 1];
} sb_icp_result;

/* slam::LoopClosureConfig (loop_closure.hpp:14-19) + the constants loop_closure.hpp:105-107 / icp.hpp:170 hard-code. */
typedef struct sb_loop_config {
    int32_t frame_gap;              /* 50   */
    int32_t max_candidates;         /* 3    */
    double sc_distance_threshold;   /* 0.25 */
    double icp_fitness_threshold;   /* 0.3  */
    int32_t icp_max_iterations;     /* 30   */
    int32_t normals_k;              /* 20   */
    double icp_tolerance;           /* 1e-6 */
    int32_t verify_chunk;           /* candidates ICP-verified concurrently per round (0 -> max_candidates)      */
    int32_t reserved;
} sb_loop_config;

/* slam::LoopClosureResult (loop_closure.hpp:25-31). */
typedef struct sb_loop_result {
    int32_t query_frame;
    int32_t match_frame;
    double transform[16];
    double scan_context_distance;
    double icp_fitness;
} sb_loop_result;

/* ---------------------------------------------------------------- context ---------------------------------- */
const char* sb_version(void);
/* stream: a cudaStream_t to enqueue on (e.g. torch's current stream) or NULL to let the context create its own. */
int sb_ctx_create(int device, void* stream, sb_ctx** out);
void sb_ctx_destroy(sb_ctx* ctx);
const char* sb_last_error(const sb_ctx* ctx);
int sb_ctx_synchronize(sb_ctx* ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
int64_t sb_ctx_launch_count(const sb_ctx* ctx);
/* Measurement hooks (not part of the reference API).  With profiling on, sb_register_batch[_dev] brackets its stages
 * with CUDA events on the context's stream; sb_ctx_stage_ms returns the milliseconds of the last call per stage:
 * 0 h2d, 1 voxel, 2 scan_context, 3 index_build, 4 normals, 5 icp_loop, 6 d2h (SB_STAGE_COUNT values).
 * sb_ctx_last_counts: [0] raw rows, [1] rows after the voxel grid, [2] indexed target rows,
 * [3] sum over pairs of (source rows x nearest-neighbour passes), [4] launches of the ICP iteration kernel. */
#define SB_STAGE_COUNT 7
int sb_ctx_set_profiling(sb_ctx* ctx, int enable);
int sb_ctx_stage_ms(sb_ctx* ctx, double* ms7);
/* host wall-clock milliseconds between the same marks (enqueue + host-side bookkeeping of each stage) */
int sb_ctx_stage_host_ms(sb_ctx* ctx, double* ms7);
int sb_ctx_last_counts(sb_ctx* ctx, int64_t* counts5);
/* which voxel-grid pipeline the last call on this context used: 1 = one-pass hashed fixed-point sums (float32-born
 * scans), 2 = sort-based (any fp64 input, any key range); 0 = none yet.  Both give the same rows, bit for bit. */
int sb_ctx_last_voxel_path(const sb_ctx* ctx);
void sb_default_icp_config(sb_icp_config* cfg);
void sb_default_loop_config(sb_loop_config* cfg);

/* ---------------------------------------------------------------- voxel grid ------------------------------- */
/* Replaces slam::voxel_downsample (file_utils.hpp:41-44, file_utils.cpp:148-196).
 * key = (long long)floor(coord / voxel) per axis with true IEEE division; centroid = sum over the voxel's points
 * in ascending input index, divided by the count.  Output rows are in ascending (kx,ky,kz) order (the reference's
 * unordered_map order is unspecified).  voxel <= 0 returns the input unchanged (file_utils.cpp:152).
 * out_xyz must hold n*3 doubles; out_keys (optional) n*3 int64. */
int sb_voxel_downsample(sb_ctx* ctx, const double* xyz, int64_t n, double voxel, double* out_xyz, int64_t* out_m,
                        int64_t* out_keys);
/* Batch of clouds in CSR form: cloud c is rows [offsets[c], offsets[c+1]).  out_offsets has n_clouds+1 entries. */
int sb_voxel_downsample_batch(sb_ctx* ctx, const double* xyz, const int64_t* offsets, int32_t n_clouds, double voxel,
                              double* out_xyz, int64_t* out_offsets, int64_t* out_keys);
/* Device variant: d_xyz / d_out_xyz / d_out_keys are device pointers (d_out_* sized for the INPUT row count),
 * offsets are host arrays.  Synchronises once to learn the output sizes. */
int sb_voxel_downsample_batch_dev(sb_ctx* ctx, const double* d_xyz, const int64_t* offsets, int32_t n_clouds,
                                  double voxel, double* d_out_xyz, int64_t* out_offsets, int64_t* d_out_keys);

/* ---------------------------------------------------------------- spatial index ---------------------------- */
/* Replaces slam::KDTree::KDTree (kdtree.hpp:20-26): copies the points to the device and builds the index. */
int sb_index_build(sb_ctx* ctx, const double* xyz, int64_t n, sb_index** out);
void sb_index_free(sb_index* index);
int64_t sb_index_size(const sb_index* index);
/* Replaces KDTree::nearest / nearest_batch (kdtree.hpp:32-59): exact 1-NN, squared distance
 * (dx*dx + dy*dy) + dz*dz in fp64 without FMA, smallest index among exact ties.  out_d2 may be NULL.
 * An empty index yields index -1 and DBL_MAX like kdtree.hpp:33-36. */
int sb_index_nearest_batch(sb_index* index, const double* queries, int64_t nq, int32_t* out_idx, double* out_d2);
/* Replaces KDTree::k_nearest (kdtree.hpp:65-78) for nq queries: row q holds min(k, size) indices ascending by
 * (d2, index), padded with -1 (and DBL_MAX in out_d2, optional).  1 <= k <= SB_MAX_K. */
int sb_index_knn(sb_index* index, const double* queries, int64_t nq, int32_t k, int32_t* out_idx, double* out_d2);
/* Replaces NearestNeighborSearch::find_correspondences (kdtree.hpp:198-214): matched target rows and sqrt(d2). */
int sb_index_find_correspondences(sb_index* index, const double* source, int64_t ns, double* matched_xyz,
                                  double* distances);
/* Replaces slam::estimate_normals(points, tree, k) (icp.hpp:23-67) for points == the indexed cloud.
 * out_normals: size*3 doubles, row i for input row i.  out_evals (optional): the 3 eigenvalues ascending per point. */
int sb_estimate_normals(sb_index* index, int32_t k, double* out_normals, double* out_evals);

/* ---------------------------------------------------------------- ICP -------------------------------------- */
/* Replaces slam::solve_point_to_plane (icp.hpp:89-144): one Gauss-Newton step from given correspondences. */
int sb_solve_point_to_plane(sb_ctx* ctx, const double* source, const double* target, const double* normals,
                            int64_t n, double* out_T16);
/* Replaces slam::icp_point_to_plane(source, target, config) (icp.hpp:157-258). */
int sb_icp_point_to_plane(sb_ctx* ctx, const double* source, int64_t ns, const double* target, int64_t nt,
                          const sb_icp_config* cfg, sb_icp_result* out);
/* Batched registration of independent pairs over a set of clouds (CSR).  pair p registers source cloud
 * pair_src[p] onto target cloud pair_tgt[p]; every cloud used as a target gets ONE index + normals.
 * voxel > 0 first applies sb_voxel_downsample to every cloud (slam_node.cpp:122).  sc_desc (optional) receives
 * the Scan Context of every (downsampled) cloud, n_clouds*1200 doubles (loop_closure.hpp:53-59). */
int sb_register_batch(sb_ctx* ctx, const double* xyz, const int64_t* offsets, int32_t n_clouds, double voxel,
                      const int32_t* pair_src, const int32_t* pair_tgt, int32_t n_pairs, const sb_icp_config* cfg,
                      sb_icp_result* results, double* sc_desc);
/* Same with the clouds already in device memory; results/sc_desc are host buffers (one D2H copy at the end). */
int sb_register_batch_dev(sb_ctx* ctx, const double* d_xyz, const int64_t* offsets, int32_t n_clouds, double voxel,
                          const int32_t* pair_src, const int32_t* pair_tgt, int32_t n_pairs,
                          const sb_icp_config* cfg, sb_icp_result* results, double* sc_desc);

/* float32 ingest (SURVEY.md 8f N1).  The reference reads x, y, z as float32 from binary PLY and KITTI .bin records
 * and widens them to double on the host (file_utils.cpp:91-97, 133-136; tools/convert_to_ply.cpp:14-67 writes
 * x, y, z, intensity).  These entry points take the float32 records as they are on disk — rows of `stride_floats`
 * floats with x, y, z first (3 for xyz, 4 for KITTI) — and widen on the device: half (or a third) of the
 * host-to-device bytes, identical results.  Host rows are uploaded in chunks that overlap with the voxel grid. */
int sb_register_batch_f32(sb_ctx* ctx, const float* xyz, int32_t stride_floats, const int64_t* offsets, int32_t n_clouds,
                          double voxel, const int32_t* pair_src, const int32_t* pair_tgt, int32_t n_pairs,
                          const sb_icp_config* cfg, sb_icp_result* results, double* sc_desc);
int sb_register_batch_f32_dev(sb_ctx* ctx, const float* d_xyz, int32_t stride_floats, const int64_t* offsets,
                              int32_t n_clouds, double voxel, const int32_t* pair_src, const int32_t* pair_tgt,
                              int32_t n_pairs, const sb_icp_config* cfg, sb_icp_result* results, double* sc_desc);
int sb_voxel_downsample_batch_f32(sb_ctx* ctx, const float* xyz, int32_t stride_floats, const int64_t* offsets,
                                  int32_t n_clouds, double voxel, double* out_xyz, int64_t* out_offsets,
                                  int64_t* out_keys);

/* ---------------------------------------------------------------- Scan Context ----------------------------- */
/* Replaces slam::ScanContext::compute (scan_context.hpp:44-82).  desc: 1200 doubles, COLUMN-major 20x60 like
 * Eigen::MatrixXd::data(): element (ring i, sector j) at desc[j*20 + i]. */
int sb_sc_compute(sb_ctx* ctx, const double* xyz, int64_t n, double* desc);
/* Replaces ScanContext::distance (scan_context.hpp:90-102,121-142): min over the 60 column shifts of b. */
int sb_sc_distance(sb_ctx* ctx, const double* desc_a, const double* desc_b, double* out);
/* One query against n_db database descriptors (contiguous, 1200 doubles each): out_dist[n_db]. */
int sb_sc_distance_batch(sb_ctx* ctx, const double* query, const double* db, int32_t n_db, double* out_dist);
/* ScanContext::ring_key / sector_key (scan_context.hpp:107-118): row means (20) / column means (60). */
int sb_sc_keys(sb_ctx* ctx, const double* desc, double* ring_key20, double* sector_key60);

/* ---------------------------------------------------------------- loop closure ----------------------------- */
/* Replaces slam::LoopClosureDetector (loop_closure.hpp:41-149).  The descriptor database and the cloud copies live
 * in device memory.  rank/world shard the database by entry id (entry i is owned by rank i % world): every rank
 * adds every frame, keeps the descriptors and clouds it owns, and sb_loop_candidates_local returns the local
 * part of the candidate list; the caller gathers (NCCL) and passes the merged list to sb_loop_verify. */
int sb_loop_create(sb_ctx* ctx, const sb_loop_config* cfg, int32_t rank, int32_t world, sb_loop** out);
void sb_loop_free(sb_loop* loop);
/* Optional: size the device pools for n_entries descriptors and total_rows cloud rows (what this rank will own) so
 * that no later addFrame allocates.  Without it the pools start at 4096 descriptors / 11 M rows and double. */
int sb_loop_reserve(sb_loop* loop, int64_t n_entries, int64_t total_rows);
int sb_loop_add_frame(sb_loop* loop, const double* xyz, int64_t n, int32_t frame_idx);      /* addFrame, :53-59  */
/* Adds a frame whose Scan Context is already known (database bulk load; the cloud is still copied). */
int sb_loop_add_frame_desc(sb_loop* loop, const double* xyz, int64_t n, int32_t frame_idx, const double* desc);
int64_t sb_loop_size(const sb_loop* loop);                                                    /* size(), :131      */
int sb_loop_clear(sb_loop* loop);                                                             /* clear(), :136-141 */
/* detect() (loop_closure.hpp:66-126) on a single rank (world == 1). */
int sb_loop_detect(sb_loop* loop, sb_loop_result* results, int32_t capacity, int32_t* count);
/* Stage 1 of detect(): candidates with frame gap >= frame_gap and distance < threshold among the entries this
 * rank owns, ascending by (distance, entry id) (loop_closure.hpp:75-92); at most `capacity` are returned,
 * *count is the number found. */
int sb_loop_candidates_local(sb_loop* loop, double* dist, int32_t* entry, int32_t capacity, int32_t* count);
/* Stage 2 for the listed entries (this rank must own them): ICP(query cloud -> entry cloud) for each,
 * loop_closure.hpp:99-109.  Fills results[i] for every listed entry (icp_fitness = final_error) and converged[i]. */
int sb_loop_verify_entries(sb_loop* loop, const int32_t* entry, const double* dist, int32_t n, sb_loop_result* results,
                           int32_t* converged);

/* Loop-closure detection over a whole recorded sequence.  The node calls addFrame and detect() once per keyframe
 * (slam_node.cpp:159-167, loop_closure.hpp:53-126); detect() for the query entry q reads only entries 0..q-1, so the
 * detections of many query entries are independent and run here as one many-query search and batched ICP rounds.
 *
 * addFrame for n_frames clouds at once: host fp64 rows in CSR form (cloud f is rows [offsets[f], offsets[f+1]),
 * offsets[0] = 0), frame_idx[n_frames], desc: n_frames*1200 Scan Context descriptors or NULL (computed).  Leaves the
 * detector in exactly the state n_frames calls of sb_loop_add_frame_desc would (world > 1 included: the owned entries
 * are kept, and the newest entry as a guest).  One descriptor launch and one synchronise. */
int sb_loop_add_frames(sb_loop* loop, const double* xyz, const int64_t* offsets, int32_t n_frames,
                       const int32_t* frame_idx, const double* desc);
/* Largest k of sb_loop_candidates_batch: the short list selected on the device per query. */
#define SB_LOOP_SELECT_MAX 32
/* Stage 1 of detect() for many queries (world == 1).  query_entries: n_queries entry ids, strictly ascending, each
 * below sb_loop_size.  Query q_i sees the entries e < q_i with frame[q_i] - frame[e] >= frame_gap and distance <
 * threshold (loop_closure.hpp:75-92): the best min(k, count[i]) of them, ascending by (distance, entry), are at
 * dist / entry[i*k ...]; count[i] = how many there are.  1 <= k <= SB_LOOP_SELECT_MAX. */
int sb_loop_candidates_batch(sb_loop* loop, const int32_t* query_entries, int32_t n_queries, int32_t k,
                             double* dist, int32_t* entry, int32_t* count);
/* detect() for many queries (world == 1, same query_entries rules): the result for q_i is what sb_loop_detect returns
 * right after entry q_i was added (query_frame = frame[q_i]).  results[i*max_candidates ...] holds the count[i]
 * accepted loops of query i.  The walk down each candidate list never skips a candidate.  The detector is not
 * modified.  max_candidates <= 0 gives empty results (results may then be NULL). */
int sb_loop_detect_batch(sb_loop* loop, const int32_t* query_entries, int32_t n_queries,
                         sb_loop_result* results, int32_t* count);

/* Loop closures between detectors: robots of a fleet mapping the same place, or a restarted robot relocalizing against
 * the database of an earlier run.  dbs[0..n_dbs) are detectors on one context, each at most once, all world == 1 and
 * with one loop config (every field but frame_gap equal).  Query i is entry query_entry[i] (0-based, as
 * sb_loop_detect_batch counts) of dbs[query_db[i]]; it gets detect()'s rule (loop_closure.hpp:66-126) over the entries
 * of every OTHER detector: candidates are the entries with distance < sc_distance_threshold (frame indices of different
 * streams are unrelated, so there is no frame gap), ordered by (distance, db, entry), and the walk verifies them with
 * the loop ICP from identity (loop_closure.hpp:99-109), accepts converged ones with final_error < icp_fitness_threshold
 * and stops at max_candidates acceptances without skipping a candidate.  The query's own detector is never searched.
 * Queries may come in any order and repeat; neither call modifies a detector; n_queries == 0 does nothing.  A rule
 * broken returns SB_ERR_INVALID_ARG before any work, with a message naming the detector or query index.
 *
 * Stage 1: per query the best min(k, count[i]) candidates over the other detectors, ascending (distance, db, entry):
 * dist / db / entry [i*k ...]; count[i] = how many are under the threshold.  1 <= k <= SB_LOOP_SELECT_MAX. */
int sb_loop_candidates_across(sb_loop* const* dbs, int32_t n_dbs, const int32_t* query_db, const int32_t* query_entry,
                              int32_t n_queries, int32_t k, double* dist, int32_t* db, int32_t* entry, int32_t* count);
/* detect() across detectors: results / match_db [i*max_candidates ...] hold the count[i] accepted loops of query i
 * (query_frame = frame of the query entry, match_frame = frame of the matched entry in dbs[match_db]).
 * max_candidates <= 0 gives empty results (results and match_db may then be NULL). */
int sb_loop_detect_across(sb_loop* const* dbs, int32_t n_dbs, const int32_t* query_db, const int32_t* query_entry,
                          int32_t n_queries, sb_loop_result* results, int32_t* match_db, int32_t* count);

/* ---------------------------------------------------------------- streaming odometry session --------------- */
/* SlamNode::process_frame (slam_node.cpp:118-175) one scan per call, with the previous frame kept on the device: its
 * downsampled cloud, index and normals serve as the next frame's ICP target, so no frame is uploaded or indexed twice.
 * A session belongs to one context; the optional loop-closure detector must be created on the same context and must
 * outlive the session.  Per push:
 *   1. voxel grid (slam_node.cpp:122); fewer than min_points rows: the frame is SKIPPED (slam_node.cpp:125-130): the
 *      pose is repeated, the previous frame stays the ICP target, nothing is added and detect does not run;
 *   2. ICP of this frame (source) onto the previous one (target), exactly sb_icp_point_to_plane(current, previous, icp);
 *   3. pose = previous pose * delta with sb_odometry_poses's rule and arithmetic (the first frame: the initial pose);
 *   4. the world-frame cloud as PointCloud2 float32 records (sb_transform_clouds_f32) and the Scan Context (sb_sc_compute);
 *   5. SB_ODOM_ADD_FRAME: the detector is left in the state sb_loop_add_frame(cloud, frame_idx) leaves (world > 1 too);
 *   6. SB_ODOM_DETECT (world == 1 only): loops = what sb_loop_detect_batch returns for the detector's newest entry.
 * A call that fails (SB_ERR_INVALID_ARG, SB_ERR_EMPTY, SB_ERR_RANGE, ...) leaves the session and the detector as they
 * were: the next push behaves as if the failed one had never been made. */
typedef struct sb_odom sb_odom;
typedef struct sb_odom_config {
    double voxel;              /* 0.5   slam_node voxel_size; <= 0: no voxel grid                                     */
    int32_t min_points;        /* 1000  slam_node.hpp:29: fewer rows after the voxel grid -> the frame is skipped      */
    int32_t reserved;
    double max_error;          /* 1.0   slam_node.cpp:139-140: delta = identity if final_error > max_error            */
    sb_icp_config icp;         /* sb_default_icp_config                                                              */
    double initial_pose[16];   /* row-major 4x4, identity                                                            */
} sb_odom_config;
void sb_default_odom_config(sb_odom_config* cfg);
/* loop: NULL for no loop closure, else a detector created on ctx */
int sb_odom_create(sb_ctx* ctx, const sb_odom_config* cfg, sb_loop* loop, sb_odom** out);
void sb_odom_free(sb_odom* odom);
/* Optional: size every device and pinned buffer for frames of up to max_raw_rows rows, so that no push allocates. */
int sb_odom_reserve(sb_odom* odom, int64_t max_raw_rows);
/* Continue the pose chain from pose16 (row-major), e.g. an optimised pose (slam_node.cpp:177-185). */
int sb_odom_set_pose(sb_odom* odom, const double* pose16);
/* The pose of the newest registered (or first) frame. */
int sb_odom_get_pose(const sb_odom* odom, double* pose16);

enum { SB_ODOM_ADD_FRAME = 1, SB_ODOM_DETECT = 2 };          /* per-push flags */
enum { SB_ODOM_FIRST = 0, SB_ODOM_REGISTERED = 1, SB_ODOM_SKIPPED = 2 };
typedef struct sb_odom_frame {
    int32_t frame_idx, state;  /* state: SB_ODOM_FIRST | SB_ODOM_REGISTERED | SB_ODOM_SKIPPED                         */
    int64_t n_points;          /* rows after the voxel grid                                                          */
    double pose[16];           /* pose of this frame after the chain step (skipped: the previous pose)                */
    sb_icp_result icp;         /* state == SB_ODOM_REGISTERED, else zero                                             */
    int32_t n_loops, pad;      /* accepted loop closures (SB_ODOM_DETECT), counted like sb_loop_detect's *count       */
} sb_odom_frame;
/* xyz: n host fp64 rows (pinned rows are copied without staging; a device pointer is SB_ERR_INVALID_ARG).  Outputs (NULL: not wanted): out_xyz n_points*3 doubles (downsampled rows, sensor frame; also
 * for a skipped frame), out_world_f32 n_points*3 floats and out_desc 1200 doubles (not for a skipped frame), loops: the
 * first min(n_loops, loop_capacity) accepted loop closures (NULL only with loop_capacity == 0).  The output buffers must
 * hold n rows: n_points is not known before the call. */
int sb_odom_push(sb_odom* odom, const double* xyz, int64_t n, int32_t frame_idx, int32_t flags, sb_odom_frame* out,
                 double* out_xyz, float* out_world_f32, double* out_desc, sb_loop_result* loops, int32_t loop_capacity);
/* The float32 records of a PLY / KITTI file: rows of stride_floats (>= 3) floats, x, y, z first, widened on the device
 * (as sb_register_batch_f32): the same results as sb_odom_push of the widened rows. */
int sb_odom_push_f32(sb_odom* odom, const float* xyz, int32_t stride_floats, int64_t n, int32_t frame_idx,
                     int32_t flags, sb_odom_frame* out, double* out_xyz, float* out_world_f32, double* out_desc,
                     sb_loop_result* loops, int32_t loop_capacity);

/* ---------------------------------------------------------------- after the path: world frame, map -------- */
/* The data-parallel steps that follow registration in slam_node.cpp (SURVEY.md 8f N2/N3).  poses16: n_clouds
 * row-major 4x4 transforms (Transformation::matrix()), cloud c is rows [offsets[c], offsets[c+1]). */
typedef struct sb_grid_config {   /* slam::OccupancyGridConfig, slam_viz/include/slam_viz/ros/slam_node.hpp:35-40 */
    double resolution;            /* 0.2  */
    double height_min;            /* 0.3  */
    double height_max;            /* 2.0  */
    double max_range;             /* 40.0 */
} sb_grid_config;
void sb_default_grid_config(sb_grid_config* cfg);
/* world = cloud * R^T + t for every cloud (slam_node.cpp:147, 189, 201-203). out_xyz: offsets[n_clouds]*3 doubles. */
int sb_transform_clouds(sb_ctx* ctx, const double* xyz, const int64_t* offsets, int32_t n_clouds, const double* poses16,
                        double* out_xyz);
/* rebuild_occupancy_grid (slam_node.cpp:211-229): transforms every (sensor-frame) cloud with its pose, keeps points
 * with height_min <= z <= height_max and 0.5 <= horizontal range from the pose's translation <= max_range, and
 * returns the set of cells (floor(x/res), floor(y/res)), ascending in (x, y) (the reference's unordered_set has no
 * order).  out_cells: 2 ints per cell, up to `capacity` cells; *out_count = number of cells found. */
int sb_occupancy_cells(sb_ctx* ctx, const double* xyz, const int64_t* offsets, int32_t n_clouds, const double* poses16,
                       const sb_grid_config* cfg, int32_t* out_cells, int64_t capacity, int64_t* out_count);
/* build_final_global_map + the voxel grid publish_global_map applies to it (slam_node.cpp:196-209, 235-238): all
 * clouds in the world frame as one cloud, voxel-downsampled with `voxel` (the node passes 2 * voxel_size);
 * voxel <= 0 returns the concatenation.  out_xyz: offsets[n_clouds]*3 doubles. */
int sb_global_map(sb_ctx* ctx, const double* xyz, const int64_t* offsets, int32_t n_clouds, const double* poses16,
                  double voxel, double* out_xyz, int64_t* out_m);

/* The same two results as the payload of the sensor_msgs/PointCloud2 the node publishes — eigen_to_pointcloud2
 * (slam_node.cpp:299-322): x, y, z as float32 (static_cast<float>, round to nearest), point_step 12, row after row —
 * converted on the device so that half the bytes cross PCIe.  publish_current_scan (slam_node.cpp:147, 231-233) /
 * publish_global_map (slam_node.cpp:235-238).  out_xyz: offsets[n_clouds]*3 floats. */
int sb_transform_clouds_f32(sb_ctx* ctx, const double* xyz, const int64_t* offsets, int32_t n_clouds,
                            const double* poses16, float* out_xyz);
int sb_global_map_f32(sb_ctx* ctx, const double* xyz, const int64_t* offsets, int32_t n_clouds, const double* poses16,
                      double voxel, float* out_xyz, int64_t* out_m);

/* The pose chain of process_frame (slam_node.cpp:139-145), for a sequence registered as one batch: results[i] is the
 * registration of frame i+1 against frame i; delta_i = identity if !converged or final_error > max_error (the node
 * uses 1.0), else the result's transformation; poses16_out[0] = initial_pose16 (NULL: identity) and
 * poses16_out[i+1] = poses16_out[i] * delta_i.  poses16_out: (n+1)*16 doubles, row-major 4x4 — the `poses16` the three
 * entry points above take.  Host arithmetic (n 4x4 products, a serial recurrence); ctx may be NULL. */
int sb_odometry_poses(sb_ctx* ctx, const sb_icp_result* results, int32_t n, double max_error,
                      const double* initial_pose16, double* poses16_out);

/* ---------------------------------------------------------------- device-resident map ---------------------- */
/* The node's map state (slam_node.cpp:147-157, 177-238) kept in device memory: every keyframe's downsampled
 * sensor-frame cloud and its pose (the node's downsampled_clouds_ and poses_), and the occupancy cell set.  A pose
 * update after a loop closure uploads only the poses; the cell set, the global map and the world-frame window are
 * rebuilt from the resident clouds.  A map belongs to one context.
 * Every output equals the stateless entry point above on the resident clouds C and poses P, bit for bit, after any
 * sequence of add / set_poses: sb_map_occupancy_cells = sb_occupancy_cells(C, P, grid), sb_map_global[_f32] =
 * sb_global_map[_f32](C, P, voxel), sb_map_world_f32 = sb_transform_clouds_f32 of the listed entries.
 * A call that fails leaves the map as it was: a non-finite row or pose, or a cell index that does not fit an int,
 * is SB_ERR_RANGE. */
typedef struct sb_map sb_map;
/* grid: NULL -> sb_default_grid_config */
int sb_map_create(sb_ctx* ctx, const sb_grid_config* grid, sb_map** out);
void sb_map_free(sb_map* map);
/* Optional: room for n_entries entries, total_rows rows and n_cells occupancy cells, so that no later call allocates
 * while the map stays within them.  Without it the buffers start small and double. */
int sb_map_reserve(sb_map* map, int64_t n_entries, int64_t total_rows, int64_t n_cells);
int64_t sb_map_size(const sb_map* map);          /* entries */
int64_t sb_map_rows(const sb_map* map);          /* rows over all entries: what sb_map_global's output must hold */
/* Measurement hook: [0] entries, [1] rows, [2] cell-table slots the device buffers hold now */
int sb_map_capacity(const sb_map* map, int64_t* caps3);
int sb_map_clear(sb_map* map);
/* One entry: a sensor-frame cloud (n host fp64 rows, n may be 0) and its pose (row-major 4x4); its cells are inserted
 * at once (update_occupancy_grid, slam_node.cpp:152, 211-221). */
int sb_map_add(sb_map* map, const double* xyz, int64_t n, const double* pose16);
/* The poses of entries [first, first + n) replaced (PoseGraph::getAllPoses after optimize, slam_node.cpp:177-185);
 * the cell set is rebuilt on the device from every resident cloud (rebuild_occupancy_grid, slam_node.cpp:222-229). */
int sb_map_set_poses(sb_map* map, int32_t first, int32_t n, const double* poses16);
int sb_map_get_poses(const sb_map* map, int32_t first, int32_t n, double* poses16);
/* The cells, ascending in (x, y), 2 ints each, up to `capacity`; *out_count = all of them. */
int sb_map_occupancy_cells(sb_map* map, int32_t* out_cells, int64_t capacity, int64_t* out_count);
/* Entries [first, first + n) in the world frame as PointCloud2 float32 records (the node's window of the last 20
 * world clouds, publish_current_scan): *out_rows rows; out_xyz must hold them. */
int sb_map_world_f32(sb_map* map, int32_t first, int32_t n, float* out_xyz, int64_t* out_rows);
/* All entries in the world frame, voxel grid at `voxel` (<= 0: the concatenation), as fp64 rows or float32 records
 * (publish_global_map, slam_node.cpp:196-209, 235-238).  out_xyz must hold sb_map_rows rows. */
int sb_map_global(sb_map* map, double voxel, double* out_xyz, int64_t* out_m);
int sb_map_global_f32(sb_map* map, double voxel, float* out_xyz, int64_t* out_m);

/* A streaming session that also feeds a map (sb_odom_create for map == NULL).  With SB_ODOM_ADD_MAP a push adds the
 * frame to the map: its downsampled rows (copied device to device) and its pose; a SKIPPED frame adds an entry with no
 * rows and the repeated pose, so that map entry i is the node's poses_[i].  The map must be created on ctx and must
 * outlive the session.  A push that fails leaves the map as it was too. */
enum { SB_ODOM_ADD_MAP = 4 };
int sb_odom_create2(sb_ctx* ctx, const sb_odom_config* cfg, sb_loop* loop, sb_map* map, sb_odom** out);

/* ---------------------------------------------------------------- many streaming sessions in one call ------ */
/* One frame into each of n sessions (SB_ODOM_* semantics per session), with one voxel grid, one index build and one ICP
 * batch for all of them: many live streams (a fleet of robots, several LiDARs, replayed sequences) on one GPU.  The
 * result is exactly what n calls of sb_odom_push would give, in array order: every output and every session, detector
 * and map state afterwards, bit for bit; single and many pushes may be mixed on the same sessions.  Arrays are indexed
 * by session: xyz[i] holds n_rows[i] rows, out[i] receives the frame, and out_xyz[i], out_world_f32[i], out_desc[i],
 * loops[i] / loop_capacity[i] are sb_odom_push's outputs.  Each of those per-session pointer arrays may be NULL (that
 * output is not wanted by any session); an entry may be NULL too.  flags may be NULL (0 for every session).
 * Rules, checked before any work is enqueued (SB_ERR_INVALID_ARG): all sessions belong to one context, no session
 * appears twice, no two sessions share a loop-closure detector or a map, all sessions have the same voxel and icp
 * config (min_points, max_error and the pose may differ), and every session's arguments pass sb_odom_push's checks.
 * Failure is all or nothing: a call that fails for any session leaves every session, detector and map as it was, and
 * the message (sb_last_error) names the index of that session.  n == 0 does nothing.  Per call the host waits as often
 * as one push does, whatever n is. */
int sb_odom_push_many(sb_odom* const* sessions, int32_t n, const double* const* xyz, const int64_t* n_rows,
                      const int32_t* frame_idx, const int32_t* flags, sb_odom_frame* out, double* const* out_xyz,
                      float* const* out_world_f32, double* const* out_desc, sb_loop_result* const* loops,
                      const int32_t* loop_capacity);
/* The same for float32 records of stride_floats (>= 3) floats, x, y, z first (sb_odom_push_f32), one stride for all. */
int sb_odom_push_many_f32(sb_odom* const* sessions, int32_t n, const float* const* xyz, int32_t stride_floats,
                          const int64_t* n_rows, const int32_t* frame_idx, const int32_t* flags, sb_odom_frame* out,
                          double* const* out_xyz, float* const* out_world_f32, double* const* out_desc,
                          sb_loop_result* const* loops, const int32_t* loop_capacity);

/* ---------------------------------------------------------------- multi-GPU exchanges (SURVEY.md 8e) -------- */
/* One process per GPU; the caller owns the NCCL communicator (an ncclComm_t passed as void*; NCCL itself is looked up
 * in the already-loaded libnccl.so.2 at first use, it is not a link dependency of this library).  The reference has no
 * counterpart: these are the two exchanges of the sharded paths, KB-sized, once per batch / per detect().
 *
 * Batched independent pair ICP (config C5): unit (pair) u is registered by rank u % world as that rank's local result
 * u / world (sb_register_batch on the rank's own pairs).  Every rank receives all n_total results in unit order.
 * local: this rank's results (NULL allowed when it owns none); all: n_total records. */
int sb_gather_results(sb_ctx* ctx, void* nccl_comm, int32_t rank, int32_t world, const sb_icp_result* local,
                      int32_t n_total, sb_icp_result* all);
/* Sharded loop-closure search (config C4): every rank contributes up to `capacity` local candidates
 * (sb_loop_candidates_local: ascending (distance, entry)); every rank receives the `capacity` best of the job in the
 * order of loop_closure.hpp:92.  Each rank then verifies the entries it owns (sb_loop_verify_entries) and the
 * records go through sb_gather_results-style exchange or the caller's own. */
int sb_gather_candidates(sb_ctx* ctx, void* nccl_comm, int32_t world, const double* dist, const int32_t* entry,
                         int32_t n_local, int32_t capacity, double* out_dist, int32_t* out_entry, int32_t* out_count);

/* ---------------------------------------------------------------- pose-graph hand-off (SURVEY.md 8f N4) ----- */
/* The pose graph itself (slam::PoseGraph, GTSAM) stays on the host and is not part of this library.  These two
 * entries turn a batch of registration / loop-closure results into the factors process_frame hands to it one frame
 * at a time, as plain records in the order the node would have produced them. */
enum { SB_FACTOR_ODOMETRY = 0, SB_FACTOR_LOOP = 1 };
typedef struct sb_pose_factor {
    int32_t kind;          /* SB_FACTOR_ODOMETRY | SB_FACTOR_LOOP */
    int32_t from;          /* odometry: frame i-1 (slam_node.cpp:145); loop: match_frame (slam_node.cpp:165) */
    int32_t to;            /* odometry: frame i; loop: query_frame */
    int32_t pad;
    double relative[16];   /* row-major 4x4 transform from `from` to `to`, as PoseGraph::add* take it */
    double fitness;        /* odometry: ICP final_error, passed as fitness_score; loop: icp_fitness */
    double noise_scale;    /* odometry: 1 + 10 * fitness, the sigma multiplier of pose_graph.cpp:88; loop: 1 */
} sb_pose_factor;
/* results[i] = registration of frame first_frame+i+1 against frame first_frame+i.  relative = identity if the pair
 * did not converge or final_error > max_error (slam_node.cpp:139-140; the node uses 1.0) — the fitness passed on is the
 * result's final_error either way (slam_node.cpp:145).  out: n records.  Host arithmetic; ctx may be NULL. */
int sb_odometry_factors(sb_ctx* ctx, const sb_icp_result* results, int32_t n, int32_t first_frame, double max_error,
                        sb_pose_factor* out);
/* Accepted loop closures (sb_loop_detect / sb_loop_verify_entries) -> addLoopClosure(match, query, transform)
 * records (slam_node.cpp:163-167).  out: n records.  Host arithmetic; ctx may be NULL. */
int sb_loop_factors(sb_ctx* ctx, const sb_loop_result* results, int32_t n, sb_pose_factor* out);

/* ---------------------------------------------------------------- bench/test input generator --------------- */
/* Synthetic 64/128-beam raycast straight into device memory (synth/lidar_synth.h).  boxes: host, n_boxes*6 floats;
 * poses: host, n_scans*3 doubles (x, y, yaw); d_xyz: device, n_scans*beams*azimuth_steps*3 doubles capacity;
 * out_offsets: host, n_scans+1.  Not part of the reference's API. */
int sb_synth_scans_dev(sb_ctx* ctx, int32_t beams, int32_t azimuth_steps, float elev_top_deg, float elev_bot_deg,
                       float max_range, float noise_sigma, float sensor_height, const float* boxes, int32_t n_boxes,
                       const double* poses, int32_t n_scans, uint64_t noise_seed, double* d_xyz,
                       int64_t* out_offsets);

#ifdef __cplusplus
}
#endif
#endif /* SLAM_B200_H */
