/* liorf_b200.h — C ABI of the B200-native scan-to-map hot path of liorf.
 *
 * The reference (jimmyshe/liorf) has no plugin / FFI layer: the path sits behind `void()` C++ member functions that
 * talk through class members (SURVEY.md §8b).  Each entry point below replaces ONE of those member-function bodies
 * and makes the implicit member state explicit.  The file:line after "replaces" is the reference interface.
 *
 * Conventions: plain pointers and sizes, no C++/torch types.  Return value 0 = success, negative = error code
 * (never throws).  The caller owns host buffers.  The opaque context owns all device memory and ONE CUDA stream;
 * like the reference's `mtx` (src/mapOptmization.cpp:136,252) a context is not thread-safe.
 * Pose layout everywhere: float[6] = (roll, pitch, yaw, x, y, z) = transformTobeMapped (src/mapOptmization.cpp:134).
 * There is NO CPU fallback: every call needs a CUDA device and fails with LIORF_ERR_CUDA otherwise.
 */
#ifndef LIORF_B200_H
#define LIORF_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define LIORF_MAX_ITERS 64

/* return codes (token-identical to csrc/common.cuh, which the implementation includes after this header) */
#define LIORF_OK 0
#define LIORF_ERR_CUDA -1           /* no device / a CUDA call failed (the message goes to stderr) */
#define LIORF_ERR_ARG -2            /* NULL context, NULL mandatory pointer, size or parameter out of range */
#define LIORF_ERR_STATE -3          /* call order / ownership: e.g. a query before the database exists, shard extents that differ from the ones agreed at connect time */
#define LIORF_ERR_DEVICE_FLAG -4    /* a bounded device-side wait gave up (look-back predecessor, solver hand-off, a peer's exchange flag); the context stays failed */

typedef struct liorf_ctx liorf_ctx;

/* pcl::PointXYZI payload (include/utility.h:61); device layout is the same 16 bytes */
typedef struct { float x, y, z, intensity; } liorf_point;
/* VelodynePointXYZIRT payload (src/imageProjection.cpp:4-15), 24 bytes */
typedef struct { float x, y, z, intensity; uint16_t ring; uint16_t _pad; float time; } liorf_point_xyzirt;

/* The ParamServer subset the path reads (include/utility.h:100-105, 227-241) */
typedef struct {
    int   N_SCAN;                               /* utility.h:100 */
    int   downsampleRate;                       /* utility.h:102 */
    int   point_filter_num;                     /* utility.h:103 */
    float lidarMinRange, lidarMaxRange;         /* utility.h:104-105 */
    float mappingSurfLeafSize;                  /* utility.h:227  (downsampleCurrentScan) */
    float surroundingKeyframeMapLeafSize;       /* utility.h:240-ish (extractCloud VoxelGrid) */
    float surroundingKeyframeSearchRadius;      /* extractCloud distance gate, src/mapOptmization.cpp:1018 */
    int   grid_dim_x, grid_dim_y, grid_dim_z;   /* voxel-hash torus (powers of two, cell = 1 m); 0 → 256,256,32 */
    int   device;                               /* CUDA device ordinal */
} liorf_params;

/* per-iteration record of scan2MapOptimization (poses AFTER each LMOptimization call) */
typedef struct {
    float pose[LIORF_MAX_ITERS][6];
    int   nsel[LIORF_MAX_ITERS];                /* laserCloudSelNum of the iteration */
    int   iters;                                /* iterations executed */
    int   converged;                            /* LMOptimization returned true */
    int   degenerate;                           /* isDegenerate after the call */
    int   ran;                                  /* 0 when the guards of :1297/:1300 skipped the solve */
} liorf_lm_trace;

void liorf_default_params(liorf_params* p);                      /* config/kitti.yaml values */
int  liorf_create(const liorf_params* p, liorf_ctx** out);
void liorf_destroy(liorf_ctx* ctx);
/* pre-size all device work buffers (no allocation, hence no device-wide sync, inside later calls) */
int  liorf_reserve(liorf_ctx* ctx, int n_scan_max, int m_raw_max, int n_keyframe_points_max, int sc_entries_max);
int  liorf_sync(liorf_ctx* ctx);                                 /* cudaStreamSynchronize + sticky device error flags */
void* liorf_stream(liorf_ctx* ctx);                              /* the context's cudaStream_t (for CUDA-event timing) */
const char* liorf_version(void);

/* ---- imageProjection ------------------------------------------------------------------------------------------ */
/* replaces ImageProjection::projectPointCloud() (src/imageProjection.cpp:568) incl. deskewPoint (:536) and
 * findRotation (:493).  imu_time / imu_rot_{x,y,z} are the tables filled by imuDeskewInfo (:350-409), rows
 * 0..imu_pointer_cur valid.  deskew_enabled = !(deskewFlag == -1 || !cloudInfo.imuAvailable) (:538).
 * Result = fullCloud: kept on the device as the context's laserCloudSurfLast and, if out != NULL, copied to
 * out[0..*n_out) (capacity n).  kept_index (nullable, capacity n) receives the raw index of every kept point. */
int liorf_project_point_cloud(liorf_ctx* ctx, const liorf_point_xyzirt* pts, int n, double time_scan_cur,
                              const double* imu_time, const double* imu_rot_x, const double* imu_rot_y, const double* imu_rot_z,
                              int imu_pointer_cur, int deskew_enabled, liorf_point* out, int* n_out, int* kept_index);
/* same, raw points already in device memory (bench "inputs resident in HBM"); nothing is copied back */
int liorf_project_point_cloud_dev(liorf_ctx* ctx, const void* d_pts, int n, double time_scan_cur, const double* imu_time,
                                  const double* imu_rot_x, const double* imu_rot_y, const double* imu_rot_z, int imu_pointer_cur,
                                  int deskew_enabled);

/* ---- mapOptimization ------------------------------------------------------------------------------------------ */
/* sets laserCloudSurfLast from a host cloud (what pcl::fromROSMsg does at src/mapOptmization.cpp:244) */
int liorf_set_current_scan(liorf_ctx* ctx, const liorf_point* scan, int n);
int liorf_set_current_scan_dev(liorf_ctx* ctx, const void* d_scan, int n);
/* laserCloudSurfLast straight from cloud_info.cloud_deskewed (msg/cloud_info.msg:27, src/mapOptmization.cpp:245): the PointCloud2 data block with
 * `point_step` bytes per point (32 for PCL's padded PointXYZI, include/utility.h:61), xyz at offset_xyz, intensity at offset_intensity (16) */
int liorf_set_current_scan_strided(liorf_ctx* ctx, const void* data, int n, int point_step, int offset_xyz, int offset_intensity, int data_on_device);
/* replaces mapOptimization::downsampleCurrentScan() (src/mapOptmization.cpp:1061): VoxelGrid(mappingSurfLeafSize) of
 * laserCloudSurfLast → laserCloudSurfLastDS.  out (nullable, capacity = input size), n_ds (nullable: skip the read-back).
 * membership (nullable, capacity = input size): output slot of every input point (bit-exact voxel membership). */
int liorf_downsample_current_scan(liorf_ctx* ctx, liorf_point* out, int* n_ds, int* membership);
/* generic VoxelGrid on host data (same kernels; used by parity tests and the global-map filters) */
int liorf_voxel_grid(liorf_ctx* ctx, const liorf_point* in, int n, float leaf, liorf_point* out, int* n_out, int* membership, int* out_keys);

/* stores laserCloudSurfLastDS as surfCloudKeyFrames[id] with its pose / time (saveKeyFramesAndFactor, :1576-1580);
 * returns the new keyframe id (>= 0) or a negative error */
int liorf_add_keyframe(liorf_ctx* ctx, const float pose6[6], double time);
/* same with an explicit host cloud (tests / map loading) */
int liorf_add_keyframe_cloud(liorf_ctx* ctx, const liorf_point* cloud, int n, const float pose6[6], double time);
int liorf_update_keyframe_pose(liorf_ctx* ctx, int id, const float pose6[6]);           /* correctPoses, :1611-1642 */
int liorf_num_keyframes(liorf_ctx* ctx);
/* replaces extractCloud (src/mapOptmization.cpp:1012-1044) for the keyframe ids chosen by extractNearby (:975-1010):
 * transform + concatenate in selection order (duplicates allowed, as the reference), VoxelGrid
 * (surroundingKeyframeMapLeafSize) → laserCloudSurfFromMapDS, then builds the voxel-hash grid that replaces
 * kdtreeSurfFromMap->setInputCloud (:1302).  m_ds nullable (skip the read-back). */
int liorf_extract_surrounding_keyframes(liorf_ctx* ctx, const int* keyframe_ids, int n_ids, int* m_ds);
/* sets laserCloudSurfFromMapDS directly from a host cloud and builds the grid (parity tests / static maps) */
int liorf_set_local_map(liorf_ctx* ctx, const liorf_point* map_ds, int m);
int liorf_get_local_map(liorf_ctx* ctx, liorf_point* out, int capacity, int* m_ds);
/* replaces kdtreeSurfFromMap->setInputCloud(laserCloudSurfFromMapDS) (src/mapOptmization.cpp:1302): rebuilds the voxel-hash grid over the
 * resident laserCloudSurfFromMapDS.  liorf_extract_surrounding_keyframes / liorf_set_local_map already do this once per map; the entry
 * lets a caller (bench.py) repeat the step the reference repeats in every scan2MapOptimization call.  Asynchronous. */
int liorf_kdtree_set_input_cloud(liorf_ctx* ctx);
int liorf_get_scan_ds(liorf_ctx* ctx, liorf_point* out, int capacity, int* n_ds);

/* keyframe SELECTION of extractNearby (src/mapOptmization.cpp:975-1010) over the context's key poses: radius search
 * around the newest key pose, VoxelGrid(surroundingKeyframeDensity) of the poses, nearest-1 id recovery, plus every
 * keyframe younger than 10 s, each passed through extractCloud's distance gate (:1018) on the position the reference tests (the
 * voxel centroid for the thinned set, the real pose for the tail).  Host-side scalar code.  ids capacity = cap; *n_ids = count. */
int liorf_extract_nearby(liorf_ctx* ctx, double time_laser_info_cur, float surrounding_keyframe_density, int* ids, int cap, int* n_ids);
/* replaces mapOptimization::saveFrame() (src/mapOptmization.cpp:1365-1384): 1 = make a keyframe, 0 = skip */
int liorf_save_frame(liorf_ctx* ctx, const float pose6[6], float adding_dist_threshold, float adding_angle_threshold);
/* the clamps of transformUpdate (src/mapOptmization.cpp:1348-1350) */
void liorf_transform_update_clamp(float pose6_inout[6], float rotation_tollerance, float z_tollerance);
/* context-free forms (host only, usable without a GPU): poses6 = n x (roll,pitch,yaw,x,y,z), times = n stamps */
int liorf_host_extract_nearby(const float* poses6, const double* times, int n, double time_laser_info_cur, float search_radius,
                              float keyframe_density, int* ids, int cap, int* n_ids);
/* mapOptimization::updateInitialGuess (src/mapOptmization.cpp:899-958), host scalar code.  `state` replaces the function's
 * static locals (zero-initialise it once: identity transforms are filled in on first use).  cloud_info fields as in
 * msg/cloud_info.msg.  tf = transformTobeMapped (roll, pitch, yaw, x, y, z), updated in place. */
typedef struct { float lastImuTransformation[12]; float lastImuPreTransformation[12]; int lastImuPreTransAvailable; int initialised; } liorf_guess_state;
typedef struct {
    int imuAvailable, odomAvailable;
    float imuRollInit, imuPitchInit, imuYawInit;
    float initialGuessX, initialGuessY, initialGuessZ, initialGuessRoll, initialGuessPitch, initialGuessYaw;
} liorf_cloud_info_guess;
int liorf_host_update_initial_guess(liorf_guess_state* state, int no_keyframes_yet, const liorf_cloud_info_guess* cloud_info,
                                    int use_imu_heading_initialization, int imu_type, float transformTobeMapped[6]);
/* mapOptimization::transformUpdate (:1323-1353) in full: 9-axis roll / pitch slerp towards the IMU attitude (tf::Quaternion
 * arithmetic in double) when imuAvailable && imuType, then the clamps */
int liorf_host_transform_update(float transformTobeMapped[6], int imu_available, int imu_type, float imu_roll_init, float imu_pitch_init,
                                float imu_rpy_weight, float rotation_tollerance, float z_tollerance);
int liorf_host_save_frame(const float* last_pose6 /*nullable*/, const float pose6[6], float adding_dist_threshold, float adding_angle_threshold);
/* replaces ImageProjection::imuDeskewInfo() (src/imageProjection.cpp:350-409) and the IMU gate of deskewInfo() (:337, check_gate != 0): from
 * the queued IMU samples (stamp[n] ascending, gyro_xyz[n][3] = angular velocity after imuConverter, include/utility.h:257-272) builds the
 * table liorf_project_point_cloud reads — row 0 = zeros at the first stamp >= time_scan_cur - 0.01, then rot[k] = rot[k-1] + w[k] dt
 * (rectangle rule), last row = first stamp > time_scan_end + 0.01 exclusive.  capacity = queueLength (2000, :62).
 * Outputs: imu_time / imu_rot_{x,y,z}[capacity], *imu_pointer_cur (:403), *n_pop (samples the reference pops from the queue front, :354-360),
 * *rpy_index (sample whose orientation gives imuRoll/Pitch/YawInit for imuType != 0, :371-375; -1 = none).  Host-side scalar code, no GPU.
 * Returns 1 = cloudInfo.imuAvailable, 0 = not available, negative = error. */
int liorf_host_imu_deskew_info(const double* stamp, const double* gyro_xyz, int n, double time_scan_cur, double time_scan_end, int check_gate,
                               double* imu_time, double* imu_rot_x, double* imu_rot_y, double* imu_rot_z, int capacity, int* imu_pointer_cur, int* n_pop, int* rpy_index);

/* replaces mapOptimization::scan2MapOptimization() (src/mapOptmization.cpp:1295) up to, not including, transformUpdate:
 * ≤ max_iters × {surfOptimization, combineOptimizationCoeffs, LMOptimization} in one persistent kernel.
 * force_all_iters != 0 disables the convergence break (benchmark).  trace nullable. */
int liorf_scan2map_optimization(liorf_ctx* ctx, float pose6_inout[6], int max_iters, int force_all_iters, liorf_lm_trace* trace);
/* asynchronous variant: pose stays on the device (liorf_get_pose reads it); returns right after the launch */
int liorf_scan2map_optimization_async(liorf_ctx* ctx, const float pose6_in[6] /*nullable: keep device pose*/, int max_iters, int force_all_iters);
int liorf_get_pose(liorf_ctx* ctx, float pose6[6], liorf_lm_trace* trace /*nullable*/);

/* per-function parity hooks.
 * surfOptimization (:1074): per point i of laserCloudSurfLastDS: coeff (coeffSelSurfVec), flag (laserCloudOriSurfFlag),
 * nn_idx[5] = indices into laserCloudSurfFromMapDS by (distance, index) (only meaningful where the 5th distance < 1.0,
 * else -1 fills), nn_d2[5], plane[4] = (pa,pb,pc,pd), sel = pointSel.  All nullable except coeff/flag. */
int liorf_surf_optimization(liorf_ctx* ctx, const float pose6[6], liorf_point* coeff, uint8_t* flag, int* nn_idx, float* nn_d2,
                            float* plane, liorf_point* sel);
/* combineOptimizationCoeffs (:1145): compacts the result of the last liorf_surf_optimization → laserCloudOri / coeffSel */
int liorf_combine_optimization_coeffs(liorf_ctx* ctx, liorf_point* ori /*nullable*/, liorf_point* coeff /*nullable*/, int* n_sel);
/* LMOptimization(iterCount) (:1158) on the compacted arrays; isDegenerate / matP persist in the context.
 * Returns 1 = converged, 0 = keep optimizing, negative = error. */
int liorf_lm_optimization(liorf_ctx* ctx, int iter_count, float pose6_inout[6], float AtA[36], float AtB[6], float X[6], int* n_sel);
int liorf_get_lm_state(liorf_ctx* ctx, int* is_degenerate, float matP[36]);
int liorf_set_lm_state(liorf_ctx* ctx, int is_degenerate, const float matP[36]);

/* ---- ScanContext ---------------------------------------------------------------------------------------------- */
/* replaces SCManager::makeAndSaveScancontextAndKeys(scan) (include/Scancontext.h:72).  cloud == NULL → use the
 * context's laserCloudSurfLast (the full deskewed cloud, as src/mapOptmization.cpp:1587-1595 passes). */
int liorf_sc_make_and_save(liorf_ctx* ctx, const liorf_point* cloud, int n);
/* appends ready-made descriptors (20x60 fp64 row-major [ring][sector]); keys are derived on the device (a11/a12) */
int liorf_sc_add_descriptors(liorf_ctx* ctx, const double* descs, int count);
int liorf_sc_size(liorf_ctx* ctx);
int liorf_sc_get(liorf_ctx* ctx, int i, double desc[1200], float ringkey[20], double sectorkey[60]);
/* replaces SCManager::detectLoopClosureID() (include/Scancontext.h:73) with the reference's semantics incl. the stale
 * tree (rebuilt every 10th call over keys[0 : n-30]).  cand3 / min_dist nullable diagnostics. */
int liorf_sc_detect_loop_closure_id(liorf_ctx* ctx, int* loop_id, float* yaw_diff_rad, double* min_dist, int* cand3);
/* detectLoopClosureID for Q calls at once.  Answer q is exactly what liorf_sc_detect_loop_closure_id returns when the database
 * held its first n_db[q] entries (query = row n_db[q] - 1) and the stale tree covered keys [0, n_tree[q]) — every output
 * bit-identical, whatever Q, the order of the queries or the search path.  Read-only: the context's own detector state (call
 * counter, tree snapshot), its database and every other search are untouched; works on a borrowed database.
 *   n_db[q] < 31        : loop_id -1, yaw 0, min_dist / cand3 entries untouched (the single call's early-out); never reaches the device
 *   n_tree[q] < 3       : unfilled kNN slots are candidate 0, as in the single call; cand3 holds the substituted ids
 *   LIORF_ERR_ARG, outputs untouched, nothing enqueued: a NULL mandatory array with Q > 0, n_db[q] outside [1, liorf_sc_size],
 *                   or n_db[q] >= 31 with n_tree[q] outside [1, n_db[q] - 30].  Q = 0 is LIORF_OK.
 * One upload of the indices, one download of the answers and one synchronisation, whatever Q.  The ring-key search takes the path
 * liorf_sc_set_search_path selects for a batch of this size.  Python's liorf_b200.sc_tree_schedule gives the n_tree a call history saw. */
int liorf_sc_detect_loop_closure_id_batch(liorf_ctx* ctx, const int* n_db, const int* n_tree, int Q,
                                          int* loop_id, float* yaw_diff_rad, double* min_dist /*nullable*/, int* cand3 /*nullable, [Q][3]*/);
/* batched search (BASELINE config 5): Q queries against the context's database rows [0, n_db) which represent GLOBAL
 * rows [global_offset, global_offset + n_db) (single GPU: offset 0).  The steps of one batch on DEVICE buffers (d_* are device pointers):
 *   prepare: ring keys (a11) of Q query descriptors → d_qkeys [Q][20] f32 (d_qsk / d_qcn, nullable: sector keys / column norms [Q][60] f64)
 *   stage 1: exact top-3 per query → (dist[Q*3], idx[Q*3]); unfilled slots carry idx INT_MAX
 *   stage 2: distanceBtnScanContext for the candidates in [global_offset, global_offset + n_db); every other output slot is left
 *            untouched, except that a candidate of INT_MAX (unfilled) or below 0 gives dist +inf and shift 0 in every context.  The
 *            query's sector key and column norms are derived inside the kernel from its descriptor
 *   decide : strict-< argmin in kNN order + threshold (include/Scancontext.cpp:302-340)
 * Query descriptors (here and in liorf_sc_shard_query_dev / _phases_dev) need only 8-byte alignment in every stage, e.g. a float64
 * tensor view at an odd element offset; 16-byte-aligned ones take the faster loads. */
int liorf_sc_prepare_queries_dev(liorf_ctx* ctx, const void* d_qdescs, int Q, void* d_qkeys /*Q*20 f32*/, void* d_qsk /*Q*60 f64, nullable*/, void* d_qcn /*Q*60 f64, nullable*/);
int liorf_sc_knn_batch_dev(liorf_ctx* ctx, const void* d_qkeys, int Q, int global_offset, void* d_dist, void* d_idx);
int liorf_sc_distance_batch_dev(liorf_ctx* ctx, const void* d_qdescs, const void* d_cand_idx, int Q, int global_offset, void* d_pair_dist /*Q*3 f64*/, void* d_pair_shift /*Q*3 i32*/);
int liorf_sc_decide_dev(liorf_ctx* ctx, const void* d_pair_dist, const void* d_pair_shift, const void* d_cand_idx, int Q,
                        void* d_loop_id, void* d_shift, void* d_dist);
/* tests: out = {SMs, stage-2 CTAs per SM for 16-byte-aligned query descriptors, the same for 8-byte-aligned ones} */
int liorf_debug_sc_distance_occupancy(liorf_ctx* ctx, int out[3]);
/* Ring-key search implementation used by liorf_sc_knn_batch_dev / liorf_sc_query_batch / the sharded search:
 *   0 auto (tensor cores for batches of >= 64 queries against >= 4096 keys), 1 CUDA-core brute force,
 *   2 tcgen05 coarse filter + exact re-rank (csrc/sc_tensor.cuh).  All three return the same exact top-3
 *   (nanoflann arithmetic, include/nanoflann.hpp:383-408, ties by (dist, idx)). */
int liorf_sc_set_search_path(liorf_ctx* ctx, int mode);
/* last tensor-core search: candidates the coarse filter passed to the exact re-rank (summed over the queries) and the
 * number of queries whose candidate list overflowed (answered by an exact scan of all keys instead) */
int liorf_sc_tensor_stats(liorf_ctx* ctx, long long* n_candidates, int* n_overflow);
/* test hook: raw tensor-core distances of Q host ring keys against the database, out[q * ld + k] */
int liorf_sc_tensor_dump(liorf_ctx* ctx, const float* qkeys, int Q, float* out, long long out_capacity, int* ld, float center[20]);
/* single-GPU convenience with host buffers: descriptors of the Q queries → loop ids / shifts / distances */
int liorf_sc_query_batch(liorf_ctx* ctx, const double* qdescs, int Q, int* loop_id, int* shift, double* dist, int* cand3 /*nullable*/);

/* ---- database sharded across GPUs, exchanged through NVLink peer memory (SURVEY §8e, BASELINE config 5) -----------------
 * "Replicated index, sharded payload" — the split the reference's SCManager already has between its search index
 * (polarcontext_invkeys_mat_ / polarcontext_tree_) and the descriptors it indexes (polarcontexts_), include/Scancontext.h:104-113:
 *   rank g holds the descriptor, sector key and column norms of rows [row_begin[g], row_begin[g+1]) (10 560 B per row); the 80-byte fp32
 *   ring key of EVERY row is replicated on every rank (pushed over NVLink by liorf_sc_shard_sync_keys when the database was loaded or grew).
 * One batch = the same Q queries on every rank:
 *   stage 1 (ring-key top-3, include/Scancontext.cpp:289-295) is split by QUERY — rank g answers queries [g Q/G, (g+1) Q/G) against all
 *     keys, which yields the global top-3 directly — and its re-rank kernel writes the result into every rank's window (phase C);
 *   stage 2 (distanceBtnScanContext, :302-317) is split by OWNER of the candidate row; the warp that evaluates a pair writes
 *     {f64 dist, i32 shift} into every rank's window (phase D); every rank then takes the decision (:319-340) for all queries.
 * The kernels push with plain stores over NVLink, fence at system scope, raise flags, and wait on flags in their own window — no
 * NCCL call and no host round trip inside a batch (csrc/sc_shard.cuh).  Exactly the global top-3 are evaluated, so loop ids / shifts /
 * distances / candidate triples equal the unsharded search bit for bit.
 *   liorf_sc_shard_init    : allocate this rank's window for batches of up to q_max queries and a replicated index of up to k_total_max
 *                            rows (0 = this context borrows the index, see liorf_sc_borrow_database); returns the window's cudaIpc handle
 *                            (64 bytes, for peers in other processes) and / or its device pointer (peers in this process)
 *   liorf_sc_shard_connect : map the peers' windows (array of `world` handles or pointers, own entry ignored).  row_begin[world + 1],
 *                            row_begin[0] = 0; the context must hold exactly rows [row_begin[rank], row_begin[rank+1]) (else LIORF_ERR_STATE)
 *   liorf_sc_shard_sync_keys: collective; replicate the ring keys (call again, after a new connect, when the database has grown)
 *   liorf_sc_shard_query_dev: one batch, asynchronous on the context's stream; every rank passes the same queries in the same order;
 *                            global_offset must equal row_begin[rank]; d_cand (nullable) receives the global candidate triples [Q][3] */
/* a second context on the same device searching the SAME database without copying it (several query batches in flight per GPU, one
 * context / stream each); the borrower is read-only, the owner must outlive it and not grow the database meanwhile.  Borrowing from a
 * sharded owner AFTER its liorf_sc_shard_sync_keys also shares the replicated index. */
int liorf_sc_borrow_database(liorf_ctx* dst, liorf_ctx* src);
int liorf_sc_shard_init(liorf_ctx* ctx, int rank, int world, int q_max, int k_total_max, void* ipc_handle_out, void** window_out);
int liorf_sc_shard_connect(liorf_ctx* ctx, const void* ipc_handles, void* const* window_ptrs, const int* row_begin /* world + 1: rows [row_begin[g], row_begin[g+1]) on rank g */);
int liorf_sc_shard_sync_keys(liorf_ctx* ctx);
/* the same in steps (bit 0: push this rank's keys + raise the flags, bit 1: wait for every peer's keys) so that several ranks sharing ONE
 * device (tests) can enqueue every push before any wait */
int liorf_sc_shard_sync_keys_phases(liorf_ctx* ctx, int phases);
int liorf_sc_shard_wait_stats(liorf_ctx* ctx, unsigned long long wait_ns[4], unsigned* batches);   /* time spent waiting for peers per phase (C, D, KEYS, -), measurement */
int liorf_sc_shard_query_dev(liorf_ctx* ctx, const void* d_qdescs, int Q, int global_offset, void* d_loop_id, void* d_shift, void* d_dist, void* d_cand);
/* the same batch enqueued in steps (bit 0: stage 1 of this rank's query slice + push C, bit 1: collect + stage 2 of the owned pairs + push D,
 * bit 2: decision; 7 = everything) so that several ranks sharing ONE device (tests) can interleave their steps and never wait on work that
 * has not been enqueued yet */
int liorf_sc_shard_query_phases_dev(liorf_ctx* ctx, const void* d_qdescs, int Q, int global_offset, void* d_loop_id, void* d_shift, void* d_dist, void* d_cand, int phases);
/* the same batch from HOST buffers: H2D of the Q descriptors (9 600 B each), the search, D2H of the answers, all asynchronous on the context's
 * stream — results are defined after liorf_sync; pinned host buffers make the copies truly asynchronous.  cand3 ([Q][3] global rows) nullable. */
int liorf_sc_shard_query_async(liorf_ctx* ctx, const double* qdescs, int Q, int global_offset, int* loop_id, int* shift, double* dist, int* cand3);
int liorf_sc_shard_debug_nowait(liorf_ctx* ctx, int on);
int liorf_sc_shard_debug_state(liorf_ctx* ctx, unsigned out[68]);   /* debugging: batch / raise / owned-pair counters, error flag, then flag[src][phase] of this rank's window */   /* measurement: consumers skip the flag waits (one rank of G timed alone, tools/profile_sc_shard.py) */

/* ---- loop-closure registration (SURVEY §8f-3) ------------------------------------------------------------------- */
/* The ICP of mapOptimization::performSCLoopClosure (src/mapOptmization.cpp:624-730) without the factor graph:
 * cureKeyframeCloud = loopFindNearKeyframes(loop_key_cur, 0, loop_index), prevKeyframeCloud = loopFindNearKeyframes(loop_key_pre,
 * history_search_num, loop_index) (:821-844; loop_index = the keyframe whose pose transforms every cloud, the reference passes
 * base_key = 0; -1 = each cloud by its own pose as performRSLoopClosure does), VoxelGrid(icp_leaf = loopClosureICPSurfLeafSize),
 * guards (< 300 / < 1000 points → ran = 0), pcl::IterativeClosestPoint with max correspondence distance max_corr_dist
 * (= 2 historyKeyframeSearchRadius), max_iters (100), transformation / fitness epsilons 1e-6, no RANSAC, then getFitnessScore().
 * The caller applies `converged && fitness <= historyKeyframeFitnessScore` (:677). */
typedef struct {
    int ran, converged, convergence_state /* 1 iterations, 2 transform, 3 abs mse, 4 rel mse, 5 no correspondences */, iterations;
    int n_source, n_target;
    float fitness;
    float transform[16];            /* icp.getFinalTransformation(), row-major 4x4 */
    float pose6[6];                 /* its (roll, pitch, yaw, x, y, z) by pcl::getTranslationAndEulerAngles (:707) */
} liorf_icp_result;
int liorf_loop_closure_icp(liorf_ctx* ctx, int loop_key_cur, int loop_key_pre, int history_search_num, int loop_index, float icp_leaf, float max_corr_dist,
                           int max_iters, liorf_icp_result* out);
int liorf_icp_get_clouds(liorf_ctx* ctx, liorf_point* source, int cap_source, liorf_point* target, int cap_target);   /* test hook */
/* performSCLoopClosure's registration for n_pairs keyframe pairs at once (batched verification of loop-closure candidates): pair p is
 * exactly liorf_loop_closure_icp(ctx, loop_key_cur[p], loop_key_pre[p], history_search_num, loop_index[p], icp_leaf, max_corr_dist,
 * max_iters, &out[p]) — every field of out[p] bit-identical to that call, whatever the batch size, order or grouping.  Duplicate pairs
 * and cur == pre are allowed; a pair that fails the size guards gets ran = 0 with n_source / n_target filled in while the others run.
 * Every argument is checked before any work is enqueued: a NULL array (n_pairs > 0), a key outside [0, n_keyframes), a loop_index
 * outside [-1, n_keyframes) or a scalar the single-pair call refuses returns LIORF_ERR_ARG with out untouched; n_pairs = 0 is LIORF_OK.
 * The pairs run in waves of consecutive pairs whose work buffers fit LIORF_ICP_BATCH_WAVE_BYTES of device memory (96 B per raw point
 * of the two selections plus 16 MiB of grid cells per pair, at most 256 pairs; a larger pair runs alone).  The buffers are the call's
 * own and stay allocated with the context, sized by the largest wave so far.  A wave synchronises with the host once after its clouds
 * are built, once per 8 ICP iterations and once for the fitness scores, independently of its pair count; the batch checks the device
 * error flag once.  liorf_icp_get_clouds keeps returning the clouds of the last single-pair call; keyframes, local map and front
 * end are not touched. */
#define LIORF_ICP_BATCH_WAVE_BYTES (4ull << 30)
int liorf_loop_closure_icp_batch(liorf_ctx* ctx, const int* loop_key_cur, const int* loop_key_pre, const int* loop_index, int n_pairs,
                                 int history_search_num, float icp_leaf, float max_corr_dist, int max_iters, liorf_icp_result* out);
int liorf_debug_icp_batch_wave(liorf_ctx* ctx, int max_pairs);   /* tests: at most max_pairs pairs per internal wave (0 = the memory-bounded default) */

/* ---- global map (SURVEY §8f-4) ---------------------------------------------------------------------------------- */
/* mapOptimization::publishGlobalMap (src/mapOptmization.cpp:453-502): key poses within search_radius
 * (globalMapVisualizationSearchRadius) of the newest, thinned by a VoxelGrid of pose_density
 * (globalMapVisualizationPoseDensity), their keyframe clouds transformed by their own poses, concatenated and VoxelGrid(leaf =
 * globalMapVisualizationLeafSize).  search_radius <= 0 takes every keyframe and leaf <= 0 skips the last filter — the map of
 * saveMapService (:379-432, req.resolution).  out == NULL / capacity 0 just returns the size in *n_out. */
int liorf_build_global_map(liorf_ctx* ctx, float search_radius, float pose_density, float leaf, liorf_point* out, int capacity, int* n_out);

/* ---- one LiDAR frame through the whole path ------------------------------------------------------------------- */
/* The call sequence of ImageProjection::cloudHandler (src/imageProjection.cpp:191-204) followed by
 * mapOptimization::laserCloudInfoHandler (src/mapOptmization.cpp:236-275) for a merged node: projectPointCloud →
 * extractSurroundingKeyFrames → downsampleCurrentScan → scan2MapOptimization → transformUpdate clamps → saveFrame →
 * keyframe store + makeAndSaveScancontextAndKeys, and detectLoopClosureID every `loop_every`-th frame (0 = never).
 * One host↔device round trip per frame (the pose).  pts_on_device != 0 → `pts` is a device pointer. */
typedef struct {
    const void* pts; int n; int pts_on_device;
    double time_scan_cur;
    const double *imu_time, *imu_rot_x, *imu_rot_y, *imu_rot_z; int imu_pointer_cur; int deskew_enabled;
    float initial_guess[6];                     /* transformTobeMapped after updateInitialGuess (:899-958) */
    float surrounding_keyframe_density;         /* utility.h:139 */
    float adding_dist_threshold, adding_angle_threshold;   /* utility.h:137-138 */
    float rotation_tollerance, z_tollerance;    /* utility.h:129-130 */
    int max_iters; int loop_every; int frame_index;
    /* use_cloud_info != 0: the initial guess is produced by updateInitialGuess (:899-958) from the context's previous pose and
     * these cloud_info fields (initial_guess[] is ignored), and transformUpdate (:1323-1353) runs in full after the solve */
    int use_cloud_info; liorf_cloud_info_guess cloud_info; int imu_type; int use_imu_heading_initialization; float imu_rpy_weight;
    /* optional look-ahead: the liorf_frame_in of the FOLLOWING frame (NULL = none).  Its cloudHandler part (projectPointCloud) and
     * downsampleCurrentScan are enqueued on a second stream as soon as this frame's solver has been launched and run while the
     * solver iterates — the reference runs imageProjection and mapOptimization as two concurrent nodes with a queue in between
     * (src/imageProjection.cpp:191-204 publishes, src/mapOptmization.cpp:236 consumes).  Only pts / n / pts_on_device / time_scan_cur /
     * imu_* / deskew_enabled / frame_index / surrounding_keyframe_density of `next` are read (the last two also let a frame that
     * became a keyframe start the next frame's extractSurroundingKeyFrames before the call returns); its buffers must stay valid until the call that processes that frame
     * (same frame_index, pts, n) returns.  Results are bit-identical with and without look-ahead. */
    const void* next;
} liorf_frame_in;
typedef struct {
    float pose[6];
    int is_keyframe, keyframe_id;
    int n_kept, n_ds, m_ds, iters, converged, degenerate, ran;
    int loop_checked, loop_id; float loop_yaw;
} liorf_frame_out;
int liorf_process_frame(liorf_ctx* ctx, const liorf_frame_in* in, liorf_frame_out* out);
/* ImageProjection::cloudHandler (src/imageProjection.cpp:191-204) for a frame that a later liorf_process_frame call (same
 * frame_index, pts, n) will consume: asynchronous, second stream, second set of scan buffers.  Primes the pipeline for frame 0;
 * afterwards liorf_frame_in.next does the same from inside liorf_process_frame. */
int liorf_cloud_handler_async(liorf_ctx* ctx, const liorf_frame_in* frame);

/* ---- measurement / introspection (bench.py) ------------------------------------------------------------------- */
/* per-section CUDA-event timing on the context's stream: sections 0 deskew, 1 downsample, 2 map build (transform +
 * VoxelGrid), 3 grid build, 4 scan2map solver, 5 ScanContext make, 6 ScanContext ring-key search, 7 the tcgen05 GEMM
 * kernel inside 6 */
int liorf_enable_timing(liorf_ctx* ctx, int on);
int liorf_enable_timing_mask(liorf_ctx* ctx, unsigned mask);         /* only the sections whose bit is set record events */
int liorf_get_timing(liorf_ctx* ctx, double ms[8], long long calls[8]);
long long liorf_get_launch_count(liorf_ctx* ctx);                     /* kernels launched by this context so far */
int liorf_get_last_counts(liorf_ctx* ctx, int* n_scan, int* n_ds, int* m_ds, int* iters);   /* as of the last liorf_get_pose */
int liorf_debug_qr_solve6(liorf_ctx* ctx, const float* A, const float* b, int n, float* x);   /* tests: the device routine behind cv::solve(DECOMP_QR) 6x6 (src/mapOptmization.cpp:1240) */
int liorf_debug_force_large_voxelgrid(liorf_ctx* ctx, int on);   /* tests: multi-kernel VoxelGrid path on every cloud */
int liorf_debug_voxelgrid_stamps(liorf_ctx* ctx, int enable, unsigned long long* out /* 32, nullable */);   /* debug: phase stamps of the one-kernel VoxelGrid */
int liorf_debug_force_fused_voxelgrid(liorf_ctx* ctx, int on);   /* tests: one-kernel cooperative VoxelGrid path on small clouds too */
int liorf_debug_voxelgrid_grid(liorf_ctx* ctx, int ctas);       /* tests: CTAs of liorf_voxel_grid's one-kernel VoxelGrid, 1..co-resident limit (0 = all SMs) */
int liorf_debug_s2m_global_state(liorf_ctx* ctx, int on);          /* tests: solver keeps per-query state in global memory (the multi-round layout) */
int liorf_debug_s2m_disable_cache(liorf_ctx* ctx, int on);        /* tests: full 27-cell search + plane refit every iteration */
int liorf_debug_s2m_grid(liorf_ctx* ctx, int ctas);               /* tests: solver CTAs of every launch, 2..SMs (0 = defaults) */
int liorf_debug_s2m_clocks(liorf_ctx* ctx, int enable, long long* out /* 64*8, nullable */);
int liorf_debug_s2m_arrivals(liorf_ctx* ctx, int enable, unsigned long long* out /* 64*160, nullable */);   /* %globaltimer stamps (debug) */   /* solver phase clocks (debug) */
int liorf_get_keyframe(liorf_ctx* ctx, int id, liorf_point* out, int capacity, int* n, float pose6[6], double* time);

#ifdef __cplusplus
}
#endif
#endif
