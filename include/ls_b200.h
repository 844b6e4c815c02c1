/* ls_b200.h -- C ABI of the B200-native laser_slam hot path (libls_b200.so).
 *
 * Plain C, plain pointers and sizes; no torch / CUDA types cross this boundary.  Each entry point
 * names the reference interface it replaces (paths relative to the reference repo root).
 *
 * Conventions
 *   - Clouds use the libpointmatcher DataPoints memory layout the reference passes around
 *     (laser_slam/include/laser_slam/common.hpp:14-15,113-120): `features` is a column-major
 *     4xN float matrix, i.e. N consecutive {x, y, z, 1} quadruples; a `normals` descriptor is read
 *     through (pointer, stride-in-floats) so a DxN descriptor block can be passed without copying.
 *   - 4x4 transforms are 16 floats, column-major (PointMatcher::TransformationParameters::data()).
 *   - Host buffers are owned by the caller and only read/written during the call.  Device memory
 *     is owned by the library (ls_ctx / ls_map) and freed by the matching *_destroy.
 *   - Return value: 0 ok; > 0 algorithmic condition (LS_ERR_CONVERGENCE maps to
 *     PointMatcher::ConvergenceError, which laser_slam/src/laser_track.cpp:495-502 catches and
 *     turns into "keep the initial guess"; laser_slam/src/incremental_estimator.cpp:108 lets it
 *     propagate); < 0 argument / CUDA / resource error.  There is no CPU fallback: without a usable
 *     CUDA device ls_b200_init fails with LS_ERR_CUDA.
 *   - Calls on one ls_ctx are serialised by the caller (the reference holds
 *     full_laser_track_mutex_ / full_class_mutex_ around them); distinct contexts are independent
 *     (own stream, own buffers).  Calls are synchronous: results are on the host at return.
 */
#ifndef LS_B200_H_
#define LS_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LS_OK 0
#define LS_ERR_CONVERGENCE 1 /* no point to minimise / NaN  -> PointMatcher::ConvergenceError */
#define LS_ERR_ARG (-1)
#define LS_ERR_CUDA (-2)
#define LS_ERR_NOMEM (-3)
#define LS_ERR_STATE (-4)
#define LS_ERR_NCCL (-5)

typedef struct ls_ctx ls_ctx;
typedef struct ls_map ls_map;

/* ICP chain parameters = the subset of laser_slam/configurations/icp_default.yaml the path uses. */
typedef struct ls_icp_params {
  int max_iterations;   /* CounterTransformationChecker.maxIterationCount      yaml:22-23 */
  float trim_ratio;     /* TrimmedDistOutlierFilter.ratio                      yaml:14-16 */
  int use_differential; /* DifferentialTransformationChecker present           yaml:24-27 */
  float min_diff_rot;   /* minDiffRotErr [rad] */
  float min_diff_trans; /* minDiffTransErr [m] */
  int smooth_length;    /* smoothLength (<= 15) */
  /* spatial-hash tuning (no reference counterpart; results do not depend on these) */
  float cell_size;      /* level-0 cell edge [m]; <= 0 -> 1.0 */
  int leaf_split;       /* subdivide cells holding more points; <= 0 -> 32 (min 16) */
  int max_cells;        /* cap on level-0 cells; <= 0 -> 4194304 */
  /* The DataPointsFilters sections of the chain (icp_default.yaml:1-7).  ls_icp_params_from_yaml reports them here; the
   * registration entry points do NOT apply them -- they take clouds as given, normals included -- the caller does, with
   * ls_keep_point / ls_estimate_normals (what PointMatcher::ICP::compute in include/laser_slam_compat/compat.hpp does). */
  float reading_sampling_prob;    /* readingDataPointsFilters: RandomSamplingDataPointsFilter.prob; 1 = absent */
  int reference_normals_knn;      /* referenceDataPointsFilters: (Sampling)SurfaceNormalDataPointsFilter.knn; 0 = absent */
  float reference_sampling_ratio; /* its ratio (SamplingSurfaceNormal keeps that fraction); 1 = absent */
  int unapplied_modules;          /* YAML modules present that the registration itself does not run (the filter sections above) */
} ls_icp_params;

typedef struct ls_icp_stats {
  int iterations;       /* ICP iterations executed */
  int converged;        /* stopped by the differential checker */
  int max_iter_reached; /* stopped by the counter (flag, not an error) */
  int last_kept;        /* matches with weight 1 in the last iteration */
  float last_limit;     /* trimmed squared-distance limit of the last iteration */
  float used_ratio;     /* last_kept / n (libpointmatcher pointUsedRatio) */
  float device_ms;      /* CUDA-event time of the device work of this call */
  float build_ms;       /* of which: sub-map assembly + spatial-hash build */
  int grid_cells;       /* level-0 cells */
  int grid_tables;      /* fine (8x8x8) tables allocated */
  int grid_overflow;    /* 1 if a table pool overflowed (slower, still exact) */
  float icp_ms;         /* CUDA-event duration of the persistent ICP kernel launch (shared by a batch) */
} ls_icp_stats;

/* ---- context ------------------------------------------------------------------------------- */
int ls_b200_init(int device, ls_ctx** out);
void ls_b200_destroy(ls_ctx* ctx);
const char* ls_b200_last_error(const ls_ctx* ctx); /* text of the last failure on this context */
int ls_b200_version(void);
/* Cap the number of CTAs the persistent ICP kernel of this context may occupy (0 = all that can be co-resident, the
 * default).  Two contexts that each take half of the device run their cooperative launches side by side, so the map build
 * and host-side staging of one overlap the ICP iterations of the other (bench.py drives two such contexts).  A batch of
 * more problems than the budget still gets one CTA per problem, so its launch then occupies more CTAs than the budget. */
int ls_b200_set_icp_cta_budget(ls_ctx* ctx, int ctas);
int ls_b200_icp_cta_budget(const ls_ctx* ctx); /* CTAs the next launch will use at most */
/* Number of this library's kernel launches issued on the context so far (bench "gpu_launches"). */
uint64_t ls_b200_launch_count(const ls_ctx* ctx);

/* icp_.setDefault()-like defaults, but with the values of icp_default.yaml:9-27
 * (replaces PointMatcher::ICP::loadFromYaml at laser_slam/src/laser_track.cpp:14-21). */
void ls_icp_default_params(ls_icp_params* p);
/* Parse the keys of icp_default.yaml this path honours out of a YAML text; unsupported matcher / minimiser / outlier
 * filter names return LS_ERR_ARG; reading / reference DataPointsFilters are reported in the params (see the struct:
 * `unapplied_modules` counts them) because they run upstream of the registration; inspector / logger are ignored. */
int ls_icp_params_from_yaml(const char* yaml_text, ls_icp_params* p);

/* Deterministic stand-in for RandomSamplingDataPointsFilter's `rand() / RAND_MAX < prob`
 * (laser_slam/configurations/icp_default.yaml:1-3; libpointmatcher draws from the process-global libc generator, which is
 * not reproducible): point `index` of a cloud is kept iff hash32(index, salt) < prob * 2^32, a counter-based rule that
 * host, device and oracle evaluate identically.  Returns 1 (keep) or 0. */
int ls_keep_point(uint32_t index, uint32_t salt, float prob);

/* ---- one-shot registration ----------------------------------------------------------------------
 * Replaces PointMatcher::ICP::compute(reading, reference, T0) at
 *   laser_slam/src/laser_track.cpp:496              (scan -> sub-map)
 *   laser_slam/src/incremental_estimator.cpp:108    (sub-map b -> sub-map a on loop closure)
 * reading: 4xN features; reference: 4xM features + normals.  T_out = T_ref<-reading.
 * On LS_ERR_CONVERGENCE T_out == T0.  opt_ids / opt_d2 (may be NULL, length n) receive the
 * correspondence indices (into the reference, -1 = none) and squared distances of the LAST
 * iteration; opt_T_iter_hist (may be NULL, max_iterations*16 floats) the accumulated T_iter after
 * every iteration (centred frame). */
int ls_icp_register(ls_ctx* ctx, const ls_icp_params* prm, const float* reading4, int n,
                    const float* ref4, const float* ref_normals, int normals_stride, int m,
                    const float T0[16], float T_out[16], ls_icp_stats* stats, int32_t* opt_ids,
                    float* opt_d2, float* opt_T_iter_hist);

/* KDTreeMatcher-level entry (icp_default.yaml:9-12): nearest reference point of T0*reading for
 * every reading point, with the reference centred exactly as ICP::compute does.  ids index the
 * reference as given; d2 are squared float32 distances. */
int ls_nn_query(ls_ctx* ctx, const ls_icp_params* prm, const float* reading4, int n, const float* ref4,
                int m, const float T0[16], int32_t* ids, float* d2);

/* RigidTransformation::compute (laser_slam/src/laser_track.cpp:265,485,508,511,630,643):
 * out = T * features, normals rotated by the 3x3 block.  normals/out_normals may be NULL. */
int ls_transform_cloud(ls_ctx* ctx, const float T[16], const float* in4, const float* normals,
                       int normals_stride, int n, float* out4, float* out_normals3);
/* RigidTransformation::checkParameters / correctParameters as used by
 * correctTransformationMatrix (laser_slam/include/laser_slam/common.hpp:136-149).  Host-side. */
int ls_check_rigid(const float T[16]);
void ls_correct_rigid(const float T_in[16], float T_out[16]);

/* ---- device-resident rolling map ------------------------------------------------------------------
 * Replaces LaserTrack::laser_scans_ + the per-scan copy/transform/concatenate loop of
 * LaserTrack::localScanToSubMap (laser_slam/src/laser_track.cpp:466-486) and
 * LaserTrack::buildSubMapAroundTime (laser_track.cpp:602-651): scans are uploaded once, kept in
 * their own sensor frame, and sub-maps are assembled on the device. */
int ls_map_create(ls_ctx* ctx, int capacity_scans, int max_pts_per_scan, ls_map** out);
void ls_map_destroy(ls_map* map);
/* Upload one scan; returns its id through *scan_id (ids grow monotonically; the scan stays
 * addressable until `capacity_scans` newer scans have been pushed). */
int ls_map_push_scan(ls_map* map, const float* features4, const float* normals, int normals_stride, int n,
                     uint64_t* scan_id);
/* The same, enqueued on the map's own upload stream; returns at once.  The host buffers must stay valid (pinned
 * memory, or the copies are synchronous after all) until ls_map_sync() or until a registration that uses the scan
 * has returned.  Registrations wait for exactly the uploads they depend on, so the next scan can go up while the
 * current one is being registered (the reference copies every scan twice on the host before its ICP starts,
 * laser_track.cpp:143,197).  3 <= normals_stride <= 8. */
int ls_map_push_scan_async(ls_map* map, const float* features4, const float* normals, int normals_stride, int n,
                           uint64_t* scan_id);
/* 1 if `p` points into page-locked (pinned) host memory known to the CUDA driver, 0 if not, < 0 on error.  The host
 * layer uses it to pick ls_map_push_scan_async (no staging copy) for DataPoints whose storage is pinned. */
int ls_host_is_pinned(const void* p);
int ls_map_sync(ls_map* map); /* wait for every asynchronous upload of this map */
int ls_map_scan_size(const ls_map* map, uint64_t scan_id); /* points, or <0 if evicted/unknown */

/* Surface normals on the device (SURVEY.md §8 row f1): replaces the SurfaceNormal / SamplingSurfaceNormal
 * DataPointsFilters the reference applies to every input scan and to the sub-map
 * (laser_slam/configurations/icp_default.yaml:5-7, laser_slam/src/laser_track.cpp:27,146).  For every point: exact
 * `knn` nearest neighbours (self included), covariance, eigenvector of the smallest eigenvalue, flipped towards the
 * sensor (origin of the scan frame).  Points with fewer than 3 neighbours get a zero normal.  3 <= knn <= 16.
 * Unlike the reference's filter this one is deterministic (no rand()-based sub-sampling). */
int ls_estimate_normals(ls_ctx* ctx, const float* features4, int n, int knn, float* out_normals3);
/* ls_map_push_scan for clouds that arrive without normals: they are estimated on the device into the slot. */
int ls_map_push_scan_estimate_normals(ls_map* map, const float* features4, int n, int knn, uint64_t* scan_id);

/* Scan -> sub-map registration on resident data.  The reference is the concatenation, in order,
 * of scans part_ids[0..n_parts) each transformed by T_parts[16*p..] (float32, already passed
 * through correctTransformationMatrix by the caller; an exact identity matrix copies the scan
 * verbatim as laser_track.cpp:476 does).  Reading = scan reading_id, untransformed.
 * Correspondence ids index that concatenation. */
int ls_icp_register_submap(ls_ctx* ctx, const ls_icp_params* prm, const ls_map* map, uint64_t reading_id,
                           int n_parts, const uint64_t* part_ids, const float* T_parts, const float T0[16],
                           float T_out[16], ls_icp_stats* stats, int32_t* opt_ids, float* opt_d2,
                           float* opt_T_iter_hist);

/* `batch` independent scan -> sub-map registrations in ONE cooperative launch (several LaserTracks hosted on one
 * GPU: the reference's n_laser_slam_workers tracks, laser_slam/src/incremental_estimator.cpp:22-26).  Problem b
 * uses reading_ids[b], its n_parts[b] parts follow each other in part_ids / T_parts (16 floats per part),
 * T0s / T_outs hold 16 floats per problem, statuses[b] is LS_OK or LS_ERR_CONVERGENCE (then T_out == T0).
 * Results are bit-identical to separate ls_icp_register_submap calls.  1 <= batch <= 160. */
int ls_icp_register_submap_batch(ls_ctx* ctx, const ls_icp_params* prm, const ls_map* map, int batch,
                                 const uint64_t* reading_ids, const int* n_parts, const uint64_t* part_ids,
                                 const float* T_parts, const float* T0s, float* T_outs, ls_icp_stats* stats,
                                 int* statuses);
/* The same in two halves.  begin() stages every problem and launches; end() waits and fetches the results (same
 * T_outs / stats / statuses as above).  In between the host is free -- typically to post the next scans with
 * ls_map_push_scan_async -- but every other call that needs the context's workspaces returns LS_ERR_STATE. */
int ls_icp_register_submap_batch_begin(ls_ctx* ctx, const ls_icp_params* prm, const ls_map* map, int batch,
                                       const uint64_t* reading_ids, const int* n_parts, const uint64_t* part_ids,
                                       const float* T_parts, const float* T0s);
int ls_icp_register_submap_batch_end(ls_ctx* ctx, float* T_outs, ls_icp_stats* stats, int* statuses);

/* ---- one registration sharded by queries over the GPUs of a node (SURVEY.md 8 e-2) -------------------------
 * The scan-matching of LaserTrack::processPoseAndLaserScan (laser_slam/src/laser_track.cpp:196-292) for ONE scan,
 * with the reading split over the GPUs of a node (one process / context per GPU, at most 8).  Every shard pushes the
 * same scans into its own map and makes the same call; per iteration each GPU stores its partial trimmed-select
 * histograms and normal-equation sums into a slot of every peer's exchange buffer over NVLink (CUDA IPC mapping), from
 * inside the persistent kernel.  The result is bit-identical to ls_icp_register_submap on every shard.
 *
 * Setup, once: every shard calls ls_shard_exchange_create (allocates its buffer, returns 64 handle bytes); the handles
 * are gathered in rank order by any means (torch.distributed all_gather, a pipe ...) and passed to
 * ls_shard_exchange_connect on every shard.  After that ls_icp_register_submap_sharded is a COLLECTIVE: every shard
 * makes the same sequence of calls with the same arguments.  A shard that does not show up trips the kernel's watchdog
 * on the others (the launch fails after 8 s; it does not hang).  Close only after every shard is done (the peers store
 * into the buffer). */
#define LS_IPC_HANDLE_BYTES 64
int ls_shard_exchange_create(ls_ctx* ctx, int shard_rank, int shard_count, unsigned char handle[LS_IPC_HANDLE_BYTES]);
int ls_shard_exchange_connect(ls_ctx* ctx, const unsigned char* handles /* shard_count x LS_IPC_HANDLE_BYTES, rank order */);
void ls_shard_exchange_close(ls_ctx* ctx);
int ls_icp_register_submap_sharded(ls_ctx* ctx, const ls_icp_params* prm, const ls_map* map, uint64_t reading_id,
                                   int n_parts, const uint64_t* part_ids, const float* T_parts, const float T0[16],
                                   float T_out[16], ls_icp_stats* stats);

/* Sub-map <-> sub-map registration on resident data: the loop-closure ICP of
 * IncrementalEstimator::processLoopClosure (laser_slam/src/incremental_estimator.cpp:90-115) without the two
 * buildSubMapAroundTime clouds (laser_slam/src/laser_track.cpp:602-651) visiting the host.  Reference = parts of
 * ref_map (normals included), reading = parts of reading_map, each part transformed by its T (an exact identity
 * copies the scan verbatim); the two maps may be the same object.  T_out maps reading coordinates into reference
 * coordinates.  Bit-identical to ls_map_assemble of both sides followed by ls_icp_register. */
int ls_icp_register_submaps(ls_ctx* ctx, const ls_icp_params* prm, const ls_map* ref_map, int n_ref_parts,
                            const uint64_t* ref_part_ids, const float* T_ref_parts, const ls_map* reading_map,
                            int n_reading_parts, const uint64_t* reading_part_ids, const float* T_reading_parts,
                            const float T0[16], float T_out[16], ls_icp_stats* stats);

/* Assemble a sub-map and download it (LaserTrack::buildSubMapAroundTime,
 * LaserTrack::getLocalCloudInWorldFrame laser_track.cpp:247-266).  out4: 4*M floats,
 * out_normals3: 3*M floats (may be NULL); returns M through *m_out. */
int ls_map_assemble(ls_ctx* ctx, const ls_map* map, int n_parts, const uint64_t* part_ids,
                    const float* T_parts, float* out4, float* out_normals3, int* m_out);

/* ---- input side and map maintenance (SURVEY.md §8 row f4) ---------------------------------------------------
 * The steps laser_slam_ros runs on the CPU either side of the registration, on the device.  Host buffers in and out;
 * `device` selects the GPU (no context needed).
 *   ls_ingest_pointcloud2   sensor_msgs/PointCloud2 payload -> DataPoints features: x, y, z floats at byte offsets
 *                           off_* inside records of point_step bytes -> {x, y, z, 1}
 *                           (laser_slam_ros/src/laser_slam_worker.cpp:125, pcl::fromROSMsg + conversion)
 *   ls_filter_cylinder      applyCylindricalFilter (laser_slam_ros/include/laser_slam_ros/common.hpp:194-223, used by
 *                           LaserSlamWorker::getFilteredMap, laser_slam_worker.cpp:415-488): keeps the points inside
 *                           (remove_points_inside == 0: d_xy^2 <= r^2 and |dz| <= h/2) or outside (>= on either) the
 *                           cylinder, in input order; out4 holds up to n points, *n_out the number kept
 *   ls_voxel_grid           pcl::VoxelGrid as getFilteredMap uses it (laser_slam_worker.cpp:434-441): one centroid per
 *                           occupied voxel of edge leaf_size, voxels in ascending cell-index order (x fastest); the
 *                           centroid is the exact mean of the voxel's points (fixed-point sums), rounded once
 *   ls_deskew_revolution    the point arithmetic of the Velodyne assembler
 *                           (sensor_drivers/velodyne_assembler/src/velodyne_assembler_ros.cpp:57-143): the packets of one
 *                           revolution, concatenated (packet k = points [packet_offsets[k], packet_offsets[k+1])), each
 *                           transformed by its T_packets[k] (column-major 4x4: sensor at the packet's time -> sensor at the
 *                           revolution's start, :124-130) and then all by T_final (start -> last packet, :107-108), as two
 *                           float32 transforms like the reference; an exact identity copies verbatim.  The wrap detection
 *                           and the composition of the transforms stay on the host:
 *                           include/laser_slam/velodyne_assembler.hpp */
int ls_ingest_pointcloud2(int device, const void* data, int point_step, int off_x, int off_y, int off_z, int n, float* out4);
int ls_filter_cylinder(int device, const float* in4, int n, const double center[3], double radius_m, double height_m,
                       int remove_points_inside, float* out4, int* n_out);
int ls_voxel_grid(int device, const float* in4, int n, const float leaf_size[3], float* out4, int* n_out);
int ls_deskew_revolution(int device, const float* points4, const int* packet_offsets, int n_packets, const float* T_packets,
                         const float T_final[16], float* out4);

/* ---- pose graph ------------------------------------------------------------------------------------
 * Replaces gtsam::ISAM2 as IncrementalEstimator uses it (laser_slam/src/incremental_estimator.cpp:17-20,
 * 151-163 estimate, 165-266 estimateAndRemove, 268-291 registerPrior).  Poses are 7 doubles
 * {qw,qx,qy,qz,tx,ty,tz}; a factor is what LaserTrack::makeMeasurementFactor /
 * makeRelativeMeasurementFactor build (laser_slam/src/laser_track.cpp:431-458):
 *   LS_FACTOR_PRIOR    error = Local(meas, T(key_a))
 *   LS_FACTOR_BETWEEN  error = Local(meas, T(key_a)^-1 * T(key_b)); fix_a != 0 freezes node a at fixed_a
 * whitened by sigma[6] ([translation x3; rotation x3], gtsam::noiseModel::Diagonal::Sigmas); robust != 0
 * wraps it in Robust(Cauchy(1)) (laser_track.cpp:37-64, incremental_estimator.cpp:29-48). */
#define LS_FACTOR_PRIOR 0
#define LS_FACTOR_BETWEEN 1

typedef struct ls_pg ls_pg;

typedef struct ls_factor {
  int32_t type;
  int32_t robust;
  int32_t fix_a;
  int32_t reserved;
  uint64_t key_a, key_b; /* prior: key_a (key_b ignored) */
  double meas[7];
  double sigma[6];
  double fixed_a[7];
} ls_factor;

typedef struct ls_pg_stats {
  int iterations, n_poses, n_factors, n_border; /* n_border = factors outside the per-track chains */
  double cost_first, cost_last;                 /* robust cost at the first / last linearisation point */
  double last_step_max;                         /* max |component| of the last update */
  float device_ms;
} ls_pg_stats;

int ls_pg_create(int device, ls_pg** out);
void ls_pg_destroy(ls_pg* pg);
const char* ls_pg_last_error(const ls_pg* pg);
uint64_t ls_pg_launch_count(const ls_pg* pg);
int ls_pg_num_poses(const ls_pg* pg);
int ls_pg_num_factors(const ls_pg* pg);
/* gtsam::Values::insert for new nodes; within one track_id the insertion order is the time order
 * (curves::DiscreteSE3Curve::extend, laser_track.cpp:573-582).  track_ids may be NULL (all track 0). */
int ls_pg_add_poses(ls_pg* pg, const uint64_t* keys, const uint32_t* track_ids, const double* poses7, int n);
int ls_pg_set_poses(ls_pg* pg, const uint64_t* keys, const double* poses7, int n);
/* isam2.update(newFactors, ...): out_indices (may be NULL) receives ISAM2Result::newFactorsIndices. */
int ls_pg_add_factors(ls_pg* pg, const ls_factor* factors, int n, uint64_t* out_indices);
/* isam2.update(..., removeFactorIndices) (incremental_estimator.cpp:258). */
int ls_pg_remove_factors(ls_pg* pg, const uint64_t* indices, int n);
/* gn_iters Gauss-Newton iterations over the whole graph on the device (3 = one estimate() call:
 * update(new) + update() + update(), incremental_estimator.cpp:156-159). */
int ls_pg_optimize(ls_pg* pg, int gn_iters, ls_pg_stats* stats);
/* gtsam::Marginals(graph, values).marginalCovariance(key) for each of keys[0..n)
 * (LaserTrack::updateCovariancesFromGTSAMValues, laser_slam/src/laser_track.cpp:421-429): the 6x6 block of the inverse
 * Gauss-Newton Hessian at the CURRENT estimate (robust factors at their current Cauchy weights), tangent order
 * [translation; rotation], row-major, 36 doubles per key. */
int ls_pg_marginals(ls_pg* pg, const uint64_t* keys, int n, double* out_cov36);
/* isam2.calculateEstimate(): all keys and poses (either pointer may be NULL); *n = number of poses. */
int ls_pg_get_poses(const ls_pg* pg, uint64_t* out_keys, double* out_poses7, int* n);

/* ---- multi-GPU -----------------------------------------------------------------------------------------
 * The path shards by independent tracks, one per GPU (the reference's n_laser_slam_workers LaserTracks,
 * laser_slam/src/incremental_estimator.cpp:22-26); the only exchange is one 32-byte record per rank per step
 * so that every rank can feed the shared estimator: a single ncclAllGather over NVLink.  NCCL is resolved at
 * run time (dlopen), so single-GPU users need no NCCL at all. */
typedef struct ls_comm ls_comm;

typedef struct ls_pose_record {
  float delta[6];  /* translation x3, rotation vector x3 of the step's T_a_b */
  int32_t status;  /* return code of the registration that produced it */
  int32_t key;     /* caller-defined (e.g. scan counter) */
} ls_pose_record;  /* 32 bytes */

int ls_comm_unique_id(void* id128);                       /* rank 0: ncclGetUniqueId -> 128 bytes to broadcast */
int ls_comm_init(int device, int rank, int nranks, const void* id128, ls_comm** out);
void ls_comm_destroy(ls_comm* comm);
const char* ls_comm_last_error(const ls_comm* comm);
/* all[nranks] <- every rank's record (rank order). */
int ls_comm_allgather_pose_records(ls_comm* comm, const ls_pose_record* mine, ls_pose_record* all);
/* The same in two halves: begin() only enqueues (copy in, ncclAllGather, copy out) on the communicator's stream
 * and returns; end() waits for it.  A track posts its step's record and collects it before posting the next one,
 * so the slowest rank of a step no longer stalls the others on the host (the estimator consumes the factors
 * asynchronously anyway, reference incremental_estimator.cpp:151-163).  One exchange in flight at a time
 * (LS_ERR_STATE otherwise). */
int ls_comm_allgather_pose_records_begin(ls_comm* comm, const ls_pose_record* mine);
int ls_comm_allgather_pose_records_end(ls_comm* comm, ls_pose_record* all);

#ifdef __cplusplus
}
#endif
#endif /* LS_B200_H_ */
