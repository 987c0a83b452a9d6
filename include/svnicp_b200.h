/*
 * svnicp_b200.h -- C ABI of the B200-native SVN-ICP registration inner loop.
 *
 * This is the drop-in boundary for the reference's registration-class interface
 * (svnicp::SVGDICP / svnicp::SVNICP, reference svn-icp/include/core/SVGDICP.h:64-211 and
 * SVNICP.h:29-80).  Each entry point names the reference member it replaces.  Plain pointers
 * and sizes only: no torch, no C++ types, no exceptions cross this boundary.  A header-only C++
 * mirror of the reference classes on top of this ABI is in
 * svn_icp_b200/include/svnicp/SVNICP.hpp; INTEGRATION.md shows the binding a reference
 * maintainer would add.
 *
 * Conventions
 *   - one handle per caller thread (the reference class is not thread safe either,
 *     OdometryPipeline.cpp:106-110); calls on a handle are blocking unless stated.
 *   - every function returns SVNICP_OK (0) or a negative svnicp_status; svnicp_align returns the
 *     reference's SteinICPState (1 = ALIGN_SUCCESS, 2 = NO_OPTIMIZER) or a negative status.
 *     svnicp_last_error() gives the message (CUDA / NCCL error text included).
 *   - there is NO CPU fallback: without a CUDA device svnicp_create fails with
 *     SVNICP_ERR_NO_DEVICE.
 *   - clouds are float64 [N][3] row-major exactly like the reference's tensors
 *     (SVGDICP.h:207 data_type = kFloat64); particles are [6][P] component-major
 *     (x,y,z,rx,ry,rz rows), the layout of init_pose [6,P,1] and of get_particles()
 *     (SVGDICP.cpp:515-520).
 */
#ifndef SVNICP_B200_H
#define SVNICP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SVNICP_B200_ABI_VERSION 2

typedef struct svnicp_handle_t *svnicp_handle;

typedef enum {
  SVNICP_OK = 0,
  SVNICP_ERR_INVALID = -1,    /* bad argument / call order                       */
  SVNICP_ERR_NO_DEVICE = -2,  /* no CUDA device or wrong architecture (need sm_100) */
  SVNICP_ERR_CUDA = -3,       /* CUDA runtime error, see svnicp_last_error       */
  SVNICP_ERR_NCCL = -4,       /* NCCL error / libnccl not loadable               */
  SVNICP_ERR_OOM = -5
} svnicp_status;

/* SteinICPState, SVGDICP.h:59-62 */
#define SVNICP_ALIGN_SUCCESS 1
#define SVNICP_NO_OPTIMIZER 2

/* class_type switch of OdometryPipeline.cpp:282-288 */
#define SVNICP_CLASS_SVNICP 0
#define SVNICP_CLASS_SVGDICP 1

/* largest particle_count svnicp_create accepts: the bandwidth median counts the P^2 pairwise distances in 32-bit bins */
#define SVNICP_MAX_PARTICLES 65535

/* SteinICPParam (SVGDICP.h:41-57) + ParticleWeightOpt (SVNICP.h:25-27); same defaults. */
typedef struct {
  int32_t iterations;            /* 50   */
  int32_t use_minibatch;         /* 0    (never enabled by the reference, SVGDICP.cpp:178-185) */
  int32_t batch_size;            /* 50   (overwritten with N_s, SVGDICP.cpp:181)               */
  double lr;                     /* 0.02 */
  double max_dist;               /* 1.0  */
  int32_t normalize_cloud;       /* 1    (unused by the hot path)                              */
  char optimizer[16];            /* "Adam" | "RMSprop" | "SGD" | "Adagrad" (SVGDICP only)     */
  int32_t check_early_stop;      /* 0    */
  int32_t convergence_steps;     /* 5    (unused by the hot path)                              */
  double convergence_threshold;  /* 1e-5 */
  int32_t KNN_count;             /* 100  */
  int32_t SVN_full_grad;         /* 1    */
  int32_t use_weight_mean;       /* 0    ParticleWeightOpt                                     */
  /* ---- extensions (0 = default); not in the reference ---- */
  double grid_cell;              /* candidate-builder voxel-hash cell edge in metres (0 -> 1.5) */
  int32_t debug_corr;            /* 1 -> keep per-(particle,point) correspondences of the LAST executed
                                    iteration for svnicp_get_correspondences (parity tests)    */
  int32_t flags;                 /* SVNICP_FLAG_* bit mask, read once by svnicp_create (A/B measurements; 0 = the
                                    measured-best default path)                                  */
  int32_t gn_stages;             /* bits 0-7: TMA ring depth of the Gauss-Newton kernel (0 -> 4); bits 8-15: refill lag in tiles (0 -> 2 when depth >= 4, else 1) */
  int32_t gn_smem_kb;            /* shared-memory budget of the Gauss-Newton tile ring in KiB (0 -> 110, at most 150) */
} svnicp_params;

/* svnicp_params.flags (all default off; none changes a result beyond the documented summation-order effects) */
#define SVNICP_FLAG_NO_PARTICLE_SORT 1  /* keep the caller's particle order internally (no pose-space ordering)      */
#define SVNICP_FLAG_FILTER_FULL 2       /* prune from the full K-slot candidate table every iteration (no list reuse) */
#define SVNICP_FLAG_NCCL_GATHER 8       /* sharded: ncclAllGather per iteration instead of the peer-memory exchange    */
#define SVNICP_FLAG_DEBUG_SYNC 32       /* synchronise after every launch group of an iteration and log it to stderr      */
#define SVNICP_FLAG_WATCHDOG 64         /* svnicp_align polls the streams instead of blocking and reports a scan that does not
                                           finish within 8 s (which stream, the device-side iteration state) as an error     */
#define SVNICP_FLAG_NO_GRAPH 128        /* never replay iterations as CUDA graphs (A/B measurements)                      */
#define SVNICP_FLAG_FORCE_GRAPH 256     /* replay iterations >= 1 as CUDA graphs whatever the problem size (default: only
                                           unsharded SVN-ICP handles without early stop and N_s * P <= 1e7: host-enqueue bound) */
#define SVNICP_FLAG_REUSE_STATS 16      /* svnicp_get_prune_stats reports the fraction of rows served by list reuse    */

/* Fill with the defaults of SteinICPParam (SVGDICP.h:41-57). */
void svnicp_default_params(svnicp_params *p);

int svnicp_abi_version(void);

/* SVNICP::SVNICP / SVGDICP::SVGDICP (SVNICP.cpp:20-38, SVGDICP.cpp:22-44).
 * init_pose: [6][P] host doubles, may be NULL (zeros).  device: CUDA ordinal (-1 = current).
 * class_type SVNICP_CLASS_SVNICP: particles are [t ; Log R] (axis-angle), Gauss-Newton + Stein Variational Newton step.
 * class_type SVNICP_CLASS_SVGDICP: particles are (x,y,z,roll,pitch,yaw) ZYX Euler (SVGDICP.cpp:226-260), first-order
 *   gradient (:398-455), RBF SVGD step (:457-474), params->optimizer update (:142-170, :476-494); svnicp_align returns
 *   SVNICP_NO_OPTIMIZER for an unknown optimizer name.  The constructor's init_pose seeds pose_particles_, which
 *   add_cloud does not refresh (:46-62): iteration 0 of a scan evaluates the kernel on the previous result.
 * use_minibatch != 0 is rejected (the reference never enables it, :178-185); so is particle_count > SVNICP_MAX_PARTICLES. */
int svnicp_create(svnicp_handle *out, const svnicp_params *params, int particle_count, const double *init_pose,
                  int class_type, int device);
void svnicp_destroy(svnicp_handle h);
const char *svnicp_last_error(svnicp_handle h); /* h may be NULL: last creation error */

/* Launch everything on this CUDA stream (cudaStream_t as void*; NULL = the handle's own stream).
 * The reference uses the current CUDA stream (knn.cu:331). */
int svnicp_set_stream(svnicp_handle h, void *cuda_stream);

/* Particle sharding across the GPUs of one box (no reference counterpart, SURVEY.md 8(e)):
 * every rank owns particles [rank*P/n, (rank+1)*P/n).  SVN-ICP class: the ranks map each other's record buffers through
 * CUDA IPC and the owner of a particle stores its record straight into every peer over NVLink (no collective call per
 * iteration; needs one process per GPU); if that cannot be set up, or with SVNICP_FLAG_NCCL_GATHER, and for the SVGD-ICP
 * class, one ncclAllGather per iteration carries the packed per-particle records instead.  unique_id: 128 bytes from svnicp_nccl_unique_id on rank 0,
 * distributed by the caller (MPI / torch.distributed / files).  libnccl.so.2 is dlopen'ed. */
int svnicp_nccl_unique_id(void *id128);
int svnicp_init_sharding(svnicp_handle h, const void *unique_id128, int rank, int n_ranks);

/* SVGDICP::add_cloud (SVGDICP.cpp:46-62).  source [n_s][3], target [n_t][3], init_pose [6][P]
 * (host).  Clouds are copied (the reference clones, :55-56).  *_device: 1 if the cloud pointer is
 * device memory on the handle's GPU. */
int svnicp_add_cloud(svnicp_handle h, const double *source, int64_t n_s, int source_on_device, const double *target,
                     int64_t n_t, int target_on_device, const double *init_pose);

/* SVGDICP::set_initial_mean (SVGDICP.h:102-110).  R0 row-major 3x3 (= gtsam Rot3::matrix()), t0[3]. */
int svnicp_set_initial_mean(svnicp_handle h, const double R0[9], const double t0[3]);

/* SVNICP::stein_align / SVGDICP::stein_align (SVNICP.cpp:41-114, SVGDICP.cpp:66-140).  Blocking. */
int svnicp_align(svnicp_handle h);

/* getters: SVNICP.cpp:281-308, SVGDICP.cpp:497-534, SVGDICP.h:94-100 */
int svnicp_get_transformation(svnicp_handle h, double out6[6]);
int svnicp_get_distribution(svnicp_handle h, double out6[6]);
int svnicp_get_cov_matrix(svnicp_handle h, double out36[36]);
int svnicp_get_particles(svnicp_handle h, double *out_6xP);
int svnicp_get_particle_weight(svnicp_handle h, double *out_P);
int svnicp_get_particle_history(svnicp_handle h, float *out_Ix6xP, int32_t *rows /* = iterations */);
int svnicp_get_runtime(svnicp_handle h, double out3[3]); /* {knn s, update s, finish_iter} */
int svnicp_set_k(svnicp_handle h, int k);
int svnicp_set_threshold(svnicp_handle h, double max_dist);

/* initialize_particles (ICPUtils.cpp:45-58) and initialize_particles_gaussian (:60-75): fills
 * [6][P] host doubles from a counter-based RNG (seeded; torch::rand is not reproducible). */
int svnicp_initialize_particles(int particle_count, const double ub[6], const double lb[6], uint64_t seed, double *out_6xP);
int svnicp_initialize_particles_gaussian(int particle_count, const double cov_diag[6], uint64_t seed, double *out_6xP);

/* ---- parity / debug taps (no reference counterpart; used by tests and bench only) ---- */
int svnicp_iterations_done(svnicp_handle h, int32_t *out);
/* candidate table of the last scan: global map indices [n_s][K], ascending (d0^2, index).  On a sharded handle the
 * index table is only all-gathered when the handle was created with debug_corr (out_idx then errors otherwise). */
int svnicp_get_candidates(svnicp_handle h, int32_t *out_idx /*[n_s][K]*/, float *out_rel_xyz /*[n_s][K][3] or NULL*/);
/* fp32 source as the kernels see it: R0*s [n_s][3] */
int svnicp_get_source_f32(svnicp_handle h, float *out_xyz);
/* last executed iteration (needs debug_corr): fp32 particle transforms [P_local][12] (A' row-major 9, tau 3),
 * chosen global map index [P_local][n_s] and mask [P_local][n_s]. */
int svnicp_get_correspondences(svnicp_handle h, float *out_transforms, int32_t *out_idx, uint8_t *out_mask);
/* Gauss-Newton system of the last executed iteration for ALL particles: H [P][36], b [P][6], x [P][6]. */
int svnicp_get_gn_system(svnicp_handle h, double *out_H, double *out_b, double *out_x);
/* Stein step of the last executed iteration, local slice: delta [P_local][6]; bandwidth h. */
int svnicp_get_stein(svnicp_handle h, double *out_delta, double *out_bandwidth);
/* mean candidates per (point) kept by the exact pruning pass, per iteration [iterations]
 * (handle created with SVNICP_FLAG_REUSE_STATS: the fraction of rows pruned from the previous iteration's list) */
int svnicp_get_prune_stats(svnicp_handle h, double *out_mean_kept, int32_t *rows);
/* how each iteration's bandwidth median was found, per iteration [iterations]: 0 sort of all pairs (P <= 64), 1 linear
 * histogram around the previous median, 2 radix select (iteration 0, or the median left that histogram's window), 3 radix
 * select after the histogram bin held too many values to pick from; -1 none (P == 1, iterations that did not run) */
int svnicp_get_median_paths(svnicp_handle h, int32_t *out, int32_t *rows);
/* device time of the phases of the last scan in ms: {setup, iterations, epilogue, total} */
int svnicp_get_timing(svnicp_handle h, double out4[4]);
/* local particle slice [lo, hi) */
int svnicp_get_slice(svnicp_handle h, int32_t *lo, int32_t *hi);
/* per-phase device timing of the next scans (events around every launch group; small overhead).
 * phase ms summed over the iterations of the last scan: {prep, filter, gn, finalize, gather, stein, setup, #iterations} */
int svnicp_set_profiling(svnicp_handle h, int on);
int svnicp_get_phase_times(svnicp_handle h, double out8[8]);
/* {n_s, n_t, K, brute-force fallback queries of the candidate builder, TB, n_slices, n_pgroups, iterations enqueued} */
int svnicp_get_scan_info(svnicp_handle h, int64_t out8[8]);
/* globaltimer stamps (ns) inside the last k_tail launch of the last scan (profiling on): CTA 0 {start, after the peer wait,
 * after the Stein sums, after the pose update}, last CTA {start of the ball reduction, end}; tuning aid */
int svnicp_get_tail_stamps(svnicp_handle h, double out8[8]);
/* number of kernel launches issued by the last svnicp_align */
int svnicp_get_launch_count(svnicp_handle h, int64_t *out);

/* Registration objective of the LAST scan at M caller-given poses (no reference counterpart): a fitness score to gate the map
 * update on, to compare hypotheses (e.g. an IMU prediction against the registered pose), and the information matrix H at a pose.
 * poses: [6][M] host doubles in the handle's particle convention (SVN-ICP: [t ; Log R]; SVGD-ICP: x,y,z,roll,pitch,yaw ZYX
 *   Euler), relative to the scan's initial mean exactly like the particles: T_world = T0 * T(x).  get_transformation() and
 *   all-zeros (= T0) are valid inputs.
 * For every pose, against the candidate table of the last stein_align (1-NN among the K candidates of each source point,
 *   the same fp32 arithmetic and tie-break as the registration; mask d^2 < max_dist, Q1; the current set_threshold value):
 *   out_stats [M][3]  {inlier count, inlier fraction = count / N_s, inlier RMSE in metres (0 when there are no inliers)}
 *   out_H [M][36], out_b [M][6]  (may be NULL)  Newton_grad_right at that pose (SVNICP.cpp:116-164, with Q1-Q3), in the
 *     layout of svnicp_get_gn_system -- for both classes (right perturbation in [t ; omega])
 *   out_mask [M][N_s] (may be NULL)  1 where the source point is an inlier
 *   out_idx [M][N_s]  (may be NULL; needs debug_corr)  global map index of the chosen candidate
 * Blocking, on the handle's stream; changes no state of the handle (particles, getters, history, timing, launch count).
 * Sharded handles hold the whole table: rank-local, no communication, the same result on every rank.
 * SVNICP_ERR_INVALID before the first stein_align, or after add_cloud / set_initial_mean / set_k until the next one. */
int svnicp_evaluate(svnicp_handle h, int n_poses, const double *poses_6xM, double *out_stats, double *out_H, double *out_b,
                    uint8_t *out_mask, int32_t *out_idx);

/* ---------------------------------------------------------------------------------------------
 * Throughput mode: S independent odometry streams on one GPU (BASELINE.json configs[3]; no reference counterpart -- the
 * reference runs one SVNICP instance per node process).  A batch owns one SVN-ICP handle per stream; use
 * svnicp_batch_stream(b, s) with svnicp_add_cloud / svnicp_set_initial_mean / the getters exactly as for a single handle
 * (do not destroy it, do not call svnicp_set_stream on it), and svnicp_batch_align instead of svnicp_align: it enqueues the
 * scans of all streams iteration by iteration so that they overlap on the GPU, then waits for all of them.  Each stream's
 * result is bit-identical to svnicp_align on that handle.  init_pose: [S][6][P] or NULL.  states: [S] SteinICPState or a
 * negative status per stream; the return value is SVNICP_ALIGN_SUCCESS or the last negative status.
 * --------------------------------------------------------------------------------------------- */
typedef struct svnicp_batch_t *svnicp_batch;
int svnicp_batch_create(svnicp_batch *out, const svnicp_params *params, int n_streams, int particle_count, const double *init_pose,
                        int device);
void svnicp_batch_destroy(svnicp_batch b);
const char *svnicp_batch_last_error(svnicp_batch b);
int svnicp_batch_size(svnicp_batch b);
svnicp_handle svnicp_batch_stream(svnicp_batch b, int s);
int svnicp_batch_align(svnicp_batch b, int32_t *states);

/* ---------------------------------------------------------------------------------------------
 * Device-resident local map: svnicp::VoxelHashMap (svn-icp/include/core/VoxelHashMap.h:28-72,
 * src/core/VoxelHashMap.cpp:22-101) kept in HBM, so the target cloud of svnicp_add_cloud
 * (target_on_device = 1) never crosses PCIe (the reference rebuilds and re-uploads it every scan,
 * OdometryPipeline.cpp:577-581, :630).  Same status codes; no CPU fallback.
 * --------------------------------------------------------------------------------------------- */
typedef struct svnicp_map_t *svnicp_map;
/* VoxelHashMap(voxel_size, max_range, max_pointscount) (VoxelHashMap.h:40-43); capacity_voxels bounds the
 * number of live voxels (the table holds 2x that many slots); max_pointscount <= 32. */
int svnicp_map_create(svnicp_map *out, double voxel_size, double max_range, int max_pointscount, int64_t capacity_voxels, int device);
void svnicp_map_destroy(svnicp_map m);
const char *svnicp_map_last_error(svnicp_map m);
/* Clear() (VoxelHashMap.h:54) */
int svnicp_map_clear(svnicp_map m);
/* AddPointCloud(new_cloud, new_pose) (VoxelHashMap.cpp:22-43) including RemoveFarPointCloud(new_pose.translation())
 * (:93-101).  xyz: [n][3] sensor-frame points, float (dtype_f64 = 0, pcl::PointXYZ) or double; host or device.
 * R row-major 3x3, t[3] = new_pose.  A voxel keeps its first max_pointscount points in cloud order. */
int svnicp_map_add_cloud(svnicp_map m, const void *xyz, int64_t n, int dtype_f64, int on_device, const double R[9], const double t[3]);
/* GetMap() (position = NULL, VoxelHashMap.cpp:45-51) / GetMap(pose, max_range) (:53-63; position = pose.translation()).
 * *device_xyz: device pointer to [*n][3] doubles owned by the map, valid until the next call on it -- pass it to
 * svnicp_add_cloud with target_on_device = 1.  Point order is arbitrary (as the reference's hash-map iteration). */
int svnicp_map_get(svnicp_map m, const double position[3], double max_range, const double **device_xyz, int64_t *n);
/* copy the first n points of the last svnicp_map_get result to the host (tests / visualisation) */
int svnicp_map_download(svnicp_map m, double *out_xyz, int64_t n);
/* Size() / Empty() (VoxelHashMap.h:55-56): live voxels and stored points */
int svnicp_map_size(svnicp_map m, int64_t *voxels, int64_t *points);
/* Registration objective of a scan at M caller-given poses against the map itself (no reference counterpart): score initial
 * guesses before registration, gate a scan against the map, check relocalisation or loop-closure poses.
 * source: [n][3] sensor-frame points, float (dtype_f64 = 0) or double, host or device (as svnicp_map_add_cloud).
 * poses: [6][M] host doubles x = [t ; omega] relative to T0 = (R0 row-major, t0), the SVN-ICP particle convention:
 *   T_world = T0 * (Exp(omega), t), i.e. R~ = R0 Exp(omega), t~ = t0 + R0 t.  x = 0 scores T0 itself.
 * Per pose and source point: q = R~ s + t~ in fp64 (the fma order of the scan's q0; x = 0 gives q0 bit for bit) and the
 *   EXACT nearest stored map point m (float widened to double, d^2 in the fp64 fma order of the candidate builder) among those
 *   with d^2 < max_dist; an exact tie goes to the lexicographically smallest (x, y, z).  The same choice as a brute-force sweep
 *   over GetMap().  max_dist has the registration's meaning (squared metres, Q1) and is also the robust scale D.
 *   A non-finite query has no correspondence.
 *   out_stats [M][3]  {inlier count, count / n, inlier RMSE in metres (0 without inliers)}
 *   out_H [M][36], out_b [M][6]  (may be NULL)  Newton_grad_right at that pose on these correspondences (Q1-Q3: points without
 *     a correspondence add I3 to the translation block), the layout of svnicp_get_gn_system
 *   out_mask [M][n]  (may be NULL)  1 where the point has a correspondence
 *   out_nearest [M][n][3]  (may be NULL)  float coordinates of the chosen map point, zeros where there is none
 * Each pose's outputs are the same bits whatever M, its position among the poses, or the call.  Blocking, on the map's stream;
 * changes no state of the map (Size(), the table, the last svnicp_map_get result stay valid).
 * SVNICP_ERR_INVALID for null pointers, n outside [1, 2^30], n_poses < 1, a non-finite or non-positive max_dist, and a search
 * radius sqrt(max_dist) beyond 4 voxels (ceil(sqrt(max_dist) / voxel_size) > 4). */
int svnicp_map_evaluate(svnicp_map m, const void *source, int64_t n, int dtype_f64, int on_device, const double R0[9],
                        const double t0[3], int n_poses, const double *poses_6xM, double max_dist, double *out_stats,
                        double *out_H, double *out_b, uint8_t *out_mask, float *out_nearest);
/* Exhaustive search of a scan against the map over a regular grid of poses (no reference counterpart): relocalisation,
 * loop-closure checks, recovery from a lost track.  Pose convention, source, max_dist, the search-radius limit and the inlier
 * test are those of svnicp_map_evaluate.
 * Grid: axis a = 0..5 of x = [t ; omega] has counts[a] >= 1 values x_a(i) = ((double)i - 0.5 * (double)(counts[a] - 1)) * steps[a],
 *   i = 0 .. counts[a]-1 (centred on T0; steps finite and >= 0).  M = prod(counts) <= 2^31 - 1.  Flat grid index
 *   g = i0 + counts[0] * (i1 + counts[1] * (i2 + ...)), axis 0 (t_x) fastest.
 * Score of a pose = its inlier count: source points with a stored map point at d^2 < max_dist -- the count svnicp_map_evaluate
 *   returns for the same pose, bit for bit.
 * Ranking: count descending, then g ascending (a total order: the result does not depend on scheduling or slot layout).
 *   out_index [k] int64  the winners' g, best first
 *   out_poses [6][k]     their grid values, to pass on to svnicp_map_evaluate or svnicp_set_initial_mean (through T0)
 *   out_stats [k][3]     svnicp_map_evaluate's {count, fraction, RMSE} of each winner, bit for bit
 *   out_counts [M] int32 (may be NULL)  the score of every grid pose, in g order
 * Host outputs.  Blocking, on the map's stream; changes no state of the map.  SVNICP_ERR_INVALID: svnicp_map_evaluate's argument
 * errors, null counts / steps / outputs, a count < 1, a negative or non-finite step, M > 2^31 - 1, top_k outside
 * [1, min(M, 1024)].
 * Path: with out_counts == NULL, a grid of at least 16 * top_k poses whose translation axes can be cut into blocks takes a
 * branch-and-bound path that counts only the blocks whose inlier bound can still reach the k-th count; every other call counts
 * every pose.  Both return the same bits (svnicp_map_search_info reports which ran). */
int svnicp_map_search(svnicp_map m, const void *source, int64_t n, int dtype_f64, int on_device, const double R0[9], const double t0[3],
                      const int32_t counts[6], const double steps[6], double max_dist, int top_k, int64_t *out_index,
                      double *out_poses_6xK, double *out_stats, int32_t *out_counts);
/* The work done by the last svnicp_map_search on this map that returned SVNICP_OK (SVNICP_ERR_INVALID before the first one):
 *   out8 = {path (0 every pose counted, 1 pruned), grid poses M, poses per full block, blocks, blocks counted, poses counted
 *           exactly, bound queries (blocks * n), bound violations (a pose counting more than its block's bound: always 0)}
 * On path 0: poses per block 0, blocks 0, blocks counted 0, poses counted M, bound queries 0, violations -1. */
int svnicp_map_search_info(svnicp_map m, int64_t out8[8]);
/* Gauss-Newton refinement of M pose hypotheses of one scan against the map (no reference counterpart): the continuous step after
 * svnicp_map_search, whose out_poses may be passed in unchanged.  Source, pose convention, correspondences (exact nearest stored
 * point with d^2 < max_dist), max_dist as the robust scale and the search-radius limit are those of svnicp_map_evaluate.
 * One iteration of one pose (the single-particle SVN-ICP step, SVNICP.cpp:41-114 with P = 1, :268-279):
 *   H, b = svnicp_map_evaluate's system at x (the same bits); delta = -H^-1 b (LDL^T, H carries + 1e-6 I);
 *   R' = Exp(omega) Exp(delta_w), t' = R' J_l(delta_w) delta_t + t with J_l = I at delta_w = 0 exactly (the reference gives NaN);
 *   x' = [t' ; Log(R')] with the principal Log (|omega| <= pi, accurate at pi); an exactly zero delta leaves x unchanged.
 * A pose stops after the update with |delta|_2 < tol, or after `iterations` updates (tol = 0 runs them all); poses are independent.
 *   out_poses [6][M]      the final x (may alias poses)
 *   out_iterations [M]    updates applied
 *   out_step [M]          |delta|_2 of the last update (may be NULL)
 *   out_stats [M][3], out_H [M][36], out_b [M][6]  svnicp_map_evaluate at the final x, bit for bit (H, b may be NULL)
 * Each pose's outputs are the same bits whatever M, its position, the call or the slot layout.  The loop runs on the map's
 * stream without host round trips; blocking; changes no state of the map.  SVNICP_ERR_INVALID: svnicp_map_evaluate's argument
 * errors, null poses / out_poses / out_iterations / out_stats, n_poses outside [1, 65536], iterations outside [1, 1000], a
 * negative or non-finite tol. */
int svnicp_map_refine(svnicp_map m, const void *source, int64_t n, int dtype_f64, int on_device, const double R0[9], const double t0[3],
                      int n_poses, const double *poses_6xM, double max_dist, int iterations, double tol, double *out_poses_6xM,
                      int32_t *out_iterations, double *out_step, double *out_stats, double *out_H, double *out_b);
/* Snapshot of the map's content (no reference counterpart), to save a map and restore it bit for bit with svnicp_map_import:
 *   voxels [V][3] int32  voxel indices (vx, vy, vz) in ascending lexicographic order
 *   counts [V]    int32  points per voxel, 1 <= count <= max_pointscount
 *   xyz [Npts][3] float  each voxel's points one after another, in the voxel order, and inside a voxel in stored order
 *                        (arrival order: the first point is the one GetMap(pose, r) and RemoveFarPointCloud test)
 * n_voxels / n_points must equal svnicp_map_size (V, Npts).  The snapshot depends on the content only, not on the slot layout,
 * the table capacity or the map's history: two maps that hold the same content give the same bytes.  Outputs are host memory,
 * or device memory on the map's GPU with on_device = 1.  Blocking, on the map's stream.  Changes no state of the map (the table,
 * Size(), the last svnicp_map_get result and its device pointer stay valid). */
int svnicp_map_export(svnicp_map m, int32_t *voxels, int32_t *counts, float *xyz, int64_t n_voxels, int64_t n_points, int on_device);
/* Replace the map's content by a snapshot in the layout of svnicp_map_export (any earlier content is discarded; no transform, no
 * RemoveFarPointCloud).  The voxels may come in any order; each voxel's points are stored in the order given.  Inputs are host
 * memory, or device memory on the map's GPU with on_device = 1.  Blocking.  All or nothing: on any error the map is exactly as
 * before.  SVNICP_ERR_INVALID for null pointers with a size > 0, negative sizes, n_points != sum of counts, and -- naming the
 * lowest offending voxel index in svnicp_map_last_error -- a count outside [1, max_pointscount], a voxel index outside
 * [-2^20, 2^20), a duplicate voxel (the later one is named), or a point that does not belong to its voxel: (int)(p /
 * float(voxel_size)) per axis, the arithmetic of AddPointCloud, so anything the map can hold round-trips (NaN points sit in
 * voxel 0).  SVNICP_ERR_OOM when n_voxels exceeds the table (2x capacity_voxels slots hold at least capacity_voxels voxels).
 * n_voxels = 0 has the effect of svnicp_map_clear. */
int svnicp_map_import(svnicp_map m, const int32_t *voxels, const int32_t *counts, const float *xyz, int64_t n_voxels, int64_t n_points,
                      int on_device);

/* ---------------------------------------------------------------------------------------------
 * Scan pre-processing on the device, the step right before add_cloud in the reference's node
 * (OdometryPipeline.cpp:555-560): crop_pointcloud (:692-704) and downsample_uniform (:684-690 =
 * pcl::UniformSampling, leaf = the radius argument).  Clouds are float xyz triples (pcl::PointXYZI without the
 * intensity).  Outputs live in buffers owned by the handle and stay valid until the next-but-one call on it, so
 * crop -> downsample -> downsample chains without copies; an output may be fed to svnicp_map_add_cloud (float, device)
 * or, through svnicp_pre_to_f64, to svnicp_add_cloud (double, device).
 * --------------------------------------------------------------------------------------------- */
typedef struct svnicp_pre_t *svnicp_pre;
int svnicp_pre_create(svnicp_pre *out, int64_t max_points, int device);
void svnicp_pre_destroy(svnicp_pre p);
const char *svnicp_pre_last_error(svnicp_pre p);
/* crop_pointcloud: keeps min_range^2 < |p|^2 < max_range^2 in input order.  *max_sq_norm = max |p|^2 over ALL input
 * points: the reference keeps the running maximum of this SQUARED norm in scan_max_range_ (:699). */
int svnicp_pre_crop(svnicp_pre p, const float *xyz, int64_t n, int on_device, double min_range, double max_range,
                    const float **dev_out, int64_t *n_out, double *max_sq_norm);
/* downsample_uniform(cloud, voxel_size): one point per leaf of size `leaf`; PCL's rule (distance to the leaf's integer
 * index, first point on ties).  Output order is arbitrary (PCL iterates an unordered_map). */
int svnicp_pre_downsample_uniform(svnicp_pre p, const float *xyz, int64_t n, int on_device, double leaf, const float **dev_out,
                                  int64_t *n_out);
/* deskew_pointcloud (OdometryPipeline.cpp:357-447): every point is moved by Pose3::Expmap((s - 0.5) * delta) with
 * delta = Pose3::Logmap(start^-1 * finish) (the two newest entries of the node's pose buffer, :419-424) and s its time
 * stamp normalised to [0,1] over the scan (:411-420).  stamps: [n] doubles in any unit (the `t` / `timestamp` / `time` field
 * of the PointCloud2 message widened to double, :400-410), host or device; kitti != 0 reproduces the KITTI branch instead
 * (:385-399: 0.205 deg tilt about p x z, stamp from the azimuth; stamps may be NULL).  *moved = 0 when all stamps are equal:
 * the cloud is returned unchanged (:415).  Poses: rotation row-major 3x3 + translation.  GTSAM's closed forms (4.2) are restated. */
int svnicp_pre_deskew(svnicp_pre p, const float *xyz, int64_t n, int on_device, const double *stamps, int stamps_on_device, int kitti,
                      const double R_start[9], const double t_start[3], const double R_finish[9], const double t_finish[3],
                      const float **dev_out, int32_t *moved);
/* The hand-off after the getters in ICP mode (updater_, OdometryPipeline.cpp:37-45; tensor2gtsamPose3, ICPUtils.cpp:84-98):
 * pose = initial_guess * Pose3(Rot3::Expmap(mean[3:6]), mean[0:3]) with mean6 = svnicp_get_transformation().  Host arithmetic. */
int svnicp_pose_compose(const double R0[9], const double t0[3], const double mean6[6], double R_out[9], double t_out[3]);
/* float device cloud -> double device cloud (owned by the handle) for svnicp_add_cloud(source_on_device = 1) */
int svnicp_pre_to_f64(svnicp_pre p, const float *dev_xyz, int64_t n, const double **dev_out);
int svnicp_pre_download(svnicp_pre p, const float *dev_xyz, int64_t n, float *out);

#ifdef __cplusplus
}
#endif
#endif /* SVNICP_B200_H */
