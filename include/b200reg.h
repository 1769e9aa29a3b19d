/* b200reg.h -- C ABI of the B200-native loop-closure registration engine.
 *
 * This is the drop-in boundary for the ONE hot path of engcang/FAST-LIO-SAM-QN that
 * this repository replaces: the registration that FastLioSamQn::loopTimerFunc
 * (fast_lio_sam_qn/src/fast_lio_sam_qn.cpp:203-252) reaches through
 * LoopClosure::performLoopClosure (fast_lio_sam_qn/src/loop_closure.cpp:168-205), i.e.
 * everything behind nano_gicp::NanoGICP<PointType,PointType>
 * (third_party/nano_gicp/include/nano_gicp/nano_gicp.hpp:58-137) and quatro<PointType>
 * (third_party/Quatro/include/quatro/quatro_module.h:19-37).
 *
 * The reference has no FFI: both libraries are linked C++ templates.  The host-side
 * facade classes in fast-lio-sam-qn_b200/host/ keep those class surfaces and call the
 * functions below; INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - every function returns 0 on success, a negative B200REG_E* code otherwise; nothing
 *     throws across this boundary;
 *   - all 4x4 matrices are ROW-MAJOR (Eigen is column-major: the facade transposes);
 *   - a context is bound to one CUDA device and one stream; use one context per host
 *     thread / per GPU rank (LoopClosure itself is single-instance and not re-entrant,
 *     fast_lio_sam_qn/src/fast_lio_sam_qn.cpp:81);
 *   - point buffers are (x, y, z [, ...]) fp32 records `stride_bytes` apart, so
 *     pcl::PointXYZI (32 B: x,y,z,1,intensity,pad) uploads without repacking;
 *   - host buffers passed to a call (pinned or pageable) have been consumed when the call returns; device buffers passed
 *     with on_device != 0 must stay valid until the context's stream has been synchronised or the call has returned a result;
 *   - b200reg_ctx_set_stream may only be called while the context is idle (everything it owns is ordered on ONE stream);
 *   - there is NO CPU fallback: if no sm_100 device is present b200reg_ctx_create fails.
 */
#ifndef B200REG_H
#define B200REG_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200REG_OK 0
#define B200REG_EINVAL (-1)   /* bad argument */
#define B200REG_ECUDA (-2)    /* CUDA runtime error (see b200reg_last_error) */
#define B200REG_ENODEV (-3)   /* no usable GPU */
#define B200REG_ESTATE (-4)   /* call order violated (e.g. align before covariances) */
#define B200REG_ENCCL (-5)    /* collective layer error */

typedef struct b200reg_ctx b200reg_ctx;
typedef struct b200reg_cloud b200reg_cloud;

/* Mirrors NanoGICPConfig (fast_lio_sam_qn/include/loop_closure.h:25-36) + the LsqRegistration
 * constructor defaults (third_party/nano_gicp/include/nano_gicp/impl/lsq_registration_impl.hpp:49-63). */
typedef struct b200reg_gicp_params {
  int32_t k_correspondences;     /* setCorrespondenceRandomness, loop_closure.cpp:10 (15)   */
  int32_t max_iterations;        /* setMaximumIterations, loop_closure.cpp:11 (32)          */
  double max_corr_dist;          /* setMaxCorrespondenceDistance, loop_closure.cpp:13 (52.5)*/
  double transformation_eps;     /* setTransformationEpsilon, loop_closure.cpp:14 (0.01)    */
  double rotation_eps;           /* lsq_registration_impl.hpp:53 (2e-3)                     */
  int32_t lm_max_iterations;     /* lsq_registration_impl.hpp:58 (10)                       */
  int32_t regularization;        /* RegularizationMethod (gicp/gicp_settings.hpp:47): 0 NONE, 1 MIN_EIG,
                                    2 NORMALIZED_MIN_EIG, 3 PLANE (default, nano_gicp_impl.hpp:61), 4 FROBENIUS */
  double lm_init_lambda_factor;  /* lsq_registration_impl.hpp:59 (1e-9)                     */
  double icp_score_thr;          /* validity gate, loop_closure.cpp:129 (config.yaml:21: 1.5) */
} b200reg_gicp_params;

/* RegistrationOutput (fast_lio_sam_qn/include/loop_closure.h:64-70) plus solver telemetry. */
typedef struct b200reg_result {
  double T[16];        /* final SE(3), fp64, row-major: maps src onto dst                      */
  float Tf[16];        /* x0.cast<float>() -- what getFinalTransformation() returns            */
  double pose_between[16]; /* RegistrationOutput::pose_between_eig_ exactly as the reference leaves it
                          (loop_closure.cpp:129-134, 156): icpAlignment: Tf.cast<double>() when valid, Identity otherwise;
                          coarseToFineAlignment: (valid fine stage ? Tf_fine : Identity) * T_quatro, or the coarse
                          stage's own output when Quatro itself is invalid; Identity for the dummy output        */
  double final_hessian[36]; /* LsqRegistration::getFinalHessian() (lsq_registration.hpp:88): H of the last linearize,
                          6x6 row-major (symmetric); Identity before any (lsq_registration_impl.hpp:62)            */
  double fitness;      /* getFitnessScore(): mean 1-NN d^2 over ALL source points              */
  int32_t converged;   /* hasConverged()                                                       */
  int32_t valid;       /* converged && fitness < icp_score_thr (loop_closure.cpp:129)          */
  int32_t iterations;  /* nr_iterations_ (index of the last outer iteration)                   */
  int32_t n_linearize; /* number of linearize() passes (= 1-NN passes)                         */
  int32_t n_error;     /* number of compute_error() passes                                     */
  int32_t lm_failed;   /* "lm not converged!!" (lsq_registration_impl.hpp:105-108)             */
  int32_t status;      /* 0 ok; <0 error for this pair                                         */
  int32_t tag;         /* caller-defined, set to 0 by the engine and carried through b200reg_allgather_results
                          (e.g. the global pair index of a sharded batch)                                      */
} b200reg_result;

/* Mirrors QuatroConfig (fast_lio_sam_qn/include/loop_closure.h:38-50) and the quatro<T> constructor arguments
 * (third_party/Quatro/include/quatro/quatro_module.h:30-32), with the EFFECTIVE deployment values as defaults
 * (SURVEY.md App. A.1: normal radius 0.9, FPFH radius 1.5, max correspondences 200 because of the rosparam typo). */
typedef struct b200reg_quatro_params {
  double fpfh_normal_radius;   /* fpfh_normal_radi (0.9)                                              */
  double fpfh_radius;          /* fpfh_radi (1.5)                                                     */
  double noise_bound;          /* 0.3                                                                 */
  double rot_gnc_factor;       /* 1.4                                                                 */
  double rot_cost_thr;         /* 1e-4                                                                */
  int32_t rot_max_iter;        /* 50                                                                  */
  int32_t max_corres;          /* num_max_corres (200); must be <= 509                                */
  double distance_threshold;   /* FEATURE-space gate of optimizedMatching (matcher.cc:422/444) (35)   */
  double tuple_scale;          /* 0.95 (quatro_module.cc:61)                                          */
  uint64_t seed;               /* replaces srand(time(NULL)) (matcher.cc:465) by a counter-based RNG  */
  int32_t estimate_scale;      /* must be 0 (QN/config: estimating_scale false)                       */
  int32_t use_optimized_matching; /* 1 (config.yaml:32): optimizedMatching; 0: advancedMatching       */
} b200reg_quatro_params;

/* Telemetry of one quatro<T>::align call. */
typedef struct b200reg_quatro_info {
  double T[16];          /* out_tf_ (row-major); Identity when !valid                                  */
  int32_t valid;         /* if_valid (quatro_module.cc:63-72)                                          */
  int32_t n_mutual;      /* correspondences after the mutual check                                     */
  int32_t n_corr;        /* after the tuple test (<= max_corres + 3)                                   */
  int32_t clique_size;   /* max-clique inliers                                                         */
  int32_t gnc_iterations;
  int32_t reserved;
} b200reg_quatro_info;

void b200reg_default_gicp_params(b200reg_gicp_params* p);
void b200reg_default_quatro_params(b200reg_quatro_params* p);
const char* b200reg_last_error(void);                /* message of the calling thread's last failure               */
void b200reg_set_last_error(const char* message);  /* used by the batch driver to hand a worker's message over     */
const char* b200reg_version(void);
/* sizeof() of the ABI structs as compiled into the library, so that a binding (ctypes, cgo, JNI ...) can check its own
 * layout at load time: 0 gicp_params, 1 result, 2 quatro_params, 3 quatro_info, 4 loop_config, 5 loop_factor.  0 = unknown. */
size_t b200reg_struct_size(int which);

/* ---- context ---------------------------------------------------------------------- */
int b200reg_ctx_create(int device, b200reg_ctx** out);
int b200reg_ctx_destroy(b200reg_ctx* ctx);
/* Use an externally owned CUDA stream (cudaStream_t passed as void*); NULL = the context's own. */
int b200reg_ctx_set_stream(b200reg_ctx* ctx, void* cuda_stream);
int b200reg_ctx_synchronize(b200reg_ctx* ctx);
/* Number of kernels this context has launched so far (bench.py reports it as gpu_launches). */
int64_t b200reg_ctx_launch_count(const b200reg_ctx* ctx);

/* Per-kernel-family timing with CUDA events recorded on the launching stream (bench.py roofline).
 * Families: 0 index_build, 1 knn_covariance, 2 gicp_step (the LM loop as ONE graph launch), 3 misc, 4 fpfh,
 * 5 quatro_match_solve, 6 gicp_search, 7 gicp_accum, 8 gicp_control.  While profiling is enabled the LM loop is not run as
 * a graph: its three kernels are launched one by one (host-polled) so that each gets its own events -- families 6-8 fill,
 * family 2 stays empty.  algo_bytes follows SURVEY.md §8(d).                                                         */
int b200reg_ctx_set_profiling(b200reg_ctx* ctx, int enable);
int b200reg_ctx_reset_profile(b200reg_ctx* ctx);
int b200reg_ctx_get_profile(b200reg_ctx* ctx, int family, const char** name, double* ms, double* algo_bytes,
                            int64_t* launches);

/* ---- clouds: replaces KdTreeFLANN::setInputCloud / buildIndex
 *      (third_party/nano_gicp/include/nano_gicp/nanoflann.hpp:131-138) ----------------- */
/* Upload `count` clouds (host or device pointers) and build their spatial indices in one
 * batched pass.  on_device != 0: the xyz pointers are device pointers (no H2D copy).      */
int b200reg_clouds_create(b200reg_ctx* ctx, int count, const float* const* xyz, const size_t* n,
                          size_t stride_bytes, int on_device, b200reg_cloud** out);
int b200reg_cloud_destroy(b200reg_ctx* ctx, b200reg_cloud* cloud);
size_t b200reg_cloud_size(const b200reg_cloud* cloud);

/* NanoGICP::calculateSourceCovariances / calculateTargetCovariances
 * (third_party/nano_gicp/include/nano_gicp/impl/nano_gicp_impl.hpp:151-159, 298-357), batched. */
int b200reg_clouds_covariances(b200reg_ctx* ctx, int count, b200reg_cloud* const* clouds, int k);
/* NanoGICP::setSourceCovariances / setTargetCovariances (nano_gicp.hpp:91-93, nano_gicp_impl.hpp:142-150): the caller's
 * per-point covariances (n x 9 doubles: the row-major 3x3 block of each Matrix4d, ORIGINAL point order) replace the
 * computed ones; align() then does not recompute them (nano_gicp_impl.hpp:162-167) until the input cloud changes.   */
int b200reg_set_covariances(b200reg_ctx* ctx, b200reg_cloud* cloud, const double* cov9, size_t n);
/* Same with an explicit RegularizationMethod (setRegularizationMethod, nano_gicp.hpp:84); the plain call uses PLANE. */
int b200reg_clouds_covariances_ex(b200reg_ctx* ctx, int count, b200reg_cloud* const* clouds, int k, int method);

/* ---- registration ----------------------------------------------------------------- */
/* pcl::Registration::align + getFitnessScore + hasConverged + getFinalTransformation for
 * `count` (src, tgt) pairs at once (call sites fast_lio_sam_qn/src/loop_closure.cpp:124-133).
 * guess16: count x 16 doubles row-major, or NULL for identity (the reference always uses identity).
 * Covariances are computed on demand if a cloud has none (nano_gicp_impl.hpp:162-167).       */
int b200reg_gicp_align(b200reg_ctx* ctx, int count, b200reg_cloud* const* src, b200reg_cloud* const* tgt,
                       const double* guess16, const b200reg_gicp_params* params, b200reg_result* out);

/* LoopClosure::icpAlignment (loop_closure.cpp:110-136) in one call, raw buffers in, results out:
 * index build x2, covariances x2, align, fitness, validity gate -- for `count` pairs.          */
int b200reg_icp_alignment(b200reg_ctx* ctx, int count, const float* const* src_xyz, const size_t* src_n,
                          const float* const* tgt_xyz, const size_t* tgt_n, size_t stride_bytes, int on_device,
                          const b200reg_gicp_params* params, b200reg_result* out);

/* ---- Quatro (global registration) --------------------------------------------------------- */
/* teaser::FPFHEstimation::computeFPFHFeatures (third_party/Quatro/src/fpfh.cc:14-42) for `count` clouds:
 * normals (radius search, viewpoint (0,0,0)) -> SPFH -> FPFH, kept on the device with the cloud.     */
int b200reg_clouds_fpfh(b200reg_ctx* ctx, int count, b200reg_cloud* const* clouds, double normal_radius,
                        double fpfh_radius);
/* quatro<PointType>::align (third_party/Quatro/src/quatro_module.cc:48-79) for `count` pairs: FPFH on demand,
 * optimizedMatching (matcher.cc:358-561) or, with use_optimized_matching = 0, advancedMatching (matcher.cc:118-356:
 * ungated forward / reverse 1-NN, cross check, three-edge tuple test, sort + unique), then the TEASER++ QUATRO solve.
 * corr_out (optional): count x 2*CAP ints, the (src, dst) ORIGINAL indices of the final correspondences of each
 * pair, CAP = B200REG_CORR_CAPACITY (optimized) or B200REG_ADV_CORR_CAPACITY (advanced).  An advancedMatching set
 * larger than B200REG_ADV_CORR_CAPACITY fails the call with B200REG_ESTATE (nothing is truncated silently).     */
#define B200REG_CORR_CAPACITY 512
#define B200REG_ADV_CORR_CAPACITY 8192
int b200reg_quatro_align(b200reg_ctx* ctx, int count, b200reg_cloud* const* src, b200reg_cloud* const* dst,
                         const b200reg_quatro_params* params, b200reg_quatro_info* out, int32_t* corr_out);
/* LoopClosure::coarseToFineAlignment (fast_lio_sam_qn/src/loop_closure.cpp:138-159) for `count` pairs from raw
 * buffers: Quatro -> transformPcd(src, T_quatro) -> icpAlignment -> T = T_gicp * T_quatro.
 * out[i].T is the composed transform; quatro_out (optional) receives the coarse stage.                   */
int b200reg_loop_closure(b200reg_ctx* ctx, int count, const float* const* src_xyz, const size_t* src_n,
                         const float* const* tgt_xyz, const size_t* tgt_n, size_t stride_bytes, int on_device,
                         const b200reg_quatro_params* qparams, const b200reg_gicp_params* gparams,
                         b200reg_result* out, b200reg_quatro_info* quatro_out);

/* ---- "next" rows (SURVEY.md §8f): device-resident keyframes, candidate search, cloud assembly ---------- */
typedef struct b200reg_keyframes b200reg_keyframes;

/* Mirrors LoopClosureConfig (fast_lio_sam_qn/include/loop_closure.h:52-62) with the EFFECTIVE deployment values
 * (SURVEY.md §5: num_submap_keyframes 5 because of the rosparam typo). */
typedef struct b200reg_loop_config {
  int32_t enable_quatro;            /* config.yaml:29 (1)                                   */
  int32_t enable_submap_matching;   /* config.yaml:9 (0)                                    */
  int32_t num_submap_keyframes;     /* submap_range (5)                                     */
  int32_t reserved;
  double voxel_res;                 /* config.yaml:16 (0.3)                                 */
  double loop_detection_radius;     /* config.yaml:13 (35.0)                                */
  double loop_detection_timediff_threshold; /* config.yaml:14 (30.0)                        */
  b200reg_gicp_params gicp;
  b200reg_quatro_params quatro;
} b200reg_loop_config;
void b200reg_default_loop_config(b200reg_loop_config* cfg);

int b200reg_keyframes_create(b200reg_ctx* ctx, b200reg_keyframes** out);
int b200reg_keyframes_destroy(b200reg_ctx* ctx, b200reg_keyframes* kf);
/* Keyframe clouds are kept in device slabs of their own (128 MB unless reserved), apart from the context's scratch pool.
 * A node that knows roughly how many points its map will hold reserves them once at start (std::vector::reserve for
 * keyframes_, fast_lio_sam_qn.h:63): no keyframe added afterwards allocates until the reservation is used up.        */
int b200reg_keyframes_reserve(b200reg_ctx* ctx, b200reg_keyframes* kf, size_t n_points);
/* PosePcd (fast_lio_sam_qn/include/pose_pcd.hpp:7-43): cloud in the LiDAR frame as fp32 records `stride_bytes` apart (host
 * memory): packed (x, y, z, intensity) for strides below 32 bytes, the pcl::PointXYZI layout (x, y, z, 1, intensity, pad...)
 * from 32 bytes on; its corrected pose (row-major 4x4) and timestamp.  Returns the index.                          */
int b200reg_keyframes_add(b200reg_ctx* ctx, b200reg_keyframes* kf, const float* xyzi, size_t n, size_t stride_bytes,
                          const double* pose16, double timestamp);
/* The PosePcd constructor itself (pose_pcd.hpp:21-43) as a device step: the scan arrives in the WORLD frame with the odometry
 * pose as position + quaternion (x, y, z, w; nav_msgs::Odometry); pose_eig_ = [tf::Matrix3x3(q) | p], pose_corrected_eig_ =
 * pose_eig_, and the stored cloud is transformPcd(scan, pose_eig_.inverse()) (LiDAR frame).  Returns the index.        */
int b200reg_keyframes_add_world(b200reg_ctx* ctx, b200reg_keyframes* kf, const float* xyzi_world, size_t n, size_t stride_bytes,
                                const double* position3, const double* quat_xyzw, double timestamp);
/* Read a keyframe back: its LiDAR-frame cloud (n x 4 floats: x, y, z, intensity; NULL to skip), corrected pose (16 doubles,
 * row-major; NULL to skip) and timestamp (NULL to skip) -- what the reference saves per keyframe (fast_lio_sam_qn.cpp:344-376). */
int b200reg_keyframes_get(b200reg_ctx* ctx, const b200reg_keyframes* kf, int idx, float* xyzi_out, double* pose16_out,
                          double* timestamp_out);
size_t b200reg_keyframes_cloud_size(const b200reg_keyframes* kf, int idx);
/* pose_corrected_eig_ rewrite after an accepted loop (fast_lio_sam_qn/src/fast_lio_sam_qn.cpp:180-188).     */
int b200reg_keyframes_set_pose(b200reg_ctx* ctx, b200reg_keyframes* kf, int idx, const double* pose16);
int b200reg_keyframes_size(const b200reg_keyframes* kf);
/* LoopClosure::fetchClosestKeyframeIdx (loop_closure.cpp:34-56) for `count` query keyframes at once; each query
 * is treated as the latest keyframe at its time, so its candidates are the indices below it. -1 = none.       */
int b200reg_fetch_closest_keyframes(b200reg_ctx* ctx, b200reg_keyframes* kf, int count, const int32_t* query_idx,
                                    double radius, double timediff_threshold, int32_t* closest_out);
/* LoopClosure::setSrcAndDstCloud (loop_closure.cpp:58-108) for `count` (src, dst) keyframe index pairs:
 * transformPcd by the corrected poses, +-submap merge, pcl::VoxelGrid at voxel_res; the resulting clouds are
 * indexed and stay on the device.  n_keyframes = size of the keyframe vector at the time (0 = current size).  */
int b200reg_assemble_clouds(b200reg_ctx* ctx, b200reg_keyframes* kf, int count, const int32_t* src_idx,
                            const int32_t* dst_idx, const b200reg_loop_config* cfg, int n_keyframes,
                            b200reg_cloud** src_out, b200reg_cloud** dst_out);
/* Points of a cloud in their ORIGINAL order as (x, y, z) (debug tap for the assembled / voxelised clouds).    */
/* Same with the size of the keyframe vector given PER PAIR (n_keyframes[i] = latest keyframe index + 1 at the tick the
 * pair was formed): a batch that replays several loopTimerFunc ticks sees, for each query, exactly the sub-map bounds
 * `i < keyframes.size() - 1` the reference evaluated at that tick (loop_closure.cpp:72,79,100).                      */
int b200reg_assemble_clouds_at(b200reg_ctx* ctx, b200reg_keyframes* kf, int count, const int32_t* src_idx,
                               const int32_t* dst_idx, const b200reg_loop_config* cfg, const int32_t* n_keyframes,
                               b200reg_cloud** src_out, b200reg_cloud** dst_out);
int b200reg_cloud_points(b200reg_ctx* ctx, const b200reg_cloud* cloud, float* xyz_out);
/* LoopClosure::performLoopClosure (loop_closure.cpp:168-205) for `count` query keyframes with given closest
 * indices (-1 = no candidate -> invalid dummy output): assemble, then coarse-to-fine (enable_quatro) or GICP only. */
int b200reg_perform_loop_closure(b200reg_ctx* ctx, b200reg_keyframes* kf, int count, const int32_t* query_idx,
                                 const int32_t* closest_idx, const b200reg_loop_config* cfg, b200reg_result* out,
                                 b200reg_quatro_info* quatro_out);

/* The corrected global map (fast_lio_sam_qn.cpp:302-316 /corrected_map, :398-411 <seq>_map.pcd, :435-449 result.pcd):
 * every keyframe 0 .. n_keyframes-1 transformed by its CURRENT corrected pose (transformPcd: double math, float result,
 * intensity carried), merged in keyframe order, then pcl::VoxelGrid at voxel_res (centroids of x, y, z, intensity in
 * voxel-index order).  n_keyframes = 0: the whole store.  When PCL's int32 index guard trips (dx*dy*dz > INT32_MAX) the
 * map is the merged cloud unchanged, as PCL returns it.  The records stay on the device until b200reg_map_destroy.
 * B200REG_EINVAL: empty store, n_keyframes out of range, voxel_res <= 0, more than 2^30 - 1 merged points.            */
typedef struct b200reg_map b200reg_map;
int b200reg_map_build(b200reg_ctx* ctx, const b200reg_keyframes* kf, int n_keyframes, double voxel_res, b200reg_map** out);
size_t b200reg_map_size(const b200reg_map* map);       /* records (x, y, z, intensity)                                 */
int b200reg_map_voxelized(const b200reg_map* map);     /* 1: voxelised; 0: PCL's int32 guard tripped, records = merged */
int b200reg_map_get(b200reg_ctx* ctx, const b200reg_map* map, float* xyzi_out);  /* size x 4 floats, voxel-index order */
int b200reg_map_destroy(b200reg_ctx* ctx, b200reg_map* map);

/* Result consumption (SURVEY.md §8f rank 3; fast_lio_sam_qn/src/fast_lio_sam_qn.cpp:220-237): the loop constraint the
 * reference hands to GTSAM for an accepted registration,
 *   BetweenFactor<Pose3>(latest.idx_, closest_idx, pose_from.between(pose_to), Diagonal::Variances(score x 6)),
 *   pose_from = poseEigToGtsamPose(pose_between_eig_ * latest.pose_corrected_eig_)   ("take care of the order", :224)
 *   pose_to   = poseEigToGtsamPose(closest.pose_corrected_eig_)
 * with poseEigToGtsamPose's roll/pitch/yaw round trip (utilities.hpp:67-75: tf getRPY, then Rot3::RzRyRx).  The pose
 * graph itself (GTSAM iSAM2) stays with the caller; corrected poses come back through b200reg_keyframes_set_pose.   */
typedef struct b200reg_loop_factor {
  int32_t from_idx;        /* key of the latest keyframe                                        */
  int32_t to_idx;          /* key of the matched keyframe                                       */
  int32_t valid;           /* RegistrationOutput::is_valid_; 0: the reference adds no factor    */
  int32_t reserved;
  double measurement[16];  /* pose_from.between(pose_to), row-major 4x4                         */
  double variances[6];     /* score in every slot                                               */
} b200reg_loop_factor;
/* Pure host arithmetic (no context, no GPU): one factor from explicit poses.                                        */
int b200reg_loop_factor_from_poses(const double* T_between16, const double* pose_latest16, const double* pose_closest16,
                                   double score, int valid, int from_idx, int to_idx, b200reg_loop_factor* out);
/* The factors of a batch of b200reg_perform_loop_closure results, poses taken from the keyframe store.              */
int b200reg_loop_factors(b200reg_ctx* ctx, const b200reg_keyframes* kf, int count, const int32_t* query_idx,
                         const int32_t* closest_idx, const b200reg_result* results, b200reg_loop_factor* out);

/* ---- batch driver (SURVEY.md §8(b)(2) "b200reg_batch"): `depth` engine contexts, each on its own host thread with its own
 *      streams and memory pool, take alternate jobs, so the PCIe upload and the host-side polling of one job hide behind
 *      the kernels of the others.  The reference registers ONE pair per timer tick (fast_lio_sam_qn.cpp:203-219); a
 *      batch of independent candidate pairs is this engine's unit of work.
 *      Jobs are submitted from ONE host thread; the pointer arrays are copied at submit time, the point buffers and the
 *      output arrays must stay valid until the job has been waited for. ------------------------------------------------ */
typedef struct b200reg_batch b200reg_batch;
int b200reg_batch_create(int device, int depth, b200reg_batch** out);
int b200reg_batch_destroy(b200reg_batch* b);
/* LoopClosure::icpAlignment (loop_closure.cpp:110-136) for `count` pairs; returns a ticket >= 0 or a B200REG_E* code. */
int64_t b200reg_batch_submit_icp(b200reg_batch* b, int count, const float* const* src_xyz, const size_t* src_n,
                                 const float* const* tgt_xyz, const size_t* tgt_n, size_t stride_bytes, int on_device,
                                 const b200reg_gicp_params* params, b200reg_result* out);
/* LoopClosure::coarseToFineAlignment (loop_closure.cpp:138-159) for `count` pairs. */
int64_t b200reg_batch_submit_loop_closure(b200reg_batch* b, int count, const float* const* src_xyz, const size_t* src_n,
                                          const float* const* tgt_xyz, const size_t* tgt_n, size_t stride_bytes,
                                          int on_device, const b200reg_quatro_params* qparams,
                                          const b200reg_gicp_params* gparams, b200reg_result* out,
                                          b200reg_quatro_info* quatro_out);
/* Blocks until the job is done; returns ITS status (the message is then in b200reg_last_error of the calling thread).
 * latency_ms (optional): submit -> completion on the host clock.  A ticket can be waited for once.               */
int b200reg_batch_wait(b200reg_batch* b, int64_t ticket, double* latency_ms);
int b200reg_batch_wait_all(b200reg_batch* b);
int64_t b200reg_batch_launch_count(const b200reg_batch* b);
int b200reg_batch_depth(const b200reg_batch* b);

/* ---- the ONE collective of the path (SURVEY.md §8(e)): all-gather of the fixed-size result records over NCCL.
 *      Rank 0 makes the id, the caller ships its 128 bytes to the other ranks by any means (MPI, a file, torch.distributed),
 *      every rank calls b200reg_comm_init on its own context.  NCCL is loaded at run time (libnccl.so.2). -------------- */
#define B200REG_UNIQUE_ID_BYTES 128
int b200reg_comm_unique_id(void* id_out128);
int b200reg_comm_init(b200reg_ctx* ctx, const void* id128, int rank, int world);
int b200reg_comm_destroy(b200reg_ctx* ctx);
int b200reg_comm_rank(const b200reg_ctx* ctx);   /* -1 without a communicator */
int b200reg_comm_world(const b200reg_ctx* ctx);  /* 1 without a communicator  */
/* ncclAllGather of n_local records per rank on the context's stream: all_out holds world * n_local records in rank
 * order on EVERY rank (bytes identical for any world size given the same shards).  Without a communicator (world 1)
 * it is a copy.                                                                                                   */
int b200reg_allgather_results(b200reg_ctx* ctx, const b200reg_result* local, int n_local, b200reg_result* all_out);

/* Output cloud of align(): final_transformation_ applied to the source in fp32
 * (lsq_registration_impl.hpp:114).  out_xyz: n x 3 floats (host), original point order.       */
int b200reg_transform_cloud(b200reg_ctx* ctx, const b200reg_cloud* cloud, const float* Tf16, float* out_xyz);

/* ---- debug taps used by the parity tests ------------------------------------------- */
/* exact k-NN of host queries in a cloud: KdTreeFLANN::nearestKSearch (nanoflann.hpp:140-152).
 * idx_out/d2_out: nq x k, ascending; indices refer to the ORIGINAL point order; -1 pads k > n.   */
int b200reg_knn(b200reg_ctx* ctx, const b200reg_cloud* cloud, const float* queries, size_t nq,
                size_t qstride_bytes, int k, int32_t* idx_out, float* d2_out);
/* Same answer by brute force (every point tested, tiles staged into shared memory by TMA bulk copies): the on-GPU
 * anchor the tree traversal is verified against at full size (100k x 100k).                               */
int b200reg_knn_bruteforce(b200reg_ctx* ctx, const b200reg_cloud* cloud, const float* queries, size_t nq,
                           size_t qstride_bytes, int k, int32_t* idx_out, float* d2_out);
/* normals (n x 3, NaN where fewer than 3 neighbours) and FPFH (n x 33), original point order.            */
int b200reg_get_fpfh(b200reg_ctx* ctx, const b200reg_cloud* cloud, float* normals_out, float* fpfh_out);
/* n x 9 doubles (row-major 3x3 block of the reference's Matrix4d), original point order.          */
int b200reg_get_covariances(b200reg_ctx* ctx, const b200reg_cloud* cloud, double* cov9_out);
/* NanoGICP::linearize at pose T16 (nano_gicp_impl.hpp:213-270): H 6x6 row-major, b, sum of errors,
 * per-source-point correspondence (original target index or -1) and squared distance.             */
int b200reg_linearize(b200reg_ctx* ctx, const b200reg_cloud* src, const b200reg_cloud* tgt, const double* T16,
                      double max_corr_dist, double* H36, double* b6, double* err, int32_t* corr_out,
                      float* sqd_out);
/* NanoGICP::compute_error (nano_gicp_impl.hpp:272-296) in isolation: correspondences and Mahalanobis matrices are
 * taken from ONE linearize at T_lin16 (they stay stale, as in step_lm), then sum e^T M e is evaluated at T_trial16.  */
int b200reg_compute_error(b200reg_ctx* ctx, const b200reg_cloud* src, const b200reg_cloud* tgt, const double* T_lin16,
                          const double* T_trial16, double max_corr_dist, double* err);

#ifdef __cplusplus
}
#endif
#endif /* B200REG_H */
