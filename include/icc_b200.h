/* icc_b200.h — C-ABI of the B200-native continuous-time IMU-camera calibration solver.
 *
 * Drop-in boundary for the ONE hot path of urbste/OpenImuCameraCalibrator: everything below
 * OpenICC::core::ImuCameraCalibrator (include/OpenCameraCalibrator/core/imu_camera_calibrator.h:29-118)
 * and SplineTrajectoryEstimator<6> (core/spline_trajectory_estimator.h:31-218), i.e. what the reference
 * delegates to Ceres autodiff + sparse Cholesky + Theia camera projections.  The reference has no FFI layer;
 * each entry point cites the C++ member it replaces.  Plain pointers and sizes only, no torch / C++ types.
 * All arithmetic is FP64; all device work is hand-written sm_100a CUDA; there is NO CPU fallback:
 * every compute entry point fails with ICC_ERR_NO_DEVICE when no CUDA device is usable.
 *
 * Threading: one host thread per handle; one handle per GPU; handles are independent.
 * Ownership: caller owns every input array (copied during the call) and every output buffer.
 */
#ifndef ICC_B200_H_
#define ICC_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct icc_handle icc_handle;

typedef enum {
  ICC_OK = 0,
  ICC_ERR_INVALID_ARGUMENT = 1,
  ICC_ERR_NO_DEVICE = 2,       /* CUDA device / driver unusable: the product path never falls back to the CPU */
  ICC_ERR_CUDA = 3,
  ICC_ERR_STATE = 4,           /* call order violated (e.g. optimize before batch_init_spline) */
  ICC_ERR_UNSUPPORTED = 5,     /* outside the solver's limits (e.g. POINTS with more than ~133 board points: border too wide), never a silent fallback */
  ICC_ERR_NUMERIC = 6          /* factorisation broke down / non-finite cost */
} icc_status;

/* theia::CameraIntrinsicsModelType numeric values (pyTheiaSfM@69c3d37); JSON `intrinsic_type` strings are the
 * upper-case names (src/io/read_camera_calibration.cc:59-116).  Intrinsic vectors use Theia's index order:
 *   PINHOLE                   [f, ar, skew, cx, cy, k1, k2]
 *   PINHOLE_RADIAL_TANGENTIAL [f, ar, skew, cx, cy, k1, k2, k3, t1, t2]
 *   FISHEYE                   [f, ar, skew, cx, cy, k1, k2, k3, k4]
 *   FOV                       [f, ar, cx, cy, omega]          (extension: the reference never dispatches FOV)
 *   DIVISION_UNDISTORTION     [f, ar, cx, cy, k]
 *   DOUBLE_SPHERE             [f, ar, skew, cx, cy, xi, alpha]
 *   EXTENDED_UNIFIED          [f, ar, skew, cx, cy, alpha, beta] */
typedef enum {
  ICC_CAM_PINHOLE = 0,
  ICC_CAM_PINHOLE_RADIAL_TANGENTIAL = 1,
  ICC_CAM_FISHEYE = 2,
  ICC_CAM_FOV = 3,
  ICC_CAM_DIVISION_UNDISTORTION = 4,
  ICC_CAM_DOUBLE_SPHERE = 5,
  ICC_CAM_EXTENDED_UNIFIED = 6
} icc_camera_model;

/* OpenICC::core::SplineOptimFlags (core/spline_trajectory_estimator.h:17-27), same numeric values. */
enum {
  ICC_FLAG_POINTS = 1 << 0,           /* board points as parameter blocks, HomogeneousVectorParameterization(4) (impl.h:136-152): 3 tangent columns per point,
                                         last in the canonical order; read the result with icc_get_board_points */
  ICC_FLAG_T_I_C = 1 << 1,
  ICC_FLAG_IMU_BIASES = 1 << 2,
  ICC_FLAG_IMU_INTRINSICS = 1 << 3,
  ICC_FLAG_GRAVITY_DIR = 1 << 4,
  ICC_FLAG_CAM_LINE_DELAY = 1 << 5,
  ICC_FLAG_SPLINE = 1 << 6,
  ICC_FLAG_ACC_BIAS = 1 << 7,
  ICC_FLAG_GYR_BIAS = 1 << 8,
  /* Extensions named by the north-star; the reference keeps both quantities fixed (SURVEY.md "Read this first" #3), so with
   * these bits clear they are pass-through exactly like there. */
  ICC_FLAG_CAM_INTRINSICS = 1 << 9,   /* camera intrinsics (Theia parameter vector of the active model) as a parameter block */
  ICC_FLAG_TIME_OFFSET = 1 << 10      /* increment [s] of the IMU->camera time offset applied to every IMU sample time */
};

/* Arguments of ImuCameraCalibrator::BatchInitSpline (src/core/imu_camera_calibrator.cc:21-124). */
typedef struct {
  double T_i_c_init[7];        /* Sophus SE3 storage: quaternion x,y,z,w then translation (impl.h:519,579) */
  double dt_so3_s, dt_r3_s;    /* SplineWeightingData::dt_so3 / dt_r3 (seconds) */
  double std_so3, std_r3;      /* weights are 1/std (imu_camera_calibrator.cc:111,117) */
  double time_offset_imu_to_cam_s;
  double init_line_delay_s;    /* 0 => global shutter path (vision zero-weighted, SURVEY quirk q3) */
  double acc_intrinsics[6];    /* [misYZ, misZY, misZX, sX, sY, sZ]                         (impl.h:1236-1239) */
  double gyr_intrinsics[9];    /* [misYZ, misZY, misZX, misXZ, misXY, misYX, sX, sY, sZ]    (impl.h:1241-1245) */
  double acc_bias[3], gyr_bias[3];
  int32_t dispatch_fov;        /* 0 = reference behaviour (FOV fails -> 1e10 residuals); 1 = enable FOV extension */
  int32_t reserved;
} icc_init_params;

/* Solver knobs: ceres::Solver::Options as set in SplineTrajectoryEstimator::Optimize (impl.h:254-266)
 * plus the Ceres 2.1 defaults that shape the Levenberg-Marquardt path. */
typedef struct {
  double function_tolerance;        /* 1e-4  (impl.h:262) */
  double parameter_tolerance;       /* 1e-7  (impl.h:263) */
  double gradient_tolerance;        /* 1e-10 (Ceres default) */
  double initial_trust_region_radius; /* 1e4 */
  double max_trust_region_radius;   /* 1e16 */
  double min_trust_region_radius;   /* 1e-32 */
  double min_relative_decrease;     /* 1e-3 */
  double min_lm_diagonal;           /* 1e-6 */
  double max_lm_diagonal;           /* 1e32 */
  int32_t jacobi_scaling;           /* 1 */
  int32_t max_consecutive_invalid_steps; /* 5 */
} icc_solver_options;

typedef struct {
  int32_t iterations;               /* LM iterations executed (successful + unsuccessful) */
  int32_t successful_steps;
  int32_t termination;              /* 0 = max iterations, 1 = function tol, 2 = parameter tol, 3 = gradient tol, 4 = failure */
  int32_t num_residuals;            /* scalar residuals per evaluation */
  int32_t num_tangent;              /* active tangent parameters */
  int32_t jacobian_evaluations;
  int32_t cost_evaluations;
  int32_t gpu_launches;             /* CUDA kernels launched inside this optimize call */
  double initial_cost, final_cost;
  double mean_reproj_error;         /* GetMeanReprojectionError (impl.h:993-1072) — return value of Optimize */
  double seconds_total;             /* host wall clock of the optimize call */
  double seconds_jacobian;          /* device time in residual+Jacobian+normal-equation kernels (CUDA events) */
  double seconds_linear_solve;      /* device time in the banded/bordered Cholesky + step kernels */
} icc_summary;

/* Optional cross-rank reduction hook for residual sharding (SURVEY §8(e)): called on the host with the DEVICE pointer
 * of the packed FP64 normal-equation buffer {band, border coupling, border block, gradient, cost}; must sum it in place
 * across ranks (e.g. torch.distributed / ncclAllReduce on the handle's stream) before returning. */
typedef void (*icc_allreduce_fn)(void* device_ptr, int64_t n_doubles, void* cuda_stream, void* user);

/* ---- lifetime --------------------------------------------------------------------------------------------- */
icc_status icc_create(icc_handle** out, int device_ordinal);
void icc_destroy(icc_handle* h);
const char* icc_last_error(const icc_handle* h);          /* never NULL */
const char* icc_version(void);
void icc_default_solver_options(icc_solver_options* o);
icc_status icc_set_solver_options(icc_handle* h, const icc_solver_options* o);

/* ---- problem data (what main() hands to ImuCameraCalibrator, continuous_time_imu_to_camera_calibration.cc:104-199) */
/* theia::Camera intrinsics read at ceres_calib_split_residuals.h:333-336 */
icc_status icc_set_camera(icc_handle* h, int model, const double* intrinsics, int n_intrinsics, int image_width, int image_height);
/* theia::Track::Point() homogeneous board points, id = index (app :111-119).  After icc_batch_init_spline only the coordinates may change
 * (same count); the new points reach the device state at once. */
icc_status icc_set_board_points(icc_handle* h, int n_points, const double* xyzw);
/* Views of the calibration dataset (app :131-161): timestamp [s], observed corners (CSR over frames), and the per-view
 * pose prior used by BatchInitSO3R3VisPoses: q_wc (x,y,z,w) = R_cw^T and camera position p_wc (impl.h:290-300). */
icc_status icc_set_frames(icc_handle* h, int n_frames, const double* timestamps_s, const int32_t* corner_offsets /* n_frames+1 */,
                          const int32_t* point_ids, const double* uv, const double* q_wc_xyzw, const double* p_wc);
/* CameraTelemetryData accelerometer/gyroscope streams (src/io/read_telemetry.cc:49-56) */
icc_status icc_set_imu(icc_handle* h, int n_samples, const double* timestamps_s, const double* accel_xyz, const double* gyro_xyz);

/* ---- ImuCameraCalibrator API -------------------------------------------------------------------------------- */
/* BatchInitSpline (imu_camera_calibrator.cc:21-124): spline time range, knot counts, knot initialisation, bias
 * splines, measurement wiring (CalcTimes impl.h:763-788), gravity initialisation; uploads everything to HBM. */
icc_status icc_batch_init_spline(icc_handle* h, const icc_init_params* p);
/* SetKnownGravityDir (imu_camera_calibrator.cc:126-128) */
icc_status icc_set_known_gravity_dir(icc_handle* h, const double g[3]);
/* Residual sharding: keep only frames/IMU samples in shard `rank` of `world` (time-sliced, equal residual counts);
 * knots stay replicated.  Must be called before icc_batch_init_spline.  world = 1 restores the full problem. */
icc_status icc_set_shard(icc_handle* h, int rank, int world);
icc_status icc_set_allreduce(icc_handle* h, icc_allreduce_fn fn, void* user);
/* Native multi-GPU path: an NCCL communicator owned by the library (bound to the process' NCCL with dlopen).  One rank creates the
 * id, every rank creates its communicator (collective call), the handle borrows it: icc_set_comm sets the residual shard to the
 * communicator's (rank, world) and routes every cross-rank sum through ncclAllReduce on the solver's stream -- one all-reduce of the
 * packed normal equations per Jacobian evaluation, one 8-byte all-reduce per candidate cost.  One process per GPU (the drop-in
 * CLI's --gpus mode spawns one rank process per device).  Reference: SURVEY.md §8(e). */
#define ICC_COMM_ID_BYTES 128
typedef struct icc_comm icc_comm;
icc_status icc_comm_unique_id(unsigned char id[ICC_COMM_ID_BYTES]);
icc_status icc_comm_create(icc_comm** out, const unsigned char id[ICC_COMM_ID_BYTES], int rank, int world, int device_ordinal);
void icc_comm_destroy(icc_comm* c);
int icc_comm_rank(const icc_comm* c);
int icc_comm_world(const icc_comm* c);
int icc_comm_nccl_version(void);              /* 0 when NCCL could not be bound */
const char* icc_comm_last_error(void);        /* never NULL; thread local */
icc_status icc_set_comm(icc_handle* h, icc_comm* c);   /* NULL detaches (single-GPU, shard 0 of 1) */
/* Optimize (imu_camera_calibrator.cc:163-168 -> impl.h:254-276): LM over the blocks selected by `flags`. */
icc_status icc_optimize(icc_handle* h, int max_iterations, int flags, icc_summary* summary);

/* ---- getters (imu_camera_calibrator.h:48-77; impl.h:898-1072,1180-1234) -------------------------------------- */
icc_status icc_get_T_i_c(const icc_handle* h, double T_i_c[7]);
icc_status icc_get_gravity(const icc_handle* h, double g[3]);
icc_status icc_get_line_delay(const icc_handle* h, double* line_delay_s);
/* extension outputs: current camera intrinsics (n = model's parameter count) and time_offset_imu_to_cam_s (input + estimated increment) */
icc_status icc_get_camera_intrinsics(const icc_handle* h, double* intrinsics, int n);
icc_status icc_get_time_offset(const icc_handle* h, double* time_offset_s);
icc_status icc_get_num_knots(const icc_handle* h, int* n_so3, int* n_r3, int* n_acc_bias, int* n_gyr_bias);
icc_status icc_get_knots(const icc_handle* h, double* so3_xyzw, double* r3_xyz, double* acc_bias_xyz, double* gyr_bias_xyz); /* any may be NULL */
icc_status icc_set_knots(icc_handle* h, const double* so3_xyzw, const double* r3_xyz, const double* acc_bias_xyz, const double* gyr_bias_xyz);
icc_status icc_set_T_i_c(icc_handle* h, const double T_i_c[7]);
icc_status icc_set_line_delay(icc_handle* h, double line_delay_s);
icc_status icc_get_mean_reprojection_error(icc_handle* h, double* err);
/* number of IMU samples kept by BatchInitSpline and their (offset-corrected) timestamps / raw readings (app :265-327) */
icc_status icc_get_num_imu_used(const icc_handle* h, int* n);
icc_status icc_get_imu_used(const icc_handle* h, double* t_s, double* accel_xyz, double* gyro_xyz);
/* Knot-interval cells of the kept IMU samples (inspection / tests): maximal runs [i_begin, i_end) of kept samples that lie in the same
 * knot interval of all four splines, i.e. share CalcTimes' segment indices (impl.h:763-788); 6 int32 per cell:
 * s_so3, s_r3, s_acc_bias, s_gyr_bias, i_begin, i_end.  The evaluation kernels stage one knot window per cell. */
icc_status icc_get_num_imu_cells(const icc_handle* h, int* n);
icc_status icc_get_imu_cells(const icc_handle* h, int32_t* cells6);
/* GetAngularVelocity / GetAcceleration / GetGyroBias / GetAcclBias / GetPose evaluated on the GPU for n timestamps [ns];
 * valid[i] = 0 where CalcTimes rejects the timestamp (outputs left untouched there). Any output may be NULL. */
icc_status icc_eval_trajectory(icc_handle* h, int n, const int64_t* t_ns, double* gyro_xyz, double* accel_xyz,
                               double* gyro_bias_xyz, double* accel_bias_xyz, double* pose_q_xyzw, double* pose_p, int32_t* valid);

/* ---- test / measurement surface ----------------------------------------------------------------------------- */
icc_status icc_num_residuals(const icc_handle* h, int* n_vision, int* n_accel, int* n_gyro);   /* scalar residual counts */
icc_status icc_num_tangent(const icc_handle* h, int flags, int* n);
/* One evaluation at the current state.  Canonical tangent order: so3 knots (3 each), r3 knots (3 each), T_i_c (6: upsilon,
 * omega), gravity (3), line delay (1), acc-bias knots (3 each), gyr-bias knots (3 each), accelerometer intrinsics (6),
 * gyroscope intrinsics (9), camera intrinsics (model count), time-offset increment (1) — only blocks active under `flags`.
 * residuals: [vision 2/corner in frame order | accel 3/sample | gyro 3/sample].  hessian_dense: n x n row-major J^T J
 * (small problems only).  Any output may be NULL. */
icc_status icc_evaluate(icc_handle* h, int flags, double* cost, double* residuals, double* gradient, double* hessian_dense);
/* Run exactly `n` LM iterations (no convergence test) from the current state; used by bench.py as the timed "step". */
/* J^T J V for nvec caller vectors (canonical tangent order, one vector after the other) from the packed normal equations of the
 * current state: full-size parity of the reduced system without a dense Hessian (evaluation helper, like icc_evaluate). */
icc_status icc_normal_matvec(icc_handle* h, int flags, int nvec, const double* V, double* HV);
/* The elimination plan of the damped solve under `flags` (works on a host-only handle): plan[0..12] = valid, P (level-0 chunks),
 * w (separator width), len, rem (chunk c owns len + (c < rem) interior knot columns), L (cyclic-reduction levels), kd (half
 * bandwidth), nb (border columns), nk (knot columns), WS_A (level-0 window slots), cl_global, cs_global (dense border blocks in
 * global memory), stage0 (level-0 back-substitution staged in shared memory); plan[13..15] reserved (0).  chunks = 0: the
 * library's own choice; chunks > 0 forces the level-0 chunk count, then clamped and halved like the automatic choice. */
icc_status icc_get_solver_plan(icc_handle* h, int flags, int chunks, int32_t* plan16);
/* One damped solve at the current state (test surface): one Jacobian evaluation, its Jacobi scale S (options.jacobi_scaling),
 * D = clamp(diag(S H S), min_lm_diagonal, max_lm_diagonal) / radius, (S H S + D) y = -S g on the plan of `chunks` (as in
 * icc_get_solver_plan).  Outputs in canonical tangent order, each nullable: cost, gradient g and hessian_dense H (n x n, small
 * problems only) of the evaluation the solve consumed, scale S, lm_diag D, delta = S y, model_change = 1/2 (y^T D y - y^T S g).
 * The state and the LM bookkeeping are not changed.  ICC_ERR_UNSUPPORTED: no valid plan; ICC_ERR_NUMERIC: a pivot broke down. */
icc_status icc_solve_step(icc_handle* h, int flags, double radius, int chunks, double* cost, double* gradient, double* hessian_dense,
                          double* scale, double* lm_diag, double* delta, double* model_change);
icc_status icc_lm_iterations(icc_handle* h, int n, int flags, icc_summary* summary);
/* Run `n` bare residual+Jacobian+normal-equation evaluations (the residual-eval kernels only); device ms per evaluation. */
icc_status icc_time_evaluations(icc_handle* h, int n, int flags, int with_jacobian, double* ms_per_eval);
/* The handle's cudaStream_t (so that callers can bracket calls with their own CUDA events on the launching stream). */
void* icc_get_stream(icc_handle* h);

/* ---- upstream row f1 (SURVEY.md §8(f)): per-view board poses, i.e. what fills the pose dataset the hot CLI reads -----------
 * PoseEstimator::EstimatePosesFromJson (src/core/pose_estimator.cc:92-191): every corner is undistorted to the normalised image
 * plane (theia::Camera::PixelToNormalizedCoordinates, :129-130), a calibrated absolute pose is estimated (RANSAC PnP,
 * :54-66; squared normalised reprojection error threshold 0.004 * image_height / image_diagonal, :100-101; >= 6 inliers, :65),
 * then refined on the inliers by theia::BundleAdjustView with a Huber(1.345) loss (:44-48, :86-87); views with fewer than
 * `min_points` corners (pose_estimator.h:72, default 8) or a mean reprojection error above `max_reproj_error` (:181) are dropped.
 * Here: camera + board points must have been set (icc_set_camera / icc_set_board_points; the board must be planar up to a few per cent of its size -- the
 * homography only starts the refinement, which uses the real 3-D points);
 * one warp per view computes a normalised homography initialisation and the Levenberg-Marquardt refinement on the same cost,
 * so that the converged pose is the reference's BundleAdjustView optimum (RANSAC's random minimal samples are not reproduced:
 * the inlier set is taken with the same threshold around the refined pose).
 * Outputs (per view, caller-owned): q_wc (x,y,z,w) = R_cw^T and p_wc exactly as icc_set_frames consumes them, the mean
 * normalised reprojection error, valid (1 / 0).  max_reproj_error <= 0 selects 0.004 * image_height; min_points <= 0 selects 8. */
icc_status icc_estimate_board_poses(icc_handle* h, int n_frames, const int32_t* corner_offsets /* n_frames+1 */, const int32_t* point_ids,
                                    const double* uv, double max_reproj_error, int min_points,
                                    double* q_wc_xyzw, double* p_wc, double* mean_reproj_error, int32_t* valid);
/* PoseEstimator::FilterBadPoses (src/core/pose_estimator.cc:238-261), the last step of estimate_camera_poses_from_checkerboard
 * (app :66-67): views whose camera height p_wc.z differs from the median height of the valid views by more than |median| are dropped
 * (poses far away or on the wrong side of the board).  Host logic only: valid[] is updated in place; h may be NULL. */
icc_status icc_filter_bad_poses(icc_handle* h, int n_views, const double* p_wc, int32_t* valid);
/* --optimize_board_points of the pose app (app :61-65): PoseEstimator::OptimizeBoardPoints (pose_estimator.cc:193-224) =
 * theia::BundleAdjustTracks over the board points seen in more than `min_observations` (<= 0 selects min_num_obs_for_optim_ = 30,
 * pose_estimator.h:78) inlier observations, every camera constant, residual = normalised pinhole reprojection error of the
 * undistorted corners, Huber(1.345); then PoseEstimator::OptimizeAllPoses (:226-236) = BundleAdjustView of every valid view on the
 * new points.  q_wc / p_wc / valid are in-out (as returned by icc_estimate_board_poses); the handle's board points are replaced
 * (also returned in board_xyzw_out, w = 1 for optimised points).  With cameras fixed every point is an independent 3-parameter
 * problem: one warp per point on the GPU.  The empirical covariances the reference prints (:212-223) are not computed. */
icc_status icc_optimize_board_points(icc_handle* h, int n_frames, const int32_t* corner_offsets, const int32_t* point_ids, const double* uv,
                                     double max_reproj_error, int min_points, int min_observations,
                                     double* q_wc_xyzw, double* p_wc, double* mean_reproj_error /* nullable */, int32_t* valid,
                                     double* board_xyzw_out /* nullable, 4 per board point */, int32_t* n_points_optimized /* nullable */);
/* current board points of the handle (icc_set_board_points, or refined by icc_optimize_board_points / icc_calibrate_camera / a spline
 * solve with ICC_FLAG_POINTS) */
icc_status icc_get_board_points(const icc_handle* h, double* xyzw, int n);
/* theia::Camera::PixelToNormalizedCoordinates / z for `n` pixels with the handle's camera: xy_out[2n], ok[n] (nullable). */
icc_status icc_pixels_to_normalized(icc_handle* h, int n, const double* uv, double* xy_out, int32_t* ok);

/* ---- upstream row f3 (SURVEY.md §8(f)): IMU-to-camera rotation + time offset initialiser -----------------------------------
 * ImuToCameraRotationEstimator::EstimateCameraImuRotation (src/core/imu_to_camera_rotation_estimator.cc:116-274) together with
 * the preparation done by applications/estimate_imu_to_camera_rotation.cc:96-173: view rotations q_cw (quaternion of
 * theia::Camera::GetOrientationAsRotationMatrix, app :125-127) resampled to the median frame interval, interpolated to the IMU
 * rate, differentiated to a visual angular velocity, both streams smoothed by a 15-tap moving average, then a golden-section
 * search over the time offset in [-1, 1] s (tolerance 1e-4 s) around the closed-form rotation (+ gyroscope bias) fit.
 * Inputs: views (any order; timestamps already include the first-image offset of app :80-86), gyroscope samples (any order);
 * gyro_bias_in = NULL enables the bias estimation (EnableGyroBiasEstimation, app :63-67), otherwise it is subtracted from the
 * samples (app :99-100) and returned unchanged.  Outputs: q_gyro_to_cam (x,y,z,w) as written to "gyro_to_camera_rotation",
 * the time offset "time_offset_gyro_to_cam", the gyroscope bias, the final alignment error and the number of iterations.
 * One documented divergence: where the reference's InterpolateVector3d reads one element past the end of its input
 * (utils.cc:250-256, undefined behaviour) the last sample is used as is. */
icc_status icc_estimate_imu_to_camera_rotation(icc_handle* h, int n_views, const double* view_t_s, const double* q_cw_xyzw,
                                               int n_imu, const double* imu_t_s, const double* gyro_xyz, const double* gyro_bias_in /* 3 or NULL */,
                                               double* q_gyro_to_cam_xyzw /* 4 */, double* time_offset_s, double* gyro_bias_out /* 3 */,
                                               double* alignment_error, int32_t* iterations);

/* ---- upstream row f2 (SURVEY.md §8(f)): spline error weighting -----------------------------------------------------------------
 * python/sew.py:knot_spacing_and_variance (python/sew.py:201-234) as called by python/get_sew_for_dataset.py:38-48 for the
 * accelerometer (q_r3 = 0.96, dt in [0.01, 0.15]) and the gyroscope (q_so3 = 0.98, dt in [0.01, 0.2]): the largest uniform knot
 * spacing whose cubic-B-spline interpolation response keeps `quality` of the signal energy, and the variance of the spline fit
 * error at that spacing (its square root is the "weighting_factor" of spline_error_weighting_json).
 * signal_xyz: n x 3 samples; times_s: their timestamps (mean rate is used); min_dt / max_dt <= 0 select the defaults of sew.py
 * (1 / rate and n / 4 / rate).  spectrum (nullable, n doubles) receives the reference spectrum Xhat (make_reference_spectrum). */
icc_status icc_spline_error_weighting(icc_handle* h, int n, const double* times_s, const double* signal_xyz, double quality, double min_dt, double max_dt,
                                      double* knot_spacing, double* variance, double* spectrum);

/* ---- upstream row f4 (SURVEY.md §8(f)): camera intrinsic calibration ----------------------------------------------------------
 * CameraCalibrator::CalibrateCameraFromJson / RunCalibration (src/core/camera_calibrator.cc:221-389, :131-219) behind
 * applications/calibrate_camera.cc: every view of the corner file gets an initial pose and focal length, views closer than
 * `grid_size` to an already accepted camera position are skipped (:313-325), then theia::BundleAdjustViews runs three times over
 * all view poses + ONE shared intrinsic vector with a Huber(1.345) loss (:140-144):
 *   stage 1  focal length (+ radial distortion unless PINHOLE), poses free (:149-160); views with a mean error > 5 px removed (:162)
 *   stage 2  principal point only, poses constant (:167-174)
 *   stage 3  principal point + focal length + aspect ratio (+ radial for PINHOLE, + tangential for PINHOLE_RADIAL_TANGENTIAL),
 *            poses free (:184-198); views with a mean error > 2 px removed (:200); fewer than 10 views left = failure (:202-205)
 * The residual is theia::ReprojectionError: CameraToPixelCoordinates(intr, R_cw (X - c)) - feature [px].  "Radial distortion" is
 * Theia's per-model subset (k1,k2 | k1..k3 | k1..k4 | k | xi,alpha | alpha,beta | omega).  Initial intrinsics as in AddView
 * (:84-129): principal point = image centre, aspect ratio 1, skew 0, DOUBLE_SPHERE xi = -0.25 alpha = 0.5, EXTENDED_UNIFIED
 * alpha = 0.5 beta = 1, DIVISION_UNDISTORTION k = distortion_init, everything else 0.
 * Initial poses: pass q_wc_init / p_wc_init (+ init_valid) and focal_length_init > 0 to start from your own estimates (what the
 * reference gets from Theia's RANSAC minimal solvers, which are not reproduced), or NULL / <= 0 to have them estimated here:
 * focal length = median over the views of the closed-form estimate from the board homography (Zhang's constraints, principal
 * point at the image centre), poses = homography decomposition + Huber pose refinement under that pinhole camera; for the
 * non-pinhole models focal length, a division-model distortion and the poses are then refined jointly (the quantities
 * utils::initialize_radial_undistortion_camera hands the reference, :283-306) before the target model takes over.
 * Needs icc_set_board_points (planar board for the internal initialiser).
 * Outputs (caller-owned): intrinsics[10] in Theia's order for `model`; per view q_wc / p_wc (as icc_set_frames consumes them),
 * the mean reprojection error [px] (GetReprojErrorOfView) and used[v] = 1 for the views that survive to the end.
 * summary->success = 0 (status still ICC_OK) when fewer than min_num_views views remain, like RunCalibration returning false. */
typedef struct icc_camcal_options {
  double grid_size;                  /* SetGridSize (calibrate_camera.cc:33-35); < 0 selects 0.04 m, 0 keeps every view */
  double function_tolerance;         /* <= 0 selects theia's 1e-6 */
  double parameter_tolerance;        /* <= 0 selects theia's 1e-8 */
  double gradient_tolerance;         /* <= 0 selects theia's 1e-10 */
  double huber_width;                /* <= 0 selects 1.345 (camera_calibrator.cc:143) */
  double max_view_error_stage1_px;   /* <= 0 selects 5.0 (:162) */
  double max_view_error_final_px;    /* <= 0 selects 2.0 (:200) */
  int32_t min_num_views;             /* camera_calibrator.h:84; <= 0 selects 10 */
  int32_t max_num_iterations;        /* theia::BundleAdjustmentOptions (external) default 100 per stage; <= 0 selects it */
  int32_t optimize_board_points;     /* --optimize_board_points (camera_calibrator.cc:207-216): BundleAdjustTracks on the board points with
                                        constant cameras, then the full BundleAdjustViews again; read the points with icc_get_board_points */
  int32_t reserved;
} icc_camcal_options;
typedef struct icc_camcal_summary {
  int32_t success;
  int32_t n_views_initialized;       /* views with an initial pose */
  int32_t n_views_selected;          /* ... that also passed the grid filter */
  int32_t n_views_used;              /* ... that survived both removal passes */
  int32_t iterations[3];             /* LM iterations per stage */
  int32_t termination[3];            /* icc_summary.termination codes per stage */
  int32_t gpu_launches;
  int32_t init_iterations;           /* LM iterations of the internal initialiser's joint refinement (0 when poses / focal length are given) */
  int32_t n_points_optimized;        /* board points refined by optimize_board_points */
  int32_t reserved;
  double focal_length_init;
  double initial_cost;               /* cost at the start of stage 1 */
  double final_cost[3];              /* cost at the end of each stage */
  double final_reproj_error;         /* mean over the used views of their mean reprojection error [px] (camera_calibrator.cc:352-366) */
  double seconds_total;
} icc_camcal_summary;
icc_status icc_calibrate_camera(icc_handle* h, int model, int image_width, int image_height,
                                int n_views, const int32_t* corner_offsets /* n_views+1 */, const int32_t* point_ids, const double* uv,
                                const double* q_wc_init_xyzw /* nullable */, const double* p_wc_init /* nullable */, const int32_t* init_valid /* nullable */,
                                double focal_length_init, double distortion_init, const icc_camcal_options* options /* nullable */,
                                double* intrinsics /* 10 */, double* q_wc_xyzw, double* p_wc, double* view_reproj_error_px, int32_t* view_used,
                                icc_camcal_summary* summary /* nullable */);
/* One iteration body of icc_calibrate_camera's bundle adjustment at a given state (test surface): the normal equations, the damped
 * step at `radius`, the cost at the candidate, and the per-view mean reprojection error at the current state, through the same
 * launches the calibration runs.  Nothing of the handle changes except its last error.
 * Inputs: views in CSR form over the handle's board points; per view q_wc (x,y,z,w; normalised here) and p_wc as
 * icc_calibrate_camera takes them; intrinsics[10] in Theia order; `active`: n_active distinct view indices in any order (slot s
 * holds view active[s]); intr_mask: free intrinsics (bit i = Theia parameter i); pose_free; huber_width; scale_in: the Jacobi
 * scale (6 n_active + 10) of an earlier iteration of the stage, or NULL to compute it as on a stage's first iteration.
 * Tangent of slot s: [delta (right increment of R_cw = conj(q_wc)) | camera centre], then the free intrinsics in Theia order.
 * Outputs, each nullable: blocks (n_active x 153, slot-major): packed upper triangle (row by row) of slot s's 17 x 17
 * [J_pose | J_intr | r]^T [J_pose | J_intr | r] with Huber-weighted rows; sys (154): the sum over slots of the intrinsics part
 * (rows 6..16 of the same packing, other entries 0) and the cost; red (66): the Schur complement of the poses onto the intrinsics,
 * packed upper 10 x 10 (55) then the gradient part (10); Y (n_active x 66): A_s^-1 [H_pk | g_p] (6 x 11, row-major), A_s the
 * damped pose block; scale (6 n_active + 10): the scale used; dk (10): intrinsics step; scalars (8): candidate cost, g.delta,
 * delta^T D delta, |delta|^2, x^2, failed factorisations, max |g|, cost; q_wc_cand / p_wc_cand (n_views) and intr_cand (10): the
 * candidate state (inactive views unchanged); view_error_px (n_views): mean reprojection error of the active views at the current
 * state, 0 elsewhere. */
typedef struct icc_camcal_step_out {
  double* blocks; double* sys; double* red; double* Y; double* scale; double* dk; double* scalars;
  double* q_wc_cand; double* p_wc_cand; double* intr_cand; double* view_error_px;
} icc_camcal_step_out;
icc_status icc_camcal_step(icc_handle* h, int model, int n_views, const int32_t* corner_offsets, const int32_t* point_ids, const double* uv,
                           const double* q_wc_xyzw, const double* p_wc, const double* intrinsics, int n_active, const int32_t* active,
                           uint32_t intr_mask, int pose_free, double huber_width, double radius, const double* scale_in /* nullable */,
                           icc_camcal_step_out* out);

/* ---- upstream: static IMU biases, the `--imu_bias_file` input of the hot CLI ------------------------------------------------------------
 * python/get_imu_biases.py:36-53: gyroscope bias = mean of the gyroscope stream; accelerometer bias = mean of the accelerometer stream
 * after removing gravity along the axis with the largest mean magnitude, gravity = gravity_const * sign(mean) stored as float32 there
 * (np.zeros(..., dtype=np.float32), :43-44 -- the rounding is reproduced).  The two column sums are one reduction kernel on the GPU.
 * Parity of this step is pinned by the reference's own Python (tests/golden/make_imu_bias_golden.py runs the unmodified script). */
icc_status icc_estimate_imu_biases(icc_handle* h, int n, const double* accel_xyz, const double* gyro_xyz, double gravity_const,
                                   double accl_bias[3], double gyro_bias[3]);

/* Device blocks of destroyed handles are cached process-wide for the next job; this returns them to the CUDA driver. */
void icc_trim_device_cache(void);

#ifdef __cplusplus
}
#endif
#endif /* ICC_B200_H_ */
