// Shared host/device structs and kernel launch prototypes (internal to libicc_b200.so).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace icc {

constexpr int SPLINE_N = 6;   // core/imu_camera_calibrator.h:27
constexpr int BIAS_N = 3;     // basalt_spline/ceres_calib_split_residuals.h:21

// Offsets inside the "globals" block of a state: T_i_c (7), gravity (3), line delay, accelerometer / gyroscope intrinsics (6 / 9),
// camera intrinsics (<= 10, Theia order) and the time-offset increment [s] (both constant unless the extension flags free them).
enum { G_TIC = 0, G_GRAV = 7, G_LD = 10, G_ACC_INTR = 11, G_GYR_INTR = 17, G_CAM_INTR = 26, G_TOFF = 36, G_COUNT = 37 };

// One LM state in HBM.  Knots are padded to 32 B (x,y,z,w / x,y,z,0) for 16-byte vector loads.
struct DeviceState {
  double4* so3;
  double4* r3;
  double4* ba;
  double4* bg;
  double* glob;   // G_COUNT doubles
  // board points of this state: homogeneous 4-vectors (parameter blocks under SplineOptimFlags::POINTS), their de-homogenised copy the
  // evaluation kernels read, and the 4 x 3 local Jacobians of ceres::HomogeneousVectorParameterization (icc_points.cu)
  double4* pts; double4* board; double* pjac;
};

struct VisionWork { int frame, c_begin, c_end, pad; };
// Packed corner stream of the TMEM vision kernel (icc_vision_tmem.cu): the non-empty frames are laid end to end, each padded to a
// multiple of four corners (one tensor-core k-step), and the stream is cut into one item per warp at 32-lane chunk boundaries, so
// a chunk may take its first lanes from the end of one frame and the rest from the start of the next.
struct VisFrame { int poff, c0, cn, s_so3, s_r3, pad; double u_so3, u_r3; };   // poff = padded stream offset; entry [n] is a sentinel
struct VisItem { int vf0, pos_begin, pos_end, pad; };                          // first frame touched + stream range
// The same packing for the IMU stream (icc_imu_tmem.cu): knot-interval cells (runs of samples sharing all four knot windows)
struct ImuCellP { int poff, i0, n, s_so3, s_r3, s_ba, s_bg, pad; };            // entries [n], [n+1] are sentinels
struct ImuCell { int s_so3, s_r3, s_ba, s_bg; int i_begin, i_end; };

struct DeviceProblem {
  // camera
  int model, dispatch_fov, n_intr;
  const double4* board;
  // vision: frames in CSR form
  int n_frames, n_corners, rolling;
  const int* f_off;          // n_frames + 1
  const int* f_s_so3; const int* f_s_r3;
  const double* f_u_so3; const double* f_u_r3;
  const double2* uv;
  const int* pid;
  int n_vwork; const VisionWork* vwork;
  int n_vframes; const VisFrame* vframes;    // + sentinel
  int n_vitems; const VisItem* vitems;
  int n_icells; const ImuCellP* icells;      // + sentinels
  int n_iitems; const VisItem* iitems;
  int n_vchunks, n_ichunks;                  // 32-lane chunks of the two packed streams (the launcher's size test)
  // imu: samples sorted by time, grouped into cells sharing all knot windows
  int n_imu;
  const int64_t* imu_t_ns;   // relative to spline start (st_ns)
  const double* imu_acc;     // 3 per sample
  const double* imu_gyr;
  int n_cells; const ImuCell* cells;
  int n_iwork; const ImuCell* iwork;   // cells possibly split into sub-ranges
  int64_t dt_so3_ns, dt_r3_ns, dt_ba_ns, dt_bg_ns;
  double inv_so3_dt, inv_r3_dt;
  double w_acc, w_gyr;
  int n_so3, n_r3, n_ba, n_bg;
  // active-set column maps (solver ordering); -1 = constant block
  const int* so3_col; const int* r3_col; const int* ba_col; const int* bg_col;
  int col_tic, col_g, col_ld, col_ai, col_gi, col_ci, col_to, col_pts;   // col_pts: first of the 3 n_points board-point columns (POINTS)
  int n_points;
  int bias_active;           // any bias block active -> wide IMU tiles
  int intr_active;           // IMU intrinsics and/or time offset free -> widest IMU tiles
  int cam_intr_active;       // camera intrinsics free (extension) -> widest vision tiles
  // normal equations: [band nk x ldb][E nk x nb][C nb x nb (lower)][g nk+nb][cost][pad]
  int nk, nb, kd, ldb;
  double* ne;
  int64_t ne_off_E, ne_off_C, ne_off_g, ne_off_cost, ne_size;
  // residual layout
  int n_res_vis, n_res_acc, n_res_gyr;
};

struct SolveParams {
  double radius, min_diag, max_diag;
  int jacobi_scaling;
};

// scal[] layout written by the solver / update kernels and read back by the host each LM iteration
enum { SC_MODEL_CHANGE = 0, SC_STEP_SQ = 1, SC_X_SQ = 2, SC_CAND_COST = 3, SC_OK = 4, SC_GRAD_MAX = 5, SC_REPROJ_SUM = 6, SC_REPROJ_CNT = 7, SC_X_COST = 8, SC_COUNT = 10 };

// ---- launches (all asynchronous on `st`) ----------------------------------------------------------------------
// residuals + analytic Jacobians + J^T J / J^T r tiles reduced into P.ne (must be zeroed first), or cost only into *cost
// `aux` (optional): a second stream + two events; the IMU kernel then runs concurrently with the vision kernel (fork / join
// around the pair on `st`), which fills the partial last wave of either kernel.
struct EvalAux { cudaStream_t stream; cudaEvent_t fork, join; };
// Persistent TMEM-parked Jacobian evaluation, vision + IMU items in one launch (icc_eval_tmem.cu); non-zero on a launch error.
// P.vitems[k] / P.iitems[k] is the run of global warp k; the two item types go out as two launches of the same kernel.
int launch_eval_tmem(const DeviceProblem& P, const DeviceState& S, double* residuals_out, int sm_count, cudaStream_t st);
int eval_tmem_warps();
int launch_eval(const DeviceProblem& P, const DeviceState& S, bool with_jacobian, double* cost_out, double* residuals_out, double* reproj_out, cudaStream_t st, const EvalAux* aux = nullptr);
// scale[i] = 1/(1+sqrt(H_ii)) (Jacobi scaling, computed once per optimize) ; gradient inf-norm
void launch_compute_scale(const DeviceProblem& P, double* scale, int jacobi, double* scal, cudaStream_t st);
// banded + bordered Cholesky solve of (S H S + D) y = -S g ; delta = S y (solver order) ; model cost change
// returns 0, 1 = no elimination plan fits the shared-memory limits (border far too wide), 2 = a launch failed
// forced_chunks > 0 replaces the plan's own level-0 chunk count (then clamped and halved exactly like the automatic choice)
int launch_solve(const DeviceProblem& P, const double* scale, SolveParams sp, double* workspace, double* delta, double* scal, cudaStream_t st, int forced_chunks = 0);
size_t solve_workspace_doubles(const DeviceProblem& P, int forced_chunks = 0);
// the elimination plan launch_solve would run: valid, P, w, len, rem, L, kd, nb, nk, WS_A, cl_global, cs_global, stage0, 0, 0, 0
void solve_plan_info(const DeviceProblem& P, int forced_chunks, int32_t plan[16]);
// candidate = Plus(current, delta) ; step / x squared norms
void launch_update(const DeviceProblem& P, const DeviceState& cur, const DeviceState& cand, const double* delta, double max_ba, double max_bg, double* scal, cudaStream_t st);
// knot initialisation from the per-view pose priors (icc_init.cu): q_wc / p_wc / t_vis in view-time order, T_c_i = T_i_c^-1 (x,y,z,w,tx,ty,tz)
void launch_init_knots(int nv, const double* t_vis, const double* q_wc, const double* p_wc, const double T_c_i[7], int nso3, int64_t dt_so3_ns, int nr3, int64_t dt_r3_ns,
                       double4* so3_a, double4* so3_b, double4* r3_a, double4* r3_b, cudaStream_t st);
void launch_id_range(int n, const int* ids, int* out2, cudaStream_t st);
// relative integer sample times of a sorted IMU stream from its raw stamps (icc_init.cu)
void launch_imu_times(int n, const double* t_raw, double offset_s, int64_t start_ns, int64_t* st_out, cudaStream_t st);
// board points as parameters (icc_points.cu)
void launch_points_prepare(int n, const double4* pts, double4* board, double* jac, cudaStream_t st);
void launch_points_update(int n, int col_pts, const double4* cur, double4* cand, double4* board, double* jac, const double* delta, double* scal, cudaStream_t st);
void launch_points_jac(const DeviceProblem& P, const DeviceState& S, const double* pjac, int col_pts, int sm_count, cudaStream_t st);
// trajectory getters
void launch_eval_trajectory(const DeviceProblem& P, const DeviceState& S, int n, const int64_t* t_ns, int64_t start_ns, double* gyro, double* accel,
                            double* bg, double* ba, double* pose_q, double* pose_p, int* valid, cudaStream_t st);
// ---- per-view board poses (icc_pose.cu) ---------------------------------------------------------------------------
struct PoseProblem {
  int model; double intr[10];
  int n_frames, n_points, min_points;
  const double4* board; const int* f_off; const int* pid;
  double thresh_sq;            // squared normalised reprojection error of an inlier (pose_estimator.cc:100-101)
  double max_err;              // views above this mean error are dropped (pose_estimator.cc:181)
  double lm_rel_tol;           // relative cost decrease that ends the refinement (0 selects 1e-15: poses pinned to ~1e-9; an initialiser can stop far earlier)
  int refine_only;             // 1: start from the poses already in q_wc / p_wc (valid views only), no homography (OptimizeAllPoses, :226-236)
};
void launch_unproject(int model, const double* intr10, int n, const double2* uv, double2* xy, int* ok, cudaStream_t st);
void launch_board_poses(const PoseProblem& Q, const double2* xy, const int* ok, unsigned char* use, double* q_wc, double* p_wc, double* err, int* valid, cudaStream_t st);
// board point refinement with constant cameras (theia::BundleAdjustTracks), one warp per point
struct PointProblem {
  int model; double intr[10];
  int normalized;              // 1: measurements are undistorted normalised coordinates (unit pinhole), 0: pixels through `model`
  int n_points, min_obs;       // points with more than min_obs observations are optimised
  double huber;
  const double4* board_in;
  const int* pt_off; const int* pt_obs;    // CSR by point: corner indices of the observations that take part
  const int* obs_view;         // view index of every corner
  const double2* meas;         // per corner: xy (normalised) or uv (pixels)
  const double* q_cw; const double* cam_c; // per view: R_cw as (x,y,z,w), camera centre
};
void launch_point_refine(const PointProblem& Q, double4* board_out, int* optimized, cudaStream_t st);
// focal length per view from the board homography on centred pixels (f2[v] = f^2 or 0), pinhole normalisation of pixels
void launch_board_focal(const PoseProblem& Q, const double2* uv, double cx, double cy, double2* xy, unsigned char* use, double* f2, cudaStream_t st);
void launch_pinhole_normalize(int n, const double2* uv, double cx, double cy, double f, double2* xy, int* ok, cudaStream_t st);
// ---- camera intrinsic calibration: bundle adjustment of view poses + shared intrinsics (icc_camcal.cu) ----------------------
// Column order of a view's [J | r] rows: 0-2 rotation increment, 3-5 camera centre, 6-15 intrinsics (Theia order), 16 residual.
constexpr int CC_COLS = 17, CC_PACK = CC_COLS * (CC_COLS + 1) / 2, CC_Y = 66;   // packed upper triangle; Y = A^-1 [H_pk | g_p] (6 x 11)
enum { CC_CAND_COST = 0, CC_G_DELTA = 1, CC_D_DELTA = 2, CC_STEP_SQ = 3, CC_X_SQ = 4, CC_FAIL = 5, CC_GRAD_MAX = 6, CC_X_COST = 7, CC_SCAL_COUNT = 8 };
struct CamCalProblem {
  int model, n_points, n_active, pose_free;
  unsigned intr_mask;          // bit i set = intrinsic i is optimised in this stage
  double huber;                // loss width (camera_calibrator.cc:143)
  const double4* board; const int* f_off; const int* pid; const double2* uv;
  const int* active;           // indices of the views that take part (n_active)
};
struct CamCalState { double* q; double* c; double* k; };   // R_cw as (x,y,z,w) per view, camera centre per view, 10 intrinsics
// with_jacobian: per-view packed blocks (n_active x CC_PACK) + the intrinsics part and the cost summed into sys[CC_PACK + 1];
// otherwise cost only into *cost_out and (optional) the per-view mean reprojection error [px] into view_err (indexed by view)
void launch_camcal_accumulate(const CamCalProblem& Q, const CamCalState& S, bool with_jacobian, double* blocks, double* sys, double* cost_out, double* view_err, cudaStream_t st);
// one damped step: per-view Schur elimination, reduced intrinsics system, back-substitution into the candidate state
void launch_camcal_step(const CamCalProblem& Q, const CamCalState& cur, const CamCalState& cand, const double* blocks, const double* sys, double* red /* 66 */, double* Y,
                        double* scale /* 6 n_active + 10 */, int compute_scale, double radius, double min_diag, double max_diag, double* dk /* 10 */, double* scal, cudaStream_t st);
// ---- IMU-to-camera rotation + time offset initialiser (icc_rotinit.cu) -----------------------------------------------------
struct RotInitState {
  double a, b, c, d;          // golden-section bracket and its two interior candidates (time offsets, seconds)
  double sums[2][16];         // per candidate: sum vis (3), sum imu (3), sum imu x vis (9), robust error
  double R[2][9], bias[2][3]; // per candidate closed-form solution (row-major)
  double R_best[9], bias_best[3], error;
  int iterations, done;
};
struct RotInitProblem {
  int n;                      // IMU samples inside the common time window
  const double* t;            // their zero-based timestamps (sorted)
  const double* vis;          // smoothed visual angular velocity at those times (3 per sample)
  const double* imu;          // smoothed gyroscope rates (3 per sample)
  double* vis_shift;          // scratch: 2 x 3n, the shifted + interpolated visual rates of both candidates
  RotInitState* state;
  int estimate_bias;
  double tolerance;
  double bias_in[3];
};
void launch_interp_quat(int n_old, const double* t_old, const double4* q_old, int n_new, const double* t_new, double4* q_new, cudaStream_t st);
void launch_visual_angular_velocity(int n, const double4* q, double dt_imu, double* w_raw, unsigned char* bad, double* w_held, double* w_smooth, const double* imu, double* imu_smooth, cudaStream_t st);
void launch_golden_section(const RotInitProblem& Q, double max_offset, int max_iterations, int sm_count, cudaStream_t st);
// ---- spline error weighting (icc_sew.cu) ------------------------------------------------------------------------------------
int sew_fft_length(int N);      // power-of-two length of the Bluestein convolution
void launch_sew_spectrum(int N, const double* signal /* N x 3 */, double* xhat /* N */, double* energy_sum, double* scratch /* 16 * sew_fft_length(N) doubles */, cudaStream_t st);
void launch_sew_residual_energy(int N, const double* xhat, double fscale, double dt, double* out, int sm_count, cudaStream_t st);
// column sums of the accelerometer / gyroscope streams (static bias estimate, python/get_imu_biases.py)
void launch_imu_sums(int n, const double* acc, const double* gyr, double* out6, int sm_count, cudaStream_t st);
int kernel_launch_count();

}  // namespace icc
