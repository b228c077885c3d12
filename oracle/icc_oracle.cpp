// ORACLE — TEST INFRASTRUCTURE ONLY (see oracle_math.hpp header).  PARITY UNPINNED by reference tests (none exist).
//
// CPU restatement of the reference's continuous-time IMU-camera calibration hot path, exported with the same C-ABI
// shape as include/icc_b200.h but with the `icco_` prefix:
//   * problem assembly      ~ src/core/imu_camera_calibrator.cc:21-161
//                             include/OpenCameraCalibrator/core/spline_trajectory_estimator.impl.h:37-90,278-339,341-613,763-788
//   * spline initialisation ~ src/utils/utils.cc:194-261 (FindClosestTimestamp / slerp / lerp, quirks kept)
//   * residual functors     ~ include/OpenCameraCalibrator/basalt_spline/ceres_calib_split_residuals.h:52-93,133-169,319-402
//   * Jacobians             ~ ceres::DynamicAutoDiffCostFunction (stride-4 forward-mode passes over the ACTIVE ambient
//                             parameters) times LieLocalParameterization::ComputeJacobian
//                             (basalt_spline/ceres_local_param.h:96-108; Sophus so3.hpp:191-220, se3.hpp:135-200)
//   * fixed / free blocks   ~ SplineTrajectoryEstimator::SetFixedParams (impl.h:92-252)
//   * Levenberg-Marquardt   ~ ceres::Solve with the options of impl.h:254-266 and Ceres-2.1 defaults (external source;
//                             restated from its documentation: TrustRegionMinimizer + LevenbergMarquardtStrategy,
//                             Jacobi scaling, SPARSE_NORMAL_CHOLESKY replaced by an exact banded+bordered Cholesky).
//                             NOT restated: use_inner_iterations (coordinate-descent refinement; same optimum, different
//                             path) and the projected line search for bound constraints (plain projection is used).
//   * result getters        ~ impl.h:898-1072,1180-1234
// Doubles as the timed CPU baseline (std::thread over residual blocks, like Ceres' num_threads = hardware_concurrency()).
#include "oracle_math.hpp"
#include "../include/icc_b200.h"

#include <algorithm>
#include <chrono>
#include <time.h>
#include <condition_variable>
#include <memory>
#include <mutex>
#include <cstdio>
#include <functional>
#include <map>
#include <string>
#include <thread>
#include <vector>

using namespace icco;

namespace {

constexpr int SPLINE_N = 6;   // core/imu_camera_calibrator.h:27
constexpr int BIAS_N = 3;     // basalt_spline/ceres_calib_split_residuals.h:21
constexpr double S_TO_NS = 1e9, NS_TO_S = 1e-9;

enum BlockType { BLK_RS_VISION = 0, BLK_ACCEL = 1, BLK_GYRO = 2 };
enum LocalParam { LP_NONE = 0, LP_SO3 = 1, LP_SE3 = 2, LP_HOMOG4 = 3 };   // LP_HOMOG4: ceres::HomogeneousVectorParameterization(4) of a board point (impl.h:148-150)

struct ParamRef { const double* ptr; int size; int lp; int tan_off; };  // tan_off < 0 => constant block

struct Block {
  int type;
  int n_res;
  int res_off;                  // offset into the global residual vector
  int frame;                    // vision: frame index; imu: sample index
  double u_so3, u_r3, u_bias;
  std::vector<ParamRef> params;
};

struct Frame { double t_s; int c0, c1; int64_t s_so3, s_r3; double u_so3, u_r3; bool ok; };
struct ImuUsed { double t_s; double acc[3], gyr[3]; };

struct Oracle {
  std::string err;
  icc_solver_options opt;
  int n_threads = 0;
  // camera + board
  int model = -1, n_intr = 0, width = 0, height = 0; double intr[10] = {0};
  std::vector<double> points;
  // frames
  std::vector<double> frame_t; std::vector<int> corner_off, point_ids; std::vector<double> uv, q_wc, p_wc;
  // imu
  std::vector<double> imu_t, imu_acc, imu_gyr;
  // shard
  int shard_rank = 0, shard_world = 1;
  // initialised problem
  bool initialised = false;
  icc_init_params ip;
  bool dispatch_fov = false;
  int64_t dt_so3_ns = 0, dt_r3_ns = 0, start_ns = 0, end_ns = 0, dt_ba_ns = 0, dt_bg_ns = 0;
  double inv_so3_dt = 0, inv_r3_dt = 0, inv_ba_dt = 0, inv_bg_dt = 0;
  double t0_s = 0, tend_s = 0;
  std::vector<double> so3, r3, ba, bg;   // knots
  double T_ic[7], grav[3], line_delay = 0, acc_intr[6], gyr_intr[9];
  double toff_delta = 0;            // extension: increment of the IMU->camera time offset [s]
  double max_ba = 1.0, max_bg = 0.1;
  std::vector<Frame> frames;
  std::vector<ImuUsed> imu_used;
  std::vector<Block> blocks;
  std::vector<Block> vis_blocks;   // RS vision blocks of every view, always built (GetMeanReprojectionError uses them even on the GS path)
  int n_res_vis = 0, n_res_acc = 0, n_res_gyr = 0;
  // active set / ordering (rebuilt per flags)
  int cur_flags = -1;
  int n_tan = 0;
  int off_so3 = -1, off_r3 = -1, off_tic = -1, off_g = -1, off_ld = -1, off_ba = -1, off_bg = -1, off_ai = -1, off_gi = -1, off_ci = -1, off_to = -1, off_pts = -1;  // canonical offsets
  // solver ordering: canonical tangent index -> solver index
  std::vector<int> perm;      // canonical -> solver
  int n_knot_dims = 0, n_border = 0, kd = 0;
  int jac_evals = 0, cost_evals = 0;
  double pose_rel_tol = 1e-15;     // stopping tolerance of the per-view pose refinement (the camera calibrator's initialiser loosens it)
  // Ceres inner iterations (Solver::Options::use_inner_iterations, impl.h:266): off by default so that the oracle mirrors the CUDA
  // LM path; switched on by icco_set_inner_iterations for the stopping-point study (tests/test_inner_iterations.py)
  bool inner_iterations = false; double inner_iteration_tolerance = 1e-3; int inner_iteration_steps = 0;
  std::shared_ptr<struct InnerPlan> inner_plan;
  std::shared_ptr<struct EvalCtx> ctx;   // persistent worker pool + per-thread partial normal equations (created on first use)
};

int nknots(const std::vector<double>& v, int dim) { return int(v.size()) / dim; }

// impl.h:763-788
bool calc_times(int64_t sensor_ns, int64_t start_ns, int64_t dt_ns, size_t nr_knots, int N, double& u, int64_t& s) {
  const int64_t st_ns = sensor_ns - start_ns;
  if (st_ns < 0) { u = 0.0; return false; }
  s = st_ns / dt_ns;
  if (s < 0) return false;
  if (size_t(s + N) > nr_knots) return false;
  u = double(st_ns % dt_ns) / double(dt_ns);
  return true;
}

// utils.cc:194-212
size_t find_closest(double t, const std::vector<double>& ts, double& dist_out) {
  double dist = 1.7976931348623157e308; size_t idx = 0;
  for (size_t i = 0; i < ts.size(); ++i) {
    double nd = std::fabs(t - ts[i]);
    if (nd < dist) { dist_out = nd; idx = i; dist = nd; if (dist_out == 0.0) break; }
  }
  return idx;
}
// Eigen::QuaternionBase::slerp
void slerp(const double a[4], const double b[4], double t, double out[4]) {
  const double one = 1.0 - 2.220446049250313e-16;
  double d = a[0] * b[0] + a[1] * b[1] + a[2] * b[2] + a[3] * b[3];
  double ad = std::fabs(d), s0, s1;
  if (ad >= one) { s0 = 1.0 - t; s1 = t; }
  else { double th = std::acos(ad), st = std::sin(th); s0 = std::sin((1.0 - t) * th) / st; s1 = std::sin(t * th) / st; }
  if (d < 0) s1 = -s1;
  for (int i = 0; i < 4; ++i) out[i] = s0 * a[i] + s1 * b[i];
}

// -------------------------------------------------------------------------------------------------------------
// Residual functors, templated on the scalar like the reference.
// -------------------------------------------------------------------------------------------------------------
template <class T>
void rs_reprojection(const Oracle& o, const Block& b, const T* const* P, T* res) {   // residuals.h:319-402
  const int N2 = 2 * SPLINE_N;
  SE3T<T> T_i_c{{P[N2][0], P[N2][1], P[N2][2], P[N2][3]}, {P[N2][4], P[N2][5], P[N2][6]}};
  const T line_delay = P[N2 + 1][0];
  T intr[10];
  for (int i = 0; i < o.n_intr; ++i) intr[i] = P[N2 + 2][i];   // extension: intrinsics are a (normally constant) parameter block
  const Frame& f = o.frames[b.frame];
  for (int c = f.c0; c < f.c1; ++c) {
    const int i = c - f.c0;
    const double ox = o.uv[2 * c], oy = o.uv[2 * c + 1];
    const T y_coord = T(oy) * line_delay;
    const T t_so3_row = T(b.u_so3) + y_coord;
    const T t_r3_row = T(b.u_r3) + y_coord;
    Q4<T> R_w_i;
    evaluate_lie_so3<SPLINE_N, T>(P, t_so3_row, T(o.inv_so3_dt), &R_w_i, nullptr);
    V3<T> t_w_i = evaluate_r3<SPLINE_N, 0, T>(P + SPLINE_N, t_r3_row, T(o.inv_r3_dt));
    SE3T<T> T_w_c = se3_mul(SE3T<T>{R_w_i, t_w_i}, T_i_c);
    SE3T<T> T_c_w = se3_inv(T_w_c);
    M3<T> R = so3_matrix(T_c_w.q);
    const T* X = P[N2 + 3 + i];
    // (T_c_w.matrix() * X_h).hnormalized()
    T h[3];
    h[0] = R.m[0][0] * X[0] + R.m[0][1] * X[1] + R.m[0][2] * X[2] + T_c_w.t.x * X[3];
    h[1] = R.m[1][0] * X[0] + R.m[1][1] * X[1] + R.m[1][2] * X[2] + T_c_w.t.y * X[3];
    h[2] = R.m[2][0] * X[0] + R.m[2][1] * X[1] + R.m[2][2] * X[2] + T_c_w.t.z * X[3];
    T p3[3] = {h[0] / X[3], h[1] / X[3], h[2] / X[3]};
    T px[2];
    const bool ok = project<T>(o.model, intr, p3, px, o.dispatch_fov);
    if (!ok) { res[2 * i] = T(1e10); res[2 * i + 1] = T(1e10); }
    else { res[2 * i] = px[0] - T(ox); res[2 * i + 1] = px[1] - T(oy); }   // covariance = I (app :157)
  }
}

template <class T>
void accel_residual(const Oracle& o, const Block& b, const T* const* P, T* res) {   // residuals.h:52-93
  const ImuUsed& m = o.imu_used[b.frame];
  const T dto = P[2 * SPLINE_N + BIAS_N + 2][0];   // extension: time-offset increment [s]; du = dto * 1e9 / dt_ns
  Q4<T> R_w_i;
  evaluate_lie_so3<SPLINE_N, T>(P, T(b.u_so3) + dto * o.inv_so3_dt, T(o.inv_so3_dt), &R_w_i, nullptr);
  V3<T> accel_w = evaluate_r3<SPLINE_N, 2, T>(P + SPLINE_N, T(b.u_r3) + dto * o.inv_r3_dt, T(o.inv_r3_dt));
  V3<T> bias = evaluate_r3<BIAS_N, 0, T>(P + 2 * SPLINE_N, T(b.u_bias) + dto * (S_TO_NS / double(o.dt_ba_ns)), T(o.inv_ba_dt));
  const T* g = P[2 * SPLINE_N + BIAS_N];
  const T* ai = P[2 * SPLINE_N + BIAS_N + 1];
  V3<T> raw{T(m.acc[0]), T(m.acc[1]), T(m.acc[2])};
  V3<T> cal = triad_unbias_normalize<T>(ai[0], ai[1], ai[2], T(0.0), T(0.0), T(0.0), ai[3], ai[4], ai[5], bias, raw);
  V3<T> aw{accel_w.x + g[0], accel_w.y + g[1], accel_w.z + g[2]};
  V3<T> pred = so3_act(so3_inv(R_w_i), aw);
  const T w(1.0 / o.ip.std_r3);
  res[0] = w * (pred.x - cal.x); res[1] = w * (pred.y - cal.y); res[2] = w * (pred.z - cal.z);
}

template <class T>
void gyro_residual(const Oracle& o, const Block& b, const T* const* P, T* res) {   // residuals.h:133-169
  const ImuUsed& m = o.imu_used[b.frame];
  V3<T> rot_vel;
  const T dto = P[SPLINE_N + BIAS_N + 1][0];
  evaluate_lie_so3<SPLINE_N, T>(P, T(b.u_so3) + dto * o.inv_so3_dt, T(o.inv_so3_dt), nullptr, &rot_vel);
  V3<T> bias = evaluate_r3<BIAS_N, 0, T>(P + SPLINE_N, T(b.u_bias) + dto * (S_TO_NS / double(o.dt_bg_ns)), T(o.inv_bg_dt));
  const T* gi = P[SPLINE_N + BIAS_N];
  V3<T> raw{T(m.gyr[0]), T(m.gyr[1]), T(m.gyr[2])};
  V3<T> cal = triad_unbias_normalize<T>(gi[0], gi[1], gi[2], gi[3], gi[4], gi[5], gi[6], gi[7], gi[8], bias, raw);
  const T w(1.0 / o.ip.std_so3);
  res[0] = w * (rot_vel.x - cal.x); res[1] = w * (rot_vel.y - cal.y); res[2] = w * (rot_vel.z - cal.z);
}

template <class T>
void eval_block_T(const Oracle& o, const Block& b, const T* const* P, T* res) {
  switch (b.type) {
    case BLK_RS_VISION: rs_reprojection<T>(o, b, P, res); break;
    case BLK_ACCEL: accel_residual<T>(o, b, P, res); break;
    case BLK_GYRO: gyro_residual<T>(o, b, P, res); break;
  }
}

// so3.hpp:191-220 / se3.hpp:135-200 : d(this * exp(x))/dx at 0, rows = ambient coeffs, cols = tangent
void lp_jacobian_so3(const double* q, double J[4][3]) {
  const double c0 = 0.5 * q[3], c1 = 0.5 * q[2], c2 = -c1, c3 = 0.5 * q[1], c4 = 0.5 * q[0], c5 = -c4, c6 = -c3;
  J[0][0] = c0; J[0][1] = c2; J[0][2] = c3;
  J[1][0] = c1; J[1][1] = c0; J[1][2] = c5;
  J[2][0] = c6; J[2][1] = c4; J[2][2] = c0;
  J[3][0] = c5; J[3][1] = c6; J[3][2] = c2;
}
void lp_jacobian_se3(const double* T7, double J[7][6]) {
  for (int i = 0; i < 7; ++i) for (int j = 0; j < 6; ++j) J[i][j] = 0;
  double Jq[4][3]; lp_jacobian_so3(T7, Jq);
  for (int i = 0; i < 4; ++i) for (int j = 0; j < 3; ++j) J[i][3 + j] = Jq[i][j];
  Q4<double> q{T7[0], T7[1], T7[2], T7[3]};
  M3<double> R = so3_matrix(q);   // identical to the c7..c21 polynomial for unit quaternions
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) J[4 + i][j] = R.m[i][j];
}

// ceres::HomogeneousVectorParameterization(4) (Ceres 2.1 local_parameterization.cc; not in /root/reference -- restated):
// Householder vector v, beta with (I - beta v v^T) x = |x| e_4 (internal::ComputeHouseholderVector); Jacobian = |x| / 2 x the first
// three columns of H; Plus(x, d) = |x| H [sin(|d|/2) d / |d| ; cos(|d|/2)]  (Hartley & Zisserman A6.9.2-3).
void householder4(const double* x, double v[4], double& beta) {
  const double sigma = x[0] * x[0] + x[1] * x[1] + x[2] * x[2];
  v[0] = x[0]; v[1] = x[1]; v[2] = x[2]; v[3] = 1.0; beta = 0.0;
  const double xp = x[3];
  if (sigma <= 2.220446049250313e-16) { if (xp < 0.0) beta = 2.0; return; }
  const double mu = std::sqrt(xp * xp + sigma);
  const double vp = xp <= 0.0 ? xp - mu : -sigma / (xp + mu);
  beta = 2.0 * vp * vp / (sigma + vp * vp);
  v[0] /= vp; v[1] /= vp; v[2] /= vp;
}
void lp_jacobian_homog4(const double* x, double J[4][3]) {
  double v[4], beta; householder4(x, v, beta);
  const double n = std::sqrt(x[0] * x[0] + x[1] * x[1] + x[2] * x[2] + x[3] * x[3]);
  for (int i = 0; i < 3; ++i) for (int k = 0; k < 4; ++k) J[k][i] = n * (-0.5 * beta * v[i] * v[k] + (k == i ? 0.5 : 0.0));
}
void plus_homog4(double* x, const double* d) {
  const double nd = std::sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
  if (nd == 0.0) return;
  const double h = 0.5 * nd, sbd = std::sin(h) / h;
  const double y[4] = {0.5 * sbd * d[0], 0.5 * sbd * d[1], 0.5 * sbd * d[2], std::cos(h)};
  double v[4], beta; householder4(x, v, beta);
  const double n = std::sqrt(x[0] * x[0] + x[1] * x[1] + x[2] * x[2] + x[3] * x[3]);
  const double vy = v[0] * y[0] + v[1] * y[1] + v[2] * y[2] + v[3] * y[3];
  for (int k = 0; k < 4; ++k) x[k] = n * (y[k] - v[k] * (beta * vy));
}

struct Scratch {
  std::vector<Jet<4>> jets; std::vector<const Jet<4>*> jptr; std::vector<Jet<4>> jres;
  std::vector<const double*> dptr; std::vector<double> res; std::vector<double> Jamb, Jtan; std::vector<int> cols;
};

// Evaluate one block: residuals always; tangent Jacobian (row-major n_res x n_cols with global canonical column ids) if wanted.
void eval_block(const Oracle& o, const Block& b, Scratch& s, bool want_jac, int& n_cols_out) {
  const int np = int(b.params.size());
  s.dptr.resize(np);
  for (int i = 0; i < np; ++i) s.dptr[i] = b.params[i].ptr;
  s.res.assign(b.n_res, 0.0);
  n_cols_out = 0;
  if (!want_jac) { eval_block_T<double>(o, b, s.dptr.data(), s.res.data()); return; }
  // ambient layout over active params
  int A = 0, total = 0;
  for (const auto& p : b.params) { total += p.size; if (p.tan_off >= 0) A += p.size; }
  s.jets.resize(total); s.jptr.resize(np); s.jres.resize(b.n_res);
  s.Jamb.assign(size_t(b.n_res) * std::max(A, 1), 0.0);
  const int passes = (A + 3) / 4;
  bool have_res = false;
  for (int pass = 0; pass < std::max(passes, 1); ++pass) {
    int off = 0, a = 0;
    for (int i = 0; i < np; ++i) {
      const auto& p = b.params[i];
      s.jptr[i] = &s.jets[off];
      for (int k = 0; k < p.size; ++k) {
        Jet<4>& j = s.jets[off + k];
        j.a = p.ptr[k]; j.v[0] = j.v[1] = j.v[2] = j.v[3] = 0;
        if (p.tan_off >= 0) { const int lane = a - 4 * pass; if (lane >= 0 && lane < 4) j.v[lane] = 1.0; ++a; }
      }
      off += p.size;
    }
    eval_block_T<Jet<4>>(o, b, s.jptr.data(), s.jres.data());
    if (!have_res) { for (int r = 0; r < b.n_res; ++r) s.res[r] = s.jres[r].a; have_res = true; }
    for (int r = 0; r < b.n_res; ++r) for (int l = 0; l < 4; ++l) { const int col = 4 * pass + l; if (col < A) s.Jamb[size_t(r) * A + col] = s.jres[r].v[l]; }
  }
  // ambient -> tangent through the local parameterisations
  int ncols = 0;
  for (const auto& p : b.params) if (p.tan_off >= 0) ncols += (p.lp == LP_SO3 ? 3 : p.lp == LP_SE3 ? 6 : p.lp == LP_HOMOG4 ? 3 : p.size);
  s.Jtan.assign(size_t(b.n_res) * std::max(ncols, 1), 0.0); s.cols.resize(ncols);
  int a = 0, c = 0;
  for (const auto& p : b.params) {
    if (p.tan_off < 0) continue;
    if (p.lp == LP_SO3) {
      double L[4][3]; lp_jacobian_so3(p.ptr, L);
      for (int r = 0; r < b.n_res; ++r) for (int j = 0; j < 3; ++j) { double v = 0; for (int k = 0; k < 4; ++k) v += s.Jamb[size_t(r) * A + a + k] * L[k][j]; s.Jtan[size_t(r) * ncols + c + j] = v; }
      for (int j = 0; j < 3; ++j) s.cols[c + j] = p.tan_off + j;
      a += 4; c += 3;
    } else if (p.lp == LP_HOMOG4) {
      double L[4][3]; lp_jacobian_homog4(p.ptr, L);
      for (int r = 0; r < b.n_res; ++r) for (int j = 0; j < 3; ++j) { double v = 0; for (int k = 0; k < 4; ++k) v += s.Jamb[size_t(r) * A + a + k] * L[k][j]; s.Jtan[size_t(r) * ncols + c + j] = v; }
      for (int j = 0; j < 3; ++j) s.cols[c + j] = p.tan_off + j;
      a += 4; c += 3;
    } else if (p.lp == LP_SE3) {
      double L[7][6]; lp_jacobian_se3(p.ptr, L);
      for (int r = 0; r < b.n_res; ++r) for (int j = 0; j < 6; ++j) { double v = 0; for (int k = 0; k < 7; ++k) v += s.Jamb[size_t(r) * A + a + k] * L[k][j]; s.Jtan[size_t(r) * ncols + c + j] = v; }
      for (int j = 0; j < 6; ++j) s.cols[c + j] = p.tan_off + j;
      a += 7; c += 6;
    } else {
      for (int r = 0; r < b.n_res; ++r) for (int j = 0; j < p.size; ++j) s.Jtan[size_t(r) * ncols + c + j] = s.Jamb[size_t(r) * A + a + j];
      for (int j = 0; j < p.size; ++j) s.cols[c + j] = p.tan_off + j;
      a += p.size; c += p.size;
    }
  }
  n_cols_out = ncols;
}

// -------------------------------------------------------------------------------------------------------------
// Active set (SetFixedParams, impl.h:92-252) and solver ordering.
// -------------------------------------------------------------------------------------------------------------
bool configure(Oracle& o, int flags) {
  const bool pts = flags & ICC_FLAG_POINTS;     // board points as parameter blocks with HomogeneousVectorParameterization(4) (impl.h:136-152)
  const int nso3 = nknots(o.so3, 4), nr3 = nknots(o.r3, 3), nba = nknots(o.ba, 3), nbg = nknots(o.bg, 3);
  const bool spline = flags & ICC_FLAG_SPLINE, tic = flags & ICC_FLAG_T_I_C, grav = flags & ICC_FLAG_GRAVITY_DIR;
  // line delay block: only touched by SetFixedParams when != 0; a zero line delay means the GS path (no such block)
  const bool ld = (flags & ICC_FLAG_CAM_LINE_DELAY) && o.line_delay != 0.0;
  const bool abias = flags & (ICC_FLAG_ACC_BIAS | ICC_FLAG_IMU_BIASES), gbias = flags & (ICC_FLAG_GYR_BIAS | ICC_FLAG_IMU_BIASES);
  const bool imu_intr = flags & ICC_FLAG_IMU_INTRINSICS;
  int n = 0;
  o.off_so3 = spline ? n : -1; if (spline) n += 3 * nso3;
  o.off_r3 = spline ? n : -1; if (spline) n += 3 * nr3;
  o.off_tic = tic ? n : -1; if (tic) n += 6;
  o.off_g = grav ? n : -1; if (grav) n += 3;
  o.off_ld = ld ? n : -1; if (ld) n += 1;
  o.off_ba = abias ? n : -1; if (abias) n += 3 * nba;
  o.off_bg = gbias ? n : -1; if (gbias) n += 3 * nbg;
  const bool cam_intr = flags & ICC_FLAG_CAM_INTRINSICS, toff = flags & ICC_FLAG_TIME_OFFSET;
  const int off_ai = imu_intr ? n : -1; if (imu_intr) n += 6;
  const int off_gi = imu_intr ? n : -1; if (imu_intr) n += 9;
  const int off_ci = cam_intr ? n : -1; if (cam_intr) n += o.n_intr;
  const int off_to = toff ? n : -1; if (toff) n += 1;
  const int n_points = int(o.points.size() / 4);
  o.off_pts = pts ? n : -1; if (pts) n += 3 * n_points;
  o.off_ai = off_ai; o.off_gi = off_gi; o.off_ci = off_ci; o.off_to = off_to;
  o.n_tan = n; o.cur_flags = flags;
  // wire tangent offsets into the blocks
  for (auto& b : o.blocks) {
    int k = 0;
    auto so3k = [&](int64_t s) { for (int i = 0; i < SPLINE_N; ++i) b.params[k++].tan_off = spline ? o.off_so3 + 3 * int(s + i) : -1; };
    auto r3k = [&](int64_t s) { for (int i = 0; i < SPLINE_N; ++i) b.params[k++].tan_off = spline ? o.off_r3 + 3 * int(s + i) : -1; };
    if (b.type == BLK_RS_VISION) {
      const Frame& f = o.frames[b.frame];
      so3k(f.s_so3); r3k(f.s_r3);
      b.params[k++].tan_off = o.off_tic;
      b.params[k++].tan_off = o.off_ld;
      b.params[k++].tan_off = off_ci;
      for (; k < int(b.params.size()); ++k) {      // the view's board points (only the points a view sees enter the problem: tracks_in_problem_)
        const int id = int((b.params[k].ptr - o.points.data()) / 4);
        b.params[k].tan_off = pts ? o.off_pts + 3 * id : -1; b.params[k].lp = pts ? LP_HOMOG4 : LP_NONE;
      }
    } else if (b.type == BLK_ACCEL) {
      const int64_t s_so3 = (b.params[0].ptr - o.so3.data()) / 4, s_r3 = (b.params[SPLINE_N].ptr - o.r3.data()) / 3;
      const int64_t s_b = (b.params[2 * SPLINE_N].ptr - o.ba.data()) / 3;
      so3k(s_so3); r3k(s_r3);
      for (int i = 0; i < BIAS_N; ++i) b.params[k++].tan_off = abias ? o.off_ba + 3 * int(s_b + i) : -1;
      b.params[k++].tan_off = o.off_g;
      b.params[k++].tan_off = off_ai;
      b.params[k++].tan_off = off_to;
    } else {
      const int64_t s_so3 = (b.params[0].ptr - o.so3.data()) / 4, s_b = (b.params[SPLINE_N].ptr - o.bg.data()) / 3;
      so3k(s_so3);
      for (int i = 0; i < BIAS_N; ++i) b.params[k++].tan_off = gbias ? o.off_bg + 3 * int(s_b + i) : -1;
      b.params[k++].tan_off = off_gi;
      b.params[k++].tan_off = off_to;
    }
  }
  // solver ordering: spline knots sorted by knot time (so3 before r3 on ties) form the banded part, rest = border
  o.perm.assign(n, -1);
  int pos = 0;
  if (spline) {
    int i = 0, j = 0;
    while (i < nso3 || j < nr3) {
      const bool take_so3 = j >= nr3 || (i < nso3 && int64_t(i) * o.dt_so3_ns <= int64_t(j) * o.dt_r3_ns);
      const int base = take_so3 ? o.off_so3 + 3 * i++ : o.off_r3 + 3 * j++;
      for (int d = 0; d < 3; ++d) o.perm[base + d] = pos++;
    }
  }
  o.n_knot_dims = pos;
  for (int c = 0; c < n; ++c) if (o.perm[c] < 0) o.perm[c] = pos++;
  o.n_border = n - o.n_knot_dims;
  // half bandwidth from the residual blocks
  int kd = 0;
  if (spline) for (const auto& b : o.blocks) {
    int lo = 1 << 30, hi = -1;
    for (const auto& p : b.params) if (p.tan_off >= 0 && o.perm[p.tan_off] < o.n_knot_dims) { lo = std::min(lo, o.perm[p.tan_off]); hi = std::max(hi, o.perm[p.tan_off] + 2); }
    if (hi >= 0) kd = std::max(kd, hi - lo);
  }
  o.kd = kd;
  return true;
}

// -------------------------------------------------------------------------------------------------------------
// Normal equations in banded + bordered ("arrowhead") storage, solver ordering.
// -------------------------------------------------------------------------------------------------------------
struct Normal {
  int nk = 0, nb = 0, kd = 0;
  std::vector<double> band;   // nk x (kd+1): band[j*(kd+1) + (i-j)], i >= j
  std::vector<double> E;      // nb x nk : E[b*nk + j]
  std::vector<double> C;      // nb x nb (full symmetric)
  std::vector<double> g;      // nk + nb
  double cost = 0;
  void init(int nk_, int nb_, int kd_) { nk = nk_; nb = nb_; kd = kd_; band.assign(size_t(nk) * (kd + 1), 0.0); E.assign(size_t(nb) * nk, 0.0); C.assign(size_t(nb) * nb, 0.0); g.assign(nk + nb, 0.0); cost = 0; }
  inline void add(int i, int j, double v) {   // solver indices, any order; adds to the symmetric entry once
    if (i < j) std::swap(i, j);
    if (i < nk) band[size_t(j) * (kd + 1) + (i - j)] += v;
    else if (j < nk) E[size_t(i - nk) * nk + j] += v;
    else { C[size_t(i - nk) * nb + (j - nk)] += v; if (i != j) C[size_t(j - nk) * nb + (i - nk)] += v; }
  }
  void operator+=(const Normal& o) {
    for (size_t i = 0; i < band.size(); ++i) band[i] += o.band[i];
    for (size_t i = 0; i < E.size(); ++i) E[i] += o.E[i];
    for (size_t i = 0; i < C.size(); ++i) C[i] += o.C[i];
    for (size_t i = 0; i < g.size(); ++i) g[i] += o.g[i];
    cost += o.cost;
  }
  double get(int i, int j) const {
    if (i < j) std::swap(i, j);
    if (i < nk) return (i - j <= kd) ? band[size_t(j) * (kd + 1) + (i - j)] : 0.0;
    if (j < nk) return E[size_t(i - nk) * nk + j];
    return C[size_t(i - nk) * nb + (j - nk)];
  }
};

// Threads the host really grants: hardware_concurrency() capped by the cgroup CPU quota (containers on shared hosts report every core
// of the machine but are throttled to their quota; more threads than that only add contention).
int host_cpu_budget() {
  static const int n = [] {
    int hw = std::max(1, int(std::thread::hardware_concurrency()));
    if (FILE* f = fopen("/sys/fs/cgroup/cpu.max", "r")) {
      char q[64] = {0}; long period = 0;
      if (fscanf(f, "%63s %ld", q, &period) == 2 && strcmp(q, "max") != 0 && period > 0) { const long quota = atol(q); if (quota > 0) hw = std::min<long>(hw, std::max<long>(1, (quota + period - 1) / period)); }
      fclose(f);
    } else if (FILE* f1 = fopen("/sys/fs/cgroup/cpu/cpu.cfs_quota_us", "r")) {   // cgroup v1
      long quota = -1, period = 100000;
      if (fscanf(f1, "%ld", &quota) != 1) quota = -1;
      fclose(f1);
      if (FILE* f2 = fopen("/sys/fs/cgroup/cpu/cpu.cfs_period_us", "r")) { if (fscanf(f2, "%ld", &period) != 1) period = 100000; fclose(f2); }
      if (quota > 0 && period > 0) hw = std::min<long>(hw, std::max<long>(1, (quota + period - 1) / period));
    }
    return hw;
  }();
  return n;
}
int thread_count(const Oracle& o) { int n = o.n_threads > 0 ? o.n_threads : host_cpu_budget(); return std::max(1, n); }

// Persistent worker pool (Ceres keeps its thread pool for the lifetime of the problem too; spawning 128 std::threads per
// evaluation and merging 128 x 4 MB partial systems serially made the CPU baseline scale 2-5x on 16x the cores).
struct Pool {
  std::vector<std::thread> th; std::mutex m; std::condition_variable cv_start, cv_done;
  const std::function<void(int)>* job = nullptr; int gen = 0, pending = 0; bool stop = false;
  explicit Pool(int n) {
    for (int t = 0; t < n; ++t) th.emplace_back([this, t] {
      int seen = 0;
      for (;;) {
        const std::function<void(int)>* j;
        { std::unique_lock<std::mutex> l(m); cv_start.wait(l, [&] { return stop || gen != seen; }); if (stop) return; seen = gen; j = job; }
        (*j)(t);
        { std::lock_guard<std::mutex> l(m); if (--pending == 0) cv_done.notify_one(); }
      }
    });
  }
  void run(const std::function<void(int)>& f) {
    std::unique_lock<std::mutex> l(m);
    job = &f; pending = int(th.size()); ++gen; cv_start.notify_all();
    cv_done.wait(l, [&] { return pending == 0; });
  }
  ~Pool() { { std::lock_guard<std::mutex> l(m); stop = true; } cv_start.notify_all(); for (auto& t : th) t.join(); }
};
struct EvalCtx {
  int T = 0, nk = -1, nb = -1, kd = -1;
  std::unique_ptr<Pool> pool;
  std::vector<Normal> parts;            // one partial system per worker, allocated once per (nk, nb, kd)
  std::vector<int> lo, hi;              // banded columns [lo, hi) a worker touched in its last evaluation (what must be cleared / merged)
  std::vector<double> costs;
};

// Full evaluation.  residuals (optional, global order), normal equations (optional), dense J (optional, tests only).
// Work split: the block list is [vision | accelerometer | gyroscope], each in time order; worker t takes the t-th slice of EACH
// segment, so its partial system only touches the banded columns of its own time slice: clearing and the cross-thread merge are
// O(total / T) per worker instead of O(total) serial.
void evaluate(Oracle& o, double* cost_out, double* residuals, Normal* ne, std::vector<double>* Jdense, int n_res_total) {
  const int T = std::min<int>(thread_count(o), std::max<size_t>(1, o.blocks.size()));
  if (!o.ctx) o.ctx = std::make_shared<EvalCtx>();
  EvalCtx& X = *o.ctx;
  if (X.T != T) { X.pool.reset(); X.pool.reset(T > 1 ? new Pool(T) : nullptr); X.T = T; X.nk = -1; X.costs.assign(T, 0.0); }
  const int nk = o.n_knot_dims, nb = o.n_border, kd = o.kd, ld = kd + 1;
  if (ne && (X.nk != nk || X.nb != nb || X.kd != kd || (int)X.parts.size() != T)) {
    X.parts.assign(T, Normal()); for (auto& p : X.parts) p.init(nk, nb, kd);
    X.lo.assign(T, 0); X.hi.assign(T, 0); X.nk = nk; X.nb = nb; X.kd = kd;
  }
  if (Jdense) Jdense->assign(size_t(n_res_total) * o.n_tan, 0.0);
  // segment boundaries of the block list
  size_t seg[4] = {0, 0, 0, o.blocks.size()};
  { size_t i = 0; while (i < o.blocks.size() && o.blocks[i].type != BLK_ACCEL && o.blocks[i].type != BLK_GYRO) ++i; seg[1] = i; while (i < o.blocks.size() && o.blocks[i].type != BLK_GYRO) ++i; seg[2] = i; }
  static const bool dbg = getenv("ICCO_DEBUG_TIMING") != nullptr;
  const auto t_dbg = std::chrono::steady_clock::now();
  std::function<void(int)> work = [&](int tid) {
    Scratch s;
    double cost = 0;
    Normal* P = ne ? &X.parts[tid] : nullptr;
    if (P) {   // clear what the last evaluation left behind
      for (size_t i = size_t(X.lo[tid]) * ld; i < size_t(X.hi[tid]) * ld; ++i) P->band[i] = 0.0;
      for (int b = 0; b < nb; ++b) for (int j = X.lo[tid]; j < X.hi[tid]; ++j) P->E[size_t(b) * nk + j] = 0.0;
      for (int j = X.lo[tid]; j < X.hi[tid]; ++j) P->g[j] = 0.0;
      std::fill(P->C.begin(), P->C.end(), 0.0); for (int b = 0; b < nb; ++b) P->g[nk + b] = 0.0;
    }
    int lo = nk, hi = 0;
    for (int sg = 0; sg < 3; ++sg) {
      const size_t n = seg[sg + 1] - seg[sg], b0 = seg[sg] + n * tid / T, b1 = seg[sg] + n * (tid + 1) / T;
      for (size_t bi = b0; bi < b1; ++bi) {
        const Block& b = o.blocks[bi];
        int ncols = 0;
        eval_block(o, b, s, ne != nullptr || Jdense != nullptr, ncols);
        double c = 0;
        for (int r = 0; r < b.n_res; ++r) c += s.res[r] * s.res[r];
        cost += 0.5 * c;
        if (residuals) for (int r = 0; r < b.n_res; ++r) residuals[b.res_off + r] = s.res[r];
        if (Jdense) for (int r = 0; r < b.n_res; ++r) for (int k = 0; k < ncols; ++k) (*Jdense)[size_t(b.res_off + r) * o.n_tan + s.cols[k]] = s.Jtan[size_t(r) * ncols + k];
        if (P && ncols > 0) {
          std::vector<int>& cols = s.cols;
          for (int k = 0; k < ncols; ++k) {
            const int sk = o.perm[cols[k]];
            if (sk < nk) { lo = std::min(lo, sk); hi = std::max(hi, sk + 1); }
            double gk = 0;
            for (int r = 0; r < b.n_res; ++r) gk += s.Jtan[size_t(r) * ncols + k] * s.res[r];
            P->g[sk] += gk;
            for (int l = k; l < ncols; ++l) {
              double h = 0;
              for (int r = 0; r < b.n_res; ++r) h += s.Jtan[size_t(r) * ncols + k] * s.Jtan[size_t(r) * ncols + l];
              if (h != 0.0) P->add(sk, o.perm[cols[l]], h);
            }
          }
        }
      }
    }
    X.costs[tid] = cost;
    if (P) { X.lo[tid] = std::min(lo, hi); X.hi[tid] = hi; }
    if (dbg) { timespec ts; clock_gettime(CLOCK_THREAD_CPUTIME_ID, &ts); fprintf(stderr, "  tid %d cpu-clock %.1f ms (thread total)", tid, 1e3 * ts.tv_sec + 1e-6 * ts.tv_nsec); }
    if (dbg) fprintf(stderr, "  tid %d segs %zu %zu %zu %zu work %.1f ms\n", tid, seg[0], seg[1], seg[2], seg[3], 1e3 * std::chrono::duration<double>(std::chrono::steady_clock::now() - t_dbg).count());
  };
  if (T == 1) work(0); else X.pool->run(work);
  double cost = 0; for (int t = 0; t < T; ++t) cost += X.costs[t];
  if (ne) {
    if (ne->nk != nk || ne->nb != nb || ne->kd != kd) ne->init(nk, nb, kd);
    std::function<void(int)> merge = [&](int tid) {   // worker tid owns banded columns [c0, c1) of the result
      const int c0 = int(int64_t(nk) * tid / T), c1 = int(int64_t(nk) * (tid + 1) / T);
      std::fill(ne->band.begin() + size_t(c0) * ld, ne->band.begin() + size_t(c1) * ld, 0.0);
      for (int b = 0; b < nb; ++b) std::fill(ne->E.begin() + size_t(b) * nk + c0, ne->E.begin() + size_t(b) * nk + c1, 0.0);
      std::fill(ne->g.begin() + c0, ne->g.begin() + c1, 0.0);
      for (int p = 0; p < T; ++p) {
        const int a = std::max(c0, X.lo[p]), z = std::min(c1, X.hi[p]);
        if (a >= z) continue;
        const Normal& Q = X.parts[p];
        for (size_t i = size_t(a) * ld; i < size_t(z) * ld; ++i) ne->band[i] += Q.band[i];
        for (int b = 0; b < nb; ++b) for (int j = a; j < z; ++j) ne->E[size_t(b) * nk + j] += Q.E[size_t(b) * nk + j];
        for (int j = a; j < z; ++j) ne->g[j] += Q.g[j];
      }
      if (tid == 0) {
        std::fill(ne->C.begin(), ne->C.end(), 0.0); for (int b = 0; b < nb; ++b) ne->g[nk + b] = 0.0;
        for (int p = 0; p < T; ++p) { const Normal& Q = X.parts[p]; for (size_t i = 0; i < Q.C.size(); ++i) ne->C[i] += Q.C[i]; for (int b = 0; b < nb; ++b) ne->g[nk + b] += Q.g[nk + b]; }
      }
    };
    if (T == 1) merge(0); else X.pool->run(merge);
    ne->cost = cost;
  }
  if (cost_out) *cost_out = cost;
}

// In-place Cholesky of (H + diag(D2)) in arrowhead storage followed by solve of (H + D2) x = rhs.  Returns false on breakdown.
bool arrowhead_solve(Normal A, const std::vector<double>& D2, const std::vector<double>& rhs, std::vector<double>& x) {
  const int nk = A.nk, nb = A.nb, kd = A.kd, n = nk + nb, ld = kd + 1;
  for (int j = 0; j < nk; ++j) A.band[size_t(j) * ld] += D2[j];
  for (int b = 0; b < nb; ++b) A.C[size_t(b) * nb + b] += D2[nk + b];
  // factor the banded part column by column, carrying the border rows along
  for (int j = 0; j < nk; ++j) {
    double* col = &A.band[size_t(j) * ld];
    if (!(col[0] > 0.0)) return false;
    const double d = std::sqrt(col[0]), inv = 1.0 / d;
    col[0] = d;
    const int m = std::min(kd, nk - 1 - j);
    for (int i = 1; i <= m; ++i) col[i] *= inv;
    for (int b = 0; b < nb; ++b) A.E[size_t(b) * nk + j] *= inv;
    for (int k = 1; k <= m; ++k) {         // trailing band update
      const double lk = col[k]; if (lk == 0.0) continue;
      double* ck = &A.band[size_t(j + k) * ld];
      for (int i = k; i <= m; ++i) ck[i - k] -= col[i] * lk;
      for (int b = 0; b < nb; ++b) A.E[size_t(b) * nk + j + k] -= A.E[size_t(b) * nk + j] * lk;
    }
    for (int b = 0; b < nb; ++b) { const double eb = A.E[size_t(b) * nk + j]; if (eb == 0.0) continue; for (int c = 0; c <= b; ++c) A.C[size_t(b) * nb + c] -= eb * A.E[size_t(c) * nk + j]; }
  }
  // dense Cholesky of the Schur complement (lower triangle of C)
  for (int j = 0; j < nb; ++j) {
    double d = A.C[size_t(j) * nb + j];
    for (int k = 0; k < j; ++k) d -= A.C[size_t(j) * nb + k] * A.C[size_t(j) * nb + k];
    if (!(d > 0.0)) return false;
    d = std::sqrt(d); A.C[size_t(j) * nb + j] = d;
    for (int i = j + 1; i < nb; ++i) {
      double v = A.C[size_t(i) * nb + j];
      for (int k = 0; k < j; ++k) v -= A.C[size_t(i) * nb + k] * A.C[size_t(j) * nb + k];
      A.C[size_t(i) * nb + j] = v / d;
    }
  }
  // forward substitution  L y = rhs
  x = rhs;
  for (int j = 0; j < nk; ++j) {
    const double* col = &A.band[size_t(j) * ld];
    x[j] /= col[0];
    const int m = std::min(kd, nk - 1 - j);
    for (int i = 1; i <= m; ++i) x[j + i] -= col[i] * x[j];
    for (int b = 0; b < nb; ++b) x[nk + b] -= A.E[size_t(b) * nk + j] * x[j];
  }
  for (int j = 0; j < nb; ++j) { double v = x[nk + j]; for (int k = 0; k < j; ++k) v -= A.C[size_t(j) * nb + k] * x[nk + k]; x[nk + j] = v / A.C[size_t(j) * nb + j]; }
  // back substitution  L^T x = y
  for (int j = nb - 1; j >= 0; --j) { double v = x[nk + j]; for (int k = j + 1; k < nb; ++k) v -= A.C[size_t(k) * nb + j] * x[nk + k]; x[nk + j] = v / A.C[size_t(j) * nb + j]; }
  for (int j = nk - 1; j >= 0; --j) {
    const double* col = &A.band[size_t(j) * ld];
    double v = x[j];
    const int m = std::min(kd, nk - 1 - j);
    for (int i = 1; i <= m; ++i) v -= col[i] * x[j + i];
    for (int b = 0; b < nb; ++b) v -= A.E[size_t(b) * nk + j] * x[nk + b];
    x[j] = v / col[0];
  }
  (void)n;
  return true;
}

// -------------------------------------------------------------------------------------------------------------
// State vector plumbing: Plus(), norms, snapshots.
// -------------------------------------------------------------------------------------------------------------
struct State { std::vector<double> so3, r3, ba, bg, points; double T_ic[7], grav[3], ld, acc_intr[6], gyr_intr[9], intr[10], toff; };
void save_state(const Oracle& o, State& s) { s.points = o.points; s.so3 = o.so3; s.r3 = o.r3; s.ba = o.ba; s.bg = o.bg; memcpy(s.T_ic, o.T_ic, sizeof s.T_ic); memcpy(s.grav, o.grav, sizeof s.grav); s.ld = o.line_delay; memcpy(s.acc_intr, o.acc_intr, sizeof s.acc_intr); memcpy(s.gyr_intr, o.gyr_intr, sizeof s.gyr_intr); memcpy(s.intr, o.intr, sizeof s.intr); s.toff = o.toff_delta; }
void load_state(Oracle& o, const State& s) {
  // copy element-wise: residual blocks hold raw pointers into these vectors
  std::copy(s.points.begin(), s.points.end(), o.points.begin());
  std::copy(s.so3.begin(), s.so3.end(), o.so3.begin()); std::copy(s.r3.begin(), s.r3.end(), o.r3.begin());
  std::copy(s.ba.begin(), s.ba.end(), o.ba.begin()); std::copy(s.bg.begin(), s.bg.end(), o.bg.begin());
  memcpy(o.T_ic, s.T_ic, sizeof s.T_ic); memcpy(o.grav, s.grav, sizeof s.grav); o.line_delay = s.ld; memcpy(o.acc_intr, s.acc_intr, sizeof s.acc_intr); memcpy(o.gyr_intr, s.gyr_intr, sizeof s.gyr_intr);
  memcpy(o.intr, s.intr, sizeof s.intr); o.toff_delta = s.toff;
}

// x <- Plus(x, delta) with delta in CANONICAL tangent order.  Returns squared ambient step norm and squared ambient x norm (before).
void apply_plus(Oracle& o, const std::vector<double>& d, double& step_sq, double& x_sq) {
  step_sq = 0; x_sq = 0;
  auto acc = [&](double oldv, double newv) { step_sq += (newv - oldv) * (newv - oldv); x_sq += oldv * oldv; };
  const int flags = o.cur_flags;
  if (o.off_so3 >= 0) {
    const int n = nknots(o.so3, 4);
    for (int i = 0; i < n; ++i) {
      double* q = &o.so3[4 * i];
      V3<double> w{d[o.off_so3 + 3 * i], d[o.off_so3 + 3 * i + 1], d[o.off_so3 + 3 * i + 2]};
      Q4<double> r = so3_mul(Q4<double>{q[0], q[1], q[2], q[3]}, so3_exp(w));   // LieLocalParameterization::Plus (ceres_local_param.h:84-92)
      acc(q[0], r.x); acc(q[1], r.y); acc(q[2], r.z); acc(q[3], r.w);
      q[0] = r.x; q[1] = r.y; q[2] = r.z; q[3] = r.w;
    }
    const int m = nknots(o.r3, 3);
    for (int i = 0; i < 3 * m; ++i) { const double nv = o.r3[i] + d[o.off_r3 + i]; acc(o.r3[i], nv); o.r3[i] = nv; }
  }
  if (o.off_tic >= 0) {
    SE3T<double> T{{o.T_ic[0], o.T_ic[1], o.T_ic[2], o.T_ic[3]}, {o.T_ic[4], o.T_ic[5], o.T_ic[6]}};
    SE3T<double> r = se3_mul(T, se3_exp(&d[o.off_tic]));
    const double nv[7] = {r.q.x, r.q.y, r.q.z, r.q.w, r.t.x, r.t.y, r.t.z};
    for (int i = 0; i < 7; ++i) { acc(o.T_ic[i], nv[i]); o.T_ic[i] = nv[i]; }
  }
  if (o.off_g >= 0) for (int i = 0; i < 3; ++i) { const double nv = o.grav[i] + d[o.off_g + i]; acc(o.grav[i], nv); o.grav[i] = nv; }
  if (o.off_ld >= 0) { const double nv = o.line_delay + d[o.off_ld]; acc(o.line_delay, nv); o.line_delay = nv; }
  auto clampv = [](double v, double r) { return std::min(std::max(v, -r), r); };
  if (o.off_ba >= 0) for (size_t i = 0; i < o.ba.size(); ++i) { const double nv = clampv(o.ba[i] + d[o.off_ba + i], o.max_ba); acc(o.ba[i], nv); o.ba[i] = nv; }
  if (o.off_bg >= 0) for (size_t i = 0; i < o.bg.size(); ++i) { const double nv = clampv(o.bg[i] + d[o.off_bg + i], o.max_bg); acc(o.bg[i], nv); o.bg[i] = nv; }
  if (o.off_ci >= 0) for (int i = 0; i < o.n_intr; ++i) { const double nv = o.intr[i] + d[o.off_ci + i]; acc(o.intr[i], nv); o.intr[i] = nv; }
  if (o.off_to >= 0) { const double nv = o.toff_delta + d[o.off_to]; acc(o.toff_delta, nv); o.toff_delta = nv; }
  if (o.off_pts >= 0) for (size_t i = 0; i < o.points.size() / 4; ++i) {
    double nx[4] = {o.points[4 * i], o.points[4 * i + 1], o.points[4 * i + 2], o.points[4 * i + 3]};
    plus_homog4(nx, &d[o.off_pts + 3 * i]);
    for (int k = 0; k < 4; ++k) { acc(o.points[4 * i + k], nx[k]); o.points[4 * i + k] = nx[k]; }
  }
  if (flags & ICC_FLAG_IMU_INTRINSICS) {
    int off = o.off_ai;
    for (int i = 0; i < 6; ++i) { const double nv = o.acc_intr[i] + d[off + i]; acc(o.acc_intr[i], nv); o.acc_intr[i] = nv; }
    for (int i = 0; i < 9; ++i) { const double nv = o.gyr_intr[i] + d[off + 6 + i]; acc(o.gyr_intr[i], nv); o.gyr_intr[i] = nv; }
  }
}

int total_residuals(const Oracle& o) { return o.n_res_vis + o.n_res_acc + o.n_res_gyr; }

// impl.h:993-1072
double mean_reproj_error(Oracle& o) {
  double sum = 0; int num = 0;
  Scratch s;
  for (const auto& b : o.vis_blocks) {
    int nc; eval_block(o, b, s, false, nc);
    for (int i = 0; i < b.n_res / 2; ++i) {
      const double rx = s.res[2 * i], ry = s.res[2 * i + 1];
      if (rx != 0.0 && ry != 0.0) { sum += std::sqrt(rx * rx + ry * ry); ++num; }
    }
  }
  return sum / num;
}

// -------------------------------------------------------------------------------------------------------------
// Ceres inner iterations (Ruhe & Wedin "Algorithm II" as implemented by ceres::internal::CoordinateDescentMinimizer; Ceres is
// not in /root/reference -- restated from the Ceres 2.1 sources as published):
//   * ordering (inner_iteration_ordering unset): recursive independent sets of the Hessian graph of the parameter blocks
//     (vertices by increasing degree, greedy), reversed -- CoordinateDescentMinimizer::CreateOrdering;
//   * for every set in order, every parameter block of the set is minimised ALONE over the residual blocks that depend on it,
//     all other blocks constant, by a trust-region minimiser with Minimizer::Options defaults (<= 50 iterations, function
//     tolerance 1e-6, gradient 1e-10, parameter 1e-8, initial radius 1e4, Jacobi scaling, exact dense LM steps);
//   * TrustRegionMinimizer::DoInnerIterationsIfNeeded: the refined point replaces the candidate, the cost it gained is added to
//     the model cost change, the step is accepted when the refinement got below the cost of x even if the ratio is small, and
//     inner iterations are switched off for good once their relative progress 1 - cost_inner / cost_candidate <= 1e-3.
// Ceres' own tie-breaking inside the ordering follows the iteration order of an unordered_set of block pointers, i.e. it is not
// reproducible between runs of the reference itself; ties are broken here by block index.
// -------------------------------------------------------------------------------------------------------------
struct InnerBlock { double* ptr; int size, lp, tan_off, tdim; std::vector<int> res_blocks; };
struct InnerPlan { int flags = -1; std::vector<InnerBlock> blocks; std::vector<std::vector<int>> groups; };

void build_inner_plan(Oracle& o) {
  if (!o.inner_plan) o.inner_plan = std::make_shared<InnerPlan>();
  InnerPlan& P = *o.inner_plan;
  if (P.flags == o.cur_flags && !P.blocks.empty()) return;
  P.flags = o.cur_flags; P.blocks.clear(); P.groups.clear();
  std::map<int, int> by_off;
  for (size_t bi = 0; bi < o.blocks.size(); ++bi)
    for (const auto& p : o.blocks[bi].params) {
      if (p.tan_off < 0) continue;
      auto it = by_off.find(p.tan_off);
      if (it == by_off.end()) {
        it = by_off.emplace(p.tan_off, int(P.blocks.size())).first;
        P.blocks.push_back({const_cast<double*>(p.ptr), p.size, p.lp, p.tan_off, p.lp == LP_SO3 ? 3 : p.lp == LP_SE3 ? 6 : p.lp == LP_HOMOG4 ? 3 : p.size, {}});
      }
      P.blocks[it->second].res_blocks.push_back(int(bi));
    }
  const int nb = int(P.blocks.size());
  std::vector<std::vector<int>> adj(nb);
  for (const auto& b : o.blocks) {
    std::vector<int> ids;
    for (const auto& p : b.params) if (p.tan_off >= 0) ids.push_back(by_off[p.tan_off]);
    for (int a : ids) for (int c : ids) if (a != c) adj[a].push_back(c);
  }
  for (auto& v : adj) { std::sort(v.begin(), v.end()); v.erase(std::unique(v.begin(), v.end()), v.end()); }
  // ComputeRecursiveIndependentSetOrdering: peel greedy maximal independent sets (vertices by increasing CURRENT degree)
  std::vector<char> removed(nb, 0);
  int left = nb;
  while (left > 0) {
    std::vector<int> order;
    for (int v = 0; v < nb; ++v) if (!removed[v]) order.push_back(v);
    std::vector<int> deg(nb, 0);
    for (int v : order) for (int w : adj[v]) if (!removed[w]) ++deg[v];
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return deg[a] < deg[b]; });
    std::vector<char> colour(nb, 0);   // 0 white, 1 grey, 2 black
    std::vector<int> set;
    for (int v : order) { if (colour[v]) continue; colour[v] = 2; set.push_back(v); for (int w : adj[v]) if (!removed[w] && !colour[w]) colour[w] = 1; }
    for (int v : set) removed[v] = 1;
    left -= int(set.size());
    P.groups.push_back(std::move(set));
  }
  std::reverse(P.groups.begin(), P.groups.end());   // ordering->Reverse()
}

void plus_block(const Oracle& o, const InnerBlock& B, const double* d) {
  if (B.lp == LP_SO3) {
    Q4<double> r = so3_mul(Q4<double>{B.ptr[0], B.ptr[1], B.ptr[2], B.ptr[3]}, so3_exp(V3<double>{d[0], d[1], d[2]}));
    B.ptr[0] = r.x; B.ptr[1] = r.y; B.ptr[2] = r.z; B.ptr[3] = r.w;
  } else if (B.lp == LP_HOMOG4) {
    plus_homog4(B.ptr, d);
  } else if (B.lp == LP_SE3) {
    SE3T<double> T{{B.ptr[0], B.ptr[1], B.ptr[2], B.ptr[3]}, {B.ptr[4], B.ptr[5], B.ptr[6]}};
    SE3T<double> r = se3_mul(T, se3_exp(d));
    const double nv[7] = {r.q.x, r.q.y, r.q.z, r.q.w, r.t.x, r.t.y, r.t.z};
    for (int i = 0; i < 7; ++i) B.ptr[i] = nv[i];
  } else {
    const bool is_ba = !o.ba.empty() && B.ptr >= o.ba.data() && B.ptr < o.ba.data() + o.ba.size();
    const bool is_bg = !o.bg.empty() && B.ptr >= o.bg.data() && B.ptr < o.bg.data() + o.bg.size();
    for (int i = 0; i < B.size; ++i) {
      double nv = B.ptr[i] + d[i];
      if (is_ba) nv = std::min(std::max(nv, -o.max_ba), o.max_ba);
      if (is_bg) nv = std::min(std::max(nv, -o.max_bg), o.max_bg);
      B.ptr[i] = nv;
    }
  }
}

// cost (and, if wanted, the dense d x d normal equations) of the residual blocks that depend on block B, everything else constant
double inner_eval(const Oracle& o, const InnerBlock& B, std::vector<Block>& local, Scratch& s, double* H, double* g) {
  const int d = B.tdim;
  if (H) { std::fill(H, H + d * d, 0.0); std::fill(g, g + d, 0.0); }
  double cost = 0;
  for (size_t k = 0; k < local.size(); ++k) {
    const Block& b = local[k];
    int ncols = 0;
    eval_block(o, b, s, H != nullptr, ncols);
    for (int r = 0; r < b.n_res; ++r) cost += 0.5 * s.res[r] * s.res[r];
    if (H) for (int r = 0; r < b.n_res; ++r) for (int i = 0; i < ncols; ++i) {
      const int ci = s.cols[i] - B.tan_off; const double ji = s.Jtan[size_t(r) * ncols + i];
      g[ci] += ji * s.res[r];
      for (int j = 0; j < ncols; ++j) H[ci * d + (s.cols[j] - B.tan_off)] += ji * s.Jtan[size_t(r) * ncols + j];
    }
  }
  return cost;
}

// TrustRegionMinimizer with Minimizer::Options defaults on ONE parameter block (CoordinateDescentMinimizer::Solve)
void inner_solve(const Oracle& o, const InnerBlock& B, Scratch& s) {
  const int d = B.tdim;
  std::vector<Block> local; local.reserve(B.res_blocks.size());
  for (int bi : B.res_blocks) { local.push_back(o.blocks[bi]); for (auto& p : local.back().params) if (p.tan_off != B.tan_off) p.tan_off = -1; }
  std::vector<double> H(d * d), g(d), A(d * d), y(d), scale(d, 1.0), saved(B.size), diag(d);
  double radius = 1e4, decrease_factor = 2.0;
  double x_cost = inner_eval(o, B, local, s, H.data(), g.data());
  for (int i = 0; i < d; ++i) scale[i] = 1.0 / (1.0 + std::sqrt(H[i * d + i]));
  bool reuse_diag = false; int invalid = 0;
  for (int it = 0; it < 50; ++it) {
    double gmax = 0; for (int i = 0; i < d; ++i) gmax = std::max(gmax, std::fabs(g[i]));
    if (gmax <= 1e-10) break;
    if (!reuse_diag) for (int i = 0; i < d; ++i) diag[i] = std::min(std::max(H[i * d + i] * scale[i] * scale[i], 1e-6), 1e32);
    for (int i = 0; i < d; ++i) for (int j = 0; j < d; ++j) A[i * d + j] = H[i * d + j] * scale[i] * scale[j] + (i == j ? diag[i] / radius : 0.0);
    // Cholesky solve of A y = -S g
    bool ok = true;
    for (int j = 0; j < d && ok; ++j) {
      double v = A[j * d + j]; for (int k = 0; k < j; ++k) v -= A[j * d + k] * A[j * d + k];
      if (!(v > 0.0)) { ok = false; break; }
      A[j * d + j] = std::sqrt(v);
      for (int i = j + 1; i < d; ++i) { double w = A[i * d + j]; for (int k = 0; k < j; ++k) w -= A[i * d + k] * A[j * d + k]; A[i * d + j] = w / A[j * d + j]; }
    }
    double model = 0;
    if (ok) {
      for (int i = 0; i < d; ++i) { double v = -scale[i] * g[i]; for (int k = 0; k < i; ++k) v -= A[i * d + k] * y[k]; y[i] = v / A[i * d + i]; }
      for (int i = d - 1; i >= 0; --i) { double v = y[i]; for (int k = i + 1; k < d; ++k) v -= A[k * d + i] * y[k]; y[i] = v / A[i * d + i]; }
      double yg = 0, yHy = 0;
      for (int i = 0; i < d; ++i) { yg += y[i] * scale[i] * g[i]; for (int j = 0; j < d; ++j) yHy += y[i] * y[j] * H[i * d + j] * scale[i] * scale[j]; }
      model = -yg - 0.5 * yHy;
    }
    if (!ok || !(model > 0.0)) { if (++invalid >= 5) break; radius /= decrease_factor; decrease_factor *= 2.0; reuse_diag = true; continue; }
    invalid = 0;
    double delta[10], step_sq = 0, x_sq = 0;
    for (int i = 0; i < d; ++i) delta[i] = y[i] * scale[i];
    for (int i = 0; i < B.size; ++i) saved[i] = B.ptr[i];
    plus_block(o, B, delta);
    for (int i = 0; i < B.size; ++i) { step_sq += (B.ptr[i] - saved[i]) * (B.ptr[i] - saved[i]); x_sq += saved[i] * saved[i]; }
    const double cand = inner_eval(o, B, local, s, nullptr, nullptr);
    if (std::sqrt(step_sq) <= 1e-8 * (std::sqrt(x_sq) + 1e-8)) { for (int i = 0; i < B.size; ++i) B.ptr[i] = saved[i]; break; }
    const double change = x_cost - cand;
    if (std::fabs(change) <= 1e-6 * x_cost) { for (int i = 0; i < B.size; ++i) B.ptr[i] = saved[i]; break; }
    const double rho = change / model;
    if (rho > 1e-3) {
      x_cost = inner_eval(o, B, local, s, H.data(), g.data());
      radius = std::min(1e16, radius / std::max(1.0 / 3.0, 1.0 - std::pow(2.0 * rho - 1.0, 3))); decrease_factor = 2.0; reuse_diag = false;
    } else {
      for (int i = 0; i < B.size; ++i) B.ptr[i] = saved[i];
      radius /= decrease_factor; decrease_factor *= 2.0; reuse_diag = true;
      if (radius < 1e-32) break;
    }
  }
}

// CoordinateDescentMinimizer::Minimize: the blocks of an independent set share no residual block, so they run in parallel
void inner_iterations(Oracle& o) {
  build_inner_plan(o);
  const InnerPlan& P = *o.inner_plan;
  const int T = thread_count(o);
  if (!o.ctx) o.ctx = std::make_shared<EvalCtx>();
  for (const auto& grp : P.groups) {
    if (grp.empty()) continue;
    if (T == 1 || grp.size() == 1 || !o.ctx->pool || o.ctx->T != T) { Scratch s; for (int b : grp) inner_solve(o, P.blocks[b], s); continue; }
    std::function<void(int)> job = [&](int tid) { Scratch s; for (size_t k = tid; k < grp.size(); k += T) inner_solve(o, P.blocks[grp[k]], s); };
    o.ctx->pool->run(job);
  }
}

// -------------------------------------------------------------------------------------------------------------
// Levenberg-Marquardt, Ceres TrustRegionMinimizer semantics.
// -------------------------------------------------------------------------------------------------------------
struct LMResult { icc_summary sum; };

// Jacobi column scaling (solver order): S_ii = 1 / (1 + sqrt(H_ii)), or the identity without it.
std::vector<double> jacobi_scale(const Normal& ne, bool jacobi) {
  const int n = ne.nk + ne.nb;
  std::vector<double> scale(n, 1.0);
  if (jacobi) for (int i = 0; i < n; ++i) scale[i] = 1.0 / (1.0 + std::sqrt(i < ne.nk ? ne.band[size_t(i) * (ne.kd + 1)] : ne.C[size_t(i - ne.nk) * ne.nb + (i - ne.nk)]));
  return scale;
}

// One LevenbergMarquardtStrategy::ComputeStep (solver order): scaled system Hs = S H S, gs = S g; the clamped diagonal
// diag = clamp(diag(Hs), min_lm_diagonal, max_lm_diagonal) (kept from the previous call when reuse_diagonal); D2 = diag / radius;
// (Hs + D2) y = -gs; model_change = -y^T gs - 1/2 y^T Hs y.  Returns false on a Cholesky breakdown.
struct LmStep { Normal sc; std::vector<double> diag, D2, rhs, y; double model_change = 0; };
bool lm_step(const Normal& ne, const std::vector<double>& scale, double radius, const icc_solver_options& opt, bool reuse_diagonal, LmStep& st) {
  const int n = ne.nk + ne.nb;
  Normal& sc = st.sc;
  sc = ne;
  for (int j = 0; j < ne.nk; ++j) { const int m = std::min(ne.kd, ne.nk - 1 - j); for (int i = 0; i <= m; ++i) sc.band[size_t(j) * (ne.kd + 1) + i] *= scale[j] * scale[j + i]; }
  for (int b = 0; b < ne.nb; ++b) for (int j = 0; j < ne.nk; ++j) sc.E[size_t(b) * ne.nk + j] *= scale[ne.nk + b] * scale[j];
  for (int b = 0; b < ne.nb; ++b) for (int c = 0; c < ne.nb; ++c) sc.C[size_t(b) * ne.nb + c] *= scale[ne.nk + b] * scale[ne.nk + c];
  st.rhs.resize(n); st.D2.resize(n); st.diag.resize(n, 0.0);
  for (int i = 0; i < n; ++i) st.rhs[i] = -scale[i] * ne.g[i];
  if (!reuse_diagonal) for (int i = 0; i < n; ++i) { const double dv = i < sc.nk ? sc.band[size_t(i) * (sc.kd + 1)] : sc.C[size_t(i - sc.nk) * sc.nb + (i - sc.nk)]; st.diag[i] = std::min(std::max(dv, opt.min_lm_diagonal), opt.max_lm_diagonal); }
  for (int i = 0; i < n; ++i) st.D2[i] = st.diag[i] / radius;
  st.model_change = 0;
  if (!arrowhead_solve(sc, st.D2, st.rhs, st.y)) return false;
  double yg = 0, yHy = 0;
  for (int i = 0; i < n; ++i) yg += st.y[i] * (-st.rhs[i]);
  for (int j = 0; j < sc.nk; ++j) { const int m = std::min(sc.kd, sc.nk - 1 - j); yHy += sc.band[size_t(j) * (sc.kd + 1)] * st.y[j] * st.y[j]; for (int i = 1; i <= m; ++i) yHy += 2.0 * sc.band[size_t(j) * (sc.kd + 1) + i] * st.y[j] * st.y[j + i]; }
  for (int b = 0; b < sc.nb; ++b) { for (int j = 0; j < sc.nk; ++j) yHy += 2.0 * sc.E[size_t(b) * sc.nk + j] * st.y[sc.nk + b] * st.y[j]; for (int c = 0; c < sc.nb; ++c) yHy += sc.C[size_t(b) * sc.nb + c] * st.y[sc.nk + b] * st.y[sc.nk + c]; }
  st.model_change = -yg - 0.5 * yHy;
  return true;
}

void lm_solve(Oracle& o, int max_iters, int flags, bool check_convergence, icc_summary& S) {
  using clk = std::chrono::steady_clock;
  const auto t_start = clk::now();
  memset(&S, 0, sizeof S);
  const int n = o.n_tan, nres = total_residuals(o);
  S.num_residuals = nres; S.num_tangent = n;
  double t_jac = 0, t_lin = 0;
  Normal ne;
  double x_cost = 0;
  auto eval_jac = [&]() { auto t0 = clk::now(); evaluate(o, &x_cost, nullptr, &ne, nullptr, nres); t_jac += std::chrono::duration<double>(clk::now() - t0).count(); ++S.jacobian_evaluations; };
  std::vector<double> scale;   // solver order
  double radius = o.opt.initial_trust_region_radius, decrease_factor = 2.0;
  bool reuse_diagonal = false, ne_valid = false, first = true;
  std::vector<double> delta_canon(n);
  int invalid = 0;
  bool inner_enabled = o.inner_iterations;
  o.inner_iteration_steps = 0;
  S.termination = 0;
  auto grad_max = [&]() { double m = 0; for (double v : ne.g) m = std::max(m, std::fabs(v)); return m; };
  LmStep st;
  for (int it = 0; it < max_iters; ++it) {
    // Jacobian rebuilt lazily at the top of the iteration that needs it (same schedule as the CUDA driver)
    if (!ne_valid) {
      eval_jac(); ne_valid = true;
      if (first) {
        first = false; S.initial_cost = x_cost;
        scale = jacobi_scale(ne, o.opt.jacobi_scaling);
      }
      if (check_convergence && grad_max() <= o.opt.gradient_tolerance) { S.termination = 3; break; }
    }
    ++S.iterations;
    auto t0 = clk::now();
    const bool ok = lm_step(ne, scale, radius, o.opt, reuse_diagonal, st);
    t_lin += std::chrono::duration<double>(clk::now() - t0).count();
    double model_change = st.model_change;
    if (!ok || !(model_change > 0.0)) {
      if (++invalid >= o.opt.max_consecutive_invalid_steps) { S.termination = 4; break; }
      radius = radius / decrease_factor; decrease_factor *= 2.0; reuse_diagonal = true;
      if (radius < o.opt.min_trust_region_radius) { S.termination = 4; break; }   // MinTrustRegionRadiusReached is tested after every iteration
      continue;
    }
    invalid = 0;
    for (int c = 0; c < n; ++c) delta_canon[c] = st.y[o.perm[c]] * scale[o.perm[c]];
    State snap; save_state(o, snap);
    double step_sq, x_sq; apply_plus(o, delta_canon, step_sq, x_sq);
    double cand_cost; evaluate(o, &cand_cost, nullptr, nullptr, nullptr, nres); ++S.cost_evaluations;
    bool inner_useful = false;
    if (inner_enabled && cand_cost < 1.7976931348623157e308) {       // TrustRegionMinimizer::DoInnerIterationsIfNeeded
      ++o.inner_iteration_steps;
      inner_iterations(o);
      double inner_cost; evaluate(o, &inner_cost, nullptr, nullptr, nullptr, nres);
      model_change += cand_cost - inner_cost;
      inner_useful = inner_cost < x_cost;
      inner_enabled = (1.0 - inner_cost / cand_cost) > o.inner_iteration_tolerance;
      cand_cost = inner_cost;
    }
    const double step_norm = std::sqrt(step_sq), x_norm = std::sqrt(x_sq);
    if (check_convergence && step_norm <= o.opt.parameter_tolerance * (x_norm + o.opt.parameter_tolerance)) { load_state(o, snap); S.termination = 2; break; }
    const double cost_change = x_cost - cand_cost;
    if (check_convergence && std::fabs(cost_change) <= o.opt.function_tolerance * x_cost) { load_state(o, snap); S.termination = 1; break; }
    const double rel_dec = cost_change / model_change;
    if (inner_useful || rel_dec > o.opt.min_relative_decrease) {      // TrustRegionMinimizer::IsStepSuccessful
      ++S.successful_steps;
      x_cost = cand_cost; ne_valid = false;
      radius = radius / std::max(1.0 / 3.0, 1.0 - std::pow(2.0 * rel_dec - 1.0, 3)); radius = std::min(o.opt.max_trust_region_radius, radius);
      decrease_factor = 2.0; reuse_diagonal = false;
    } else {
      load_state(o, snap);
      radius = radius / decrease_factor; decrease_factor *= 2.0; reuse_diagonal = true;
      if (radius < o.opt.min_trust_region_radius) { S.termination = 4; break; }
    }
  }
  if (first) { eval_jac(); S.initial_cost = x_cost; }
  S.final_cost = x_cost;
  S.seconds_jacobian = t_jac; S.seconds_linear_solve = t_lin;
  S.seconds_total = std::chrono::duration<double>(clk::now() - t_start).count();
}

Oracle* O(void* h) { return reinterpret_cast<Oracle*>(h); }
const Oracle* O(const void* h) { return reinterpret_cast<const Oracle*>(h); }

}  // namespace

// =================================================================================================================
// C-ABI (icco_*), mirrors include/icc_b200.h
// =================================================================================================================
extern "C" {

icc_status icco_create(void** out, int n_threads) {
  Oracle* o = new Oracle();
  o->n_threads = n_threads;
  o->opt.function_tolerance = 1e-4; o->opt.parameter_tolerance = 1e-7; o->opt.gradient_tolerance = 1e-10;
  o->opt.initial_trust_region_radius = 1e4; o->opt.max_trust_region_radius = 1e16; o->opt.min_trust_region_radius = 1e-32;
  o->opt.min_relative_decrease = 1e-3; o->opt.min_lm_diagonal = 1e-6; o->opt.max_lm_diagonal = 1e32; o->opt.jacobi_scaling = 1;
  o->opt.max_consecutive_invalid_steps = 5;
  *out = o; return ICC_OK;
}
void icco_destroy(void* h) { delete O(h); }
const char* icco_last_error(const void* h) { return O(h)->err.c_str(); }
icc_status icco_set_solver_options(void* h, const icc_solver_options* p) { O(h)->opt = *p; return ICC_OK; }
// Ceres' use_inner_iterations (impl.h:266) for the stopping-point study; `steps` (optional) = outer iterations that ran them last time
icc_status icco_set_inner_iterations(void* h, int enable) { O(h)->inner_iterations = enable != 0; return ICC_OK; }
int icco_inner_iteration_steps(const void* h) { return O(h)->inner_iteration_steps; }
int icco_num_threads(const void* h) { return thread_count(*O(h)); }

icc_status icco_set_camera(void* h, int model, const double* intr, int n, int w, int hgt) {
  Oracle& o = *O(h);
  if (camera_num_params(model) < 0 || n != camera_num_params(model)) { o.err = "bad camera model / intrinsic count"; return ICC_ERR_INVALID_ARGUMENT; }
  o.model = model; o.n_intr = n; o.width = w; o.height = hgt; for (int i = 0; i < n; ++i) o.intr[i] = intr[i];
  return ICC_OK;
}
icc_status icco_set_board_points(void* h, int n, const double* xyzw) { O(h)->points.assign(xyzw, xyzw + 4 * size_t(n)); return ICC_OK; }
icc_status icco_set_frames(void* h, int nf, const double* t, const int32_t* off, const int32_t* ids, const double* uv, const double* q, const double* p) {
  Oracle& o = *O(h);
  o.frame_t.assign(t, t + nf); o.corner_off.assign(off, off + nf + 1);
  const int nc = off[nf];
  o.point_ids.assign(ids, ids + nc); o.uv.assign(uv, uv + 2 * size_t(nc)); o.q_wc.assign(q, q + 4 * size_t(nf)); o.p_wc.assign(p, p + 3 * size_t(nf));
  return ICC_OK;
}
icc_status icco_set_imu(void* h, int n, const double* t, const double* a, const double* g) {
  Oracle& o = *O(h); o.imu_t.assign(t, t + n); o.imu_acc.assign(a, a + 3 * size_t(n)); o.imu_gyr.assign(g, g + 3 * size_t(n)); return ICC_OK;
}
icc_status icco_set_shard(void* h, int rank, int world) { Oracle& o = *O(h); if (world < 1 || rank < 0 || rank >= world) { o.err = "bad shard"; return ICC_ERR_INVALID_ARGUMENT; } o.shard_rank = rank; o.shard_world = world; return ICC_OK; }

icc_status icco_batch_init_spline(void* h, const icc_init_params* ipp) {
  Oracle& o = *O(h);
  if (o.model < 0 || o.frame_t.empty() || o.points.empty()) { o.err = "camera, board points and frames must be set first"; return ICC_ERR_STATE; }
  o.ip = *ipp; o.dispatch_fov = ipp->dispatch_fov != 0;
  const int nf = int(o.frame_t.size());
  memcpy(o.T_ic, ipp->T_i_c_init, sizeof o.T_ic);
  { Q4<double> q = qnormalized(Q4<double>{o.T_ic[0], o.T_ic[1], o.T_ic[2], o.T_ic[3]}); o.T_ic[0] = q.x; o.T_ic[1] = q.y; o.T_ic[2] = q.z; o.T_ic[3] = q.w; }
  memcpy(o.acc_intr, ipp->acc_intrinsics, sizeof o.acc_intr); memcpy(o.gyr_intr, ipp->gyr_intrinsics, sizeof o.gyr_intr);
  o.line_delay = ipp->init_line_delay_s; o.toff_delta = 0.0;
  // imu_camera_calibrator.cc:37-63
  std::vector<double> cam_ts(o.frame_t); std::sort(cam_ts.begin(), cam_ts.end());
  o.t0_s = cam_ts.front(); o.tend_s = cam_ts.back();
  o.start_ns = int64_t(o.t0_s * S_TO_NS);
  o.end_ns = int64_t(o.tend_s * S_TO_NS + 0.01 * S_TO_NS + ipp->init_line_delay_s);
  o.dt_so3_ns = int64_t(ipp->dt_so3_s * S_TO_NS); o.dt_r3_ns = int64_t(ipp->dt_r3_s * S_TO_NS);
  if (o.dt_so3_ns <= 0 || o.dt_r3_ns <= 0) { o.err = "knot spacing must be positive"; return ICC_ERR_INVALID_ARGUMENT; }
  const int64_t duration = o.end_ns - o.start_ns;
  const int nso3 = int(duration / o.dt_so3_ns) + SPLINE_N, nr3 = int(duration / o.dt_r3_ns) + SPLINE_N;   // impl.h:46-48
  o.inv_so3_dt = S_TO_NS / double(o.dt_so3_ns); o.inv_r3_dt = S_TO_NS / double(o.dt_r3_ns);
  // BatchInitSO3R3VisPoses (impl.h:278-339): time-sorted map of T_w_i = T_w_c * T_i_c^-1
  std::map<double, int> by_time; for (int i = 0; i < nf; ++i) by_time[o.frame_t[i]] = i;
  std::vector<double> t_vis; std::vector<double> q_vis, p_vis;
  SE3T<double> Tic{{o.T_ic[0], o.T_ic[1], o.T_ic[2], o.T_ic[3]}, {o.T_ic[4], o.T_ic[5], o.T_ic[6]}};
  SE3T<double> Tci = se3_inv(Tic);
  for (auto& kv : by_time) {
    const int i = kv.second;
    SE3T<double> Twc{qnormalized(Q4<double>{o.q_wc[4 * i], o.q_wc[4 * i + 1], o.q_wc[4 * i + 2], o.q_wc[4 * i + 3]}), {o.p_wc[3 * i], o.p_wc[3 * i + 1], o.p_wc[3 * i + 2]}};
    SE3T<double> Twi = se3_mul(Twc, Tci);
    t_vis.push_back(kv.first);
    q_vis.insert(q_vis.end(), {Twi.q.x, Twi.q.y, Twi.q.z, Twi.q.w}); p_vis.insert(p_vis.end(), {Twi.t.x, Twi.t.y, Twi.t.z});
  }
  const int nv = int(t_vis.size());
  o.so3.assign(4 * size_t(nso3), 0.0); o.r3.assign(3 * size_t(nr3), 0.0);
  for (int i = 0; i < nso3; ++i) {       // utils.cc:221-241 (knot times are zero-based: quirk q7)
    const double t = double(i) * double(o.dt_so3_ns) * NS_TO_S;
    double dist = 0; const size_t k = find_closest(t, t_vis, dist);
    double q[4];
    if (k < size_t(nv) - 1) { const double frac = dist / (t_vis[k + 1] - t_vis[k]); slerp(&q_vis[4 * k], &q_vis[4 * (k + 1)], frac, q); }
    else memcpy(q, &q_vis[4 * k], sizeof q);
    Q4<double> qn = qnormalized(Q4<double>{q[0], q[1], q[2], q[3]});
    o.so3[4 * i] = qn.x; o.so3[4 * i + 1] = qn.y; o.so3[4 * i + 2] = qn.z; o.so3[4 * i + 3] = qn.w;
  }
  for (int i = 0; i < nr3; ++i) {        // utils.cc:243-261; the `nearest < t_new.size()` test is the reference's (quirk);
    const double t = double(i) * double(o.dt_r3_ns) * NS_TO_S;   // reading one past the end (UB there) falls back to the nearest value here
    double dist = 0; const size_t k = find_closest(t, t_vis, dist);
    if (k < size_t(nr3) && k + 1 < size_t(nv)) {
      const double frac = dist / (t_vis[k + 1] - t_vis[k]);
      for (int d = 0; d < 3; ++d) o.r3[3 * i + d] = (1.0 - frac) * p_vis[3 * k + d] + frac * p_vis[3 * (k + 1) + d];
    } else for (int d = 0; d < 3; ++d) o.r3[3 * i + d] = p_vis[3 * k + d];
  }
  // InitBiasSplines(…, 10e9, 10e9, 1.0, 0.1)  (imu_camera_calibrator.cc:80-85, impl.h:53-90)
  o.dt_ba_ns = o.dt_bg_ns = int64_t(10 * 1e9); o.max_ba = 1.0; o.max_bg = 1e-1;
  o.inv_ba_dt = 1.0 / double(o.dt_ba_ns); o.inv_bg_dt = 1.0 / double(o.dt_bg_ns);
  const int nba = int(duration / o.dt_ba_ns) + BIAS_N, nbg = int(duration / o.dt_bg_ns) + BIAS_N;
  o.ba.resize(3 * size_t(nba)); o.bg.resize(3 * size_t(nbg));
  for (int i = 0; i < nba; ++i) for (int d = 0; d < 3; ++d) o.ba[3 * i + d] = ipp->acc_bias[d];
  for (int i = 0; i < nbg; ++i) for (int d = 0; d < 3; ++d) o.bg[3 * i + d] = ipp->gyr_bias[d];

  // ---- measurement wiring ---------------------------------------------------------------------------------
  // Shards (icc_set_shard): time-sorted residual units are cut into `world` slices of equal scalar-residual count.
  o.frames.clear(); o.blocks.clear(); o.vis_blocks.clear(); o.imu_used.clear();
  o.n_res_vis = o.n_res_acc = o.n_res_gyr = 0;
  struct Unit { double t; int kind; int idx; int nres; };
  std::vector<Unit> units;
  const bool rolling = ipp->init_line_delay_s != 0.0;
  std::vector<Frame> all_frames(nf);
  for (int i = 0; i < nf; ++i) {
    Frame& f = all_frames[i]; f.t_s = o.frame_t[i]; f.c0 = o.corner_off[i]; f.c1 = o.corner_off[i + 1];
    const int64_t t_ns = int64_t(f.t_s * S_TO_NS);     // impl.h:541
    f.ok = calc_times(t_ns, o.start_ns, o.dt_r3_ns, nr3, SPLINE_N, f.u_r3, f.s_r3) && calc_times(t_ns, o.start_ns, o.dt_so3_ns, nso3, SPLINE_N, f.u_so3, f.s_so3);
    if (f.ok) units.push_back({f.t_s, 0, i, 2 * (f.c1 - f.c0)});
  }
  std::vector<ImuUsed> all_imu; std::map<double, int> imu_by_t;
  for (size_t i = 0; i < o.imu_t.size(); ++i) {           // imu_camera_calibrator.cc:102-120
    const double t = o.imu_t[i] + ipp->time_offset_imu_to_cam_s;
    if (t < o.t0_s || t >= o.tend_s) continue;
    ImuUsed m; m.t_s = t; for (int d = 0; d < 3; ++d) { m.acc[d] = o.imu_acc[3 * i + d]; m.gyr[d] = o.imu_gyr[3 * i + d]; }
    imu_by_t[t] = int(all_imu.size()); all_imu.push_back(m);
    units.push_back({t, 1, int(all_imu.size()) - 1, 6});
  }
  std::stable_sort(units.begin(), units.end(), [](const Unit& a, const Unit& b) { return a.t < b.t; });
  long total = 0; for (auto& u : units) total += u.nres;
  long lo = total * o.shard_rank / o.shard_world, hi = total * (o.shard_rank + 1) / o.shard_world, run = 0;
  int res_vis = 0;
  std::vector<int> imu_sel;
  std::vector<int> frame_sel;
  for (auto& u : units) { const bool mine = run >= lo && run < hi; run += u.nres; if (!mine) continue; if (u.kind == 0) frame_sel.push_back(u.idx); else imu_sel.push_back(u.idx); }
  std::sort(frame_sel.begin(), frame_sel.end());
  // vision blocks (RS path; the GS path is Huber(0) => zero weight, quirk q3, so no block is created)
  for (int fi : frame_sel) {
    const Frame& f = all_frames[fi];
    o.frames.push_back(f);
    Block b; b.type = BLK_RS_VISION; b.frame = int(o.frames.size()) - 1; b.n_res = 2 * (f.c1 - f.c0); b.res_off = res_vis; res_vis += b.n_res;
    b.u_so3 = f.u_so3; b.u_r3 = f.u_r3; b.u_bias = 0;
    for (int i = 0; i < SPLINE_N; ++i) b.params.push_back({&o.so3[4 * (f.s_so3 + i)], 4, LP_SO3, -1});
    for (int i = 0; i < SPLINE_N; ++i) b.params.push_back({&o.r3[3 * (f.s_r3 + i)], 3, LP_NONE, -1});
    b.params.push_back({o.T_ic, 7, LP_SE3, -1});
    b.params.push_back({&o.line_delay, 1, LP_NONE, -1});
    b.params.push_back({o.intr, o.n_intr, LP_NONE, -1});
    for (int c = f.c0; c < f.c1; ++c) b.params.push_back({&o.points[4 * size_t(o.point_ids[c])], 4, LP_NONE, -1});
    o.vis_blocks.push_back(b);
    if (rolling) o.blocks.push_back(std::move(b));
  }
  if (!rolling) res_vis = 0;
  o.n_res_vis = res_vis;
  // IMU blocks: accelerometer residuals first, then gyroscope residuals, both in time order
  std::vector<Block> acc_blocks, gyr_blocks;
  for (int mi : imu_sel) {
    const ImuUsed& m = all_imu[mi];
    o.imu_used.push_back(m);
    const int ui = int(o.imu_used.size()) - 1;
    const int64_t t_ns = int64_t(m.t_s * S_TO_NS);
    double u_r3, u_so3, u_b; int64_t s_r3, s_so3, s_b;
    if (calc_times(t_ns, o.start_ns, o.dt_r3_ns, nr3, SPLINE_N, u_r3, s_r3) && calc_times(t_ns, o.start_ns, o.dt_so3_ns, nso3, SPLINE_N, u_so3, s_so3) &&
        calc_times(t_ns, o.start_ns, o.dt_ba_ns, nba, BIAS_N, u_b, s_b)) {
      Block b; b.type = BLK_ACCEL; b.frame = ui; b.n_res = 3; b.u_so3 = u_so3; b.u_r3 = u_r3; b.u_bias = u_b;
      for (int i = 0; i < SPLINE_N; ++i) b.params.push_back({&o.so3[4 * (s_so3 + i)], 4, LP_SO3, -1});
      for (int i = 0; i < SPLINE_N; ++i) b.params.push_back({&o.r3[3 * (s_r3 + i)], 3, LP_NONE, -1});
      for (int i = 0; i < BIAS_N; ++i) b.params.push_back({&o.ba[3 * (s_b + i)], 3, LP_NONE, -1});
      b.params.push_back({o.grav, 3, LP_NONE, -1});
      b.params.push_back({o.acc_intr, 6, LP_NONE, -1});
      b.params.push_back({&o.toff_delta, 1, LP_NONE, -1});
      acc_blocks.push_back(std::move(b));
    }
    if (calc_times(t_ns, o.start_ns, o.dt_so3_ns, nso3, SPLINE_N, u_so3, s_so3) && calc_times(t_ns, o.start_ns, o.dt_bg_ns, nbg, BIAS_N, u_b, s_b)) {
      Block b; b.type = BLK_GYRO; b.frame = ui; b.n_res = 3; b.u_so3 = u_so3; b.u_r3 = 0; b.u_bias = u_b;
      for (int i = 0; i < SPLINE_N; ++i) b.params.push_back({&o.so3[4 * (s_so3 + i)], 4, LP_SO3, -1});
      for (int i = 0; i < BIAS_N; ++i) b.params.push_back({&o.bg[3 * (s_b + i)], 3, LP_NONE, -1});
      b.params.push_back({o.gyr_intr, 9, LP_NONE, -1});
      b.params.push_back({&o.toff_delta, 1, LP_NONE, -1});
      gyr_blocks.push_back(std::move(b));
    }
  }
  int off = res_vis;
  for (auto& b : acc_blocks) { b.res_off = off; off += 3; o.blocks.push_back(std::move(b)); }
  o.n_res_acc = 3 * int(acc_blocks.size());
  for (auto& b : gyr_blocks) { b.res_off = off; off += 3; o.blocks.push_back(std::move(b)); }
  o.n_res_gyr = 3 * int(gyr_blocks.size());

  // InitializeGravity (imu_camera_calibrator.cc:130-161), incl. the integer-second truncation of the accelerometer time
  bool ginit = false; double g0[3] = {0, 0, 9.81};
  for (size_t j = 0; j < cam_ts.size() && !ginit; ++j) {
    const int vi = by_time[cam_ts[j]];
    SE3T<double> Twc{qnormalized(Q4<double>{o.q_wc[4 * vi], o.q_wc[4 * vi + 1], o.q_wc[4 * vi + 2], o.q_wc[4 * vi + 3]}), {o.p_wc[3 * vi], o.p_wc[3 * vi + 1], o.p_wc[3 * vi + 2]}};
    SE3T<double> Tai = se3_mul(Twc, Tci);
    for (size_t i = 0; i < o.imu_t.size(); ++i) {
      const int64_t accl_t = int64_t(o.imu_t[i]);
      if (std::fabs(double(accl_t) - cam_ts[j]) < 1. / 30.) {
        V3<double> g = so3_act(Tai.q, V3<double>{o.imu_acc[3 * i], o.imu_acc[3 * i + 1], o.imu_acc[3 * i + 2]});
        g0[0] = g.x; g0[1] = g.y; g0[2] = g.z; ginit = true; break;
      }
    }
  }
  memcpy(o.grav, g0, sizeof g0);
  o.initialised = true; o.cur_flags = -1;
  return ICC_OK;
}

icc_status icco_set_known_gravity_dir(void* h, const double g[3]) { memcpy(O(h)->grav, g, 3 * sizeof(double)); return ICC_OK; }

icc_status icco_optimize(void* h, int max_iters, int flags, icc_summary* S) {
  Oracle& o = *O(h);
  if (!o.initialised) { o.err = "batch_init_spline first"; return ICC_ERR_STATE; }
  if (!configure(o, flags)) return ICC_ERR_UNSUPPORTED;
  icc_summary s; lm_solve(o, max_iters, flags, true, s);
  s.mean_reproj_error = o.vis_blocks.empty() ? 0.0 : mean_reproj_error(o);
  if (S) *S = s;
  return ICC_OK;
}
icc_status icco_lm_iterations(void* h, int n, int flags, icc_summary* S) {
  Oracle& o = *O(h);
  if (!o.initialised) { o.err = "batch_init_spline first"; return ICC_ERR_STATE; }
  if (!configure(o, flags)) return ICC_ERR_UNSUPPORTED;
  icc_summary s; lm_solve(o, n, flags, false, s);
  if (S) *S = s;
  return ICC_OK;
}
// One damped solve at the current state, same contract as icc_solve_step (`chunks` has no meaning here: one sequential factorisation).
icc_status icco_solve_step(void* h, int flags, double radius, int chunks, double* cost, double* gradient, double* hessian_dense,
                           double* scale, double* lm_diag, double* delta, double* model_change) {
  Oracle& o = *O(h);
  if (!o.initialised) { o.err = "batch_init_spline first"; return ICC_ERR_STATE; }
  if (!(radius > 0.0) || chunks < 0) return ICC_ERR_INVALID_ARGUMENT;
  if (!configure(o, flags)) return ICC_ERR_UNSUPPORTED;
  const int n = o.n_tan;
  if (n == 0) return ICC_ERR_INVALID_ARGUMENT;
  Normal ne; double c;
  evaluate(o, &c, nullptr, &ne, nullptr, total_residuals(o));
  const std::vector<double> s = jacobi_scale(ne, o.opt.jacobi_scaling);
  LmStep st;
  if (!lm_step(ne, s, radius, o.opt, false, st)) { o.err = "Cholesky breakdown"; return ICC_ERR_NUMERIC; }
  if (cost) *cost = c;
  for (int i = 0; i < n; ++i) {
    const int j = o.perm[i];
    if (gradient) gradient[i] = ne.g[j];
    if (scale) scale[i] = s[j];
    if (lm_diag) lm_diag[i] = st.D2[j];
    if (delta) delta[i] = st.y[j] * s[j];
  }
  if (hessian_dense) for (int i = 0; i < n; ++i) for (int j = 0; j < n; ++j) hessian_dense[size_t(i) * n + j] = ne.get(o.perm[i], o.perm[j]);
  if (model_change) *model_change = st.model_change;
  return ICC_OK;
}

icc_status icco_get_T_i_c(const void* h, double T[7]) { memcpy(T, O(h)->T_ic, 7 * sizeof(double)); return ICC_OK; }
icc_status icco_get_gravity(const void* h, double g[3]) { memcpy(g, O(h)->grav, 3 * sizeof(double)); return ICC_OK; }
icc_status icco_get_line_delay(const void* h, double* ld) { *ld = O(h)->line_delay; return ICC_OK; }
icc_status icco_get_camera_intrinsics(const void* h, double* k, int n) { for (int i = 0; i < n && i < O(h)->n_intr; ++i) k[i] = O(h)->intr[i]; return ICC_OK; }
icc_status icco_get_time_offset(const void* h, double* t) { *t = O(h)->ip.time_offset_imu_to_cam_s + O(h)->toff_delta; return ICC_OK; }
icc_status icco_get_num_knots(const void* h, int* a, int* b, int* c, int* d) { const Oracle& o = *O(h); if (a) *a = nknots(o.so3, 4); if (b) *b = nknots(o.r3, 3); if (c) *c = nknots(o.ba, 3); if (d) *d = nknots(o.bg, 3); return ICC_OK; }
icc_status icco_get_knots(const void* h, double* so3, double* r3, double* ba, double* bg) {
  const Oracle& o = *O(h);
  if (so3) std::copy(o.so3.begin(), o.so3.end(), so3);
  if (r3) std::copy(o.r3.begin(), o.r3.end(), r3);
  if (ba) std::copy(o.ba.begin(), o.ba.end(), ba);
  if (bg) std::copy(o.bg.begin(), o.bg.end(), bg);
  return ICC_OK;
}
icc_status icco_set_knots(void* h, const double* so3, const double* r3, const double* ba, const double* bg) {
  Oracle& o = *O(h);
  if (so3) std::copy(so3, so3 + o.so3.size(), o.so3.begin());
  if (r3) std::copy(r3, r3 + o.r3.size(), o.r3.begin());
  if (ba) std::copy(ba, ba + o.ba.size(), o.ba.begin());
  if (bg) std::copy(bg, bg + o.bg.size(), o.bg.begin());
  return ICC_OK;
}
icc_status icco_set_T_i_c(void* h, const double T[7]) { memcpy(O(h)->T_ic, T, 7 * sizeof(double)); return ICC_OK; }
icc_status icco_set_line_delay(void* h, double ld) { O(h)->line_delay = ld; return ICC_OK; }
icc_status icco_get_mean_reprojection_error(void* h, double* e) { Oracle& o = *O(h); if (!o.initialised) return ICC_ERR_STATE; *e = mean_reproj_error(o); return ICC_OK; }
icc_status icco_get_num_imu_used(const void* h, int* n) { *n = int(O(h)->imu_used.size()); return ICC_OK; }
icc_status icco_get_imu_used(const void* h, double* t, double* a, double* g) {
  const Oracle& o = *O(h);
  for (size_t i = 0; i < o.imu_used.size(); ++i) { if (t) t[i] = o.imu_used[i].t_s; for (int d = 0; d < 3; ++d) { if (a) a[3 * i + d] = o.imu_used[i].acc[d]; if (g) g[3 * i + d] = o.imu_used[i].gyr[d]; } }
  return ICC_OK;
}

// impl.h:898-991,1180-1234
icc_status icco_eval_trajectory(void* h, int n, const int64_t* t_ns, double* gyro, double* accel, double* bg, double* ba, double* pose_q, double* pose_p, int32_t* valid) {
  Oracle& o = *O(h);
  if (!o.initialised) return ICC_ERR_STATE;
  const int nso3 = nknots(o.so3, 4), nr3 = nknots(o.r3, 3), nba = nknots(o.ba, 3), nbg = nknots(o.bg, 3);
  for (int i = 0; i < n; ++i) {
    double u_so3, u_r3, u_b; int64_t s_so3, s_r3, s_b;
    const bool ok_so3 = calc_times(t_ns[i], o.start_ns, o.dt_so3_ns, nso3, SPLINE_N, u_so3, s_so3);
    const bool ok_r3 = calc_times(t_ns[i], o.start_ns, o.dt_r3_ns, nr3, SPLINE_N, u_r3, s_r3);
    if (valid) valid[i] = ok_so3 && ok_r3;
    const double* ks[SPLINE_N]; const double* kr[SPLINE_N];
    if (ok_so3) for (int k = 0; k < SPLINE_N; ++k) ks[k] = &o.so3[4 * (s_so3 + k)];
    if (ok_r3) for (int k = 0; k < SPLINE_N; ++k) kr[k] = &o.r3[3 * (s_r3 + k)];
    Q4<double> R{0, 0, 0, 1}; V3<double> w{0, 0, 0};
    if (ok_so3) evaluate_lie_so3<SPLINE_N, double>(ks, u_so3, o.inv_so3_dt, &R, &w);
    if (gyro && ok_so3) { gyro[3 * i] = w.x; gyro[3 * i + 1] = w.y; gyro[3 * i + 2] = w.z; }
    if (accel && ok_so3 && ok_r3) {
      V3<double> aw = evaluate_r3<SPLINE_N, 2, double>(kr, u_r3, o.inv_r3_dt);
      V3<double> a = so3_act(so3_inv(R), V3<double>{aw.x + o.grav[0], aw.y + o.grav[1], aw.z + o.grav[2]});
      accel[3 * i] = a.x; accel[3 * i + 1] = a.y; accel[3 * i + 2] = a.z;
    }
    if (pose_q && ok_so3 && ok_r3) { pose_q[4 * i] = R.x; pose_q[4 * i + 1] = R.y; pose_q[4 * i + 2] = R.z; pose_q[4 * i + 3] = R.w; }
    if (pose_p && ok_so3 && ok_r3) { V3<double> p = evaluate_r3<SPLINE_N, 0, double>(kr, u_r3, o.inv_r3_dt); pose_p[3 * i] = p.x; pose_p[3 * i + 1] = p.y; pose_p[3 * i + 2] = p.z; }
    if (bg) { double v[3] = {0, 0, 0}; if (calc_times(t_ns[i], o.start_ns, o.dt_bg_ns, nbg, BIAS_N, u_b, s_b)) { const double* kb[BIAS_N]; for (int k = 0; k < BIAS_N; ++k) kb[k] = &o.bg[3 * (s_b + k)]; V3<double> b = evaluate_r3<BIAS_N, 0, double>(kb, u_b, o.inv_bg_dt); v[0] = b.x; v[1] = b.y; v[2] = b.z; } for (int d = 0; d < 3; ++d) bg[3 * i + d] = v[d]; }
    if (ba) { double v[3] = {0, 0, 0}; if (calc_times(t_ns[i], o.start_ns, o.dt_ba_ns, nba, BIAS_N, u_b, s_b)) { const double* kb[BIAS_N]; for (int k = 0; k < BIAS_N; ++k) kb[k] = &o.ba[3 * (s_b + k)]; V3<double> b = evaluate_r3<BIAS_N, 0, double>(kb, u_b, o.inv_ba_dt); v[0] = b.x; v[1] = b.y; v[2] = b.z; } for (int d = 0; d < 3; ++d) ba[3 * i + d] = v[d]; }
  }
  return ICC_OK;
}

icc_status icco_num_residuals(const void* h, int* v, int* a, int* g) { const Oracle& o = *O(h); if (v) *v = o.n_res_vis; if (a) *a = o.n_res_acc; if (g) *g = o.n_res_gyr; return ICC_OK; }
icc_status icco_num_tangent(void* h, int flags, int* n) { Oracle& o = *O(h); if (!o.initialised) return ICC_ERR_STATE; if (!configure(o, flags)) return ICC_ERR_UNSUPPORTED; *n = o.n_tan; return ICC_OK; }

icc_status icco_evaluate(void* h, int flags, double* cost, double* residuals, double* gradient, double* hessian_dense) {
  Oracle& o = *O(h);
  if (!o.initialised) { o.err = "batch_init_spline first"; return ICC_ERR_STATE; }
  if (!configure(o, flags)) return ICC_ERR_UNSUPPORTED;
  const int nres = total_residuals(o), n = o.n_tan;
  if (!gradient && !hessian_dense) { evaluate(o, cost, residuals, nullptr, nullptr, nres); return ICC_OK; }
  Normal ne; double c;
  evaluate(o, &c, residuals, &ne, nullptr, nres);
  if (cost) *cost = c;
  if (gradient) for (int i = 0; i < n; ++i) gradient[i] = ne.g[o.perm[i]];
  if (hessian_dense) for (int i = 0; i < n; ++i) for (int j = 0; j < n; ++j) hessian_dense[size_t(i) * n + j] = ne.get(o.perm[i], o.perm[j]);
  return ICC_OK;
}
// J^T J V (canonical tangent order), same contract as icc_normal_matvec.
icc_status icco_normal_matvec(void* h, int flags, int nvec, const double* V, double* HV) {
  Oracle& o = *O(h);
  if (!o.initialised) return ICC_ERR_STATE;
  if (!configure(o, flags)) return ICC_ERR_UNSUPPORTED;
  Normal ne; double c;
  evaluate(o, &c, nullptr, &ne, nullptr, total_residuals(o));
  const int n = o.n_tan, nk = ne.nk, nb = ne.nb, kd = ne.kd;
  std::vector<double> x(n), y(n);
  for (int v = 0; v < nvec; ++v) {
    for (int i = 0; i < n; ++i) x[o.perm[i]] = V[size_t(v) * n + i];
    std::fill(y.begin(), y.end(), 0.0);
    for (int j = 0; j < nk; ++j) {
      const double* col = &ne.band[size_t(j) * (kd + 1)];
      y[j] += col[0] * x[j];
      for (int d = 1; d <= kd && j + d < nk; ++d) { y[j] += col[d] * x[j + d]; y[j + d] += col[d] * x[j]; }
      for (int b = 0; b < nb; ++b) { const double e = ne.E[size_t(b) * nk + j]; y[j] += e * x[nk + b]; y[nk + b] += e * x[j]; }
    }
    for (int a = 0; a < nb; ++a) for (int b = 0; b < nb; ++b) y[nk + a] += ne.C[size_t(a) * nb + b] * x[nk + b];
    for (int i = 0; i < n; ++i) HV[size_t(v) * n + i] = y[o.perm[i]];
  }
  return ICC_OK;
}
// Dense Jacobian (n_res x n_tan, row-major, canonical column order) — tests only.
icc_status icco_jacobian_dense(void* h, int flags, double* J) {
  Oracle& o = *O(h);
  if (!o.initialised) return ICC_ERR_STATE;
  if (!configure(o, flags)) return ICC_ERR_UNSUPPORTED;
  std::vector<double> Jd; double c;
  evaluate(o, &c, nullptr, nullptr, &Jd, total_residuals(o));
  std::copy(Jd.begin(), Jd.end(), J);
  return ICC_OK;
}
// Time `n` Jacobian (or cost-only) evaluations; seconds per evaluation on this host.
icc_status icco_time_evaluations(void* h, int n, int flags, int with_jacobian, double* ms_per_eval) {
  Oracle& o = *O(h);
  if (!o.initialised) return ICC_ERR_STATE;
  if (!configure(o, flags)) return ICC_ERR_UNSUPPORTED;
  const int nres = total_residuals(o);
  auto t0 = std::chrono::steady_clock::now();
  Normal ne;
  for (int i = 0; i < n; ++i) { double c; evaluate(o, &c, nullptr, with_jacobian ? &ne : nullptr, nullptr, nres); }
  *ms_per_eval = 1e3 * std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() / std::max(n, 1);
  return ICC_OK;
}
// Known-answer access to the blending matrices (SURVEY §8(a2)).
void icco_blending_matrix(int N, int cumulative, double* out) {
  if (N == 6) { const auto& B = blend<6>(); for (int i = 0; i < 6; ++i) for (int j = 0; j < 6; ++j) out[i * 6 + j] = cumulative ? B.Mc[i][j] : B.M[i][j]; }
  if (N == 3) { const auto& B = blend<3>(); for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) out[i * 3 + j] = cumulative ? B.Mc[i][j] : B.M[i][j]; }
}
void icco_base_coefficients(int N, double* out) {
  if (N == 6) { const auto& B = blend<6>(); for (int i = 0; i < 6; ++i) for (int j = 0; j < 6; ++j) out[i * 6 + j] = B.base[i][j]; }
}
// Camera projection (double) for generator cross-checks.
// ---- upstream row f1: per-view board poses (restates src/core/pose_estimator.cc:54-191; TEST INFRASTRUCTURE) -----------------
// Deliberately formulated differently from the CUDA path: forward-mode duals for the un-projection Jacobian, the DLT null vector
// of the full 9-parameter homography by inverse iteration, Gauss-Newton systems solved by Gaussian elimination with pivoting.
namespace {
bool gauss_solve(int n, std::vector<double>& A, std::vector<double>& b) {   // A row-major n x n, overwritten
  for (int c = 0; c < n; ++c) {
    int piv = c; for (int r = c + 1; r < n; ++r) if (std::fabs(A[r * n + c]) > std::fabs(A[piv * n + c])) piv = r;
    if (!(std::fabs(A[piv * n + c]) > 0.0)) return false;
    if (piv != c) { for (int k = 0; k < n; ++k) std::swap(A[c * n + k], A[piv * n + k]); std::swap(b[c], b[piv]); }
    for (int r = c + 1; r < n; ++r) { const double f = A[r * n + c] / A[c * n + c]; for (int k = c; k < n; ++k) A[r * n + k] -= f * A[c * n + k]; b[r] -= f * b[c]; }
  }
  for (int r = n - 1; r >= 0; --r) { double s2 = b[r]; for (int k = r + 1; k < n; ++k) s2 -= A[r * n + k] * b[k]; b[r] = s2 / A[r * n + r]; }
  return true;
}
bool oracle_unproject(int model, const double* intr, double px, double py, double* xy) {
  typedef Jet<2> J2;
  auto eval = [&](double x, double y, double* uv, double* Jm) -> bool {
    J2 k[10]; for (int i = 0; i < 10; ++i) k[i] = J2(intr[i]);
    J2 p[3]; p[0] = J2(x); p[0].v[0] = 1.0; p[1] = J2(y); p[1].v[1] = 1.0; p[2] = J2(1.0);
    J2 o[2];
    if (!project<J2>(model, k, p, o, true)) return false;
    uv[0] = o[0].a; uv[1] = o[1].a; Jm[0] = o[0].v[0]; Jm[1] = o[0].v[1]; Jm[2] = o[1].v[0]; Jm[3] = o[1].v[1];
    return true;
  };
  double uv[2], Jm[4];
  if (!eval(0.0, 0.0, uv, Jm)) return false;
  double det = Jm[0] * Jm[3] - Jm[1] * Jm[2];
  if (!(std::fabs(det) > 0.0)) return false;
  double x = (Jm[3] * (px - uv[0]) - Jm[1] * (py - uv[1])) / det, y = (-Jm[2] * (px - uv[0]) + Jm[0] * (py - uv[1])) / det;
  int guard = 0;
  while (!eval(x, y, uv, Jm)) { x *= 0.5; y *= 0.5; if (++guard > 60) return false; }
  double e = (uv[0] - px) * (uv[0] - px) + (uv[1] - py) * (uv[1] - py);
  for (int it = 0; it < 100 && e > 1e-28; ++it) {
    det = Jm[0] * Jm[3] - Jm[1] * Jm[2];
    if (!(std::fabs(det) > 1e-300)) break;
    const double ru = uv[0] - px, rv = uv[1] - py;
    const double dx = -(Jm[3] * ru - Jm[1] * rv) / det, dy = -(-Jm[2] * ru + Jm[0] * rv) / det;
    bool moved = false; double t = 1.0;
    for (int bt = 0; bt < 40; ++bt, t *= 0.5) {
      double uv2[2], J2m[4];
      if (!eval(x + t * dx, y + t * dy, uv2, J2m)) continue;
      const double en = (uv2[0] - px) * (uv2[0] - px) + (uv2[1] - py) * (uv2[1] - py);
      if (en < e) { x += t * dx; y += t * dy; e = en; uv[0] = uv2[0]; uv[1] = uv2[1]; for (int i = 0; i < 4; ++i) Jm[i] = J2m[i]; moved = true; break; }
    }
    if (!moved) break;
  }
  xy[0] = x; xy[1] = y;
  return e < 1e-12;
}
struct PoseObs { double X, Y, Z, x, y; int c; };
typedef V3<double> Vd; typedef Q4<double> Qd;
double pose_cost(const std::vector<PoseObs>& ob, const Qd& R, const Vd& t) {
  double c = 0.0;
  for (const PoseObs& o : ob) {
    const Vd Pc = so3_act(R, Vd{o.X, o.Y, o.Z}) + t;
    if (!(Pc.z > 0.0)) { c += 1e6; continue; }
    const double r0 = Pc.x / Pc.z - o.x, r1 = Pc.y / Pc.z - o.y, rn = std::sqrt(r0 * r0 + r1 * r1);
    c += rn <= 1.345 ? 0.5 * rn * rn : 1.345 * rn - 0.5 * 1.345 * 1.345;
  }
  return c;
}
void pose_gauss_newton(const std::vector<PoseObs>& ob, Qd& R, Vd& t, double rel_tol = 1e-15) {
  double lambda = 1e-4, cost = pose_cost(ob, R, t);
  for (int it = 0; it < 100; ++it) {
    std::vector<double> H(36, 0.0), g(6, 0.0);
    const M3<double> Rm = so3_matrix(R);
    for (const PoseObs& o : ob) {
      const double X[3] = {o.X, o.Y, o.Z};
      const Vd Pc = so3_act(R, Vd{o.X, o.Y, o.Z}) + t;
      if (!(Pc.z > 0.0)) continue;
      const double iz = 1.0 / Pc.z, u = Pc.x * iz, v = Pc.y * iz, r[2] = {u - o.x, v - o.y};
      const double rn = std::sqrt(r[0] * r[0] + r[1] * r[1]), w = rn <= 1.345 ? 1.0 : 1.345 / rn;
      // dPc/d(delta) = -R [X]x (right increment R exp(delta)), dPc/dt = I
      double dP[3][6];
      const double Xx[3][3] = {{0, -X[2], X[1]}, {X[2], 0, -X[0]}, {-X[1], X[0], 0}};
      for (int a2 = 0; a2 < 3; ++a2) for (int b2 = 0; b2 < 3; ++b2) { double s2 = 0; for (int k = 0; k < 3; ++k) s2 += Rm.m[a2][k] * Xx[k][b2]; dP[a2][b2] = -s2; dP[a2][3 + b2] = a2 == b2 ? 1.0 : 0.0; }
      double Jr[2][6];
      for (int b2 = 0; b2 < 6; ++b2) { Jr[0][b2] = iz * dP[0][b2] - u * iz * dP[2][b2]; Jr[1][b2] = iz * dP[1][b2] - v * iz * dP[2][b2]; }
      for (int a2 = 0; a2 < 6; ++a2) { g[a2] += w * (Jr[0][a2] * r[0] + Jr[1][a2] * r[1]); for (int b2 = 0; b2 < 6; ++b2) H[a2 * 6 + b2] += w * (Jr[0][a2] * Jr[0][b2] + Jr[1][a2] * Jr[1][b2]); }
    }
    std::vector<double> A = H, b(6);
    for (int a2 = 0; a2 < 6; ++a2) { A[a2 * 6 + a2] += lambda * (H[a2 * 6 + a2] + 1e-12); b[a2] = -g[a2]; }
    if (!gauss_solve(6, A, b)) { lambda *= 10.0; if (lambda > 1e12) break; continue; }
    const Qd Rn = qnormalized(so3_mul(R, so3_exp(Vd{b[0], b[1], b[2]})));
    const Vd tn = t + Vd{b[3], b[4], b[5]};
    const double cn = pose_cost(ob, Rn, tn), step2 = b[0] * b[0] + b[1] * b[1] + b[2] * b[2] + b[3] * b[3] + b[4] * b[4] + b[5] * b[5];
    if (cn < cost) { const double dec = cost - cn; R = Rn; t = tn; cost = cn; lambda = std::max(lambda * 0.1, 1e-12); if (dec <= rel_tol * cost || step2 < 1e-28) break; }
    else { if (step2 < 1e-28) break; lambda *= 10.0; if (lambda > 1e12) break; }
  }
}
Qd quat_from_cols(const Vd& r1, const Vd& r2, const Vd& r3) {
  const double m00 = r1.x, m10 = r1.y, m20 = r1.z, m01 = r2.x, m11 = r2.y, m21 = r2.z, m02 = r3.x, m12 = r3.y, m22 = r3.z, tr = m00 + m11 + m22;
  Qd q;
  if (tr > 0.0) { const double s2 = std::sqrt(tr + 1.0) * 2.0; q = Qd{(m21 - m12) / s2, (m02 - m20) / s2, (m10 - m01) / s2, 0.25 * s2}; }
  else if (m00 > m11 && m00 > m22) { const double s2 = std::sqrt(1.0 + m00 - m11 - m22) * 2.0; q = Qd{0.25 * s2, (m01 + m10) / s2, (m02 + m20) / s2, (m21 - m12) / s2}; }
  else if (m11 > m22) { const double s2 = std::sqrt(1.0 + m11 - m00 - m22) * 2.0; q = Qd{(m01 + m10) / s2, 0.25 * s2, (m12 + m21) / s2, (m02 - m20) / s2}; }
  else { const double s2 = std::sqrt(1.0 + m22 - m00 - m11) * 2.0; q = Qd{(m02 + m20) / s2, (m12 + m21) / s2, 0.25 * s2, (m10 - m01) / s2}; }
  return qnormalized(q);
}
double vnorm(const Vd& a) { return std::sqrt(dot(a, a)); }
// Normalised DLT homography board plane (X, Y, 1) -> image of one view; zref = height of the board plane
bool oracle_homography(const std::vector<PoseObs>& ob, double& zref, double Hm[9]) {
  const double n = (double)ob.size();
  double mX = 0, mY = 0, mx = 0, my = 0; zref = 0.0;
  for (const PoseObs& p : ob) { zref += p.Z; mX += p.X; mY += p.Y; mx += p.x; my += p.y; }
  zref /= n; mX /= n; mY /= n; mx /= n; my /= n;
  double dB = 0, dI = 0, dz = 0; for (const PoseObs& p : ob) { dB += std::hypot(p.X - mX, p.Y - mY); dI += std::hypot(p.x - mx, p.y - my); dz = std::max(dz, std::fabs(p.Z - zref)); }
  dB /= n; dI /= n;
  if (!(dB > 0.0) || !(dI > 0.0) || dz > 0.05 * dB) return false;   // degenerate, or too far from a plane for the homography initialisation
  const double sB = std::sqrt(2.0) / dB, sI = std::sqrt(2.0) / dI;
  // DLT: null vector of A^T A (9 x 9) by inverse iteration with a tiny shift
  std::vector<double> M(81, 0.0);
  for (const PoseObs& p : ob) {
    const double X = (p.X - mX) * sB, Y = (p.Y - mY) * sB, x = (p.x - mx) * sI, y = (p.y - my) * sI;
    const double ra[9] = {X, Y, 1, 0, 0, 0, -x * X, -x * Y, -x}, rb[9] = {0, 0, 0, X, Y, 1, -y * X, -y * Y, -y};
    for (int a2 = 0; a2 < 9; ++a2) for (int b2 = 0; b2 < 9; ++b2) M[a2 * 9 + b2] += ra[a2] * ra[b2] + rb[a2] * rb[b2];
  }
  double tr = 0; for (int a2 = 0; a2 < 9; ++a2) tr += M[a2 * 9 + a2];
  std::vector<double> hv(9, 1.0 / 3.0);
  bool okh = true;
  for (int it = 0; it < 8 && okh; ++it) {
    std::vector<double> A = M, b = hv;
    for (int a2 = 0; a2 < 9; ++a2) A[a2 * 9 + a2] += 1e-14 * tr;
    okh = gauss_solve(9, A, b);
    double nn = 0; for (double v : b) nn += v * v; nn = std::sqrt(nn);
    if (!(nn > 0.0)) { okh = false; break; }
    for (int a2 = 0; a2 < 9; ++a2) hv[a2] = b[a2] / nn;
  }
  if (!okh) return false;
  double G[9];
  for (int r = 0; r < 3; ++r) { G[3 * r] = hv[3 * r] * sB; G[3 * r + 1] = hv[3 * r + 1] * sB; G[3 * r + 2] = hv[3 * r + 2] - sB * (hv[3 * r] * mX + hv[3 * r + 1] * mY); }
  for (int c = 0; c < 3; ++c) { Hm[c] = G[c] / sI + mx * G[6 + c]; Hm[3 + c] = G[3 + c] / sI + my * G[6 + c]; Hm[6 + c] = G[6 + c]; }
  return true;
}
}  // namespace

icc_status icco_pixels_to_normalized(void* h, int n, const double* uv, double* xy, int32_t* ok) {
  Oracle& o = *O(h);
  for (int i = 0; i < n; ++i) { const bool g = oracle_unproject(o.model, o.intr, uv[2 * i], uv[2 * i + 1], xy + 2 * i); if (!g) { xy[2 * i] = 0; xy[2 * i + 1] = 0; } if (ok) ok[i] = g ? 1 : 0; }
  return ICC_OK;
}

}  // extern "C"
namespace {
// the per-view loop of PoseEstimator::EstimatePosesFromJson; refine_only = OptimizeAllPoses (start from the stored poses of the valid
// views, no homography); inlier (optional, one flag per corner) receives the final inlier sets
icc_status oracle_board_poses(Oracle& o, int nf, const int32_t* off, const int32_t* ids, const double* uv, double max_reproj_error, int min_points, bool refine_only,
                              double* q_wc, double* p_wc, double* mean_err, int32_t* valid, std::vector<char>* inlier) {
  const int np = (int)(o.points.size() / 4);
  const double W = o.width, Hh = o.height;
  const double max_px = max_reproj_error > 0.0 ? max_reproj_error : 0.004 * Hh;
  const double thresh_sq = (W > 0 && Hh > 0) ? max_px / std::sqrt(W * W + Hh * Hh) : 1e-3;
  if (min_points <= 0) min_points = 8;
  for (int f = 0; f < nf; ++f) {
    if (refine_only && !valid[f]) continue;
    if (!refine_only) { q_wc[4 * f] = q_wc[4 * f + 1] = q_wc[4 * f + 2] = 0.0; q_wc[4 * f + 3] = 1.0; p_wc[3 * f] = p_wc[3 * f + 1] = p_wc[3 * f + 2] = 0.0; valid[f] = 0; if (mean_err) mean_err[f] = 0.0; }
    std::vector<PoseObs> ob;
    for (int c = off[f]; c < off[f + 1]; ++c) {
      const int id = ids[c]; double xy[2];
      if (id < 0 || id >= np || !oracle_unproject(o.model, o.intr, uv[2 * c], uv[2 * c + 1], xy)) continue;
      const double* P = &o.points[4 * (size_t)id];
      ob.push_back({P[0] / P[3], P[1] / P[3], P[2] / P[3], xy[0], xy[1], c});
    }
    if (off[f + 1] - off[f] < min_points || ob.size() < 6) { if (refine_only) { q_wc[4 * f] = q_wc[4 * f + 1] = q_wc[4 * f + 2] = 0.0; q_wc[4 * f + 3] = 1.0; p_wc[3 * f] = p_wc[3 * f + 1] = p_wc[3 * f + 2] = 0.0; valid[f] = 0; if (mean_err) mean_err[f] = 0.0; } continue; }
    double zref = 0.0, Hm[9];
    Qd R; Vd t;
    if (refine_only) {   // PoseEstimator::OptimizeAllPoses (pose_estimator.cc:226-236): BundleAdjustView again from the stored pose
      R = so3_inv(qnormalized(Qd{q_wc[4 * f], q_wc[4 * f + 1], q_wc[4 * f + 2], q_wc[4 * f + 3]}));
      t = so3_act(R, Vd{p_wc[3 * f], p_wc[3 * f + 1], p_wc[3 * f + 2]}) * -1.0;
      q_wc[4 * f] = q_wc[4 * f + 1] = q_wc[4 * f + 2] = 0.0; q_wc[4 * f + 3] = 1.0; p_wc[3 * f] = p_wc[3 * f + 1] = p_wc[3 * f + 2] = 0.0; valid[f] = 0; if (mean_err) mean_err[f] = 0.0;
    } else {
    if (!oracle_homography(ob, zref, Hm)) continue;
    const Vd h1{Hm[0], Hm[3], Hm[6]}, h2{Hm[1], Hm[4], Hm[7]}, h3{Hm[2], Hm[5], Hm[8]};
    double sc = 2.0 / (vnorm(h1) + vnorm(h2));
    if (h3.z * sc < 0.0) sc = -sc;
    Vd r1 = h1 * sc, r2 = h2 * sc; t = h3 * sc;
    r1 = r1 * (1.0 / vnorm(r1)); r2 = r2 - r1 * dot(r1, r2); r2 = r2 * (1.0 / vnorm(r2));
    const Vd r3 = cross(r1, r2);
    R = quat_from_cols(r1, r2, r3);
    }
    for (PoseObs& p : ob) p.Z -= zref;
    pose_gauss_newton(ob, R, t, o.pose_rel_tol);
    std::vector<PoseObs> in;
    for (const PoseObs& p : ob) { const Vd Pc = so3_act(R, Vd{p.X, p.Y, p.Z}) + t; const double r0 = Pc.x / Pc.z - p.x, r1e = Pc.y / Pc.z - p.y; if (Pc.z > 0.0 && r0 * r0 + r1e * r1e < thresh_sq) in.push_back(p); }
    if (in.size() < 6) continue;
    if (in.size() != ob.size()) pose_gauss_newton(in, R, t, o.pose_rel_tol);
    double e = 0; for (const PoseObs& p : in) { const Vd Pc = so3_act(R, Vd{p.X, p.Y, p.Z}) + t; e += std::hypot(Pc.x / Pc.z - p.x, Pc.y / Pc.z - p.y); }
    e /= (double)in.size();
    const Vd tf = t - so3_act(R, Vd{0.0, 0.0, zref});
    const Qd Rw = so3_inv(R);
    const Vd pw = so3_act(Rw, tf) * -1.0;
    q_wc[4 * f] = Rw.x; q_wc[4 * f + 1] = Rw.y; q_wc[4 * f + 2] = Rw.z; q_wc[4 * f + 3] = Rw.w;
    p_wc[3 * f] = pw.x; p_wc[3 * f + 1] = pw.y; p_wc[3 * f + 2] = pw.z;
    if (mean_err) mean_err[f] = e;
    valid[f] = e <= max_px ? 1 : 0;
    if (inlier) for (const PoseObs& p : in) (*inlier)[p.c] = 1;
  }
  return ICC_OK;
}
}  // namespace

extern "C" {
icc_status icco_estimate_board_poses(void* h, int nf, const int32_t* off, const int32_t* ids, const double* uv, double max_reproj_error, int min_points,
                                     double* q_wc, double* p_wc, double* mean_err, int32_t* valid) {
  return oracle_board_poses(*O(h), nf, off, ids, uv, max_reproj_error, min_points, false, q_wc, p_wc, mean_err, valid, nullptr);
}

icc_status icco_filter_bad_poses(void* h, int nv, const double* p_wc, int32_t* valid) {   // PoseEstimator::FilterBadPoses (pose_estimator.cc:238-261)
  std::vector<double> z; for (int i = 0; i < nv; ++i) if (valid[i]) z.push_back(p_wc[3 * i + 2]);
  if (z.empty()) return ICC_OK;
  std::sort(z.begin(), z.end());
  const size_t n = z.size(); const double med = n % 2 == 0 ? (z[n / 2 - 1] + z[n / 2]) / 2 : z[n / 2];
  for (int i = 0; i < nv; ++i) if (valid[i] && std::fabs(p_wc[3 * i + 2] - med) > std::fabs(med)) valid[i] = 0;
  return ICC_OK;
}
icc_status icco_get_board_points(const void* h, double* xyzw, int n) { const Oracle& o = *O(h); for (size_t i = 0; i < 4 * (size_t)n && i < o.points.size(); ++i) xyzw[i] = o.points[i]; return ICC_OK; }
}  // extern "C"

namespace {
// One observation of a board point with a constant camera, as theia::BundleAdjustTracks poses it (forward-mode duals over the point).
template <class T> bool point_residual(bool normalized, int model, const double* intr, const M3<double>& Rcw, const Vd& cc, const T X[3], const double* meas, T r[2]) {
  const T d[3] = {X[0] - cc.x, X[1] - cc.y, X[2] - cc.z};
  T pc[3];
  for (int i = 0; i < 3; ++i) pc[i] = d[0] * Rcw.m[i][0] + d[1] * Rcw.m[i][1] + d[2] * Rcw.m[i][2];
  if (normalized) { if (!(jval(pc[2]) > 0.0)) return false; r[0] = pc[0] / pc[2] - meas[0]; r[1] = pc[1] / pc[2] - meas[1]; return true; }
  T k[10], px[2]; for (int i = 0; i < 10; ++i) k[i] = T(intr[i]);
  if (!project<T>(model, k, pc, px, true)) return false;
  r[0] = px[0] - meas[0]; r[1] = px[1] - meas[1];
  return true;
}
struct PointObs { M3<double> R; Vd c; double meas[2]; };
// Levenberg-Marquardt on the three coordinates of one point (same damping schedule as the pose refinement above); returns the cost
void refine_point(bool normalized, int model, const double* intr, const std::vector<PointObs>& ob, double huber, double X[3]) {
  typedef Jet<4> J4;
  auto cost_of = [&](const double* Xd) { double c = 0; for (const PointObs& o : ob) { double r[2]; if (!point_residual<double>(normalized, model, intr, o.R, o.c, Xd, o.meas, r)) { c += normalized ? 1e6 : 1e10; continue; }
      const double rn = std::sqrt(r[0] * r[0] + r[1] * r[1]); c += rn <= huber ? 0.5 * rn * rn : huber * rn - 0.5 * huber * huber; } return c; };
  double lambda = 1e-4, cost = cost_of(X);
  for (int it = 0; it < 100; ++it) {
    std::vector<double> H(9, 0.0), g(3, 0.0);
    for (const PointObs& o : ob) {
      J4 Xj[3], r[2]; for (int i = 0; i < 3; ++i) { Xj[i] = J4(X[i]); Xj[i].v[i] = 1.0; }
      if (!point_residual<J4>(normalized, model, intr, o.R, o.c, Xj, o.meas, r)) continue;
      const double rn = std::sqrt(r[0].a * r[0].a + r[1].a * r[1].a), w = rn <= huber ? 1.0 : huber / rn;
      for (int a = 0; a < 3; ++a) { g[a] += w * (r[0].v[a] * r[0].a + r[1].v[a] * r[1].a); for (int b = 0; b < 3; ++b) H[a * 3 + b] += w * (r[0].v[a] * r[0].v[b] + r[1].v[a] * r[1].v[b]); }
    }
    std::vector<double> A = H, b(3);
    for (int a = 0; a < 3; ++a) { A[a * 3 + a] += lambda * (H[a * 3 + a] + 1e-12); b[a] = -g[a]; }
    if (!gauss_solve(3, A, b)) { lambda *= 10.0; if (lambda > 1e12) break; continue; }
    const double Xn[3] = {X[0] + b[0], X[1] + b[1], X[2] + b[2]};
    const double cn = cost_of(Xn), step2 = b[0] * b[0] + b[1] * b[1] + b[2] * b[2];
    if (cn < cost) { const double dec = cost - cn; X[0] = Xn[0]; X[1] = Xn[1]; X[2] = Xn[2]; cost = cn; lambda = std::max(lambda * 0.1, 1e-12); if (dec <= 1e-15 * cost || step2 < 1e-30) break; }
    else { if (step2 < 1e-30) break; lambda *= 10.0; if (lambda > 1e12) break; }
  }
}
// theia::BundleAdjustTracks with constant cameras over the corners selected by take(c); returns the number of optimised points
template <class F>
int oracle_refine_points(Oracle& o, bool normalized, int model, const double* intr, int nv, const int32_t* off, const int32_t* ids, const double* meas,
                         const double* q_wc, const double* p_wc, F take, int min_obs, double huber) {
  const int np = (int)(o.points.size() / 4);
  std::vector<std::vector<PointObs>> per(np);
  for (int v = 0; v < nv; ++v) {
    const M3<double> R = so3_matrix(so3_inv(qnormalized(Qd{q_wc[4 * v], q_wc[4 * v + 1], q_wc[4 * v + 2], q_wc[4 * v + 3]})));
    const Vd c{p_wc[3 * v], p_wc[3 * v + 1], p_wc[3 * v + 2]};
    for (int cidx = off[v]; cidx < off[v + 1]; ++cidx) if (take(cidx)) per[ids[cidx]].push_back({R, c, {meas[2 * cidx], meas[2 * cidx + 1]}});
  }
  int n_opt = 0;
  for (int p = 0; p < np; ++p) {
    if ((int)per[p].size() <= min_obs) continue;
    double* P = &o.points[4 * (size_t)p];
    double X[3] = {P[0] / P[3], P[1] / P[3], P[2] / P[3]};
    refine_point(normalized, model, intr, per[p], huber, X);
    P[0] = X[0]; P[1] = X[1]; P[2] = X[2]; P[3] = 1.0; ++n_opt;
  }
  return n_opt;
}
}  // namespace

extern "C" {
// PoseEstimator::OptimizeBoardPoints + OptimizeAllPoses (pose_estimator.cc:193-236; app estimate_camera_poses_from_checkerboard.cc:61-65)
icc_status icco_optimize_board_points(void* h, int nf, const int32_t* off, const int32_t* ids, const double* uv, double max_reproj_error, int min_points, int min_observations,
                                      double* q_wc, double* p_wc, double* mean_err, int32_t* valid, double* board_out, int32_t* n_opt_out) {
  Oracle& o = *O(h);
  const int nc = off[nf];
  std::vector<char> inlier(std::max(1, nc), 0);
  std::vector<double> e(nf);
  oracle_board_poses(o, nf, off, ids, uv, max_reproj_error, min_points, true, q_wc, p_wc, e.data(), valid, &inlier);
  std::vector<double> xy(2 * (size_t)std::max(1, nc), 0.0);
  for (int c = 0; c < nc; ++c) if (inlier[c]) oracle_unproject(o.model, o.intr, uv[2 * c], uv[2 * c + 1], &xy[2 * c]);
  std::vector<int> view_of(std::max(1, nc)); for (int f = 0; f < nf; ++f) for (int c = off[f]; c < off[f + 1]; ++c) view_of[c] = f;
  const int n_opt = oracle_refine_points(o, true, o.model, o.intr, nf, off, ids, xy.data(), q_wc, p_wc, [&](int c) { return inlier[c] && valid[view_of[c]]; },
                                         min_observations > 0 ? min_observations : 30, 1.345);
  oracle_board_poses(o, nf, off, ids, uv, max_reproj_error, min_points, true, q_wc, p_wc, e.data(), valid, nullptr);
  if (mean_err) for (int f = 0; f < nf; ++f) mean_err[f] = e[f];
  if (board_out) std::copy(o.points.begin(), o.points.end(), board_out);
  if (n_opt_out) *n_opt_out = n_opt;
  return ICC_OK;
}

// ---- upstream row f3: IMU-to-camera rotation + time offset initialiser (TEST INFRASTRUCTURE) -------------------------------
// Restates src/core/imu_to_camera_rotation_estimator.cc:39-274 + applications/estimate_imu_to_camera_rotation.cc:96-162 serially,
// with the closed-form rotation through an SVD (one-sided Jacobi) exactly as the reference formulates it (the CUDA path uses
// Horn's quaternion method instead).  FindClosestTimestamp's linear scan is replaced by bisection (same index on sorted times).
namespace {
size_t nearest_sorted(const std::vector<double>& ts, double t, double& dist) {
  const size_t n = ts.size();
  size_t hi = std::lower_bound(ts.begin(), ts.end(), t) - ts.begin();
  size_t idx = hi == 0 ? 0 : (hi == n ? n - 1 : (std::fabs(t - ts[hi - 1]) <= std::fabs(t - ts[hi]) ? hi - 1 : hi));
  dist = std::fabs(t - ts[idx]);
  return idx;
}
void slerp_eigen(const double* a, const double* b, double t, double* o) {
  const double thresh = 1.0 - 2.220446049250313e-16;
  const double d = a[0] * b[0] + a[1] * b[1] + a[2] * b[2] + a[3] * b[3], ad = std::fabs(d);
  double s0, s1;
  if (ad >= thresh) { s0 = 1.0 - t; s1 = t; } else { const double th = std::acos(ad), sth = std::sin(th); s0 = std::sin((1.0 - t) * th) / sth; s1 = std::sin(t * th) / sth; }
  if (d < 0) s1 = -s1;
  for (int i = 0; i < 4; ++i) o[i] = s0 * a[i] + s1 * b[i];
}
void interp_quats(const std::vector<double>& t_old, const std::vector<double>& t_new, const std::vector<double>& q_old, std::vector<double>& q_new) {
  q_new.assign(4 * t_new.size(), 0.0);
  for (size_t i = 0; i < t_new.size(); ++i) {
    double dist; const size_t k = nearest_sorted(t_old, t_new[i], dist);
    if (k < t_old.size() - 1) slerp_eigen(&q_old[4 * k], &q_old[4 * (k + 1)], dist / (t_old[k + 1] - t_old[k]), &q_new[4 * i]);
    else for (int d = 0; d < 4; ++d) q_new[4 * i + d] = q_old[4 * k + d];
  }
}
// SVD of a 3x3 matrix by one-sided Jacobi: A = U diag(s) V^T
void svd3(const double A[3][3], double U[3][3], double s[3], double V[3][3]) {
  double B[3][3]; for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) { B[i][j] = A[i][j]; V[i][j] = i == j ? 1.0 : 0.0; }
  for (int sweep = 0; sweep < 60; ++sweep) {
    double off = 0.0;
    for (int p = 0; p < 3; ++p) for (int q = p + 1; q < 3; ++q) {
      double al = 0, be = 0, ga = 0;
      for (int k = 0; k < 3; ++k) { al += B[k][p] * B[k][p]; be += B[k][q] * B[k][q]; ga += B[k][p] * B[k][q]; }
      off = std::max(off, std::fabs(ga) / std::sqrt(std::max(al * be, 1e-300)));
      if (std::fabs(ga) < 1e-300) continue;
      const double zeta = (be - al) / (2.0 * ga), t = (zeta >= 0 ? 1.0 : -1.0) / (std::fabs(zeta) + std::sqrt(1.0 + zeta * zeta));
      const double c = 1.0 / std::sqrt(1.0 + t * t), sn = c * t;
      for (int k = 0; k < 3; ++k) { const double bp = B[k][p], bq = B[k][q]; B[k][p] = c * bp - sn * bq; B[k][q] = sn * bp + c * bq; const double vp = V[k][p], vq = V[k][q]; V[k][p] = c * vp - sn * vq; V[k][q] = sn * vp + c * vq; }
    }
    if (off < 1e-15) break;
  }
  for (int j = 0; j < 3; ++j) { s[j] = std::sqrt(B[0][j] * B[0][j] + B[1][j] * B[1][j] + B[2][j] * B[2][j]); }
  // U columns = B columns / s ; complete a rank-deficient basis by cross products
  for (int j = 0; j < 3; ++j) for (int k = 0; k < 3; ++k) U[k][j] = s[j] > 1e-300 ? B[k][j] / s[j] : 0.0;
  int order[3] = {0, 1, 2}; std::sort(order, order + 3, [&](int a, int b) { return s[a] > s[b]; });
  if (!(s[order[2]] > 1e-12 * std::max(s[order[0]], 1e-300))) {     // smallest singular vector: u3 = u1 x u2
    const int a = order[0], b = order[1], c = order[2];
    U[0][c] = U[1][a] * U[2][b] - U[2][a] * U[1][b]; U[1][c] = U[2][a] * U[0][b] - U[0][a] * U[2][b]; U[2][c] = U[0][a] * U[1][b] - U[1][a] * U[0][b];
  }
}
double det3(const double M[3][3]) { return M[0][0] * (M[1][1] * M[2][2] - M[1][2] * M[2][1]) - M[0][1] * (M[1][0] * M[2][2] - M[1][2] * M[2][0]) + M[0][2] * (M[1][0] * M[2][1] - M[1][1] * M[2][0]); }
struct RotFit { double R[3][3]; double bias[3]; double error; };
RotFit solve_closed_form(const std::vector<double>& angVis, const std::vector<double>& angImu, const std::vector<double>& ts, double td, bool estimate_bias) {
  const size_t n = ts.size();
  std::vector<double> two(n); for (size_t i = 0; i < n; ++i) two[i] = ts[i] - td;
  std::vector<double> iv(3 * n);
  for (size_t i = 0; i < n; ++i) {                                           // InterpolateVector3d(time_with_offset, timestamps, angVis)
    double dist; const size_t k = nearest_sorted(two, ts[i], dist);
    if (k + 1 >= n) { for (int d = 0; d < 3; ++d) iv[3 * i + d] = angVis[3 * k + d]; continue; }   // reference: out-of-bounds read (UB)
    const double f = dist / (two[k + 1] - two[k]);
    for (int d = 0; d < 3; ++d) iv[3 * i + d] = (1.0 - f) * angVis[3 * k + d] + f * angVis[3 * (k + 1) + d];
  }
  double mv[3] = {0, 0, 0}, mi[3] = {0, 0, 0};
  for (size_t i = 0; i < n; ++i) for (int d = 0; d < 3; ++d) { mi[d] += angImu[3 * i + d]; mv[d] += iv[3 * i + d]; }
  for (int d = 0; d < 3; ++d) { mi[d] /= (double)n; mv[d] /= (double)n; }
  double M[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};                         // P^T Q
  for (size_t i = 0; i < n; ++i) for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) M[a][b] += (angImu[3 * i + a] - mi[a]) * (iv[3 * i + b] - mv[b]);
  double U[3][3], sv[3], V[3][3];
  svd3(M, U, sv, V);
  double VUt[3][3]; for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) { VUt[a][b] = 0; for (int k = 0; k < 3; ++k) VUt[a][b] += V[a][k] * U[b][k]; }
  // C = diag(1, 1, -1) on the LAST column of V / U in Eigen's descending singular value order -> flip the smallest here
  RotFit r;
  int smallest = 0; for (int k = 1; k < 3; ++k) if (sv[k] < sv[smallest]) smallest = k;
  const double sgn = det3(VUt) < 0.0 ? -1.0 : 1.0;
  for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) { r.R[a][b] = 0; for (int k = 0; k < 3; ++k) r.R[a][b] += V[a][k] * (k == smallest ? sgn : 1.0) * U[b][k]; }
  for (int d = 0; d < 3; ++d) r.bias[d] = estimate_bias ? mv[d] - (r.R[d][0] * mi[0] + r.R[d][1] * mi[1] + r.R[d][2] * mi[2]) : 0.0;
  r.error = 0.0;
  for (size_t i = 0; i < n; ++i) {
    double e2 = 0;
    for (int d = 0; d < 3; ++d) { const double D = iv[3 * i + d] - (r.R[d][0] * angImu[3 * i] + r.R[d][1] * angImu[3 * i + 1] + r.R[d][2] * angImu[3 * i + 2] + r.bias[d]); e2 += D * D; }
    r.error += e2 > 1.345 ? 2.0 * 1.345 * std::sqrt(e2) - 1.345 * 1.345 : e2;
  }
  return r;
}
}  // namespace

icc_status icco_estimate_imu_to_camera_rotation(void* h, int n_views, const double* view_t, const double* q_cw, int n_imu, const double* imu_t, const double* gyro,
                                                const double* bias_in, double* q_out, double* td_out, double* bias_out, double* err_out, int32_t* iters_out) {
  (void)h;
  std::map<double, int> vmap, gmap;
  for (int i = 0; i < n_views; ++i) vmap[view_t[i]] = i;
  for (int i = 0; i < n_imu; ++i) gmap[imu_t[i]] = i;
  if (vmap.size() < 2 || gmap.size() < 2) return ICC_ERR_INVALID_ARGUMENT;
  double imu_dt = 0.0; for (int i = 1; i < n_imu; ++i) imu_dt += imu_t[i] - imu_t[i - 1]; imu_dt /= (double)(n_imu - 1);
  std::vector<double> tv, qv; for (const auto& kv : vmap) { tv.push_back(kv.first); for (int d = 0; d < 4; ++d) qv.push_back(q_cw[4 * (size_t)kv.second + d]); }
  std::vector<double> diffs; for (size_t i = 1; i < tv.size(); ++i) diffs.push_back(tv[i] - tv[i - 1]);
  std::sort(diffs.begin(), diffs.end());
  const double cam_dt = diffs.size() % 2 == 0 ? (diffs[diffs.size() / 2 - 1] + diffs[diffs.size() / 2]) / 2 : diffs[diffs.size() / 2];
  std::vector<double> grid; for (double t = tv.front(); t < tv.back(); t += cam_dt) grid.push_back(t);
  std::vector<double> qgrid; interp_quats(tv, grid, qv, qgrid);
  std::vector<double> tg, gg; for (const auto& kv : gmap) { tg.push_back(kv.first); for (int d = 0; d < 3; ++d) gg.push_back(gyro[3 * (size_t)kv.second + d] - (bias_in ? bias_in[d] : 0.0)); }
  const double t0 = grid.front() >= tg.front() ? grid.front() : tg.front(), tend = grid.back() >= tg.back() ? grid.back() : tg.back();
  std::vector<double> tI, angImu; for (size_t i = 0; i < tg.size(); ++i) if (tg[i] >= t0 && tg[i] <= tend) { tI.push_back(tg[i] - t0); for (int d = 0; d < 3; ++d) angImu.push_back(gg[3 * i + d]); }
  std::vector<double> tV, qV; for (size_t i = 0; i < grid.size(); ++i) if (grid[i] >= t0 && grid[i] <= tend) { tV.push_back(grid[i] - t0); for (int d = 0; d < 4; ++d) qV.push_back(qgrid[4 * i + d]); }
  const size_t n = tI.size();
  if (n < 2 || tV.empty()) return ICC_ERR_INVALID_ARGUMENT;
  std::vector<double> qi; interp_quats(tV, tI, qV, qi);
  std::vector<double> qd(4 * n, 0.0);
  for (size_t i = 1; i < n; ++i) for (int d = 0; d < 4; ++d) qd[4 * (i - 1) + d] = qi[4 * i + d] - qi[4 * (i - 1) + d];
  for (int d = 0; d < 4; ++d) qd[4 * (n - 1) + d] = qd[4 * (n - 2) + d];
  std::vector<double> angVis(3 * n);
  for (size_t i = 0; i < n; ++i) {
    const double* q = &qi[4 * i]; const double n2 = q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3];
    const Q4<double> inv{-q[0] / n2, -q[1] / n2, -q[2] / n2, q[3] / n2}, dq{qd[4 * i], qd[4 * i + 1], qd[4 * i + 2], qd[4 * i + 3]};
    // plain (non-normalising) quaternion product, Eigen operator*
    const double ax = dq.w * inv.x + dq.x * inv.w + dq.y * inv.z - dq.z * inv.y, ay = dq.w * inv.y + dq.y * inv.w + dq.z * inv.x - dq.x * inv.z, az = dq.w * inv.z + dq.z * inv.w + dq.x * inv.y - dq.y * inv.x;
    const double s2 = -2.0 / imu_dt; double w[3] = {s2 * ax, s2 * ay, s2 * az};
    if (std::fabs(w[0]) > 2 * M_PI || std::fabs(w[1]) > 2 * M_PI || std::fabs(w[2]) > 2 * M_PI) { for (int d = 0; d < 3; ++d) w[d] = i > 1 ? angVis[3 * (i - 1) + d] : 0.0; }
    for (int d = 0; d < 3; ++d) angVis[3 * i + d] = w[d];
  }
  auto smooth = [&](const std::vector<double>& x) { std::vector<double> y(x.size()); for (size_t i = 0; i < n; ++i) { const size_t k0 = i >= 14 ? i - 14 : 0; for (int d = 0; d < 3; ++d) { double s2 = 0; for (size_t k = k0; k <= i; ++k) s2 += x[3 * k + d]; y[3 * i + d] = s2 / (double)(i - k0 + 1); } } return y; };
  const std::vector<double> sVis = smooth(angVis), sImu = smooth(angImu);
  const double g = (1.0 + std::sqrt(5.0)) / 2.0, tol = 1e-4;
  double a = -1.0, b = 1.0, c = b - (b - a) / g, d = a + (b - a) / g, error = 0.0;
  double R[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}}, bias[3] = {bias_in ? bias_in[0] : 0.0, bias_in ? bias_in[1] : 0.0, bias_in ? bias_in[2] : 0.0};
  int iter = 0;
  while (std::fabs(c - d) > tol) {
    const RotFit fc = solve_closed_form(sVis, sImu, tI, c, !bias_in), fd = solve_closed_form(sVis, sImu, tI, d, !bias_in);
    const RotFit& k = fc.error < fd.error ? fc : fd;
    if (fc.error < fd.error) b = d; else a = c;
    for (int r = 0; r < 3; ++r) for (int cc = 0; cc < 3; ++cc) R[r][cc] = k.R[r][cc];
    if (!bias_in) for (int r = 0; r < 3; ++r) bias[r] = k.bias[r];
    error = k.error;
    c = b - (b - a) / g; d = a + (b - a) / g; ++iter;
  }
  const Q4<double> q = quat_from_cols(V3<double>{R[0][0], R[1][0], R[2][0]}, V3<double>{R[0][1], R[1][1], R[2][1]}, V3<double>{R[0][2], R[1][2], R[2][2]});
  q_out[0] = q.x; q_out[1] = q.y; q_out[2] = q.z; q_out[3] = q.w;
  *td_out = (b + a) / 2;
  if (bias_out) for (int r = 0; r < 3; ++r) bias_out[r] = bias[r];
  if (err_out) *err_out = error;
  if (iters_out) *iters_out = iter;
  return ICC_OK;
}

// ---- upstream row f2: spline error weighting (restates python/sew.py:36-234; TEST INFRASTRUCTURE) ---------------------------
// Pinned by tests/golden/sew_*.npz, which are outputs of the reference's own python/sew.py (tests/golden/make_sew_golden.py).
// Plain O(N^2) DFT with an exact twiddle table (index k n mod N) -- nothing in common with the CUDA path's Bluestein transform.
namespace {
double sew_removed_energy(const std::vector<double>& xhat, double fscale, double dt) {
  const int n = (int)xhat.size();
  double e = 0.0;
  for (int k = 0; k < n; ++k) {
    const int ik = k < (n + 1) / 2 ? k : k - n;
    const double y = (double)ik * fscale * dt;
    const double sinc = y == 0.0 ? 1.0 : std::sin(M_PI * y) / (M_PI * y);
    const double H = 3.0 * std::pow(sinc, 4) / (2.0 + std::cos(2.0 * M_PI * y));
    const double v = (1.0 - H) * xhat[k];
    e += v * v;
  }
  return e / (double)n;
}
double sew_brentq(const std::function<double(double)>& f, double xa, double xb) {    // scipy.optimize.brentq defaults
  const double xtol = 2e-12, rtol = 8.881784197001252e-16;
  double xpre = xa, xcur = xb, xblk = 0, fpre = f(xpre), fcur = f(xcur), fblk = 0, spre = 0, scur = 0;
  if (fpre == 0) return xpre;
  if (fcur == 0) return xcur;
  for (int i = 0; i < 100; ++i) {
    if (fpre != 0 && fcur != 0 && (std::signbit(fpre) != std::signbit(fcur))) { xblk = xpre; fblk = fpre; spre = scur = xcur - xpre; }
    if (std::fabs(fblk) < std::fabs(fcur)) { xpre = xcur; xcur = xblk; xblk = xpre; fpre = fcur; fcur = fblk; fblk = fpre; }
    const double delta = (xtol + rtol * std::fabs(xcur)) / 2, sbis = (xblk - xcur) / 2;
    if (fcur == 0 || std::fabs(sbis) < delta) return xcur;
    if (std::fabs(spre) > delta && std::fabs(fcur) < std::fabs(fpre)) {
      double stry;
      if (xpre == xblk) stry = -fcur * (xcur - xpre) / (fcur - fpre);
      else { const double dpre = (fpre - fcur) / (xpre - xcur), dblk = (fblk - fcur) / (xblk - xcur); stry = -fcur * (fblk * dblk - fpre * dpre) / (dblk * dpre * (fblk - fpre)); }
      if (2 * std::fabs(stry) < std::min(std::fabs(spre), 3 * std::fabs(sbis) - delta)) { spre = scur; scur = stry; } else { spre = sbis; scur = sbis; }
    } else { spre = sbis; scur = sbis; }
    xpre = xcur; fpre = fcur;
    xcur += std::fabs(scur) > delta ? scur : (sbis > 0 ? delta : -delta);
    fcur = f(xcur);
  }
  return xcur;
}
}  // namespace

icc_status icco_spline_error_weighting(void* h, int n, const double* times, const double* signal, double quality, double min_dt, double max_dt,
                                       double* dt_out, double* var_out, double* spectrum) {
  (void)h;
  if (n < 4) return ICC_ERR_INVALID_ARGUMENT;
  std::vector<double> tw_re(n), tw_im(n);
  for (int m = 0; m < n; ++m) { tw_re[m] = std::cos(-2.0 * M_PI * (double)m / (double)n); tw_im[m] = std::sin(-2.0 * M_PI * (double)m / (double)n); }
  std::vector<double> xhat(n, 0.0);
  for (int k = 1; k < n; ++k) {                    // S[:, 0] = 0 (sew.py:179)
    double s2 = 0.0;
    for (int ch = 0; ch < 3; ++ch) {
      double re = 0.0, im = 0.0; long long idx = 0;
      for (int j = 0; j < n; ++j) { const double x = signal[3 * (size_t)j + ch]; re += x * tw_re[idx]; im += x * tw_im[idx]; idx += k; if (idx >= n) idx -= n; }
      s2 += re * re + im * im;
    }
    xhat[k] = std::sqrt(1.0 / 3.0) * std::sqrt(s2);
  }
  if (spectrum) for (int k = 0; k < n; ++k) spectrum[k] = xhat[k];
  double mean_dt = 0.0; for (int i = 1; i < n; ++i) mean_dt += times[i] - times[i - 1]; mean_dt /= (double)(n - 1);
  const double sample_rate = 1.0 / mean_dt, d = 1.0 / sample_rate, fscale = 1.0 / ((double)n * d);
  if (!(min_dt > 0.0)) min_dt = 1.0 / sample_rate;
  if (!(max_dt > 0.0)) max_dt = ((double)n / 4.0) / sample_rate;
  double energy = 0.0; for (double v : xhat) energy += v * v; energy /= (double)n;
  const double max_remove = energy * (1.0 - quality);
  auto qf = [&](double dt) { return max_remove / sew_removed_energy(xhat, fscale, dt); };
  double dt = max_dt, found = 0.0;
  if (qf(dt) >= 1.0) found = dt;
  else {
    double step = max_dt * 0.5, best_q = 0.0, best_dt = dt;
    for (;;) {
      dt -= step; dt = std::max(dt, min_dt);
      const double q = qf(dt);
      if (q > 1.0) { found = sew_brentq([&](double x) { return qf(x) - 1.0; }, dt, max_dt); break; }
      step *= 0.5;
      if (q > best_q) { best_q = q; best_dt = dt; }
      if (dt <= min_dt) { found = best_dt; break; }
    }
  }
  *dt_out = found;
  *var_out = sew_removed_energy(xhat, fscale, found) / (double)n;
  return ICC_OK;
}

// ---- upstream row f4: camera intrinsic calibration (restates src/core/camera_calibrator.cc:131-389; TEST INFRASTRUCTURE) -----------
// Formulated the way theia::BundleAdjustViews poses it to Ceres (pyTheiaSfM@69c3d37, external): per view the extrinsic block
// [position (3) | angle-axis of R_cw (3)] with plain additive updates, one shared intrinsic block, residual
// theia::ReprojectionError = CameraToPixelCoordinates(intr, AngleAxisRotatePoint(aa, X - w * position)) - feature, Jacobians by
// forward-mode Jet<4> passes, ceres::HuberLoss(1.345) through Ceres' corrector (rho'' <= 0 => sqrt(rho') scaling), dense normal
// equations and dense Cholesky, Ceres' trust-region loop.  (The CUDA path uses right increments on a quaternion, closed-form
// Jacobians and per-view Schur elimination: same cost, same optimum, different route.)
}  // extern "C"
namespace {
template <class T> void angle_axis_rotate(const T* aa, const T* pt, T* out) {   // ceres/rotation.h AngleAxisRotatePoint
  const T theta2 = aa[0] * aa[0] + aa[1] * aa[1] + aa[2] * aa[2];
  if (jval(theta2) > 2.220446049250313e-16) {
    const T theta = jsqrt(theta2), ct = jcos(theta), st = jsin(theta);
    const T w[3] = {aa[0] / theta, aa[1] / theta, aa[2] / theta};
    const T wxp[3] = {w[1] * pt[2] - w[2] * pt[1], w[2] * pt[0] - w[0] * pt[2], w[0] * pt[1] - w[1] * pt[0]};
    const T tmp = (w[0] * pt[0] + w[1] * pt[1] + w[2] * pt[2]) * (T(1.0) - ct);
    for (int i = 0; i < 3; ++i) out[i] = pt[i] * ct + wxp[i] * st + w[i] * tmp;
  } else {
    const T wxp[3] = {aa[1] * pt[2] - aa[2] * pt[1], aa[2] * pt[0] - aa[0] * pt[2], aa[0] * pt[1] - aa[1] * pt[0]};
    for (int i = 0; i < 3; ++i) out[i] = pt[i] + wxp[i];
  }
}
template <class T> bool theia_reprojection_error(int model, const T* ext, const T* intr, const double* X4, const double* feat, T* res) {
  const T adj[3] = {T(X4[0]) - ext[0] * X4[3], T(X4[1]) - ext[1] * X4[3], T(X4[2]) - ext[2] * X4[3]};
  T rot[3], px[2];
  angle_axis_rotate(ext + 3, adj, rot);
  const bool ok = project<T>(model, intr, rot, px, true);
  res[0] = px[0] - feat[0]; res[1] = px[1] - feat[1];
  return ok;
}
struct CamCal {
  int model, nv; const int32_t* off; const int32_t* ids; const double* uv; const std::vector<double>* points;
  std::vector<double> ext;   // 6 per view
  double k[10];
  std::vector<int> active;
  double huber;
};
double camcal_cost(const CamCal& C, const std::vector<double>& ext, const double* k, std::vector<double>* view_err) {
  double cost = 0.0;
  for (int v : C.active) {
    double e = 0.0;
    for (int c = C.off[v]; c < C.off[v + 1]; ++c) {
      double r[2];
      if (!theia_reprojection_error<double>(C.model, &ext[6 * v], k, &(*C.points)[4 * (size_t)C.ids[c]], C.uv + 2 * c, r)) { cost += 1e10; e += 1e10; continue; }
      const double s2 = r[0] * r[0] + r[1] * r[1], rn = std::sqrt(s2);
      cost += rn <= C.huber ? 0.5 * s2 : C.huber * rn - 0.5 * C.huber * C.huber;
      e += rn;
    }
    if (view_err) (*view_err)[v] = C.off[v + 1] > C.off[v] ? e / double(C.off[v + 1] - C.off[v]) : 0.0;
  }
  return cost;
}
bool dense_cholesky_solve(int n, std::vector<double>& A, std::vector<double>& b) {   // A row-major SPD, overwritten by its factor
  for (int j = 0; j < n; ++j) {
    double d = A[(size_t)j * n + j];
    for (int m = 0; m < j; ++m) d -= A[(size_t)j * n + m] * A[(size_t)j * n + m];
    if (!(d > 0.0)) return false;
    const double l = std::sqrt(d);
    A[(size_t)j * n + j] = l;
    for (int i = j + 1; i < n; ++i) { double s2 = A[(size_t)i * n + j]; for (int m = 0; m < j; ++m) s2 -= A[(size_t)i * n + m] * A[(size_t)j * n + m]; A[(size_t)i * n + j] = s2 / l; }
  }
  for (int i = 0; i < n; ++i) { double s2 = b[i]; for (int m = 0; m < i; ++m) s2 -= A[(size_t)i * n + m] * b[m]; b[i] = s2 / A[(size_t)i * n + i]; }
  for (int i = n - 1; i >= 0; --i) { double s2 = b[i]; for (int m = i + 1; m < n; ++m) s2 -= A[(size_t)m * n + i] * b[m]; b[i] = s2 / A[(size_t)i * n + i]; }
  return true;
}
struct CamCalStage { int iterations = 0, termination = 0; double initial_cost = 0, final_cost = 0; };
// theia::BundleAdjustViews: which intrinsics are free (bit mask, Theia order) and whether the extrinsics are
CamCalStage camcal_bundle_adjust(CamCal& C, unsigned mask, bool pose_free, const icc_camcal_options& o) {
  CamCalStage R;
  const int na = (int)C.active.size();
  std::vector<int> kcol(10, -1); int n = pose_free ? 6 * na : 0;
  for (int a = 0; a < 10; ++a) if ((mask >> a) & 1u) kcol[a] = n++;
  if (n == 0 || na == 0) { R.termination = 3; return R; }
  std::vector<double> H((size_t)n * n), g(n), scale(n, 1.0), D(n);
  double x_cost = 0.0, radius = 1e4, decrease_factor = 2.0;
  int invalid = 0; bool ne_valid = false, first = true;
  typedef Jet<4> J4;
  auto build = [&]() {
    std::fill(H.begin(), H.end(), 0.0); std::fill(g.begin(), g.end(), 0.0);
    x_cost = 0.0;
    for (int s2 = 0; s2 < na; ++s2) {
      const int v = C.active[s2];
      for (int c = C.off[v]; c < C.off[v + 1]; ++c) {
        double J[2][16], r[2]; bool ok = true;
        for (int pass = 0; pass < 4; ++pass) {           // 16 ambient parameters in Jet<4> passes, like DynamicAutoDiff's strides
          J4 e[6], k[10], res[2];
          for (int i = 0; i < 6; ++i) { e[i] = J4(C.ext[6 * v + i]); const int gidx = i; if (gidx / 4 == pass) e[i].v[gidx % 4] = 1.0; }
          for (int i = 0; i < 10; ++i) { k[i] = J4(C.k[i]); const int gidx = 6 + i; if (gidx / 4 == pass) k[i].v[gidx % 4] = 1.0; }
          ok = theia_reprojection_error<J4>(C.model, e, k, &(*C.points)[4 * (size_t)C.ids[c]], C.uv + 2 * c, res) && ok;
          r[0] = res[0].a; r[1] = res[1].a;
          for (int d = 0; d < 4; ++d) { J[0][4 * pass + d] = res[0].v[d]; J[1][4 * pass + d] = res[1].v[d]; }
        }
        if (!ok) { x_cost += 1e10; continue; }
        const double sq = r[0] * r[0] + r[1] * r[1], rn = std::sqrt(sq);
        x_cost += rn <= C.huber ? 0.5 * sq : C.huber * rn - 0.5 * C.huber * C.huber;
        const double w = rn <= C.huber ? 1.0 : C.huber / rn;   // rho'
        int cols[16];
        for (int i = 0; i < 6; ++i) cols[i] = pose_free ? 6 * s2 + i : -1;
        for (int i = 0; i < 10; ++i) cols[6 + i] = kcol[i];
        for (int a = 0; a < 16; ++a) {
          if (cols[a] < 0) continue;
          g[cols[a]] += w * (J[0][a] * r[0] + J[1][a] * r[1]);
          for (int b = 0; b < 16; ++b) if (cols[b] >= 0) H[(size_t)cols[a] * n + cols[b]] += w * (J[0][a] * J[0][b] + J[1][a] * J[1][b]);
        }
      }
    }
  };
  for (int it = 0; it < o.max_num_iterations; ++it) {
    bool fresh = false;
    if (!ne_valid) { build(); ne_valid = true; fresh = true; }
    if (first) { for (int i = 0; i < n; ++i) scale[i] = 1.0 / (1.0 + std::sqrt(H[(size_t)i * n + i])); R.initial_cost = x_cost; }
    first = false;
    if (fresh) { double gm = 0; for (double v : g) gm = std::max(gm, std::fabs(v)); if (gm <= o.gradient_tolerance) { R.termination = 3; break; } }
    ++R.iterations;
    std::vector<double> A = H, b(n);
    for (int i = 0; i < n; ++i) {
      const double sc = scale[i];
      D[i] = std::min(std::max(sc * sc * H[(size_t)i * n + i], 1e-6), 1e32) / (radius * sc * sc);
      A[(size_t)i * n + i] += D[i]; b[i] = -g[i];
    }
    double model_change = 0.0; const bool solved = dense_cholesky_solve(n, A, b);
    if (solved) { double gd = 0, dd = 0; for (int i = 0; i < n; ++i) { gd += g[i] * b[i]; dd += D[i] * b[i] * b[i]; } model_change = 0.5 * (dd - gd); }
    if (!solved || !(model_change > 0.0)) { if (++invalid >= 5) { R.termination = 4; break; } radius /= decrease_factor; decrease_factor *= 2.0; continue; }
    invalid = 0;
    std::vector<double> ext = C.ext; double k[10]; memcpy(k, C.k, sizeof k);
    double step_sq = 0, x_sq = 0;
    for (int a = 0; a < 10; ++a) { x_sq += C.k[a] * C.k[a]; if (kcol[a] >= 0) { k[a] += b[kcol[a]]; step_sq += b[kcol[a]] * b[kcol[a]]; } }
    for (int s2 = 0; s2 < na; ++s2) { const int v = C.active[s2]; for (int i = 0; i < 6; ++i) { x_sq += C.ext[6 * v + i] * C.ext[6 * v + i]; if (pose_free) { ext[6 * v + i] += b[6 * s2 + i]; step_sq += b[6 * s2 + i] * b[6 * s2 + i]; } } }
    double cand_cost = camcal_cost(C, ext, k, nullptr);
    if (!std::isfinite(cand_cost)) cand_cost = 1.7976931348623157e308;
    if (std::sqrt(step_sq) <= o.parameter_tolerance * (std::sqrt(x_sq) + o.parameter_tolerance)) { R.termination = 2; break; }
    const double cost_change = x_cost - cand_cost;
    if (std::fabs(cost_change) <= o.function_tolerance * x_cost) { R.termination = 1; break; }
    const double rel = cost_change / model_change;
    if (rel > 1e-3) {
      C.ext = ext; memcpy(C.k, k, sizeof k); x_cost = cand_cost; ne_valid = false;
      radius = std::min(1e16, radius / std::max(1.0 / 3.0, 1.0 - std::pow(2.0 * rel - 1.0, 3)));
      decrease_factor = 2.0;
    } else { radius /= decrease_factor; decrease_factor *= 2.0; if (radius < 1e-32) { R.termination = 4; break; } }
  }
  R.final_cost = x_cost;
  return R;
}
double median_of(std::vector<double> v) {   // utils::MedianOfDoubleVec (src/utils/utils.cc:77-97)
  const size_t n = v.size(); std::sort(v.begin(), v.end());
  return n % 2 == 0 ? (v[n / 2 - 1] + v[n / 2]) / 2 : v[n / 2];
}
}  // namespace
extern "C" {

icc_status icco_calibrate_camera(void* h, int model, int W, int Hh, int nv, const int32_t* off, const int32_t* ids, const double* uv,
                                 const double* q_init, const double* p_init, const int32_t* init_valid, double focal_init, double distortion_init,
                                 const icc_camcal_options* options, double* intr_out, double* q_out, double* p_out, double* err_out, int32_t* used_out,
                                 icc_camcal_summary* summary) {
  Oracle& orc = *O(h);
  if (nv <= 0 || !off || !ids || !uv || camera_num_params(model) < 0 || orc.points.empty()) return ICC_ERR_INVALID_ARGUMENT;
  icc_camcal_options o; memset(&o, 0, sizeof o); if (options) o = *options;
  if (o.grid_size < 0.0) o.grid_size = 0.04;
  if (o.min_num_views <= 0) o.min_num_views = 10;
  if (o.max_num_iterations <= 0) o.max_num_iterations = 100;
  if (!(o.function_tolerance > 0.0)) o.function_tolerance = 1e-6;
  if (!(o.parameter_tolerance > 0.0)) o.parameter_tolerance = 1e-8;
  if (!(o.gradient_tolerance > 0.0)) o.gradient_tolerance = 1e-10;
  if (!(o.huber_width > 0.0)) o.huber_width = 1.345;
  if (!(o.max_view_error_stage1_px > 0.0)) o.max_view_error_stage1_px = 5.0;
  if (!(o.max_view_error_final_px > 0.0)) o.max_view_error_final_px = 2.0;
  icc_camcal_summary S; memset(&S, 0, sizeof S);
  const double cx0 = W / 2.0, cy0 = Hh / 2.0;
  const int np = (int)(orc.points.size() / 4);
  // ---- initial focal length (median of the per-view homography estimates) and poses (pinhole board poses) -------------------------
  std::vector<double> q0(4 * (size_t)nv), p0(3 * (size_t)nv); std::vector<int32_t> ok0(nv, 1);
  double f0 = focal_init;
  if (!(focal_init > 0.0)) {
    std::vector<double> fs;
    for (int v = 0; v < nv; ++v) {
      std::vector<PoseObs> ob;
      for (int c = off[v]; c < off[v + 1]; ++c) { if (ids[c] < 0 || ids[c] >= np) continue; const double* P = &orc.points[4 * (size_t)ids[c]]; ob.push_back({P[0] / P[3], P[1] / P[3], P[2] / P[3], uv[2 * c] - cx0, uv[2 * c + 1] - cy0, c}); }
      double zref, Hm[9];
      if (off[v + 1] - off[v] < 6 || ob.size() < 6 || !oracle_homography(ob, zref, Hm)) continue;
      const double a1 = Hm[0] * Hm[1] + Hm[3] * Hm[4], b1 = Hm[6] * Hm[7], a2 = Hm[0] * Hm[0] + Hm[3] * Hm[3] - Hm[1] * Hm[1] - Hm[4] * Hm[4], b2 = Hm[6] * Hm[6] - Hm[7] * Hm[7];
      const double den = b1 * b1 + b2 * b2; if (!(den > 0.0)) continue;
      const double f2 = -(a1 * b1 + a2 * b2) / den;
      if (f2 > 0.0 && std::isfinite(f2)) fs.push_back(std::sqrt(f2));
    }
    if (fs.empty()) { orc.err = "no view yields a focal length estimate"; return ICC_ERR_NUMERIC; }
    f0 = median_of(fs);
  }
  if (!q_init || !p_init) {
    const int m_save = orc.model, n_save = orc.n_intr, w_save = orc.width, h_save = orc.height; double k_save[10]; memcpy(k_save, orc.intr, sizeof k_save);
    const double kp[10] = {f0, 1.0, 0.0, cx0, cy0, 0.0, 0.0, 0.0, 0.0, 0.0};
    orc.model = 0; orc.n_intr = 7; memcpy(orc.intr, kp, sizeof kp); orc.width = W; orc.height = Hh;
    std::vector<double> e(nv);
    orc.pose_rel_tol = 1e-6;   // these poses only start the bundle adjustment
    icco_estimate_board_poses(h, nv, off, ids, uv, 1e300, 6, q0.data(), p0.data(), e.data(), ok0.data());
    orc.pose_rel_tol = 1e-15;
    orc.model = m_save; orc.n_intr = n_save; orc.width = w_save; orc.height = h_save; memcpy(orc.intr, k_save, sizeof k_save);
  } else {
    memcpy(q0.data(), q_init, 4 * (size_t)nv * sizeof(double)); memcpy(p0.data(), p_init, 3 * (size_t)nv * sizeof(double));
    if (init_valid) for (int v = 0; v < nv; ++v) ok0[v] = init_valid[v] != 0;
  }
  CamCal C; C.model = model; C.nv = nv; C.off = off; C.ids = ids; C.uv = uv; C.points = &orc.points; C.huber = o.huber_width;
  C.ext.resize(6 * (size_t)nv);
  for (int v = 0; v < nv; ++v) {
    const Qd qcw = so3_inv(qnormalized(Qd{q0[4 * v], q0[4 * v + 1], q0[4 * v + 2], q0[4 * v + 3]}));
    const Vd aa = so3_log(qcw);
    C.ext[6 * v] = p0[3 * v]; C.ext[6 * v + 1] = p0[3 * v + 1]; C.ext[6 * v + 2] = p0[3 * v + 2]; C.ext[6 * v + 3] = aa.x; C.ext[6 * v + 4] = aa.y; C.ext[6 * v + 5] = aa.z;
  }
  for (int v = 0; v < nv; ++v) if (ok0[v]) C.active.push_back(v);
  S.n_views_initialized = (int)C.active.size();
  // joint refinement of (focal length, division distortion, poses): what utils::initialize_radial_undistortion_camera hands the
  // reference for every non-pinhole model (:283-306)
  if ((!q_init || !p_init) && !(focal_init > 0.0) && model != 0 && model != 1) {
    C.model = 4;
    for (int i = 0; i < 10; ++i) C.k[i] = 0.0;
    C.k[0] = f0; C.k[1] = 1.0; C.k[2] = cx0; C.k[3] = cy0; C.k[4] = -1e-2 / ((double)W * W + (double)Hh * Hh);
    const CamCalStage pre = camcal_bundle_adjust(C, (1u << 0) | (1u << 4), true, o);
    S.init_iterations = pre.iterations;
    C.model = model;
    if (C.k[0] > 0.0 && std::isfinite(C.k[0])) { f0 = C.k[0]; if (model == 4) distortion_init = C.k[4]; }
  }
  S.focal_length_init = f0;
  {                                                                                         // grid filter (:313-325)
    std::vector<int> sel;
    for (int v : C.active) {
      bool take = true;
      for (int a : sel) { const double dx = C.ext[6 * v] - C.ext[6 * a], dy = C.ext[6 * v + 1] - C.ext[6 * a + 1], dz = C.ext[6 * v + 2] - C.ext[6 * a + 2]; if (std::sqrt(dx * dx + dy * dy + dz * dz) < o.grid_size) { take = false; break; } }
      if (take) sel.push_back(v);
    }
    C.active.swap(sel);
  }
  S.n_views_selected = (int)C.active.size();
  for (int i = 0; i < 10; ++i) C.k[i] = 0.0;
  C.k[0] = f0; C.k[1] = 1.0;
  const bool noskew = model == 3 || model == 4;
  if (noskew) { C.k[2] = cx0; C.k[3] = cy0; } else { C.k[3] = cx0; C.k[4] = cy0; }
  if (model == 4) C.k[4] = distortion_init;
  if (model == 3) C.k[4] = distortion_init != 0.0 ? distortion_init : 1e-3;
  if (model == 5) { C.k[5] = -0.25; C.k[6] = 0.5; }
  if (model == 6) { C.k[5] = 0.5; C.k[6] = 1.0; }
  auto bits = [](std::initializer_list<int> l) { unsigned m = 0; for (int i : l) m |= 1u << i; return m; };
  const unsigned focal = 1u, aspect = 2u, principal = noskew ? bits({2, 3}) : bits({3, 4});
  unsigned radial = 0, tangential = 0;
  switch (model) { case 0: radial = bits({5, 6}); break; case 1: radial = bits({5, 6, 7}); tangential = bits({8, 9}); break; case 2: radial = bits({5, 6, 7, 8}); break;
                   case 3: case 4: radial = bits({4}); break; default: radial = bits({5, 6}); break; }
  std::vector<double> verr(nv, 0.0);
  auto remove_views = [&](double max_err) { camcal_cost(C, C.ext, C.k, &verr); std::vector<int> keep; for (int v : C.active) if (!(verr[v] > max_err)) keep.push_back(v); C.active.swap(keep); };
  auto finish = [&](bool success) {
    camcal_cost(C, C.ext, C.k, &verr);
    for (int v = 0; v < nv; ++v) {
      const Qd qcw = so3_exp(Vd{C.ext[6 * v + 3], C.ext[6 * v + 4], C.ext[6 * v + 5]});
      q_out[4 * v] = -qcw.x; q_out[4 * v + 1] = -qcw.y; q_out[4 * v + 2] = -qcw.z; q_out[4 * v + 3] = qcw.w;
      for (int d = 0; d < 3; ++d) p_out[3 * v + d] = C.ext[6 * v + d];
      used_out[v] = 0; if (err_out) err_out[v] = 0.0;
    }
    double tot = 0; for (int v : C.active) { used_out[v] = 1; if (err_out) err_out[v] = verr[v]; tot += verr[v]; }
    for (int i = 0; i < 10; ++i) intr_out[i] = C.k[i];
    S.success = success ? 1 : 0; S.n_views_used = (int)C.active.size(); S.final_reproj_error = C.active.empty() ? 0.0 : tot / double(C.active.size());
    if (summary) *summary = S;
    return ICC_OK;
  };
  if ((int)C.active.size() < o.min_num_views) return finish(false);
  CamCalStage st = camcal_bundle_adjust(C, focal | (model != 0 ? radial : 0u), true, o);
  S.iterations[0] = st.iterations; S.termination[0] = st.termination; S.initial_cost = st.initial_cost; S.final_cost[0] = st.final_cost;
  remove_views(o.max_view_error_stage1_px);
  st = camcal_bundle_adjust(C, principal, false, o);
  S.iterations[1] = st.iterations; S.termination[1] = st.termination; S.final_cost[1] = st.final_cost;
  if ((int)C.active.size() < o.min_num_views) return finish(false);
  st = camcal_bundle_adjust(C, principal | focal | aspect | (model == 0 ? radial : 0u) | (model == 1 ? tangential : 0u), true, o);
  S.iterations[2] = st.iterations; S.termination[2] = st.termination; S.final_cost[2] = st.final_cost;
  remove_views(o.max_view_error_final_px);
  if ((int)C.active.size() < o.min_num_views) return finish(false);
  if (o.optimize_board_points) {   // camera_calibrator.cc:207-216: BundleAdjustTracks (cameras constant), then BundleAdjustViews once more
    std::vector<double> qv(4 * (size_t)nv), pv(3 * (size_t)nv); std::vector<char> in_active(nv, 0), take(std::max(1, off[nv]), 0);
    for (int v : C.active) { in_active[v] = 1; for (int c = off[v]; c < off[v + 1]; ++c) take[c] = 1; }
    for (int v = 0; v < nv; ++v) {
      const Qd qcw = so3_exp(Vd{C.ext[6 * v + 3], C.ext[6 * v + 4], C.ext[6 * v + 5]});
      qv[4 * v] = -qcw.x; qv[4 * v + 1] = -qcw.y; qv[4 * v + 2] = -qcw.z; qv[4 * v + 3] = qcw.w;
      for (int d = 0; d < 3; ++d) pv[3 * v + d] = C.ext[6 * v + d];
    }
    S.n_points_optimized = oracle_refine_points(orc, false, model, C.k, nv, off, ids, uv, qv.data(), pv.data(), [&](int c) { return take[c] != 0; }, 1, o.huber_width);
    const int it3 = S.iterations[2];
    st = camcal_bundle_adjust(C, principal | focal | aspect | (model == 0 ? radial : 0u) | (model == 1 ? tangential : 0u), true, o);
    S.iterations[2] = it3 + st.iterations; S.termination[2] = st.termination; S.final_cost[2] = st.final_cost;
  }
  return finish(true);
}

// python/get_imu_biases.py:36-53 (TEST INFRASTRUCTURE): means by plain sequential sums, gravity removed on the dominant accelerometer axis
icc_status icco_estimate_imu_biases(void* h, int n, const double* acc, const double* gyr, double gravity_const, double accl_bias[3], double gyro_bias[3]) {
  long double sa[3] = {0, 0, 0}, sg[3] = {0, 0, 0};
  for (int i = 0; i < n; ++i) for (int d = 0; d < 3; ++d) { sa[d] += acc[3 * i + d]; sg[d] += gyr[3 * i + d]; }
  double ma[3], mg[3]; for (int d = 0; d < 3; ++d) { ma[d] = (double)(sa[d] / n); mg[d] = (double)(sg[d] / n); }
  int ax = 0; for (int d = 1; d < 3; ++d) if (std::fabs(ma[d]) > std::fabs(ma[ax])) ax = d;
  const float g32 = (float)(gravity_const * (ma[ax] > 0.0 ? 1.0 : (ma[ax] < 0.0 ? -1.0 : 0.0)));
  for (int d = 0; d < 3; ++d) { accl_bias[d] = ma[d] - (d == ax ? (double)g32 : 0.0); gyro_bias[d] = mg[d]; }
  return ICC_OK;
}

int icco_project(int model, const double* intr, const double* p3, double* px, int dispatch_fov) { return project<double>(model, intr, p3, px, dispatch_fov != 0) ? 1 : 0; }

// n camera-frame points through project<T> (FOV dispatched, as the CUDA calibration does) with Jet<4> passes over the 13 inputs
// [point (3) | intrinsics (10)]: pixel px[2n], point Jacobian Jp[6n] (2 x 3 row-major per point), intrinsic Jacobian Jk[20n]
// (2 x 10 row-major), ok[n].  Returns the number of points that project.
int icco_project_jacobian(int model, const double* intr, int n, const double* p3, double* px, double* Jp, double* Jk, int32_t* ok) {
  typedef Jet<4> J4;
  int n_ok = 0;
  for (int i = 0; i < n; ++i) {
    bool good = true;
    for (int pass = 0; pass < 4; ++pass) {
      J4 p[3], k[10], r[2];
      for (int a = 0; a < 3; ++a) { p[a] = J4(p3[3 * i + a]); if (a / 4 == pass) p[a].v[a % 4] = 1.0; }
      for (int a = 0; a < 10; ++a) { k[a] = J4(intr[a]); if ((3 + a) / 4 == pass) k[a].v[(3 + a) % 4] = 1.0; }
      good = project<J4>(model, k, p, r, true) && good;
      for (int row = 0; row < 2; ++row) {
        px[2 * i + row] = r[row].a;
        for (int d = 0; d < 4; ++d) {
          const int col = 4 * pass + d;
          if (col < 3) Jp[6 * i + 3 * row + col] = r[row].v[d];
          else if (col < 13) Jk[20 * i + 10 * row + col - 3] = r[row].v[d];
        }
      }
    }
    ok[i] = good ? 1 : 0; n_ok += good;
  }
  return n_ok;
}

}  // extern "C"
