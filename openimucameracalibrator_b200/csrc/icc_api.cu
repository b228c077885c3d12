// C-ABI + host logic of the B200 calibration solver (see include/icc_b200.h for the boundary contract).
//
// Host side mirrors, in its own structure, what the reference does on one thread before/around ceres::Solve:
//   ImuCameraCalibrator::BatchInitSpline / InitializeGravity / Optimize   src/core/imu_camera_calibrator.cc:21-168
//   SplineTrajectoryEstimator::SetTimes / InitBiasSplines / BatchInitSO3R3VisPoses / Add*Measurement / CalcTimes /
//   SetFixedParams / Optimize / getters       include/OpenCameraCalibrator/core/spline_trajectory_estimator.impl.h
//   InterpolateQuaternions / InterpolateVector3d                           src/utils/utils.cc:194-261
// Everything numerical per LM iteration runs on the GPU (icc_eval.cu, icc_solver.cu); the host only sequences launches
// and applies the trust-region accept/reject logic to a few scalars read back per iteration.  There is no CPU fallback.
#include "../../include/icc_b200.h"
#include "icc_camera.cuh"
#include "icc_kernels.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

using namespace icc;

namespace {

constexpr double S_TO_NS = 1e9, NS_TO_S = 1e-9;

// Process-wide caching allocator for device blocks: a calibration job allocates ~30 buffers and the CUDA driver's
// cudaMalloc / cudaFree cost 0.1-1 ms each, which would dominate the whole-job wall clock of back-to-back jobs.
// Freed blocks are kept (per device) and handed out again best-fit; icc_trim_device_cache() returns them to the driver.
struct BlockCache {
  std::mutex mu;
  std::multimap<size_t, std::pair<int, void*>> free_blocks;   // bytes -> (device, ptr)
  cudaError_t get(size_t bytes, void** out) {
    int dev = 0; cudaGetDevice(&dev);
    {
      std::lock_guard<std::mutex> lk(mu);
      for (auto it = free_blocks.lower_bound(bytes); it != free_blocks.end() && it->first <= 2 * bytes + 4096; ++it)
        if (it->second.first == dev) { *out = it->second.second; free_blocks.erase(it); return cudaSuccess; }
    }
    return cudaMalloc(out, bytes);
  }
  void put(size_t bytes, void* p) { int dev = 0; cudaGetDevice(&dev); std::lock_guard<std::mutex> lk(mu); free_blocks.emplace(bytes, std::make_pair(dev, p)); }
  void trim() { std::lock_guard<std::mutex> lk(mu); for (auto& kv : free_blocks) { cudaSetDevice(kv.second.first); cudaFree(kv.second.second); } free_blocks.clear(); }
};
BlockCache& block_cache() { static BlockCache* c = new BlockCache(); return *c; }   // intentionally leaked: outlives every handle

template <class T>
struct DevBuf {
  T* p = nullptr; size_t n = 0, cap_bytes = 0;
  ~DevBuf() { release(); }
  void release() { if (p) block_cache().put(cap_bytes, p); p = nullptr; n = 0; cap_bytes = 0; }
  cudaError_t alloc(size_t count) {
    const size_t bytes = (count * sizeof(T) + 255) / 256 * 256;
    if (p && cap_bytes >= bytes) { n = count; return cudaSuccess; }
    release(); n = count; if (!count) return cudaSuccess;
    void* q = nullptr; cudaError_t e = block_cache().get(bytes, &q); if (e != cudaSuccess) { n = 0; return e; }
    p = static_cast<T*>(q); cap_bytes = bytes; return cudaSuccess;
  }
  cudaError_t upload(const std::vector<T>& v) { cudaError_t e = alloc(v.size()); if (e != cudaSuccess || v.empty()) return e; return cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice); }
};

// Host staging of the large measurement arrays (corners, IMU samples): page-locked blocks from a process-wide cache (the first
// job pays cudaHostAlloc, later ones reuse), so that the uploads of BatchInitSpline are asynchronous DMA transfers that overlap the
// host assembly.  Host-only handles (and a failed cudaHostAlloc) use ordinary memory; the copies then stage through the driver.
struct PinnedCache {
  std::mutex mu;
  std::multimap<size_t, void*> free_blocks;
  void* get(size_t bytes, size_t* cap) {
    {
      std::lock_guard<std::mutex> lk(mu);
      auto it = free_blocks.lower_bound(bytes);
      if (it != free_blocks.end() && it->first <= 2 * bytes + 4096) { void* q = it->second; *cap = it->first; free_blocks.erase(it); return q; }
    }
    void* q = nullptr;
    if (cudaHostAlloc(&q, bytes, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    *cap = bytes; return q;
  }
  void put(size_t bytes, void* q) { std::lock_guard<std::mutex> lk(mu); free_blocks.emplace(bytes, q); }
  void trim() { std::lock_guard<std::mutex> lk(mu); for (auto& kv : free_blocks) cudaFreeHost(kv.second); free_blocks.clear(); }
};
PinnedCache& pinned_cache() { static PinnedCache* c = new PinnedCache(); return *c; }

template <class T>
struct HostBuf {
  T* p = nullptr; size_t n = 0, cap_bytes = 0; bool pinned = false;
  HostBuf() = default; HostBuf(const HostBuf&) = delete; HostBuf& operator=(const HostBuf&) = delete;
  ~HostBuf() { release(); }
  void release() { if (p) { if (pinned) pinned_cache().put(cap_bytes, p); else free(p); } p = nullptr; n = 0; cap_bytes = 0; pinned = false; }
  void resize(size_t count, bool want_pinned) {    // contents are NOT preserved
    const size_t bytes = std::max<size_t>(256, (count * sizeof(T) + 255) / 256 * 256);
    if (!(p && cap_bytes >= bytes && (pinned || !want_pinned))) {
      release();
      if (want_pinned) { size_t cap = 0; p = static_cast<T*>(pinned_cache().get(bytes, &cap)); if (p) { pinned = true; cap_bytes = cap; } }
      if (!p) { p = static_cast<T*>(malloc(bytes)); cap_bytes = bytes; pinned = false; }
    }
    n = count;
  }
  void assign(const T* src, size_t count, bool want_pinned) { resize(count, want_pinned); if (count) memcpy(p, src, count * sizeof(T)); }   // (splitting this copy over threads was measured: the later DMA / reads get slower by more than the copy gains)
  void clear() { n = 0; }
  T* data() { return p; } const T* data() const { return p; }
  size_t size() const { return n; } bool empty() const { return n == 0; }
  T& operator[](size_t i) { return p[i]; } const T& operator[](size_t i) const { return p[i]; }
  const T* begin() const { return p; } const T* end() const { return p + n; }
};

// Bump allocator over one page-locked block: the many small arrays a job uploads (frame tables, work lists, knots) are staged here
// and copied asynchronously, instead of one blocking pageable cudaMemcpy each.  reset() only after the stream has drained.
struct PinnedArena {
  HostBuf<unsigned char> buf; size_t used = 0;
  void reset(size_t capacity, bool pin) { if (buf.size() < capacity) buf.resize(capacity, pin); used = 0; }
  void* take(size_t bytes) { const size_t o = (used + 255) & ~size_t(255); if (o + bytes > buf.size()) return nullptr; used = o + bytes; return buf.data() + o; }
};

struct StateBufs {
  DevBuf<double4> so3, r3, ba, bg; DevBuf<double> glob;
  DevBuf<double4> pts, board; DevBuf<double> pjac;   // board points of the state (icc_points.cu)
  DeviceState view() const { DeviceState s; s.so3 = so3.p; s.r3 = r3.p; s.ba = ba.p; s.bg = bg.p; s.glob = glob.p; s.pts = pts.p; s.board = board.p; s.pjac = pjac.p; return s; }
};

struct FrameHost { double t_s; int c0, c1; int s_so3, s_r3; double u_so3, u_r3; };

}  // namespace

struct icc_handle {
  std::string err = "";
  int device = -1;
  icc_solver_options opt;
  // ---- raw inputs -------------------------------------------------------------------------------------------
  int model = -1, n_intr = 0, width = 0, height = 0; double intr[10] = {0};
  std::vector<double> points;
  std::vector<double> frame_t; std::vector<int> corner_off; HostBuf<int> point_ids; HostBuf<double> uv; std::vector<double> q_wc, p_wc;
  HostBuf<double> imu_t, imu_acc, imu_gyr;
  int id_lo = 0, id_hi = -1;                 // range of the corner point ids (found while set_frames copies them)
  // Page-locked caller buffers (cudaHostAlloc / cudaHostRegister / torch pin_memory): set_frames / set_imu send the big arrays straight to the
  // device by DMA and wait for it, instead of staging them through a host copy first; the host then only keeps what it reads (time stamps,
  // offsets, poses) and fetches the rest back from the device in the rare paths that gather (unsorted streams, non-contiguous shards).
  bool frames_dev = false, imu_dev = false; size_t n_corners_in = 0, n_imu_in = 0;
  bool imu_sorted = false;                   // imu_t is non-decreasing (found while set_imu copies it)
  int shard_rank = 0, shard_world = 1;
  icc_allreduce_fn allreduce = nullptr; void* allreduce_user = nullptr;
  icc_comm* comm = nullptr;                  // borrowed NCCL communicator (icc_set_comm): the native cross-rank sum
  // ---- assembled problem (host) -----------------------------------------------------------------------------
  bool initialised = false;
  icc_init_params ip;
  int64_t dt_so3_ns = 0, dt_r3_ns = 0, dt_ba_ns = 0, dt_bg_ns = 0, start_ns = 0, end_ns = 0;
  double t0_s = 0, tend_s = 0, max_ba = 1.0, max_bg = 0.1;
  std::vector<double> so3, r3, ba, bg;       // host mirror of the state (4/3/3/3 doubles per knot)
  double glob[G_COUNT] = {0};
  std::vector<FrameHost> frames;             // frames in the problem (this shard)
  std::vector<double> used_uv; std::vector<int> used_pid;   // gathered corners -- only when the used frames are not one contiguous run
  bool used_contig = false; int used_c0 = 0, used_n = 0;    // ... otherwise corners [used_c0, used_c0 + used_n) of uv / point_ids are used in place
  bool imu_contig = false; int imu_src0 = 0;                // same for the accelerometer / gyroscope samples
  std::vector<double> imu_used_t, imu_used_acc, imu_used_gyr; HostBuf<int64_t> imu_used_st;
  size_t n_imu_used = 0;                     // kept samples; imu_used_t / imu_used_st are only materialised off the sorted fast path (imu_lazy == false)
  bool imu_lazy = false;                     // sorted fast path: kept samples = imu_t[imu_src0 .. +n_imu_used) + time offset, relative times derived on the device
  std::vector<ImuCell> cells;
  int dropped_frames = 0, dropped_imu = 0;
  // ---- device ---------------------------------------------------------------------------------------------------
  cudaStream_t stream = nullptr;
  EvalAux aux{};            // second stream + fork/join events: vision and IMU kernels of one evaluation run concurrently
  bool aux_ok = false;
  int sm_count = 148;
  StateBufs st[2]; int cur = 0;
  HostBuf<unsigned char> small_pinned; DevBuf<int> d_idrange;
  void* arena_small(size_t bytes) { if (small_pinned.size() < bytes) small_pinned.resize(std::max<size_t>(bytes, 256), true); return small_pinned.pinned ? small_pinned.data() : nullptr; }
  DevBuf<double2> d_uv_all; DevBuf<int> d_pid_all; DevBuf<double> d_acc_all, d_gyr_all;   // complete input arrays (frames_dev / imu_dev)
  DevBuf<double4> d_board; DevBuf<int> d_f_off, d_f_s_so3, d_f_s_r3, d_pid; DevBuf<double> d_f_u_so3, d_f_u_r3; DevBuf<double2> d_uv;
  DevBuf<double> d_view_t, d_view_q, d_view_p;   // per-view pose priors in time order (knot initialisation kernel)
  DevBuf<VisFrame> d_vframes; DevBuf<VisItem> d_vitems;
  DevBuf<ImuCellP> d_icells; DevBuf<VisItem> d_iitems;
  DevBuf<double> d_imu_traw; DevBuf<VisionWork> d_vwork; DevBuf<int64_t> d_imu_t; DevBuf<double> d_imu_acc, d_imu_gyr; DevBuf<ImuCell> d_cells, d_iwork;
  DevBuf<int> d_so3_col, d_r3_col, d_ba_col, d_bg_col;
  DevBuf<double> d_ne, d_scale, d_ws, d_delta, d_scal, d_res;
  PinnedArena arena;        // staging of the small uploads of BatchInitSpline
  DeviceProblem P;
  bool state_dirty_host = false;   // device state newer than host mirror
  bool glob_host_current = false;  // ... but the small block of globals (T_i_c, gravity, line delay, intrinsics) was already read back
  bool knots_dirty_host = false;   // only the spline knots are newer on the device (device-side initialisation): globals / biases on the host are current
  // ---- active set ------------------------------------------------------------------------------------------------
  int cur_flags = -1;
  std::vector<int> so3_col, r3_col, ba_col, bg_col;   // solver index of first dim or -1
  int col_tic = -1, col_g = -1, col_ld = -1;
  int n_tan = 0;
  std::vector<int> perm;           // canonical tangent index -> solver index
  int launches_at_start = 0;
};

namespace {

icc_status fail(icc_handle* h, icc_status s, const std::string& m) { if (h) h->err = m; return s; }
// ICC_TRACE_PHASES=1: host wall clock between the marked points of a call, to stderr (diagnosis only; synchronises the stream at every mark)
struct PhaseTrace {
  bool on; cudaStream_t st; std::chrono::steady_clock::time_point t;
  PhaseTrace(cudaStream_t s) : on(getenv("ICC_TRACE_PHASES") != nullptr), st(s), t(std::chrono::steady_clock::now()) {}
  void lap(const char* what) {
    if (!on) return;
    const auto a = std::chrono::steady_clock::now(); if (st) cudaStreamSynchronize(st); const auto b = std::chrono::steady_clock::now();
    fprintf(stderr, "[icc phase] %-28s %8.3f ms host + %7.3f ms stream drain\n", what, std::chrono::duration<double, std::milli>(a - t).count(), std::chrono::duration<double, std::milli>(b - a).count());
    t = std::chrono::steady_clock::now();
  }
};
#define CU(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return fail(h, ICC_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); } while (0)
#define NEED_DEVICE() do { if (h->device < 0) return fail(h, ICC_ERR_NO_DEVICE, "no CUDA device bound to this handle (host-only handle): compute entry points are unavailable"); } while (0)

Q4 qn(const double* q) { return qnormalized(q4(q[0], q[1], q[2], q[3])); }

// CalcTimes (impl.h:763-788)
bool calc_times(int64_t sensor_ns, int64_t start_ns, int64_t dt_ns, size_t nr_knots, int N, double& u, int64_t& s) {
  const int64_t st = sensor_ns - start_ns;
  if (st < 0) { u = 0.0; return false; }
  s = st / dt_ns;
  if (s < 0) return false;
  if (size_t(s + N) > nr_knots) return false;
  u = double(st % dt_ns) / double(dt_ns);
  return true;
}

// CSR by board point of the corners selected by `take(c)`: pt_off[np + 1], pt_obs[...] (counting sort, stable in corner order)
template <class F>
void build_point_adjacency(int np, int nc, const int32_t* ids, F take, std::vector<int>& pt_off, std::vector<int>& pt_obs) {
  pt_off.assign(np + 1, 0);
  for (int c = 0; c < nc; ++c) if (take(c)) ++pt_off[ids[c] + 1];
  for (int p = 0; p < np; ++p) pt_off[p + 1] += pt_off[p];
  pt_obs.resize(pt_off[np]);
  std::vector<int> fill(pt_off.begin(), pt_off.end() - 1);
  for (int c = 0; c < nc; ++c) if (take(c)) pt_obs[fill[ids[c]]++] = c;
}

size_t nearest_index(double t, const std::vector<double>& ts, double& dist_out) {   // utils.cc:194-212
  // FindClosestTimestamp is a linear scan keeping the FIRST strict minimum of |t - ts[i]|; on the time-sorted, distinct
  // view timestamps used here the same index is found by bisection + comparison of the two neighbours.
  const size_t n = ts.size();
  size_t hi = std::lower_bound(ts.begin(), ts.end(), t) - ts.begin();   // first ts >= t
  size_t idx;
  if (hi == 0) idx = 0;
  else if (hi == n) idx = n - 1;
  else idx = (std::fabs(t - ts[hi - 1]) <= std::fabs(t - ts[hi])) ? hi - 1 : hi;   // tie -> earlier index, like the scan
  dist_out = std::fabs(t - ts[idx]);
  return idx;
}

void quat_slerp(const double* a, const double* b, double t, double* o) {   // Eigen::Quaternion::slerp semantics (utils.cc:234)
  const double thresh = 1.0 - 2.220446049250313e-16;
  const double d = a[0] * b[0] + a[1] * b[1] + a[2] * b[2] + a[3] * b[3], ad = std::fabs(d);
  double s0, s1;
  if (ad >= thresh) { s0 = 1.0 - t; s1 = t; }
  else { const double th = std::acos(ad), sth = std::sin(th); s0 = std::sin((1.0 - t) * th) / sth; s1 = std::sin(t * th) / sth; }
  if (d < 0) s1 = -s1;
  for (int i = 0; i < 4; ++i) o[i] = s0 * a[i] + s1 * b[i];
}

struct Pose { Q4 q; V3 t; };
Pose pose_mul(const Pose& a, const Pose& b) { return {qnormalized(qmul(a.q, b.q)), a.t + qrot(a.q, b.t)}; }
Pose pose_inv(const Pose& a) { const Q4 qi = qnormalized(qconj(a.q)); return {qi, qrot(qi, -a.t)}; }

std::vector<double4> pad4(const std::vector<double>& v, int dim) {
  const size_t n = v.size() / dim; std::vector<double4> o(n);
  for (size_t i = 0; i < n; ++i) o[i] = make_double4(v[dim * i], v[dim * i + 1], v[dim * i + 2], dim == 4 ? v[dim * i + 3] : 0.0);
  return o;
}

// v -> d through the handle's staging arena (asynchronous on the handle's stream); falls back to the blocking copy when the arena is full
template <class T>
cudaError_t upload_staged(icc_handle* h, DevBuf<T>& d, const std::vector<T>& v) {
  cudaError_t e = d.alloc(v.size()); if (e != cudaSuccess || v.empty()) return e;
  const size_t bytes = v.size() * sizeof(T);
  void* stage = h->arena.take(bytes);
  if (!stage) return cudaMemcpy(d.p, v.data(), bytes, cudaMemcpyHostToDevice);
  memcpy(stage, v.data(), bytes);
  return cudaMemcpyAsync(d.p, stage, bytes, cudaMemcpyHostToDevice, h->stream);
}

// board points of state `which`: homogeneous vectors up, de-homogenised copy + local Jacobians derived on the device
icc_status upload_points(icc_handle* h, int which, bool staged) {
  StateBufs& s = h->st[which];
  const size_t np = h->points.size() / 4;
  if (!np) return ICC_OK;
  CU(s.board.alloc(np)); CU(s.pjac.alloc(12 * np));
  if (staged) { CU(upload_staged(h, s.pts, pad4(h->points, 4))); }
  else { CU(cudaStreamSynchronize(h->stream)); CU(s.pts.upload(pad4(h->points, 4))); }
  launch_points_prepare((int)np, s.pts.p, s.board.p, s.pjac.p, h->stream);
  if (!staged) CU(cudaStreamSynchronize(h->stream));
  return ICC_OK;
}

bool host_is_pinned(const void* p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return at.type == cudaMemoryTypeHost;
}
// host copies of the arrays that went straight to the device, for the paths that gather on the host
icc_status ensure_host_corners(icc_handle* h) {
  if (!h->frames_dev || h->uv.size() == 2 * h->n_corners_in) return ICC_OK;
  h->uv.resize(2 * h->n_corners_in, true); h->point_ids.resize(h->n_corners_in, true);
  CU(cudaStreamSynchronize(h->stream));
  if (h->n_corners_in) { CU(cudaMemcpy(h->uv.data(), h->d_uv_all.p, h->n_corners_in * sizeof(double2), cudaMemcpyDeviceToHost)); CU(cudaMemcpy(h->point_ids.data(), h->d_pid_all.p, h->n_corners_in * sizeof(int), cudaMemcpyDeviceToHost)); }
  return ICC_OK;
}
icc_status ensure_host_imu(icc_handle* h) {
  if (!h->imu_dev || h->imu_acc.size() == 3 * h->n_imu_in) return ICC_OK;
  h->imu_acc.resize(3 * h->n_imu_in, true); h->imu_gyr.resize(3 * h->n_imu_in, true);
  CU(cudaStreamSynchronize(h->stream));
  if (h->n_imu_in) { CU(cudaMemcpy(h->imu_acc.data(), h->d_acc_all.p, 3 * h->n_imu_in * sizeof(double), cudaMemcpyDeviceToHost)); CU(cudaMemcpy(h->imu_gyr.data(), h->d_gyr_all.p, 3 * h->n_imu_in * sizeof(double), cudaMemcpyDeviceToHost)); }
  return ICC_OK;
}

icc_status upload_state(icc_handle* h, int which, bool staged = false) {
  StateBufs& s = h->st[which];
  std::vector<double> g(h->glob, h->glob + G_COUNT);
  { icc_status r = upload_points(h, which, staged); if (r != ICC_OK) return r; }
  if (staged) {
    CU(upload_staged(h, s.so3, pad4(h->so3, 4))); CU(upload_staged(h, s.r3, pad4(h->r3, 3))); CU(upload_staged(h, s.ba, pad4(h->ba, 3))); CU(upload_staged(h, s.bg, pad4(h->bg, 3)));
    CU(upload_staged(h, s.glob, g));
    return ICC_OK;
  }
  CU(cudaStreamSynchronize(h->stream));   // a staged upload of the same buffers may still be in flight
  CU(s.so3.upload(pad4(h->so3, 4))); CU(s.r3.upload(pad4(h->r3, 3))); CU(s.ba.upload(pad4(h->ba, 3))); CU(s.bg.upload(pad4(h->bg, 3)));
  CU(s.glob.upload(g));
  return ICC_OK;
}

icc_status sync_state_to_host(icc_handle* h) {
  if (!(h->state_dirty_host || h->knots_dirty_host) || h->device < 0) return ICC_OK;
  const StateBufs& s = h->st[h->cur];
  auto pull = [&](const DevBuf<double4>& d, std::vector<double>& v, int dim) -> cudaError_t {
    std::vector<double4> tmp(d.n);
    if (d.n) { cudaError_t e = cudaMemcpy(tmp.data(), d.p, d.n * sizeof(double4), cudaMemcpyDeviceToHost); if (e != cudaSuccess) return e; }
    for (size_t i = 0; i < d.n; ++i) { v[dim * i] = tmp[i].x; v[dim * i + 1] = tmp[i].y; v[dim * i + 2] = tmp[i].z; if (dim == 4) v[dim * i + 3] = tmp[i].w; }
    return cudaSuccess;
  };
  CU(cudaStreamSynchronize(h->stream));
  CU(pull(s.so3, h->so3, 4)); CU(pull(s.r3, h->r3, 3)); CU(pull(s.ba, h->ba, 3)); CU(pull(s.bg, h->bg, 3));
  CU(cudaMemcpy(h->glob, s.glob.p, G_COUNT * sizeof(double), cudaMemcpyDeviceToHost));
  if (h->state_dirty_host && s.pts.n * 4 == h->points.size()) CU(pull(s.pts, h->points, 4));
  h->state_dirty_host = false; h->knots_dirty_host = false;
  return ICC_OK;
}

// getters of the globals (T_i_c, gravity, line delay, ...) after a solve: 25 doubles instead of every knot
icc_status sync_globals_to_host(icc_handle* h) {
  if (!h->state_dirty_host || h->glob_host_current || h->device < 0) return ICC_OK;
  CU(cudaMemcpyAsync(h->glob, h->st[h->cur].glob.p, G_COUNT * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->glob_host_current = true;
  return ICC_OK;
}

icc_status push_state_to_device(icc_handle* h) {
  if (h->device < 0 || !h->initialised) return ICC_OK;
  icc_status s = upload_state(h, h->cur);
  h->state_dirty_host = false; h->knots_dirty_host = false;
  return s;
}

// Active set (SetFixedParams, impl.h:92-252) -> column maps in SOLVER order: spline knots sorted by knot time (SO3 before
// R3 on ties) form the banded part; T_i_c, gravity, line delay and bias knots form the border.
icc_status configure(icc_handle* h, int flags) {
  if ((flags & ICC_FLAG_POINTS) && (flags & ICC_FLAG_CAM_INTRINSICS)) return fail(h, ICC_ERR_UNSUPPORTED, "POINTS together with CAM_INTRINSICS (an extension flag of this library) is not supported");
  if (h->cur_flags == flags) return ICC_OK;
  const int nso3 = (int)h->so3.size() / 4, nr3 = (int)h->r3.size() / 3, nba = (int)h->ba.size() / 3, nbg = (int)h->bg.size() / 3;
  const bool spline = flags & ICC_FLAG_SPLINE, tic = flags & ICC_FLAG_T_I_C, grav = flags & ICC_FLAG_GRAVITY_DIR;
  const bool ld = (flags & ICC_FLAG_CAM_LINE_DELAY) && h->ip.init_line_delay_s != 0.0;
  const bool ab = flags & (ICC_FLAG_ACC_BIAS | ICC_FLAG_IMU_BIASES), gb = flags & (ICC_FLAG_GYR_BIAS | ICC_FLAG_IMU_BIASES);
  const bool intr = flags & ICC_FLAG_IMU_INTRINSICS, cam_intr = flags & ICC_FLAG_CAM_INTRINSICS, toff = flags & ICC_FLAG_TIME_OFFSET;
  const int npts = (int)(h->points.size() / 4);
  const bool pts = (flags & ICC_FLAG_POINTS) && npts > 0;      // every track a view sees (impl.h:136-152); points no view sees get zero columns
  // canonical offsets
  int n = 0;
  const int c_so3 = spline ? n : -1; if (spline) n += 3 * nso3;
  const int c_r3 = spline ? n : -1; if (spline) n += 3 * nr3;
  const int c_tic = tic ? n : -1; if (tic) n += 6;
  const int c_g = grav ? n : -1; if (grav) n += 3;
  const int c_ld = ld ? n : -1; if (ld) n += 1;
  const int c_ba = ab ? n : -1; if (ab) n += 3 * nba;
  const int c_bg = gb ? n : -1; if (gb) n += 3 * nbg;
  const int c_ai = intr ? n : -1; if (intr) n += 6;
  const int c_gi = intr ? n : -1; if (intr) n += 9;
  const int c_ci = cam_intr ? n : -1; if (cam_intr) n += h->n_intr;
  const int c_to = toff ? n : -1; if (toff) n += 1;
  const int c_pts = pts ? n : -1; if (pts) n += 3 * npts;
  h->n_tan = n;
  h->so3_col.assign(nso3, -1); h->r3_col.assign(nr3, -1); h->ba_col.assign(nba, -1); h->bg_col.assign(nbg, -1);
  int pos = 0;
  if (spline) {
    int i = 0, j = 0;
    while (i < nso3 || j < nr3) {
      const bool take_so3 = j >= nr3 || (i < nso3 && int64_t(i) * h->dt_so3_ns <= int64_t(j) * h->dt_r3_ns);
      if (take_so3) h->so3_col[i++] = pos; else h->r3_col[j++] = pos;
      pos += 3;
    }
  }
  const int nk = pos;
  h->col_tic = tic ? pos : -1; if (tic) pos += 6;
  h->col_g = grav ? pos : -1; if (grav) pos += 3;
  h->col_ld = ld ? pos : -1; if (ld) pos += 1;
  if (ab) for (int k = 0; k < nba; ++k) { h->ba_col[k] = pos; pos += 3; }
  if (gb) for (int k = 0; k < nbg; ++k) { h->bg_col[k] = pos; pos += 3; }
  const int col_ai = intr ? pos : -1; if (intr) pos += 6;
  const int col_gi = intr ? pos : -1; if (intr) pos += 9;
  const int col_ci = cam_intr ? pos : -1; if (cam_intr) pos += h->n_intr;
  const int col_to = toff ? pos : -1; if (toff) pos += 1;
  const int col_pts = pts ? pos : -1; if (pts) pos += 3 * npts;
  const int nb = pos - nk;
  h->perm.assign(n, -1);
  if (spline) { for (int k = 0; k < nso3; ++k) for (int d = 0; d < 3; ++d) h->perm[c_so3 + 3 * k + d] = h->so3_col[k] + d; for (int k = 0; k < nr3; ++k) for (int d = 0; d < 3; ++d) h->perm[c_r3 + 3 * k + d] = h->r3_col[k] + d; }
  if (tic) for (int d = 0; d < 6; ++d) h->perm[c_tic + d] = h->col_tic + d;
  if (grav) for (int d = 0; d < 3; ++d) h->perm[c_g + d] = h->col_g + d;
  if (ld) h->perm[c_ld] = h->col_ld;
  if (ab) for (int k = 0; k < nba; ++k) for (int d = 0; d < 3; ++d) h->perm[c_ba + 3 * k + d] = h->ba_col[k] + d;
  if (gb) for (int k = 0; k < nbg; ++k) for (int d = 0; d < 3; ++d) h->perm[c_bg + 3 * k + d] = h->bg_col[k] + d;
  if (intr) { for (int d = 0; d < 6; ++d) h->perm[c_ai + d] = col_ai + d; for (int d = 0; d < 9; ++d) h->perm[c_gi + d] = col_gi + d; }
  if (cam_intr) for (int d = 0; d < h->n_intr; ++d) h->perm[c_ci + d] = col_ci + d;
  if (toff) h->perm[c_to] = col_to;
  if (pts) for (int d = 0; d < 3 * npts; ++d) h->perm[c_pts + d] = col_pts + d;
  // half bandwidth: widest knot window touched by one residual block
  int kd = 0;
  if (spline) {
    auto span = [&](int s_so3, int s_r3, bool use_r3) {
      int lo = h->so3_col[s_so3], hi = h->so3_col[s_so3 + SPLINE_N - 1] + 2;
      if (use_r3) { lo = std::min(lo, h->r3_col[s_r3]); hi = std::max(hi, h->r3_col[s_r3 + SPLINE_N - 1] + 2); }
      kd = std::max(kd, hi - lo);
    };
    if (h->ip.init_line_delay_s != 0.0) for (const auto& f : h->frames) span(f.s_so3, f.s_r3, true);
    for (const auto& c : h->cells) span(c.s_so3, c.s_r3, true);
    if (h->shard_world > 1) {   // every rank must agree on the layout: use the global worst case of the time-sorted order
      for (int s = 0; s + SPLINE_N <= nso3; ++s) { const int64_t t = int64_t(s) * h->dt_so3_ns; const int sr = (int)std::min<int64_t>(t / h->dt_r3_ns, nr3 - SPLINE_N); span(s, sr, true); }
      for (int s = 0; s + SPLINE_N <= nr3; ++s) { const int64_t t = int64_t(s) * h->dt_r3_ns; const int ss = (int)std::min<int64_t>(t / h->dt_so3_ns, nso3 - SPLINE_N); span(ss, s, true); }
    }
  }
  if (kd > 255) return fail(h, ICC_ERR_UNSUPPORTED, "knot-spacing ratio produces a half bandwidth > 255");
  h->cur_flags = flags;
  DeviceProblem& P = h->P;
  P.nk = nk; P.nb = nb; P.kd = kd; P.ldb = kd + 1;
  P.col_tic = h->col_tic; P.col_g = h->col_g; P.col_ld = h->col_ld; P.col_ai = col_ai; P.col_gi = col_gi; P.col_ci = col_ci; P.col_to = col_to; P.col_pts = col_pts; P.n_points = npts;
  P.bias_active = (ab || gb) ? 1 : 0; P.intr_active = (intr || toff) ? 1 : 0; P.cam_intr_active = cam_intr ? 1 : 0;
  P.ne_off_E = (int64_t)nk * P.ldb; P.ne_off_C = P.ne_off_E + (int64_t)nk * nb; P.ne_off_g = P.ne_off_C + (int64_t)nb * nb;
  P.ne_off_cost = P.ne_off_g + nk + nb; P.ne_size = (P.ne_off_cost + 1 + 3) / 4 * 4;
  if (h->device >= 0) {
    // (staged through the page-locked arena while it has room: asynchronous, ordered before the kernels on the solver's stream)
    CU(upload_staged(h, h->d_so3_col, h->so3_col)); CU(upload_staged(h, h->d_r3_col, h->r3_col)); CU(upload_staged(h, h->d_ba_col, h->ba_col)); CU(upload_staged(h, h->d_bg_col, h->bg_col));
    P.so3_col = h->d_so3_col.p; P.r3_col = h->d_r3_col.p; P.ba_col = h->d_ba_col.p; P.bg_col = h->d_bg_col.p;
    CU(h->d_ne.alloc((size_t)P.ne_size)); P.ne = h->d_ne.p;
    CU(h->d_scale.alloc((size_t)std::max(1, nk + nb))); CU(h->d_delta.alloc((size_t)std::max(1, nk + nb)));
    CU(h->d_ws.alloc(solve_workspace_doubles(P)));
  }
  return ICC_OK;
}

extern "C" int icc_comm_allreduce_sum(icc_comm* c, double* dev, int64_t n, void* stream);
// Cross-rank sum of a device buffer on the solver's stream: the library's own NCCL communicator, else the caller's hook.  Every rank
// must enter every sum (also with an empty slice), and a failing collective fails the call.
icc_status cross_rank_sum(icc_handle* h, double* dev, int64_t n) {
  if (h->shard_world <= 1) return ICC_OK;
  if (h->comm) return icc_comm_allreduce_sum(h->comm, dev, n, (void*)h->stream) ? fail(h, ICC_ERR_CUDA, std::string("all-reduce failed: ") + icc_comm_last_error()) : ICC_OK;
  if (h->allreduce) { h->allreduce(dev, n, (void*)h->stream, h->allreduce_user); return ICC_OK; }
  return ICC_OK;   // shards evaluated on their own (tests add them up on the host)
}

// One Jacobian evaluation on the current state: zero the packed normal equations, run the kernels, cross-rank reduce.
icc_status eval_jacobian(icc_handle* h, const DeviceState& S, double* residuals_dev) {
  CU(cudaMemsetAsync(h->P.ne, 0, (size_t)h->P.ne_size * sizeof(double), h->stream));
  if (launch_eval(h->P, S, true, nullptr, residuals_dev, nullptr, h->stream, h->aux_ok ? &h->aux : nullptr)) return fail(h, ICC_ERR_CUDA, std::string("eval launch: ") + cudaGetErrorString(cudaGetLastError()));
  if (h->P.col_pts >= 0 && h->P.rolling) launch_points_jac(h->P, S, S.pjac, h->P.col_pts, h->sm_count, h->stream);   // board-point columns (POINTS)
  return cross_rank_sum(h, h->P.ne, h->P.ne_size);
}
icc_status eval_cost(icc_handle* h, const DeviceState& S, double* cost_dev, double* residuals_dev, double* reproj_dev) {
  if (launch_eval(h->P, S, false, cost_dev, residuals_dev, reproj_dev, h->stream, h->aux_ok ? &h->aux : nullptr)) return fail(h, ICC_ERR_CUDA, std::string("eval launch: ") + cudaGetErrorString(cudaGetLastError()));
  return cost_dev ? cross_rank_sum(h, cost_dev, 1) : ICC_OK;
}

icc_status mean_reproj(icc_handle* h, double* out) {
  // GetMeanReprojectionError (impl.h:993-1072): RS functor on every view, values only
  if (h->P.n_vwork == 0 && h->shard_world <= 1) { *out = 0.0; return ICC_OK; }
  CU(cudaMemsetAsync(h->d_scal.p, 0, SC_COUNT * sizeof(double), h->stream));
  if (h->P.n_vwork > 0) {
    DeviceProblem P = h->P; P.n_iwork = 0; P.rolling = 1;
    if (launch_eval(P, h->st[h->cur].view(), false, h->d_scal.p + SC_CAND_COST, nullptr, h->d_scal.p + SC_REPROJ_SUM, h->stream)) return fail(h, ICC_ERR_CUDA, "eval launch failed");
  }
  { icc_status r = cross_rank_sum(h, h->d_scal.p + SC_REPROJ_SUM, 2); if (r != ICC_OK) return r; }   // a rank without vision work still enters the sum
  double sc[SC_COUNT];
  CU(cudaMemcpyAsync(sc, h->d_scal.p, sizeof sc, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  if (!(sc[SC_REPROJ_CNT] > 0.0)) { *out = 0.0; return ICC_OK; }
  *out = sc[SC_REPROJ_SUM] / sc[SC_REPROJ_CNT];
  return ICC_OK;
}

// Dense J^T J (canonical tangent order, row-major) from the packed banded + bordered normal equations read back to the host.
void dense_hessian(const icc_handle* h, const std::vector<double>& ne, double* out) {
  const DeviceProblem& P = h->P;
  const int n = h->n_tan;
  auto get = [&](int a, int b) -> double {
    const int lo = std::min(a, b), hi = std::max(a, b);
    if (hi < P.nk) return hi - lo <= P.kd ? ne[(size_t)lo * P.ldb + (hi - lo)] : 0.0;
    if (lo < P.nk) return ne[P.ne_off_E + (size_t)lo * P.nb + (hi - P.nk)];
    return ne[P.ne_off_C + (size_t)(hi - P.nk) * P.nb + (lo - P.nk)];
  };
  for (int i = 0; i < n; ++i) for (int j = 0; j < n; ++j) out[(size_t)i * n + j] = get(h->perm[i], h->perm[j]);
}

// Levenberg-Marquardt with Ceres TrustRegionMinimizer semantics (options: impl.h:254-266 + Ceres 2.1 defaults).
icc_status run_lm(icc_handle* h, int max_iters, int flags, bool check_convergence, icc_summary* out) {
  using clk = std::chrono::steady_clock;
  const auto t_start = clk::now();
  PhaseTrace trace(h->stream);
  icc_status rc = configure(h, flags);
  if (rc != ICC_OK) return rc;
  trace.lap("run_lm: configure");
  icc_summary S; memset(&S, 0, sizeof S);
  const DeviceProblem& P = h->P;
  const int n = P.nk + P.nb;
  S.num_residuals = P.n_res_vis + P.n_res_acc + P.n_res_gyr; S.num_tangent = n;
  const int launches0 = kernel_launch_count();
  std::vector<cudaEvent_t> ev;
  auto mark = [&]() { cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, h->stream); ev.push_back(e); return (int)ev.size() - 1; };
  std::vector<std::pair<int, int>> jac_spans, lin_spans;
  double sc[SC_COUNT];
  double x_cost = 0.0;
  auto jac = [&]() -> icc_status {
    const int a = mark();
    icc_status r = eval_jacobian(h, h->st[h->cur].view(), nullptr);
    if (r != ICC_OK) return r;
    const int b = mark(); jac_spans.push_back({a, b});
    ++S.jacobian_evaluations;
    return ICC_OK;
  };
  // After a Jacobian evaluation: Jacobi scaling (first time) + gradient max-norm, and the cost at x parked next to the other
  // per-iteration scalars, so that ONE device->host read-back (and one stream synchronisation) serves the whole LM iteration.
  auto after_jacobian = [&](bool compute_scale) -> icc_status {
    CU(cudaMemsetAsync(h->d_scal.p + SC_GRAD_MAX, 0, sizeof(double), h->stream));
    launch_compute_scale(P, compute_scale ? h->d_scale.p : nullptr, h->opt.jacobi_scaling, h->d_scal.p, h->stream);
    return ICC_OK;
  };
  auto read_scalars = [&]() -> icc_status {
    CU(cudaMemcpyAsync(sc, h->d_scal.p, sizeof sc, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return ICC_OK;
  };
  if (n == 0) { if (out) *out = S; return ICC_OK; }
  double radius = h->opt.initial_trust_region_radius, decrease_factor = 2.0;
  int invalid = 0;
  bool ne_valid = false, first = true;
  S.termination = 0;
  for (int it = 0; it < max_iters; ++it) {
    // The Jacobian / normal equations are (re)built lazily at the top of the iteration that needs them, so that n
    // iterations cost n linear solves + n cost evaluations + one Jacobian evaluation per accepted step (and the first).
    bool fresh_jacobian = false;
    if (!ne_valid) {
      rc = jac(); if (rc != ICC_OK) return rc;
      rc = after_jacobian(first); if (rc != ICC_OK) return rc;
      ne_valid = true; fresh_jacobian = true;
    }
    SolveParams sp; sp.radius = radius; sp.min_diag = h->opt.min_lm_diagonal; sp.max_diag = h->opt.max_lm_diagonal; sp.jacobi_scaling = h->opt.jacobi_scaling;
    const int a = mark();
    { const int se = launch_solve(P, h->d_scale.p, sp, h->d_ws.p, h->d_delta.p, h->d_scal.p, h->stream);
      if (se == 1) return fail(h, ICC_ERR_UNSUPPORTED, "the border (bias knots + globals) is too wide for the solver's shared-memory plans");
      if (se) return fail(h, ICC_ERR_CUDA, std::string("solver launch: ") + cudaGetErrorString(cudaGetLastError())); }
    const int b = mark(); lin_spans.push_back({a, b});
    const int cand = 1 - h->cur;
    launch_update(P, h->st[h->cur].view(), h->st[cand].view(), h->d_delta.p, h->max_ba, h->max_bg, h->d_scal.p, h->stream);
    if (P.col_pts >= 0) launch_points_update(P.n_points, P.col_pts, h->st[h->cur].pts.p, h->st[cand].pts.p, h->st[cand].board.p, h->st[cand].pjac.p, h->d_delta.p, h->d_scal.p, h->stream);
    rc = eval_cost(h, h->st[cand].view(), h->d_scal.p + SC_CAND_COST, nullptr, nullptr); if (rc != ICC_OK) return rc;
    rc = read_scalars(); if (rc != ICC_OK) return rc;
    trace.lap("run_lm: iteration");
    if (fresh_jacobian) {
      x_cost = sc[SC_X_COST];
      if (first) { S.initial_cost = x_cost; first = false; if (!std::isfinite(x_cost)) return fail(h, ICC_ERR_NUMERIC, "non-finite initial cost"); }
      // Ceres tests the gradient right after the Jacobian evaluation; the step computed above is simply discarded
      if (check_convergence && sc[SC_GRAD_MAX] <= h->opt.gradient_tolerance) { S.termination = 3; break; }
    }
    ++S.iterations; ++S.cost_evaluations;
    const double model_change = sc[SC_MODEL_CHANGE];
    if (sc[SC_OK] == 0.0 || !(model_change > 0.0)) {          // invalid step (HandleInvalidStep)
      if (++invalid >= h->opt.max_consecutive_invalid_steps) { S.termination = 4; break; }
      radius /= decrease_factor; decrease_factor *= 2.0;
      if (radius < h->opt.min_trust_region_radius) { S.termination = 4; break; }   // Ceres tests MinTrustRegionRadiusReached after every iteration
      continue;
    }
    invalid = 0;
    const double step_norm = std::sqrt(sc[SC_STEP_SQ]), x_norm = std::sqrt(sc[SC_X_SQ]);
    double cand_cost = sc[SC_CAND_COST];
    if (!std::isfinite(cand_cost)) cand_cost = 1.7976931348623157e308;
    if (check_convergence && step_norm <= h->opt.parameter_tolerance * (x_norm + h->opt.parameter_tolerance)) { S.termination = 2; break; }
    const double cost_change = x_cost - cand_cost;
    if (check_convergence && std::fabs(cost_change) <= h->opt.function_tolerance * x_cost) { S.termination = 1; break; }
    const double rel = cost_change / model_change;
    if (rel > h->opt.min_relative_decrease) {               // HandleSuccessfulStep
      ++S.successful_steps;
      h->cur = cand; h->state_dirty_host = true; h->glob_host_current = false;
      x_cost = cand_cost; ne_valid = false;
      radius = radius / std::max(1.0 / 3.0, 1.0 - std::pow(2.0 * rel - 1.0, 3));
      radius = std::min(h->opt.max_trust_region_radius, radius);
      decrease_factor = 2.0;
    } else {                                                  // StepRejected
      radius /= decrease_factor; decrease_factor *= 2.0;
      if (radius < h->opt.min_trust_region_radius) { S.termination = 4; break; }
    }
  }
  if (first) { rc = jac(); if (rc != ICC_OK) return rc; rc = after_jacobian(true); if (rc != ICC_OK) return rc; rc = read_scalars(); if (rc != ICC_OK) return rc; x_cost = sc[SC_X_COST]; S.initial_cost = x_cost; }
  if (P.col_pts >= 0 && S.successful_steps > 0) {   // both state buffers carry the accepted points again (runs without POINTS never copy them)
    const StateBufs& a = h->st[h->cur]; StateBufs& b = h->st[1 - h->cur];
    CU(cudaMemcpyAsync(b.pts.p, a.pts.p, a.pts.n * sizeof(double4), cudaMemcpyDeviceToDevice, h->stream));
    CU(cudaMemcpyAsync(b.board.p, a.board.p, a.board.n * sizeof(double4), cudaMemcpyDeviceToDevice, h->stream));
    CU(cudaMemcpyAsync(b.pjac.p, a.pjac.p, a.pjac.n * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  }
  CU(cudaStreamSynchronize(h->stream));
  S.final_cost = x_cost;
  auto span_s = [&](const std::vector<std::pair<int, int>>& v) { double tot = 0; for (auto& p : v) { float ms = 0; cudaEventElapsedTime(&ms, ev[p.first], ev[p.second]); tot += ms; } return tot * 1e-3; };
  S.seconds_jacobian = span_s(jac_spans); S.seconds_linear_solve = span_s(lin_spans);
  for (auto e : ev) cudaEventDestroy(e);
  S.gpu_launches = kernel_launch_count() - launches0;
  S.seconds_total = std::chrono::duration<double>(clk::now() - t_start).count();
  trace.lap("run_lm: epilogue");
  if (out) *out = S;
  return ICC_OK;
}

}  // namespace

// =================================================================================================================
extern "C" {

const char* icc_version(void) { return "icc_b200 0.1 (sm_100a, fp64)"; }

void icc_default_solver_options(icc_solver_options* o) {
  o->function_tolerance = 1e-4; o->parameter_tolerance = 1e-7; o->gradient_tolerance = 1e-10;
  o->initial_trust_region_radius = 1e4; o->max_trust_region_radius = 1e16; o->min_trust_region_radius = 1e-32;
  o->min_relative_decrease = 1e-3; o->min_lm_diagonal = 1e-6; o->max_lm_diagonal = 1e32; o->jacobi_scaling = 1; o->max_consecutive_invalid_steps = 5;
}

// device_ordinal >= 0 binds a GPU (required for every compute entry point).  device_ordinal == -1 creates a host-only
// handle whose sole use is inspecting the problem ASSEMBLY (knot initialisation, counts) without a GPU; it cannot compute.
icc_status icc_create(icc_handle** out, int device_ordinal) {
  if (!out) return ICC_ERR_INVALID_ARGUMENT;
  icc_handle* h = new icc_handle();
  icc_default_solver_options(&h->opt);
  memset(&h->P, 0, sizeof h->P);
  *out = h;
  if (device_ordinal < 0) { h->device = -1; return ICC_OK; }
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count <= 0 || device_ordinal >= count) {
    h->err = std::string("no usable CUDA device (") + (e != cudaSuccess ? cudaGetErrorString(e) : "device ordinal out of range") + "); this library has no CPU fallback";
    return ICC_ERR_NO_DEVICE;
  }
  if (cudaSetDevice(device_ordinal) != cudaSuccess) { h->err = "cudaSetDevice failed"; return ICC_ERR_NO_DEVICE; }
  h->device = device_ordinal;
  cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device_ordinal);
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) { h->err = "cudaStreamCreate failed"; h->device = -1; return ICC_ERR_CUDA; }
  if (h->d_scal.alloc(SC_COUNT) != cudaSuccess) { h->err = "cudaMalloc failed"; return ICC_ERR_CUDA; }
  h->aux_ok = cudaStreamCreateWithFlags(&h->aux.stream, cudaStreamNonBlocking) == cudaSuccess &&
              cudaEventCreateWithFlags(&h->aux.fork, cudaEventDisableTiming) == cudaSuccess && cudaEventCreateWithFlags(&h->aux.join, cudaEventDisableTiming) == cudaSuccess;
  if (!h->aux_ok) { h->err = "cudaStreamCreate failed"; return ICC_ERR_CUDA; }
  return ICC_OK;
}
void icc_destroy(icc_handle* h) { if (!h) return; if (h->device >= 0) { cudaSetDevice(h->device); if (h->stream) { cudaStreamSynchronize(h->stream); cudaStreamDestroy(h->stream); } if (h->aux_ok) { cudaStreamDestroy(h->aux.stream); cudaEventDestroy(h->aux.fork); cudaEventDestroy(h->aux.join); } } delete h; }
const char* icc_last_error(const icc_handle* h) { return h ? h->err.c_str() : "null handle"; }
icc_status icc_set_solver_options(icc_handle* h, const icc_solver_options* o) { if (!h || !o) return ICC_ERR_INVALID_ARGUMENT; h->opt = *o; return ICC_OK; }

icc_status icc_set_camera(icc_handle* h, int model, const double* intr, int n, int w, int hgt) {
  if (!h || !intr) return ICC_ERR_INVALID_ARGUMENT;
  if (camera_num_params(model) < 0 || n != camera_num_params(model)) return fail(h, ICC_ERR_INVALID_ARGUMENT, "unknown camera model or wrong intrinsic count");
  h->model = model; h->n_intr = n; h->width = w; h->height = hgt; for (int i = 0; i < n; ++i) h->intr[i] = intr[i];
  return ICC_OK;
}
icc_status icc_set_board_points(icc_handle* h, int n, const double* xyzw) {
  if (!h || n <= 0 || !xyzw) return ICC_ERR_INVALID_ARGUMENT;
  const bool same_board = h->points.size() == 4 * (size_t)n;
  if (h->initialised && h->device >= 0 && same_board) { icc_status s = sync_state_to_host(h); if (s != ICC_OK) return s; }
  h->points.assign(xyzw, xyzw + 4 * (size_t)n);
  if (h->initialised && h->device >= 0) {      // an assembled problem keeps its corners: only the coordinates may change
    if (!same_board) return fail(h, ICC_ERR_STATE, "the number of board points cannot change after batch_init_spline");
    for (int k = 0; k < 2; ++k) { icc_status s = upload_points(h, k, false); if (s != ICC_OK) return s; }
  }
  return ICC_OK;
}
icc_status icc_set_frames(icc_handle* h, int nf, const double* t, const int32_t* off, const int32_t* ids, const double* uv, const double* q, const double* p) {
  if (!h || nf <= 0 || !t || !off || !ids || !uv || !q || !p) return ICC_ERR_INVALID_ARGUMENT;
  const int nc = off[nf];
  for (int i = 0; i < nf; ++i) if (off[i + 1] < off[i]) return fail(h, ICC_ERR_INVALID_ARGUMENT, "corner offsets must be non-decreasing");
  if (h->device >= 0 && h->stream) cudaStreamSynchronize(h->stream);   // an asynchronous upload may still be reading the staging buffers
  const bool pin = h->device >= 0;
  h->frame_t.assign(t, t + nf); h->corner_off.assign(off, off + nf + 1);
  h->n_corners_in = (size_t)nc;
  h->frames_dev = pin && nc > 0 && host_is_pinned(uv) && host_is_pinned(ids);
  if (h->frames_dev) {   // page-locked caller buffers: DMA straight to the device, the id range is found while it runs
    CU(cudaSetDevice(h->device));
    CU(h->d_uv_all.alloc((size_t)nc)); CU(h->d_pid_all.alloc((size_t)nc));
    CU(cudaMemcpyAsync(h->d_uv_all.p, uv, (size_t)nc * sizeof(double2), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_pid_all.p, ids, (size_t)nc * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    // the id range is reduced on the device behind the copy (two ints come back with the synchronisation this call ends with anyway)
    int* rng = static_cast<int*>(h->arena_small(2 * sizeof(int)));
    if (rng) {
      rng[0] = 0; rng[1] = -1;
      CU(h->d_idrange.alloc(2));
      CU(cudaMemcpyAsync(h->d_idrange.p, rng, 2 * sizeof(int), cudaMemcpyHostToDevice, h->stream));
      launch_id_range(nc, h->d_pid_all.p, h->d_idrange.p, h->stream);
      CU(cudaMemcpyAsync(rng, h->d_idrange.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    }
    h->uv.clear(); h->point_ids.clear();
    CU(cudaStreamSynchronize(h->stream));   // the caller's arrays are not referenced after this call returns
    if (rng) { h->id_lo = rng[0]; h->id_hi = rng[1]; }
    else { int lo = 0, hi = -1; for (int i = 0; i < nc; ++i) { const int v = ids[i]; lo = v < lo ? v : lo; hi = v > hi ? v : hi; } h->id_lo = lo; h->id_hi = hi; }
  } else {
    h->uv.assign(uv, 2 * (size_t)nc, pin);
    // the ids are copied and range-checked in one pass (the check of batch_init_spline would read them again, cold)
    h->point_ids.resize((size_t)nc, pin);
    int lo = 0, hi = -1; int* dst = h->point_ids.data();
    for (int i = 0; i < nc; ++i) { const int v = ids[i]; dst[i] = v; lo = v < lo ? v : lo; hi = v > hi ? v : hi; }
    h->id_lo = lo; h->id_hi = hi;
  }
  h->q_wc.assign(q, q + 4 * (size_t)nf); h->p_wc.assign(p, p + 3 * (size_t)nf);
  return ICC_OK;
}
icc_status icc_set_imu(icc_handle* h, int n, const double* t, const double* a, const double* g) {
  if (!h || n < 0 || (n > 0 && (!t || !a || !g))) return ICC_ERR_INVALID_ARGUMENT;
  if (h->device >= 0 && h->stream) cudaStreamSynchronize(h->stream);
  const bool pin = h->device >= 0;
  h->n_imu_in = (size_t)n;
  h->imu_dev = pin && n > 0 && host_is_pinned(a) && host_is_pinned(g);
  if (h->imu_dev) {
    CU(cudaSetDevice(h->device));
    CU(h->d_acc_all.alloc(3 * (size_t)n)); CU(h->d_gyr_all.alloc(3 * (size_t)n));
    CU(cudaMemcpyAsync(h->d_acc_all.p, a, 3 * (size_t)n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_gyr_all.p, g, 3 * (size_t)n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    h->imu_acc.clear(); h->imu_gyr.clear();
  } else { h->imu_acc.assign(a, 3 * (size_t)n, pin); h->imu_gyr.assign(g, 3 * (size_t)n, pin); }
  {   // time stamps: copied and tested for order in one pass (the sorted stream takes the bisection path of batch_init_spline)
    h->imu_t.resize((size_t)n, pin);
    double* dst = h->imu_t.data(); int unsorted = 0; double prev = n > 0 ? t[0] : 0.0;
    for (int i = 0; i < n; ++i) { const double v = t[i]; dst[i] = v; unsorted |= !(v >= prev); prev = v; }
    h->imu_sorted = !unsorted;
  }
  if (h->imu_dev) CU(cudaStreamSynchronize(h->stream));   // the caller's arrays are not referenced after this call returns
  return ICC_OK;
}
icc_status icc_set_shard(icc_handle* h, int rank, int world) { if (!h || world < 1 || rank < 0 || rank >= world) return fail(h, ICC_ERR_INVALID_ARGUMENT, "bad shard"); h->shard_rank = rank; h->shard_world = world; return ICC_OK; }
icc_status icc_set_comm(icc_handle* h, icc_comm* c) {
  if (!h) return ICC_ERR_INVALID_ARGUMENT;
  h->comm = c;
  h->shard_rank = c ? icc_comm_rank(c) : 0; h->shard_world = c ? icc_comm_world(c) : 1;
  return ICC_OK;
}
icc_status icc_set_allreduce(icc_handle* h, icc_allreduce_fn fn, void* user) { if (!h) return ICC_ERR_INVALID_ARGUMENT; h->allreduce = fn; h->allreduce_user = user; return ICC_OK; }

icc_status icc_batch_init_spline(icc_handle* h, const icc_init_params* ipp) {
  if (!h || !ipp) return ICC_ERR_INVALID_ARGUMENT;
  if (h->model < 0 || h->frame_t.empty() || h->points.empty()) return fail(h, ICC_ERR_STATE, "camera, board points and frames must be set before batch_init_spline");
  PhaseTrace trace(h->device >= 0 ? h->stream : nullptr);
  if (h->id_lo < 0 || (size_t)(h->id_hi + 1) > h->points.size() / 4) return fail(h, ICC_ERR_INVALID_ARGUMENT, "corner references an unknown board point");
  h->ip = *ipp;
  const int nf = (int)h->frame_t.size();
  trace.lap("batch_init: id range check");
  // T_i_c, IMU intrinsics, line delay (imu_camera_calibrator.cc:30-47)
  { const Q4 q = qn(ipp->T_i_c_init); h->glob[G_TIC + 0] = q.x; h->glob[G_TIC + 1] = q.y; h->glob[G_TIC + 2] = q.z; h->glob[G_TIC + 3] = q.w; for (int i = 4; i < 7; ++i) h->glob[G_TIC + i] = ipp->T_i_c_init[i]; }
  for (int i = 0; i < 6; ++i) h->glob[G_ACC_INTR + i] = ipp->acc_intrinsics[i];
  for (int i = 0; i < 9; ++i) h->glob[G_GYR_INTR + i] = ipp->gyr_intrinsics[i];
  h->glob[G_LD] = ipp->init_line_delay_s;
  for (int i = 0; i < 10; ++i) h->glob[G_CAM_INTR + i] = i < h->n_intr ? h->intr[i] : 0.0;
  h->glob[G_TOFF] = 0.0;
  // spline time range and knot counts (imu_camera_calibrator.cc:49-72, impl.h:37-51)
  std::vector<double> cam_ts(h->frame_t); std::sort(cam_ts.begin(), cam_ts.end());
  h->t0_s = cam_ts.front(); h->tend_s = cam_ts.back();
  h->start_ns = (int64_t)(h->t0_s * S_TO_NS);
  h->end_ns = (int64_t)(h->tend_s * S_TO_NS + 0.01 * S_TO_NS + ipp->init_line_delay_s);
  h->dt_so3_ns = (int64_t)(ipp->dt_so3_s * S_TO_NS); h->dt_r3_ns = (int64_t)(ipp->dt_r3_s * S_TO_NS);
  if (h->dt_so3_ns <= 0 || h->dt_r3_ns <= 0) return fail(h, ICC_ERR_INVALID_ARGUMENT, "knot spacing must be positive");
  const int64_t duration = h->end_ns - h->start_ns;
  const int nso3 = (int)(duration / h->dt_so3_ns) + SPLINE_N, nr3 = (int)(duration / h->dt_r3_ns) + SPLINE_N;
  // knot initialisation from the per-view pose priors (impl.h:278-339)
  const Pose Tic{q4(h->glob[0], h->glob[1], h->glob[2], h->glob[3]), v3(h->glob[4], h->glob[5], h->glob[6])};
  const Pose Tci = pose_inv(Tic);
  // the reference walks its views through a std::map keyed by timestamp (time order, a repeated timestamp keeps the LAST view);
  // strictly increasing timestamps -- the usual case -- give that order without the tree
  bool increasing = true; for (int i = 1; i < nf && increasing; ++i) increasing = h->frame_t[i] > h->frame_t[i - 1];
  std::vector<int> view_order;
  if (increasing) { view_order.resize(nf); for (int i = 0; i < nf; ++i) view_order[i] = i; }
  else { std::map<double, int> by_time; for (int i = 0; i < nf; ++i) by_time[h->frame_t[i]] = i; for (const auto& kv : by_time) view_order.push_back(kv.second); }
  std::vector<double> t_vis, q_vis, p_vis;
  t_vis.reserve(view_order.size()); q_vis.reserve(4 * view_order.size()); p_vis.reserve(3 * view_order.size());
  for (const int i : view_order) {
    const Pose Twc{qn(&h->q_wc[4 * i]), v3(h->p_wc[3 * i], h->p_wc[3 * i + 1], h->p_wc[3 * i + 2])};
    const Pose Twi = pose_mul(Twc, Tci);
    t_vis.push_back(h->frame_t[i]);
    q_vis.push_back(Twi.q.x); q_vis.push_back(Twi.q.y); q_vis.push_back(Twi.q.z); q_vis.push_back(Twi.q.w);
    p_vis.push_back(Twi.t.x); p_vis.push_back(Twi.t.y); p_vis.push_back(Twi.t.z);
  }
  const size_t nv = t_vis.size();
  h->so3.assign(4 * (size_t)nso3, 0.0); h->r3.assign(3 * (size_t)nr3, 0.0);
  // With a device the knots are initialised by init_knots_kernel (icc_init.cu) straight into both state copies, from the uploaded
  // view poses; the host statement below serves the host-only handle (device -1: assembly checks against the oracle on CPU).
  if (h->device < 0) {
  for (int i = 0; i < nso3; ++i) {   // InterpolateQuaternions (utils.cc:221-241); knot times are zero based (SURVEY quirk q7)
    const double t = double(i) * double(h->dt_so3_ns) * NS_TO_S;
    double dist = 0; const size_t k = nearest_index(t, t_vis, dist);
    double q[4];
    if (k < nv - 1) quat_slerp(&q_vis[4 * k], &q_vis[4 * (k + 1)], dist / (t_vis[k + 1] - t_vis[k]), q); else memcpy(q, &q_vis[4 * k], sizeof q);
    const Q4 r = qn(q);
    h->so3[4 * i] = r.x; h->so3[4 * i + 1] = r.y; h->so3[4 * i + 2] = r.z; h->so3[4 * i + 3] = r.w;
  }
  for (int i = 0; i < nr3; ++i) {    // InterpolateVector3d (utils.cc:243-261) incl. its `nearest < t_new.size()` test; the reference's
    const double t = double(i) * double(h->dt_r3_ns) * NS_TO_S;   // out-of-range read past the last view falls back to the nearest value
    double dist = 0; const size_t k = nearest_index(t, t_vis, dist);
    if (k < (size_t)nr3 && k + 1 < nv) { const double f = dist / (t_vis[k + 1] - t_vis[k]); for (int d = 0; d < 3; ++d) h->r3[3 * i + d] = (1.0 - f) * p_vis[3 * k + d] + f * p_vis[3 * (k + 1) + d]; }
    else for (int d = 0; d < 3; ++d) h->r3[3 * i + d] = p_vis[3 * k + d];
  }
  }
  // bias splines: InitBiasSplines(bias, bias, 10 s, 10 s, 1.0, 0.1) (imu_camera_calibrator.cc:80-85, impl.h:53-90)
  h->dt_ba_ns = h->dt_bg_ns = (int64_t)(10 * 1e9); h->max_ba = 1.0; h->max_bg = 1e-1;
  const int nba = (int)(duration / h->dt_ba_ns) + BIAS_N, nbg = (int)(duration / h->dt_bg_ns) + BIAS_N;
  h->ba.resize(3 * (size_t)nba); h->bg.resize(3 * (size_t)nbg);
  for (int i = 0; i < nba; ++i) for (int d = 0; d < 3; ++d) h->ba[3 * i + d] = ipp->acc_bias[d];
  for (int i = 0; i < nbg; ++i) for (int d = 0; d < 3; ++d) h->bg[3 * i + d] = ipp->gyr_bias[d];

  trace.lap("batch_init: ranges, view order, bias knots");
  // ---- measurement wiring (imu_camera_calibrator.cc:87-120; Add*Measurement impl.h:341-613) ----------------------
  const bool pin = h->device >= 0;
  std::vector<FrameHost> all_frames(nf);
  std::vector<char> frame_ok(nf);
  h->dropped_frames = h->dropped_imu = 0;
  for (int i = 0; i < nf; ++i) {
    FrameHost& f = all_frames[i]; f.t_s = h->frame_t[i]; f.c0 = h->corner_off[i]; f.c1 = h->corner_off[i + 1];
    const int64_t t_ns = (int64_t)(f.t_s * S_TO_NS);
    int64_t s1 = 0, s2 = 0;
    const bool ok = calc_times(t_ns, h->start_ns, h->dt_r3_ns, nr3, SPLINE_N, f.u_r3, s1) && calc_times(t_ns, h->start_ns, h->dt_so3_ns, nso3, SPLINE_N, f.u_so3, s2);
    f.s_r3 = (int)s1; f.s_so3 = (int)s2;
    frame_ok[i] = ok; if (!ok) ++h->dropped_frames;
  }
  struct ImuHost { double t_s; int64_t st; int s_so3, s_r3, s_ba, s_bg; int src; };
  // CalcTimes' segment index s = st / dt of a time-sorted stream only ever steps forward: track it with comparisons and fall back
  // to the division when a sample is not where the previous one left off (unsorted input); the results are identical
  struct SegTrack { int64_t dt, s = 0, lo = 0, hi = -1;   // [lo, hi) = time range of segment s; hi < lo until the first sample
    int64_t seg(int64_t st) {
      if (st >= lo && st < hi) return s;
      if (hi > lo && st >= hi && st < hi + 63 * dt) { do { ++s; lo = hi; hi += dt; } while (st >= hi); return s; }
      s = st / dt; lo = s * dt; hi = lo + dt; return s;
    } };
  const size_t n_imu_in = h->imu_t.size();
  h->imu_used_t.clear(); h->imu_used_acc.clear(); h->imu_used_gyr.clear(); h->cells.clear();
  h->imu_used_st.resize(n_imu_in, pin);
  std::vector<ImuHost> all_imu;
  // One pass over the IMU stream.  `direct` (one shard): the kept samples go straight into the problem arrays in arrival order,
  // which IS the time order as long as the stream is sorted -- the pass gives up (returns false) at the first sample that is not.
  // Otherwise they are collected for the general path below (time merge with the frames, residual-count sharding).
  auto imu_pass = [&](bool direct) -> bool {
    SegTrack tr_r3{h->dt_r3_ns}, tr_so3{h->dt_so3_ns}, tr_ba{h->dt_ba_ns}, tr_bg{h->dt_bg_ns};
    h->dropped_imu = 0; h->imu_used_t.clear(); h->cells.clear(); all_imu.clear();
    if (direct) h->imu_used_t.resize(n_imu_in); else all_imu.reserve(n_imu_in);
    double* t_out = h->imu_used_t.data();
    int64_t* st_out = h->imu_used_st.data();
    double last_t = -1.7976931348623157e308; int prev_src = -1; bool contig = true; size_t k = 0;
    const double* imu_t = h->imu_t.data(); const double toff = ipp->time_offset_imu_to_cam_s, t0 = h->t0_s, tend = h->tend_s;
    for (size_t i = 0; i < n_imu_in; ++i) {
      const double t = imu_t[i] + toff;
      if (t < t0 || t >= tend) continue;
      const int64_t t_ns = (int64_t)(t * S_TO_NS), st = t_ns - h->start_ns;
      bool ok = st >= 0;
      int64_t a = 0, b = 0, c = 0, d = 0;
      if (ok) { a = tr_r3.seg(st); b = tr_so3.seg(st); c = tr_ba.seg(st); d = tr_bg.seg(st);
                ok = size_t(a + SPLINE_N) <= (size_t)nr3 && size_t(b + SPLINE_N) <= (size_t)nso3 && size_t(c + BIAS_N) <= (size_t)nba && size_t(d + BIAS_N) <= (size_t)nbg; }
      if (!ok) { ++h->dropped_imu; continue; }
      if (!direct) { all_imu.push_back({t, st, (int)b, (int)a, (int)c, (int)d, (int)i}); continue; }
      if (t < last_t) { h->imu_used_t.clear(); return false; }
      last_t = t;
      if (prev_src >= 0 && (int)i != prev_src + 1) contig = false;
      if (prev_src < 0) h->imu_src0 = (int)i;
      prev_src = (int)i;
      t_out[k] = t; st_out[k] = st;
      if (h->cells.empty() || h->cells.back().s_so3 != (int)b || h->cells.back().s_r3 != (int)a || h->cells.back().s_ba != (int)c || h->cells.back().s_bg != (int)d)
        h->cells.push_back({(int)b, (int)a, (int)c, (int)d, (int)k, (int)k});
      h->cells.back().i_end = (int)k + 1;
      ++k;
    }
    if (direct) { h->imu_contig = k > 0 && contig; if (k == 0) h->imu_src0 = 0; h->imu_used_st.n = k; h->imu_used_t.resize(k); }
    return true;
  };
  // Sorted stream (the usual case; known from set_imu): the kept samples [ka, kb) of imu_t are used in place, and the cells -- maximal runs of
  // samples inside the same knot interval of all four splines -- are found by galloping + bisection for the next interval boundary
  // (CalcTimes' st is monotone in t), so the host touches O(cells log run) time stamps instead of every sample.  The relative times
  // st = int64((t + offset) 1e9) - start themselves are derived on the device from the uploaded stamps (imu_times_kernel), bit for bit.
  auto cells_by_bisection = [&](size_t ka, size_t kb) {
    const double* imu_t = h->imu_t.data(); const double toff = ipp->time_offset_imu_to_cam_s;
    auto st_of = [&](size_t i) { return (int64_t)((imu_t[i] + toff) * S_TO_NS) - h->start_ns; };
    h->cells.clear(); h->imu_used_t.clear(); h->imu_used_st.n = 0;
    size_t k = ka;
    while (k < kb) {
      const int64_t st = st_of(k);
      const int64_t a = st / h->dt_r3_ns, b = st / h->dt_so3_ns, c = st / h->dt_ba_ns, d = st / h->dt_bg_ns;
      const int64_t edge = std::min(std::min((a + 1) * h->dt_r3_ns, (b + 1) * h->dt_so3_ns), std::min((c + 1) * h->dt_ba_ns, (d + 1) * h->dt_bg_ns));
      size_t prev = k, probe = k + 1, step = 1;                     // first index in (k, kb) with st >= edge: gallop, then bisect
      while (probe < kb && st_of(probe) < edge) { prev = probe; probe += step; step *= 2; }
      size_t lo = prev + 1, hi = std::min(probe, kb);                // st_of(prev) < edge <= st_of(probe) (or probe is past the end)
      while (lo < hi) { const size_t m = (lo + hi) / 2; if (st_of(m) < edge) lo = m + 1; else hi = m; }
      h->cells.push_back({(int)b, (int)a, (int)c, (int)d, (int)(k - ka), (int)(lo - ka)});
      k = lo;
    }
    h->imu_lazy = true; h->n_imu_used = kb - ka; h->imu_contig = kb > ka; h->imu_src0 = kb > ka ? (int)ka : 0;
  };
  auto imu_sorted_pass = [&]() -> bool {
    if (h->shard_world != 1 || !h->imu_sorted || n_imu_in == 0 || getenv("ICC_NO_BISECTION")) return false;   // (the switch forces the sample-by-sample pass: tests)
    const double* imu_t = h->imu_t.data(); const double toff = ipp->time_offset_imu_to_cam_s, t0 = h->t0_s, tend = h->tend_s;
    auto bisect = [&](size_t a, size_t b, auto pred) { while (a < b) { const size_t m = (a + b) / 2; if (pred(m)) a = m + 1; else b = m; } return a; };   // first index where pred is false
    auto fits = [&](size_t i) {   // upper-side validity of CalcTimes for all four splines (monotone: true, then false)
      const double t = imu_t[i] + toff;
      if (t >= tend) return false;
      const int64_t st = (int64_t)(t * S_TO_NS) - h->start_ns;
      return size_t(st / h->dt_r3_ns + SPLINE_N) <= (size_t)nr3 && size_t(st / h->dt_so3_ns + SPLINE_N) <= (size_t)nso3 && size_t(st / h->dt_ba_ns + BIAS_N) <= (size_t)nba && size_t(st / h->dt_bg_ns + BIAS_N) <= (size_t)nbg;
    };
    const size_t ia = bisect(0, n_imu_in, [&](size_t i) { const double t = imu_t[i] + toff; return t < t0 || (int64_t)(t * S_TO_NS) - h->start_ns < 0; });
    const size_t ib = bisect(ia, n_imu_in, fits);
    if (ib <= ia) return false;                                     // nothing kept: the sequential pass reports it
    const size_t in_window = bisect(ia, n_imu_in, [&](size_t i) { return imu_t[i] + toff < tend; }) - ia;
    h->dropped_imu = (int)(in_window - (ib - ia));
    cells_by_bisection(ia, ib);
    return true;
  };
  std::vector<int> frame_sel;
  // (a stream with holes inside the kept range -- samples dropped in the middle -- takes the general path, which gathers the readings)
  trace.lap("batch_init: frame times");
  h->imu_lazy = false; h->n_imu_used = 0;
  const bool direct = imu_sorted_pass() || (h->shard_world == 1 && imu_pass(true) && h->imu_contig);
  trace.lap("batch_init: imu pass");
  if (direct) {
    for (int i = 0; i < nf; ++i) if (frame_ok[i]) frame_sel.push_back(i);
  } else if ([&]() -> bool {
    // Sharded fast path (every stream in time order, the usual case): the shard rule -- unit `mine` iff the scalar residuals of all
    // units before it in the time-merged order (frames before IMU samples on ties) fall in [lo, hi) -- is evaluated on counts only:
    // kept IMU samples of a sorted stream are ONE index range (the validity tests of CalcTimes are monotone in time), frames are
    // break points found by bisection, and only the shard's own samples are then walked.  O(frames log samples + samples / world)
    // instead of O(samples) per rank; same decisions as the general path below (tests/test_capi_boundary.py, test_sharding_gloo.py).
    const double* imu_t = h->imu_t.data(); const double toff = ipp->time_offset_imu_to_cam_s, t0 = h->t0_s, tend = h->tend_s;
    if (!increasing || !h->imu_sorted) return false;
    auto fits = [&](size_t i) {   // upper-side validity (monotone: true, then false)
      const double t = imu_t[i] + toff;
      if (t >= tend) return false;
      const int64_t st = (int64_t)(t * S_TO_NS) - h->start_ns;
      return size_t(st / h->dt_r3_ns + SPLINE_N) <= (size_t)nr3 && size_t(st / h->dt_so3_ns + SPLINE_N) <= (size_t)nso3 && size_t(st / h->dt_ba_ns + BIAS_N) <= (size_t)nba && size_t(st / h->dt_bg_ns + BIAS_N) <= (size_t)nbg;
    };
    std::vector<size_t> idx(0);
    struct It { size_t i; };   // bisection over indices
    auto bisect = [&](size_t a, size_t b, auto pred) { while (a < b) { const size_t m = (a + b) / 2; if (pred(m)) a = m + 1; else b = m; } return a; };   // first index where pred is false
    const size_t ia = bisect(0, n_imu_in, [&](size_t i) { const double t = imu_t[i] + toff; return t < t0 || (int64_t)(t * S_TO_NS) - h->start_ns < 0; });
    const size_t ib = bisect(ia, n_imu_in, fits);
    const size_t in_window = bisect(ia, n_imu_in, [&](size_t i) { return imu_t[i] + toff < tend; }) - ia;
    h->dropped_imu = (int)(in_window - (ib - ia));
    std::vector<int> fk; fk.reserve(nf);
    for (int i = 0; i < nf; ++i) if (frame_ok[i]) fk.push_back(i);
    long total = 6 * (long)(ib - ia);
    for (int j : fk) total += 2 * (all_frames[j].c1 - all_frames[j].c0);
    const long lo = total * h->shard_rank / h->shard_world, hi = total * (h->shard_rank + 1) / h->shard_world;
    auto ceil_div6 = [](long v) { return v <= 0 ? 0L : (v + 5) / 6; };
    size_t ka = ib, kb = ia, prev_p = ia;   // this shard's sample range [ka, kb)
    long Rf = 0;                            // residuals of the kept frames seen so far
    auto take_imu = [&](size_t a, size_t b) {   // samples [a, b) lie between two frames: run_before(i) = Rf + 6 (i - ia)
      const size_t first = std::max(a, ia + (size_t)ceil_div6(lo - Rf)), last = std::min(b, ia + (size_t)ceil_div6(hi - Rf));
      if (first < last) { ka = std::min(ka, first); kb = std::max(kb, last); }
    };
    for (int j : fk) {
      const double tf = all_frames[j].t_s;
      const size_t p = bisect(prev_p, ib, [&](size_t i) { return imu_t[i] + toff < tf; });   // samples strictly before the frame
      take_imu(prev_p, p);
      const long run = Rf + 6 * (long)(p - ia);
      if (run >= lo && run < hi) frame_sel.push_back(j);
      Rf += 2 * (all_frames[j].c1 - all_frames[j].c0);
      prev_p = p;
    }
    take_imu(prev_p, ib);
    if (ka > kb) ka = kb = ia;
    // the shard's own samples: cells by bisection, readings used in place
    cells_by_bisection(ka, kb);

    return true;
  }()) {
  } else {
    frame_sel.clear();
    imu_pass(false);
    struct Unit { double t; int kind, idx, nres; };
    std::vector<Unit> units; units.reserve(nf + all_imu.size());
    for (int i = 0; i < nf; ++i) if (frame_ok[i]) units.push_back({all_frames[i].t_s, 0, i, 2 * (all_frames[i].c1 - all_frames[i].c0)});
    const size_t nfu = units.size();
    for (size_t i = 0; i < all_imu.size(); ++i) units.push_back({all_imu[i].t_s, 1, (int)i, 6});
    {   // time order with frames before IMU samples on ties (== stable sort of [frames..., imu...]); both streams are normally
        // already sorted, so merge in O(n) and only fall back to sorting when they are not
      auto lt = [](const Unit& x, const Unit& y) { return x.t < y.t; };
      if (!std::is_sorted(units.begin(), units.begin() + nfu, lt)) std::stable_sort(units.begin(), units.begin() + nfu, lt);
      if (!std::is_sorted(units.begin() + nfu, units.end(), lt)) std::stable_sort(units.begin() + nfu, units.end(), lt);
      std::vector<Unit> merged(units.size());
      std::merge(units.begin(), units.begin() + nfu, units.begin() + nfu, units.end(), merged.begin(), lt);
      units.swap(merged);
    }
    long total = 0; for (const auto& u : units) total += u.nres;
    const long lo = total * h->shard_rank / h->shard_world, hi = total * (h->shard_rank + 1) / h->shard_world;
    long run = 0;
    std::vector<int> imu_sel;
    for (const auto& u : units) { const bool mine = run >= lo && run < hi; run += u.nres; if (!mine) continue; (u.kind == 0 ? frame_sel : imu_sel).push_back(u.idx); }
    std::sort(frame_sel.begin(), frame_sel.end());
    h->imu_contig = !imu_sel.empty();
    for (size_t k = 1; k < imu_sel.size() && h->imu_contig; ++k) h->imu_contig = all_imu[imu_sel[k]].src == all_imu[imu_sel[k - 1]].src + 1;
    h->imu_src0 = imu_sel.empty() ? 0 : all_imu[imu_sel.front()].src;
    h->imu_used_t.resize(imu_sel.size()); h->imu_used_st.n = imu_sel.size();
    if (!h->imu_contig) { icc_status es = ensure_host_imu(h); if (es != ICC_OK) return es; }
    if (!h->imu_contig) { h->imu_used_acc.resize(3 * imu_sel.size()); h->imu_used_gyr.resize(3 * imu_sel.size()); }
    for (size_t k = 0; k < imu_sel.size(); ++k) {
      const ImuHost& m = all_imu[imu_sel[k]];
      const int idx = (int)k;
      h->imu_used_t[k] = m.t_s; h->imu_used_st[k] = m.st;
      if (!h->imu_contig) { memcpy(&h->imu_used_acc[3 * k], &h->imu_acc[3 * (size_t)m.src], 3 * sizeof(double)); memcpy(&h->imu_used_gyr[3 * k], &h->imu_gyr[3 * (size_t)m.src], 3 * sizeof(double)); }
      if (h->cells.empty() || h->cells.back().s_so3 != m.s_so3 || h->cells.back().s_r3 != m.s_r3 || h->cells.back().s_ba != m.s_ba || h->cells.back().s_bg != m.s_bg)
        h->cells.push_back({m.s_so3, m.s_r3, m.s_ba, m.s_bg, idx, idx});
      h->cells.back().i_end = idx + 1;
    }
  }
  h->frames.clear(); h->used_uv.clear(); h->used_pid.clear();
  h->frames.reserve(frame_sel.size());
  bool consecutive = !frame_sel.empty();
  for (size_t k = 1; k < frame_sel.size() && consecutive; ++k) consecutive = frame_sel[k] == frame_sel[k - 1] + 1;
  h->used_contig = consecutive; h->used_c0 = 0; h->used_n = 0;
  if (consecutive) {   // the usual case (all frames, or one contiguous shard): the corners are used in place, no host copy
    const int cb = all_frames[frame_sel.front()].c0, ce = all_frames[frame_sel.back()].c1;
    h->used_c0 = cb; h->used_n = ce - cb;
    for (int fi : frame_sel) { FrameHost f = all_frames[fi]; f.c0 -= cb; f.c1 -= cb; h->frames.push_back(f); }
  } else {
    { icc_status es = ensure_host_corners(h); if (es != ICC_OK) return es; }
    for (int fi : frame_sel) {
      FrameHost f = all_frames[fi];
      const int c0 = (int)h->used_pid.size();
      for (int c = f.c0; c < f.c1; ++c) { h->used_pid.push_back(h->point_ids[c]); h->used_uv.push_back(h->uv[2 * c]); h->used_uv.push_back(h->uv[2 * c + 1]); }
      f.c0 = c0; f.c1 = (int)h->used_pid.size();
      h->frames.push_back(f);
    }
    h->used_n = (int)h->used_pid.size();
  }
  trace.lap("batch_init: host assembly");
  // gravity initialisation (imu_camera_calibrator.cc:130-161) incl. the integer-second truncation of the accelerometer time
  auto view_of_time = [&](double t) { const size_t k = std::lower_bound(t_vis.begin(), t_vis.end(), t) - t_vis.begin(); return view_order[std::min(k, view_order.size() - 1)]; };
  bool ginit = false; double g0[3] = {0.0, 0.0, 9.81};   // GRAVITY_MAGN (spline_trajectory_estimator.h:29) when never initialised
  for (size_t j = 0; j < cam_ts.size() && !ginit; ++j) {
    const int vi = view_of_time(cam_ts[j]);
    const Pose Twc{qn(&h->q_wc[4 * vi]), v3(h->p_wc[3 * vi], h->p_wc[3 * vi + 1], h->p_wc[3 * vi + 2])};
    const Pose Tai = pose_mul(Twc, Tci);
    for (size_t i = 0; i < h->imu_t.size(); ++i) {
      const int64_t accl_t = (int64_t)h->imu_t[i];
      if (std::fabs(double(accl_t) - cam_ts[j]) < 1. / 30.) {
        double a3[3];
        if (h->imu_dev && h->imu_acc.size() != 3 * h->n_imu_in) { CU(cudaMemcpy(a3, h->d_acc_all.p + 3 * i, sizeof a3, cudaMemcpyDeviceToHost)); }   // one reading
        else { a3[0] = h->imu_acc[3 * i]; a3[1] = h->imu_acc[3 * i + 1]; a3[2] = h->imu_acc[3 * i + 2]; }
        const V3 g = qrot(Tai.q, v3(a3[0], a3[1], a3[2])); g0[0] = g.x; g0[1] = g.y; g0[2] = g.z; ginit = true; break; }
    }
  }
  for (int d = 0; d < 3; ++d) h->glob[G_GRAV + d] = g0[d];

  // ---- device upload ----------------------------------------------------------------------------------------------
  DeviceProblem& P = h->P;
  memset(&P, 0, sizeof P);
  P.model = h->model; P.dispatch_fov = ipp->dispatch_fov; P.n_intr = h->n_intr;
  P.n_frames = (int)h->frames.size(); P.n_corners = h->used_n; P.rolling = ipp->init_line_delay_s != 0.0 ? 1 : 0;
  if (!h->imu_lazy) h->n_imu_used = h->imu_used_t.size();
  P.n_imu = (int)h->n_imu_used; P.n_cells = (int)h->cells.size();
  P.dt_so3_ns = h->dt_so3_ns; P.dt_r3_ns = h->dt_r3_ns; P.dt_ba_ns = h->dt_ba_ns; P.dt_bg_ns = h->dt_bg_ns;
  P.inv_so3_dt = S_TO_NS / double(h->dt_so3_ns); P.inv_r3_dt = S_TO_NS / double(h->dt_r3_ns);
  P.w_acc = 1.0 / ipp->std_r3; P.w_gyr = 1.0 / ipp->std_so3;
  P.n_so3 = nso3; P.n_r3 = nr3; P.n_ba = nba; P.n_bg = nbg;
  P.n_res_vis = P.rolling ? 2 * P.n_corners : 0; P.n_res_acc = 3 * P.n_imu; P.n_res_gyr = 3 * P.n_imu;
  h->cur_flags = -1; h->initialised = true; h->cur = 0; h->state_dirty_host = false; h->knots_dirty_host = false;
  if (h->device < 0) return ICC_OK;
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));   // nothing may still read the staging arena of an earlier call
  trace.lap("batch_init: gravity init");
  h->arena.reset((size_t)(1 << 17) + 64 * (size_t)nf + 48 * (size_t)(nf + 4) + 16 * (size_t)(h->sm_count * 16 + 16) + 48 * (size_t)(nf + h->used_n / 32 + 64) + (96 + 40) * (h->cells.size() + (size_t)P.n_imu / 32 + 64)
                 + 8 * 8 * (size_t)(nf + 8) + 2 * 40 * (size_t)(nso3 + nr3 + nba + nbg + 16) + 3 * (32 * (h->points.size() / 4 + 8) + 256) + 3 * (4 * (size_t)(nso3 + nr3 + nba + nbg) + 1024), true);
  trace.lap("batch_init: pinned arena");
  {
    std::vector<double4> board(h->points.size() / 4);
    // hnormalized(T^-1 X_h) of the functor (residuals.h:357-362) == T^-1 (X / w): the division is done once here
    for (size_t i = 0; i < board.size(); ++i) { const double iw = 1.0 / h->points[4 * i + 3]; board[i] = make_double4(h->points[4 * i] * iw, h->points[4 * i + 1] * iw, h->points[4 * i + 2] * iw, 1.0); }
    CU(upload_staged(h, h->d_board, board)); P.board = h->d_board.p;   // (the evaluation kernels read the copy that belongs to the state: DeviceState::board)
    std::vector<int> off, s1, s2; std::vector<double> u1, u2;
    for (const auto& f : h->frames) { off.push_back(f.c0); s1.push_back(f.s_so3); s2.push_back(f.s_r3); u1.push_back(f.u_so3); u2.push_back(f.u_r3); }
    off.push_back(P.n_corners);
    CU(upload_staged(h, h->d_f_off, off)); CU(upload_staged(h, h->d_f_s_so3, s1)); CU(upload_staged(h, h->d_f_s_r3, s2)); CU(upload_staged(h, h->d_f_u_so3, u1)); CU(upload_staged(h, h->d_f_u_r3, u2));
    P.f_off = h->d_f_off.p; P.f_s_so3 = h->d_f_s_so3.p; P.f_s_r3 = h->d_f_s_r3.p; P.f_u_so3 = h->d_f_u_so3.p; P.f_u_r3 = h->d_f_u_r3.p;
    const bool corners_in_place = h->frames_dev && h->used_contig;   // already on the device (set_frames): used where they lie
    if (corners_in_place) { P.uv = h->d_uv_all.p + h->used_c0; P.pid = h->d_pid_all.p + h->used_c0; }
    else { CU(h->d_uv.alloc(P.n_corners)); CU(h->d_pid.alloc(P.n_corners)); P.uv = h->d_uv.p; P.pid = h->d_pid.p; }   // (u, v) pairs are already laid out as double2
    if (P.n_corners > 0 && !corners_in_place) {
      const double* uv_src = h->used_contig ? h->uv.data() + 2 * (size_t)h->used_c0 : h->used_uv.data();
      const int* pid_src = h->used_contig ? h->point_ids.data() + h->used_c0 : h->used_pid.data();
      // page-locked sources (HostBuf): the DMA transfers run behind the rest of this function; kernels follow on the same stream
      CU(cudaMemcpyAsync(h->d_uv.p, uv_src, (size_t)P.n_corners * sizeof(double2), cudaMemcpyHostToDevice, h->stream));
      CU(cudaMemcpyAsync(h->d_pid.p, pid_src, (size_t)P.n_corners * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    }
    // work lists: one warp per item; items sized so that the grid fills the GPU but every item amortises its tile flush
    const int target_items = h->sm_count * 8;
    auto round32 = [](long v) { return (int)((v + 31) / 32 * 32); };
    const int per_v = std::max(32, round32(P.n_corners / std::max(1, target_items)));
    std::vector<VisionWork> vw;
    for (int fi = 0; fi < P.n_frames; ++fi) for (int c = h->frames[fi].c0; c < h->frames[fi].c1; c += per_v) vw.push_back({fi, c, std::min(c + per_v, h->frames[fi].c1), 0});
    CU(upload_staged(h, h->d_vwork, vw)); P.vwork = h->d_vwork.p; P.n_vwork = (int)vw.size();
    const int per_i = std::max(32, round32(P.n_imu / std::max(1, target_items)));
    std::vector<ImuCell> iw;
    for (const auto& c : h->cells) for (int i = c.i_begin; i < c.i_end; i += per_i) { ImuCell s = c; s.i_begin = i; s.i_end = std::min(i + per_i, c.i_end); iw.push_back(s); }
    CU(upload_staged(h, h->d_iwork, iw)); P.iwork = h->d_iwork.p; P.n_iwork = (int)iw.size();
    CU(upload_staged(h, h->d_cells, h->cells)); P.cells = h->d_cells.p;
    {
      // Schedule of the persistent TMEM evaluation kernel (icc_eval_tmem.cu).  Both streams -- the corners of the non-empty frames and
      // the samples of the knot-interval cells, units padded to a multiple of 4 = one m8n8k4 k-step -- are walked with the kernel's own
      // chunk rule (a chunk = up to 32 stream positions from at most two consecutive units) and cut into even per-warp runs.
      struct Walk { std::vector<int> pos, unit; int total = 0; };
      auto walk = [](const std::vector<int>& poff, int n_units) { Walk w; w.total = poff[n_units];
        for (int pos = 0, u = 0; pos < w.total;) {
          while (poff[u + 1] <= pos) ++u;
          w.pos.push_back(pos); w.unit.push_back(u);
          const int nA = std::min(32, poff[u + 1] - pos);
          int n = nA;
          if (nA < 32 && u + 1 < n_units) n += std::min(32 - nA, poff[u + 2] - poff[u + 1]);
          pos += n;
        }
        return w; };
      std::vector<VisFrame> vf; vf.reserve(h->frames.size() + 2);
      std::vector<int> vpoff;
      int poff = 0;
      if (P.rolling) for (const auto& f : h->frames) {
        const int cn = f.c1 - f.c0;
        if (cn <= 0) continue;
        vf.push_back({poff, f.c0, cn, f.s_so3, f.s_r3, 0, f.u_so3, f.u_r3}); vpoff.push_back(poff);
        poff += (cn + 3) / 4 * 4;
      }
      const int nvf = (int)vf.size();
      vf.push_back({poff, 0, 0, 0, 0, 0, 0.0, 0.0}); vf.push_back({poff, 0, 0, 0, 0, 0, 0.0, 0.0});   // sentinels [n], [n+1]
      vpoff.push_back(poff); vpoff.push_back(poff);
      std::vector<ImuCellP> ic; ic.reserve(h->cells.size() + 2);
      std::vector<int> ipoff;
      poff = 0;
      for (const auto& c : h->cells) {
        const int n = c.i_end - c.i_begin;
        if (n <= 0) continue;
        ic.push_back({poff, c.i_begin, n, c.s_so3, c.s_r3, c.s_ba, c.s_bg, 0}); ipoff.push_back(poff);
        poff += (n + 3) / 4 * 4;
      }
      const int nic = (int)ic.size();
      ic.push_back({poff, 0, 0, 0, 0, 0, 0, 0}); ic.push_back({poff, 0, 0, 0, 0, 0, 0, 0});
      ipoff.push_back(poff); ipoff.push_back(poff);
      const Walk wv = walk(vpoff, nvf), wi = walk(ipoff, nic);
      const int nVc = (int)wv.pos.size(), nIc = (int)wi.pos.size(), W = h->sm_count * eval_tmem_warps();
      auto split = [W](const Walk& w) {      // even runs, one per warp
        const int nc = (int)w.pos.size(), n_items = std::min(W, nc);
        std::vector<VisItem> items((size_t)n_items);
        for (int k = 0; k < n_items; ++k) {
          const int a = (int)((int64_t)nc * k / n_items), b = (int)((int64_t)nc * (k + 1) / n_items);
          items[(size_t)k] = {w.unit[a], w.pos[a], b < nc ? w.pos[b] : w.total, 0};
        }
        return items; };
      const std::vector<VisItem> vi = split(wv), ii = split(wi);
      const int n_iit = (int)ii.size();
      P.n_vchunks = nVc; P.n_ichunks = nIc;
      CU(upload_staged(h, h->d_vframes, vf)); P.vframes = h->d_vframes.p; P.n_vframes = nvf;
      CU(upload_staged(h, h->d_vitems, vi)); P.vitems = h->d_vitems.p; P.n_vitems = (int)vi.size();
      CU(upload_staged(h, h->d_icells, ic)); P.icells = h->d_icells.p; P.n_icells = nic;
      CU(upload_staged(h, h->d_iitems, ii)); P.iitems = h->d_iitems.p; P.n_iitems = n_iit;
    }
    CU(h->d_imu_t.alloc(h->n_imu_used));
    if (h->imu_lazy && h->n_imu_used) {   // sorted fast path: the raw stamps go up, the relative integer times are derived there
      CU(h->d_imu_traw.alloc(h->n_imu_used));
      CU(cudaMemcpyAsync(h->d_imu_traw.p, h->imu_t.data() + h->imu_src0, h->n_imu_used * sizeof(double), cudaMemcpyHostToDevice, h->stream));
      launch_imu_times((int)h->n_imu_used, h->d_imu_traw.p, ipp->time_offset_imu_to_cam_s, h->start_ns, h->d_imu_t.p, h->stream);
    } else if (h->n_imu_used) CU(cudaMemcpyAsync(h->d_imu_t.p, h->imu_used_st.data(), h->n_imu_used * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
    const bool imu_in_place = h->imu_dev && h->imu_contig;   // already on the device (set_imu): used where they lie
    if (imu_in_place) { P.imu_acc = h->d_acc_all.p + 3 * (size_t)h->imu_src0; P.imu_gyr = h->d_gyr_all.p + 3 * (size_t)h->imu_src0; }
    else { CU(h->d_imu_acc.alloc(3 * (size_t)P.n_imu)); CU(h->d_imu_gyr.alloc(3 * (size_t)P.n_imu)); P.imu_acc = h->d_imu_acc.p; P.imu_gyr = h->d_imu_gyr.p; }
    if (P.n_imu > 0 && !imu_in_place) {
      const double* a_src = h->imu_contig ? h->imu_acc.data() + 3 * (size_t)h->imu_src0 : h->imu_used_acc.data();
      const double* g_src = h->imu_contig ? h->imu_gyr.data() + 3 * (size_t)h->imu_src0 : h->imu_used_gyr.data();
      CU(cudaMemcpyAsync(h->d_imu_acc.p, a_src, 3 * (size_t)P.n_imu * sizeof(double), cudaMemcpyHostToDevice, h->stream));
      CU(cudaMemcpyAsync(h->d_imu_gyr.p, g_src, 3 * (size_t)P.n_imu * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    }
    P.imu_t_ns = h->d_imu_t.p;
  }
  trace.lap("batch_init: problem upload");
  icc_status s = upload_state(h, 0, true); if (s != ICC_OK) return s;
  s = upload_state(h, 1, true); if (s != ICC_OK) return s;
  trace.lap("batch_init: state upload");
  {   // knots: BatchInitSO3R3VisPoses on the device, written into both state copies (the zero knots uploaded above only sized them)
    std::vector<double> tv, qv, pv;
    tv.reserve(view_order.size()); qv.reserve(4 * view_order.size()); pv.reserve(3 * view_order.size());
    for (const int i : view_order) { tv.push_back(h->frame_t[i]); for (int d = 0; d < 4; ++d) qv.push_back(h->q_wc[4 * i + d]); for (int d = 0; d < 3; ++d) pv.push_back(h->p_wc[3 * i + d]); }
    CU(upload_staged(h, h->d_view_t, tv)); CU(upload_staged(h, h->d_view_q, qv)); CU(upload_staged(h, h->d_view_p, pv));
    const double Tci7[7] = {Tci.q.x, Tci.q.y, Tci.q.z, Tci.q.w, Tci.t.x, Tci.t.y, Tci.t.z};
    launch_init_knots((int)tv.size(), h->d_view_t.p, h->d_view_q.p, h->d_view_p.p, Tci7, nso3, h->dt_so3_ns, nr3, h->dt_r3_ns,
                      h->st[0].so3.p, h->st[1].so3.p, h->st[0].r3.p, h->st[1].r3.p, h->stream);
    h->knots_dirty_host = true;     // the device holds the knots; the host mirror is refreshed on demand (getters / setters)
  }
  trace.lap("batch_init: knot init");
  return ICC_OK;
}

icc_status icc_set_known_gravity_dir(icc_handle* h, const double g[3]) {
  if (!h || !g) return ICC_ERR_INVALID_ARGUMENT;
  if (h->state_dirty_host) { icc_status s = sync_state_to_host(h); if (s != ICC_OK) return s; }   // (knots alone being newer on the device does not matter here)
  for (int d = 0; d < 3; ++d) h->glob[G_GRAV + d] = g[d];
  if (h->device >= 0 && h->initialised) {   // only the globals block changed: one small staged copy instead of the whole state
    CU(cudaSetDevice(h->device));
    CU(upload_staged(h, h->st[h->cur].glob, std::vector<double>(h->glob, h->glob + G_COUNT)));
    return ICC_OK;
  }
  return push_state_to_device(h);
}

icc_status icc_optimize(icc_handle* h, int max_iterations, int flags, icc_summary* summary) {
  if (!h) return ICC_ERR_INVALID_ARGUMENT;
  NEED_DEVICE();
  if (!h->initialised) return fail(h, ICC_ERR_STATE, "icc_batch_init_spline must be called first");
  CU(cudaSetDevice(h->device));
  icc_summary S;
  icc_status s = run_lm(h, max_iterations, flags, true, &S); if (s != ICC_OK) return s;
  const int l0 = kernel_launch_count();
  PhaseTrace trace(h->stream);
  s = mean_reproj(h, &S.mean_reproj_error); if (s != ICC_OK) return s;
  trace.lap("optimize: mean reprojection error");
  S.gpu_launches += kernel_launch_count() - l0;
  if (summary) *summary = S;
  return ICC_OK;
}
icc_status icc_lm_iterations(icc_handle* h, int n, int flags, icc_summary* summary) {
  if (!h) return ICC_ERR_INVALID_ARGUMENT;
  NEED_DEVICE();
  if (!h->initialised) return fail(h, ICC_ERR_STATE, "icc_batch_init_spline must be called first");
  CU(cudaSetDevice(h->device));
  return run_lm(h, n, flags, false, summary);
}

icc_status icc_get_T_i_c(const icc_handle* hc, double T[7]) { icc_handle* h = const_cast<icc_handle*>(hc); if (!h || !T) return ICC_ERR_INVALID_ARGUMENT; icc_status s = sync_globals_to_host(h); if (s != ICC_OK) return s; memcpy(T, h->glob + G_TIC, 7 * sizeof(double)); return ICC_OK; }
icc_status icc_get_gravity(const icc_handle* hc, double g[3]) { icc_handle* h = const_cast<icc_handle*>(hc); if (!h || !g) return ICC_ERR_INVALID_ARGUMENT; icc_status s = sync_globals_to_host(h); if (s != ICC_OK) return s; memcpy(g, h->glob + G_GRAV, 3 * sizeof(double)); return ICC_OK; }
icc_status icc_get_line_delay(const icc_handle* hc, double* ld) { icc_handle* h = const_cast<icc_handle*>(hc); if (!h || !ld) return ICC_ERR_INVALID_ARGUMENT; icc_status s = sync_globals_to_host(h); if (s != ICC_OK) return s; *ld = h->glob[G_LD]; return ICC_OK; }
icc_status icc_get_camera_intrinsics(const icc_handle* hc, double* k, int n) { icc_handle* h = const_cast<icc_handle*>(hc); if (!h || !k) return ICC_ERR_INVALID_ARGUMENT; icc_status s = sync_globals_to_host(h); if (s != ICC_OK) return s; for (int i = 0; i < n && i < h->n_intr; ++i) k[i] = h->initialised ? h->glob[G_CAM_INTR + i] : h->intr[i]; return ICC_OK; }
icc_status icc_get_time_offset(const icc_handle* hc, double* t) { icc_handle* h = const_cast<icc_handle*>(hc); if (!h || !t) return ICC_ERR_INVALID_ARGUMENT; icc_status s = sync_globals_to_host(h); if (s != ICC_OK) return s; *t = h->ip.time_offset_imu_to_cam_s + h->glob[G_TOFF]; return ICC_OK; }
icc_status icc_get_num_knots(const icc_handle* h, int* a, int* b, int* c, int* d) {
  if (!h) return ICC_ERR_INVALID_ARGUMENT;
  if (a) *a = (int)h->so3.size() / 4; if (b) *b = (int)h->r3.size() / 3; if (c) *c = (int)h->ba.size() / 3; if (d) *d = (int)h->bg.size() / 3;
  return ICC_OK;
}
icc_status icc_get_knots(const icc_handle* hc, double* so3, double* r3, double* ba, double* bg) {
  icc_handle* h = const_cast<icc_handle*>(hc); if (!h) return ICC_ERR_INVALID_ARGUMENT;
  icc_status s = sync_state_to_host(h); if (s != ICC_OK) return s;
  if (so3) std::copy(h->so3.begin(), h->so3.end(), so3);
  if (r3) std::copy(h->r3.begin(), h->r3.end(), r3);
  if (ba) std::copy(h->ba.begin(), h->ba.end(), ba);
  if (bg) std::copy(h->bg.begin(), h->bg.end(), bg);
  return ICC_OK;
}
icc_status icc_set_knots(icc_handle* h, const double* so3, const double* r3, const double* ba, const double* bg) {
  if (!h) return ICC_ERR_INVALID_ARGUMENT;
  icc_status s = sync_state_to_host(h); if (s != ICC_OK) return s;
  if (so3) std::copy(so3, so3 + h->so3.size(), h->so3.begin());
  if (r3) std::copy(r3, r3 + h->r3.size(), h->r3.begin());
  if (ba) std::copy(ba, ba + h->ba.size(), h->ba.begin());
  if (bg) std::copy(bg, bg + h->bg.size(), h->bg.begin());
  return push_state_to_device(h);
}
icc_status icc_set_T_i_c(icc_handle* h, const double T[7]) { if (!h || !T) return ICC_ERR_INVALID_ARGUMENT; icc_status s = sync_state_to_host(h); if (s != ICC_OK) return s; memcpy(h->glob + G_TIC, T, 7 * sizeof(double)); return push_state_to_device(h); }
icc_status icc_set_line_delay(icc_handle* h, double ld) { if (!h) return ICC_ERR_INVALID_ARGUMENT; icc_status s = sync_state_to_host(h); if (s != ICC_OK) return s; h->glob[G_LD] = ld; return push_state_to_device(h); }
icc_status icc_get_mean_reprojection_error(icc_handle* h, double* e) {
  if (!h || !e) return ICC_ERR_INVALID_ARGUMENT;
  NEED_DEVICE();
  if (!h->initialised) return fail(h, ICC_ERR_STATE, "icc_batch_init_spline must be called first");
  CU(cudaSetDevice(h->device));
  return mean_reproj(h, e);
}
icc_status icc_get_num_imu_cells(const icc_handle* h, int* n) { if (!h || !n) return ICC_ERR_INVALID_ARGUMENT; *n = (int)h->cells.size(); return ICC_OK; }
icc_status icc_get_imu_cells(const icc_handle* h, int32_t* c6) {
  if (!h || !c6) return ICC_ERR_INVALID_ARGUMENT;
  for (size_t k = 0; k < h->cells.size(); ++k) { const ImuCell& c = h->cells[k]; int32_t* o = c6 + 6 * k; o[0] = c.s_so3; o[1] = c.s_r3; o[2] = c.s_ba; o[3] = c.s_bg; o[4] = c.i_begin; o[5] = c.i_end; }
  return ICC_OK;
}
icc_status icc_get_num_imu_used(const icc_handle* h, int* n) { if (!h || !n) return ICC_ERR_INVALID_ARGUMENT; *n = (int)h->n_imu_used; return ICC_OK; }
icc_status icc_get_imu_used(const icc_handle* hc, double* t, double* a, double* g) {
  icc_handle* h = const_cast<icc_handle*>(hc);
  if (!h) return ICC_ERR_INVALID_ARGUMENT;
  if (a || g) { icc_status es = ensure_host_imu(h); if (es != ICC_OK) return es; }
  const size_t nu = h->n_imu_used;
  if (t) { if (h->imu_lazy) { for (size_t k = 0; k < nu; ++k) t[k] = h->imu_t[h->imu_src0 + k] + h->ip.time_offset_imu_to_cam_s; } else std::copy(h->imu_used_t.begin(), h->imu_used_t.end(), t); }
  if (a) { const double* src = h->imu_contig ? h->imu_acc.data() + 3 * (size_t)h->imu_src0 : h->imu_used_acc.data(); std::copy(src, src + 3 * nu, a); }
  if (g) { const double* src = h->imu_contig ? h->imu_gyr.data() + 3 * (size_t)h->imu_src0 : h->imu_used_gyr.data(); std::copy(src, src + 3 * nu, g); }
  return ICC_OK;
}

icc_status icc_eval_trajectory(icc_handle* h, int n, const int64_t* t_ns, double* gyro, double* accel, double* gb, double* ab, double* pq, double* pp, int32_t* valid) {
  if (!h || n < 0 || (n > 0 && !t_ns)) return ICC_ERR_INVALID_ARGUMENT;
  NEED_DEVICE();
  if (!h->initialised) return fail(h, ICC_ERR_STATE, "icc_batch_init_spline must be called first");
  if (n == 0) return ICC_OK;
  CU(cudaSetDevice(h->device));
  DevBuf<int64_t> d_t; DevBuf<double> d_out; DevBuf<int> d_valid;
  std::vector<int64_t> tv(t_ns, t_ns + n);
  CU(d_t.upload(tv)); CU(d_out.alloc((size_t)n * 19)); CU(d_valid.alloc(n));
  CU(cudaMemsetAsync(d_out.p, 0, (size_t)n * 19 * sizeof(double), h->stream));
  double* o = d_out.p;
  launch_eval_trajectory(h->P, h->st[h->cur].view(), n, d_t.p, h->start_ns, o, o + 3 * n, o + 6 * n, o + 9 * n, o + 12 * n, o + 16 * n, d_valid.p, h->stream);
  std::vector<double> ho((size_t)n * 19); std::vector<int> hv(n);
  CU(cudaMemcpyAsync(ho.data(), d_out.p, ho.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(hv.data(), d_valid.p, n * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  for (int i = 0; i < n; ++i) {
    const bool v = hv[i] != 0;
    if (valid) valid[i] = hv[i];
    // like the reference getters, outputs are only written where CalcTimes accepts the timestamp (gyro needs SO3 only,
    // but the hot CLI queries inside the spline range where both hold)
    if (gyro && v) for (int d = 0; d < 3; ++d) gyro[3 * i + d] = ho[3 * i + d];
    if (accel && v) for (int d = 0; d < 3; ++d) accel[3 * i + d] = ho[3 * n + 3 * i + d];
    if (gb) for (int d = 0; d < 3; ++d) gb[3 * i + d] = ho[6 * n + 3 * i + d];
    if (ab) for (int d = 0; d < 3; ++d) ab[3 * i + d] = ho[9 * n + 3 * i + d];
    if (pq && v) for (int d = 0; d < 4; ++d) pq[4 * i + d] = ho[12 * n + 4 * i + d];
    if (pp && v) for (int d = 0; d < 3; ++d) pp[3 * i + d] = ho[16 * n + 3 * i + d];
  }
  return ICC_OK;
}

icc_status icc_num_residuals(const icc_handle* h, int* v, int* a, int* g) {
  if (!h) return ICC_ERR_INVALID_ARGUMENT;
  if (v) *v = h->P.n_res_vis; if (a) *a = h->P.n_res_acc; if (g) *g = h->P.n_res_gyr;
  return ICC_OK;
}
icc_status icc_num_tangent(const icc_handle* hc, int flags, int* n) {
  icc_handle* h = const_cast<icc_handle*>(hc);
  if (!h || !n) return ICC_ERR_INVALID_ARGUMENT;
  if (!h->initialised) return fail(h, ICC_ERR_STATE, "icc_batch_init_spline must be called first");
  icc_status s = configure(h, flags); if (s != ICC_OK) return s;
  *n = h->n_tan; return ICC_OK;
}

icc_status icc_evaluate(icc_handle* h, int flags, double* cost, double* residuals, double* gradient, double* hessian) {
  if (!h) return ICC_ERR_INVALID_ARGUMENT;
  NEED_DEVICE();
  if (!h->initialised) return fail(h, ICC_ERR_STATE, "icc_batch_init_spline must be called first");
  CU(cudaSetDevice(h->device));
  icc_status s = configure(h, flags); if (s != ICC_OK) return s;
  const DeviceProblem& P = h->P;
  const int nres = P.n_res_vis + P.n_res_acc + P.n_res_gyr, n = h->n_tan;
  double* res_dev = nullptr;
  if (residuals) { CU(h->d_res.alloc((size_t)std::max(1, nres))); CU(cudaMemsetAsync(h->d_res.p, 0, (size_t)nres * sizeof(double), h->stream)); res_dev = h->d_res.p; }
  if (!gradient && !hessian) {
    CU(cudaMemsetAsync(h->d_scal.p, 0, SC_COUNT * sizeof(double), h->stream));
    s = eval_cost(h, h->st[h->cur].view(), h->d_scal.p + SC_CAND_COST, res_dev, nullptr); if (s != ICC_OK) return s;
    double c; CU(cudaMemcpyAsync(&c, h->d_scal.p + SC_CAND_COST, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (residuals) CU(cudaMemcpyAsync(residuals, res_dev, (size_t)nres * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (cost) *cost = c;
    return ICC_OK;
  }
  s = eval_jacobian(h, h->st[h->cur].view(), res_dev); if (s != ICC_OK) return s;
  std::vector<double> ne((size_t)P.ne_size);
  CU(cudaMemcpyAsync(ne.data(), P.ne, ne.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (residuals) CU(cudaMemcpyAsync(residuals, res_dev, (size_t)nres * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  if (cost) *cost = ne[P.ne_off_cost];
  if (gradient) for (int i = 0; i < n; ++i) gradient[i] = ne[P.ne_off_g + h->perm[i]];
  if (hessian) dense_hessian(h, ne, hessian);
  return ICC_OK;
}

// J^T J products with caller-supplied vectors (canonical tangent order, nvec columns stored one after the other): the packed
// banded + bordered normal equations are read back once and multiplied on the host.  Evaluation / parity helper: a dense Hessian of
// BASELINE config 4 would be 1.2 GB, a handful of products check every stored entry of J^T J at full size.
icc_status icc_normal_matvec(icc_handle* h, int flags, int nvec, const double* V, double* HV) {
  if (!h || nvec <= 0 || !V || !HV) return ICC_ERR_INVALID_ARGUMENT;
  NEED_DEVICE();
  if (!h->initialised) return fail(h, ICC_ERR_STATE, "icc_batch_init_spline must be called first");
  CU(cudaSetDevice(h->device));
  icc_status s = configure(h, flags); if (s != ICC_OK) return s;
  const DeviceProblem& P = h->P;
  const int n = h->n_tan, nk = P.nk, nb = P.nb;
  s = eval_jacobian(h, h->st[h->cur].view(), nullptr); if (s != ICC_OK) return s;
  std::vector<double> ne((size_t)P.ne_size);
  CU(cudaMemcpyAsync(ne.data(), P.ne, ne.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  std::vector<double> x((size_t)n), y((size_t)n);
  for (int v = 0; v < nvec; ++v) {
    for (int i = 0; i < n; ++i) x[h->perm[i]] = V[(size_t)v * n + i];
    std::fill(y.begin(), y.end(), 0.0);
    for (int lo = 0; lo < nk; ++lo) {
      const double* col = &ne[(size_t)lo * P.ldb];
      y[lo] += col[0] * x[lo];
      for (int d = 1; d <= P.kd && lo + d < nk; ++d) { y[lo] += col[d] * x[lo + d]; y[lo + d] += col[d] * x[lo]; }
      const double* e = &ne[P.ne_off_E + (size_t)lo * nb];
      for (int b = 0; b < nb; ++b) { y[lo] += e[b] * x[nk + b]; y[nk + b] += e[b] * x[lo]; }
    }
    for (int hi = 0; hi < nb; ++hi) for (int lo = 0; lo <= hi; ++lo) {
      const double c = ne[P.ne_off_C + (size_t)hi * nb + lo];
      y[nk + hi] += c * x[nk + lo]; if (lo != hi) y[nk + lo] += c * x[nk + hi];
    }
    for (int i = 0; i < n; ++i) HV[(size_t)v * n + i] = y[h->perm[i]];
  }
  return ICC_OK;
}

// The elimination plan of the damped solve for `flags` (host only: works on a host-only handle).  chunks > 0 forces the level-0
// chunk count, which then goes through the same clamping and halving as the automatic choice.
icc_status icc_get_solver_plan(icc_handle* h, int flags, int chunks, int32_t* plan16) {
  if (!h || !plan16 || chunks < 0) return ICC_ERR_INVALID_ARGUMENT;
  if (!h->initialised) return fail(h, ICC_ERR_STATE, "icc_batch_init_spline must be called first");
  icc_status s = configure(h, flags); if (s != ICC_OK) return s;
  solve_plan_info(h->P, chunks, plan16);
  return ICC_OK;
}

// One damped solve at the current state, outside the LM driver: one Jacobian evaluation, the Jacobi scale of THAT evaluation, one
// launch_solve.  Outputs (canonical tangent order, each nullable) all come from the same evaluation, so a host reference can rebuild
// exactly the system the kernels factored.  Leaves the state, the LM scale and the LM bookkeeping untouched.
icc_status icc_solve_step(icc_handle* h, int flags, double radius, int chunks, double* cost, double* gradient, double* hessian_dense,
                          double* scale, double* lm_diag, double* delta, double* model_change) {
  if (!h || !(radius > 0.0) || chunks < 0) return ICC_ERR_INVALID_ARGUMENT;
  NEED_DEVICE();
  if (!h->initialised) return fail(h, ICC_ERR_STATE, "icc_batch_init_spline must be called first");
  CU(cudaSetDevice(h->device));
  icc_status s = configure(h, flags); if (s != ICC_OK) return s;
  const DeviceProblem& P = h->P;
  const int n = h->n_tan;
  if (n == 0) return fail(h, ICC_ERR_INVALID_ARGUMENT, "no free parameters for these flags");
  int32_t plan[16]; solve_plan_info(P, chunks, plan);
  if (!plan[0]) return fail(h, ICC_ERR_UNSUPPORTED, "the border (bias knots + globals) is too wide for the solver's shared-memory plans");
  DevBuf<double> d_scale, d_delta, d_scal, d_ws;
  CU(d_scale.alloc((size_t)n)); CU(d_delta.alloc((size_t)n)); CU(d_scal.alloc(SC_COUNT));
  double* ws = h->d_ws.p;
  if (chunks > 0) { CU(d_ws.alloc(solve_workspace_doubles(P, chunks))); ws = d_ws.p; }
  s = eval_jacobian(h, h->st[h->cur].view(), nullptr); if (s != ICC_OK) { cudaStreamSynchronize(h->stream); return s; }
  CU(cudaMemsetAsync(d_scal.p, 0, SC_COUNT * sizeof(double), h->stream));
  launch_compute_scale(P, d_scale.p, h->opt.jacobi_scaling, d_scal.p, h->stream);
  SolveParams sp; sp.radius = radius; sp.min_diag = h->opt.min_lm_diagonal; sp.max_diag = h->opt.max_lm_diagonal; sp.jacobi_scaling = h->opt.jacobi_scaling;
  const int se = launch_solve(P, d_scale.p, sp, ws, d_delta.p, d_scal.p, h->stream, chunks);
  if (se) { cudaStreamSynchronize(h->stream); return fail(h, ICC_ERR_CUDA, std::string("solver launch: ") + cudaGetErrorString(cudaGetLastError())); }
  std::vector<double> ne((size_t)P.ne_size), sc_h((size_t)n), dl_h((size_t)n);
  double sc[SC_COUNT];
  CU(cudaMemcpyAsync(ne.data(), P.ne, ne.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(sc_h.data(), d_scale.p, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(dl_h.data(), d_delta.p, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(sc, d_scal.p, sizeof sc, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  if (sc[SC_OK] != 1.0) return fail(h, ICC_ERR_NUMERIC, "the factorisation met a non-positive pivot");
  // diagonal of H in solver order; the LM diagonal is the same expression as the kernels' lm_d2
  auto diag = [&](int i) { return i < P.nk ? ne[(size_t)i * P.ldb] : ne[P.ne_off_C + (size_t)(i - P.nk) * P.nb + (i - P.nk)]; };
  for (int i = 0; i < n; ++i) {
    const int j = h->perm[i];
    if (gradient) gradient[i] = ne[P.ne_off_g + j];
    if (scale) scale[i] = sc_h[j];
    if (lm_diag) lm_diag[i] = std::fmin(std::fmax(diag(j) * sc_h[j] * sc_h[j], sp.min_diag), sp.max_diag) / sp.radius;
    if (delta) delta[i] = dl_h[j];
  }
  if (cost) *cost = ne[P.ne_off_cost];
  if (model_change) *model_change = sc[SC_MODEL_CHANGE];
  if (hessian_dense) dense_hessian(h, ne, hessian_dense);
  return ICC_OK;
}

icc_status icc_time_evaluations(icc_handle* h, int n, int flags, int with_jacobian, double* ms_per_eval) {
  if (!h || !ms_per_eval || n <= 0) return ICC_ERR_INVALID_ARGUMENT;
  NEED_DEVICE();
  if (!h->initialised) return fail(h, ICC_ERR_STATE, "icc_batch_init_spline must be called first");
  CU(cudaSetDevice(h->device));
  icc_status s = configure(h, flags); if (s != ICC_OK) return s;
  cudaEvent_t e0, e1; CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
  CU(cudaMemsetAsync(h->d_scal.p, 0, SC_COUNT * sizeof(double), h->stream));
  CU(cudaEventRecord(e0, h->stream));
  for (int i = 0; i < n; ++i) {
    if (with_jacobian == 1) { s = eval_jacobian(h, h->st[h->cur].view(), nullptr); }
    else if (with_jacobian == 2 || with_jacobian == 3) {   // one kernel family only (2 = vision, 3 = imu), Jacobian mode, no memset
      DeviceProblem Q = h->P; if (with_jacobian == 2) Q.n_iwork = 0; else { Q.n_vwork = 0; Q.n_vitems = 0; }
      if (with_jacobian == 2) Q.n_iitems = 0;
      s = launch_eval(Q, h->st[h->cur].view(), true, nullptr, nullptr, nullptr, h->stream) ? fail(h, ICC_ERR_CUDA, "eval launch failed") : ICC_OK;
    }
    else { s = eval_cost(h, h->st[h->cur].view(), h->d_scal.p + SC_CAND_COST, nullptr, nullptr); }
    if (s != ICC_OK) return s;
  }
  CU(cudaEventRecord(e1, h->stream));
  CU(cudaEventSynchronize(e1));
  float ms = 0; CU(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  *ms_per_eval = ms / n;
  return ICC_OK;
}

void* icc_get_stream(icc_handle* h) { return h ? (void*)h->stream : nullptr; }
// ---- upstream row f1: per-view board poses ---------------------------------------------------------------------------
icc_status icc_pixels_to_normalized(icc_handle* h, int n, const double* uv, double* xy_out, int32_t* ok) {
  if (!h || n < 0 || (n > 0 && (!uv || !xy_out))) return ICC_ERR_INVALID_ARGUMENT;
  if (h->device < 0) return fail(h, ICC_ERR_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
  if (h->model < 0) return fail(h, ICC_ERR_STATE, "icc_set_camera must be called first");
  if (n == 0) return ICC_OK;
  CU(cudaSetDevice(h->device));
  DevBuf<double2> d_uv, d_xy; DevBuf<int> d_ok;
  CU(d_uv.alloc(n)); CU(d_xy.alloc(n)); CU(d_ok.alloc(n));
  CU(cudaMemcpyAsync(d_uv.p, uv, (size_t)n * sizeof(double2), cudaMemcpyHostToDevice, h->stream));
  launch_unproject(h->model, h->intr, n, d_uv.p, d_xy.p, d_ok.p, h->stream);
  CU(cudaMemcpyAsync(xy_out, d_xy.p, (size_t)n * sizeof(double2), cudaMemcpyDeviceToHost, h->stream));
  std::vector<int> okh(ok ? n : 0);
  if (ok) CU(cudaMemcpyAsync(okh.data(), d_ok.p, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  if (ok) for (int i = 0; i < n; ++i) ok[i] = okh[i];
  return ICC_OK;
}

icc_status icc_estimate_board_poses(icc_handle* h, int nf, const int32_t* off, const int32_t* ids, const double* uv, double max_reproj_error, int min_points,
                                    double* q_wc, double* p_wc, double* mean_err, int32_t* valid) {
  if (!h || nf <= 0 || !off || !ids || !uv || !q_wc || !p_wc || !valid) return ICC_ERR_INVALID_ARGUMENT;
  if (h->device < 0) return fail(h, ICC_ERR_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
  if (h->model < 0 || h->points.empty()) return fail(h, ICC_ERR_STATE, "icc_set_camera and icc_set_board_points must be called first");
  for (int i = 0; i < nf; ++i) if (off[i + 1] < off[i]) return fail(h, ICC_ERR_INVALID_ARGUMENT, "corner offsets must be non-decreasing");
  const int nc = off[nf] - off[0];
  if (off[0] != 0) return fail(h, ICC_ERR_INVALID_ARGUMENT, "corner offsets must start at 0");
  CU(cudaSetDevice(h->device));
  const int np = (int)(h->points.size() / 4);
  std::vector<double4> board(np);
  for (int i = 0; i < np; ++i) board[i] = make_double4(h->points[4 * i], h->points[4 * i + 1], h->points[4 * i + 2], h->points[4 * i + 3]);
  DevBuf<double4> d_board; DevBuf<int> d_off, d_pid, d_ok, d_valid; DevBuf<double2> d_uv, d_xy; DevBuf<unsigned char> d_use; DevBuf<double> d_q, d_p, d_e;
  CU(d_board.upload(board));
  CU(d_off.alloc(nf + 1)); CU(d_pid.alloc(std::max(1, nc))); CU(d_uv.alloc(std::max(1, nc))); CU(d_xy.alloc(std::max(1, nc))); CU(d_ok.alloc(std::max(1, nc))); CU(d_use.alloc(std::max(1, nc)));
  CU(d_q.alloc(4 * (size_t)nf)); CU(d_p.alloc(3 * (size_t)nf)); CU(d_e.alloc(nf)); CU(d_valid.alloc(nf));
  CU(cudaMemcpyAsync(d_off.p, off, (size_t)(nf + 1) * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  if (nc > 0) {
    CU(cudaMemcpyAsync(d_pid.p, ids, (size_t)nc * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(d_uv.p, uv, (size_t)nc * sizeof(double2), cudaMemcpyHostToDevice, h->stream));
  }
  launch_unproject(h->model, h->intr, nc, d_uv.p, d_xy.p, d_ok.p, h->stream);
  PoseProblem Q; memset(&Q, 0, sizeof Q);
  Q.model = h->model; for (int i = 0; i < 10; ++i) Q.intr[i] = h->intr[i];
  Q.n_frames = nf; Q.n_points = np; Q.min_points = min_points > 0 ? min_points : 8;
  Q.board = d_board.p; Q.f_off = d_off.p; Q.pid = d_pid.p;
  const double W = h->width, H = h->height;
  const double max_px = max_reproj_error > 0.0 ? max_reproj_error : 0.004 * H;            // pose_estimator.cc:97
  Q.thresh_sq = (W > 0 && H > 0) ? max_px / std::sqrt(W * W + H * H) : 1e-3;               // :101 (compared with a SQUARED error by theia's RANSAC)
  Q.max_err = max_px;                                                                       // :181 (pixels against a normalised error, as in the reference)
  launch_board_poses(Q, d_xy.p, d_ok.p, d_use.p, d_q.p, d_p.p, d_e.p, d_valid.p, h->stream);
  std::vector<double> eh(nf); std::vector<int> vh(nf);
  CU(cudaMemcpyAsync(q_wc, d_q.p, 4 * (size_t)nf * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(p_wc, d_p.p, 3 * (size_t)nf * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(eh.data(), d_e.p, (size_t)nf * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(vh.data(), d_valid.p, (size_t)nf * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  if (cudaGetLastError() != cudaSuccess) return fail(h, ICC_ERR_CUDA, "pose kernels failed");
  for (int i = 0; i < nf; ++i) { valid[i] = vh[i]; if (mean_err) mean_err[i] = eh[i]; }
  return ICC_OK;
}

icc_status icc_filter_bad_poses(icc_handle* h, int nv, const double* p_wc, int32_t* valid) {
  if (nv <= 0 || !p_wc || !valid) return ICC_ERR_INVALID_ARGUMENT;
  std::vector<double> z; for (int i = 0; i < nv; ++i) if (valid[i]) z.push_back(p_wc[3 * i + 2]);
  if (z.empty()) return ICC_OK;
  const size_t n = z.size(); double med;   // utils::MedianOfDoubleVec (src/utils/utils.cc:77-97)
  if (n % 2 == 0) { std::nth_element(z.begin(), z.begin() + n / 2 - 1, z.end()); const double e1 = z[n / 2 - 1]; std::nth_element(z.begin(), z.begin() + n / 2, z.end()); med = (e1 + z[n / 2]) / 2; }
  else { std::nth_element(z.begin(), z.begin() + n / 2, z.end()); med = z[n / 2]; }
  for (int i = 0; i < nv; ++i) if (valid[i] && std::fabs(p_wc[3 * i + 2] - med) > std::fabs(med)) valid[i] = 0;
  (void)h;
  return ICC_OK;
}

icc_status icc_get_board_points(const icc_handle* h, double* xyzw, int n) {
  if (!h || !xyzw || n < 0) return ICC_ERR_INVALID_ARGUMENT;
  { icc_status s = sync_state_to_host(const_cast<icc_handle*>(h)); if (s != ICC_OK) return s; }   // POINTS: the optimised points live in the device state
  const size_t m = std::min<size_t>(4 * (size_t)n, h->points.size());
  std::copy(h->points.begin(), h->points.begin() + m, xyzw);
  return ICC_OK;
}

icc_status icc_optimize_board_points(icc_handle* h, int nf, const int32_t* off, const int32_t* ids, const double* uv, double max_reproj_error, int min_points,
                                     int min_observations, double* q_wc, double* p_wc, double* mean_err, int32_t* valid, double* board_out, int32_t* n_opt_out) {
  if (!h || nf <= 0 || !off || !ids || !uv || !q_wc || !p_wc || !valid) return ICC_ERR_INVALID_ARGUMENT;
  if (h->device < 0) return fail(h, ICC_ERR_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
  if (h->model < 0 || h->points.empty()) return fail(h, ICC_ERR_STATE, "icc_set_camera and icc_set_board_points must be called first");
  if (off[0] != 0) return fail(h, ICC_ERR_INVALID_ARGUMENT, "corner offsets must start at 0");
  for (int i = 0; i < nf; ++i) if (off[i + 1] < off[i]) return fail(h, ICC_ERR_INVALID_ARGUMENT, "corner offsets must be non-decreasing");
  const int nc = off[nf], np = (int)(h->points.size() / 4);
  CU(cudaSetDevice(h->device));
  cudaStream_t st = h->stream;
  std::vector<double4> board(np);
  for (int i = 0; i < np; ++i) board[i] = make_double4(h->points[4 * i], h->points[4 * i + 1], h->points[4 * i + 2], h->points[4 * i + 3]);
  std::vector<int> obs_view(std::max(1, nc));
  for (int f = 0; f < nf; ++f) for (int c = off[f]; c < off[f + 1]; ++c) obs_view[c] = f;
  DevBuf<double4> d_board, d_board2; DevBuf<int> d_off, d_pid, d_ok, d_valid, d_view, d_pt_off, d_pt_obs, d_opt; DevBuf<double2> d_uv, d_xy; DevBuf<unsigned char> d_use;
  DevBuf<double> d_q, d_p, d_e, d_qcw, d_c;
  CU(d_board.upload(board)); CU(d_board2.alloc(np)); CU(d_opt.alloc(np));
  CU(d_off.alloc(nf + 1)); CU(d_pid.alloc(std::max(1, nc))); CU(d_uv.alloc(std::max(1, nc))); CU(d_xy.alloc(std::max(1, nc))); CU(d_ok.alloc(std::max(1, nc))); CU(d_use.alloc(std::max(1, nc)));
  CU(d_q.alloc(4 * (size_t)nf)); CU(d_p.alloc(3 * (size_t)nf)); CU(d_e.alloc(nf)); CU(d_valid.alloc(nf)); CU(d_view.upload(obs_view));
  CU(cudaMemcpyAsync(d_off.p, off, (size_t)(nf + 1) * sizeof(int), cudaMemcpyHostToDevice, st));
  if (nc > 0) {
    CU(cudaMemcpyAsync(d_pid.p, ids, (size_t)nc * sizeof(int), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_uv.p, uv, (size_t)nc * sizeof(double2), cudaMemcpyHostToDevice, st));
  }
  CU(cudaMemcpyAsync(d_q.p, q_wc, 4 * (size_t)nf * sizeof(double), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d_p.p, p_wc, 3 * (size_t)nf * sizeof(double), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d_valid.p, valid, (size_t)nf * sizeof(int), cudaMemcpyHostToDevice, st));
  CU(cudaMemsetAsync(d_e.p, 0, (size_t)nf * sizeof(double), st));   // views that are not valid keep a zero error
  launch_unproject(h->model, h->intr, nc, d_uv.p, d_xy.p, d_ok.p, st);
  PoseProblem Q; memset(&Q, 0, sizeof Q);
  Q.model = h->model; for (int i = 0; i < 10; ++i) Q.intr[i] = h->intr[i];
  Q.n_frames = nf; Q.n_points = np; Q.min_points = min_points > 0 ? min_points : 8;
  Q.board = d_board.p; Q.f_off = d_off.p; Q.pid = d_pid.p; Q.refine_only = 1;
  const double W = h->width, H = h->height;
  const double max_px = max_reproj_error > 0.0 ? max_reproj_error : 0.004 * H;
  Q.thresh_sq = (W > 0 && H > 0) ? max_px / std::sqrt(W * W + H * H) : 1e-3;
  Q.max_err = max_px;
  // 1. the stored poses and their inlier sets (what the pose dataset holds after EstimatePosesFromJson)
  launch_board_poses(Q, d_xy.p, d_ok.p, d_use.p, d_q.p, d_p.p, d_e.p, d_valid.p, st);
  std::vector<unsigned char> use(std::max(1, nc)); std::vector<int> vh(nf); std::vector<double> qh(4 * (size_t)nf), ph(3 * (size_t)nf);
  CU(cudaMemcpyAsync(use.data(), d_use.p, (size_t)std::max(1, nc), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(vh.data(), d_valid.p, (size_t)nf * sizeof(int), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(qh.data(), d_q.p, qh.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(ph.data(), d_p.p, ph.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  // 2. OptimizeBoardPoints: one warp per point over its inlier observations in valid views, cameras constant
  std::vector<int> pt_off, pt_obs;
  build_point_adjacency(np, nc, ids, [&](int c) { return use[c] && vh[obs_view[c]]; }, pt_off, pt_obs);
  std::vector<double> qcw(4 * (size_t)nf);
  for (int f = 0; f < nf; ++f) { qcw[4 * f] = -qh[4 * f]; qcw[4 * f + 1] = -qh[4 * f + 1]; qcw[4 * f + 2] = -qh[4 * f + 2]; qcw[4 * f + 3] = qh[4 * f + 3]; }
  CU(d_qcw.upload(qcw)); CU(d_c.upload(ph)); CU(d_pt_off.upload(pt_off)); CU(d_pt_obs.alloc(std::max<size_t>(1, pt_obs.size())));
  if (!pt_obs.empty()) CU(cudaMemcpy(d_pt_obs.p, pt_obs.data(), pt_obs.size() * sizeof(int), cudaMemcpyHostToDevice));
  PointProblem PQ; memset(&PQ, 0, sizeof PQ);
  PQ.model = h->model; for (int i = 0; i < 10; ++i) PQ.intr[i] = h->intr[i];
  PQ.normalized = 1; PQ.n_points = np; PQ.min_obs = min_observations > 0 ? min_observations : 30; PQ.huber = 1.345;
  PQ.board_in = d_board.p; PQ.pt_off = d_pt_off.p; PQ.pt_obs = d_pt_obs.p; PQ.obs_view = d_view.p; PQ.meas = d_xy.p; PQ.q_cw = d_qcw.p; PQ.cam_c = d_c.p;
  launch_point_refine(PQ, d_board2.p, d_opt.p, st);
  // 3. OptimizeAllPoses on the new points
  Q.board = d_board2.p;
  launch_board_poses(Q, d_xy.p, d_ok.p, d_use.p, d_q.p, d_p.p, d_e.p, d_valid.p, st);
  std::vector<double> eh(nf); std::vector<int> opt(np);
  CU(cudaMemcpyAsync(board.data(), d_board2.p, (size_t)np * sizeof(double4), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(opt.data(), d_opt.p, (size_t)np * sizeof(int), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(q_wc, d_q.p, 4 * (size_t)nf * sizeof(double), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(p_wc, d_p.p, 3 * (size_t)nf * sizeof(double), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(eh.data(), d_e.p, (size_t)nf * sizeof(double), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(vh.data(), d_valid.p, (size_t)nf * sizeof(int), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  if (cudaGetLastError() != cudaSuccess) return fail(h, ICC_ERR_CUDA, "board point kernels failed");
  int n_opt = 0;
  for (int i = 0; i < np; ++i) { h->points[4 * i] = board[i].x; h->points[4 * i + 1] = board[i].y; h->points[4 * i + 2] = board[i].z; h->points[4 * i + 3] = board[i].w; n_opt += opt[i]; }
  if (board_out) std::copy(h->points.begin(), h->points.end(), board_out);
  if (n_opt_out) *n_opt_out = n_opt;
  for (int i = 0; i < nf; ++i) { valid[i] = vh[i]; if (mean_err) mean_err[i] = eh[i]; }
  return ICC_OK;
}

// ---- upstream row f3: IMU-to-camera rotation + time offset initialiser ---------------------------------------------------
namespace {
double median_like_reference(std::vector<double> v) {   // utils::MedianOfDoubleVec (src/utils/utils.cc:77-97)
  const size_t n = v.size();
  if (n % 2 == 0) {
    std::nth_element(v.begin(), v.begin() + n / 2 - 1, v.end()); const double e1 = v[n / 2 - 1];
    std::nth_element(v.begin(), v.begin() + n / 2, v.end()); const double e2 = v[n / 2];
    return (e1 + e2) / 2;
  }
  std::nth_element(v.begin(), v.begin() + n / 2, v.end());
  return v[n / 2];
}
void quat_from_rowmajor(const double* R, double* q) {    // -> x, y, z, w
  const double m00 = R[0], m01 = R[1], m02 = R[2], m10 = R[3], m11 = R[4], m12 = R[5], m20 = R[6], m21 = R[7], m22 = R[8], tr = m00 + m11 + m22;
  double x, y, z, w;
  if (tr > 0.0) { const double s = std::sqrt(tr + 1.0) * 2.0; w = 0.25 * s; x = (m21 - m12) / s; y = (m02 - m20) / s; z = (m10 - m01) / s; }
  else if (m00 > m11 && m00 > m22) { const double s = std::sqrt(1.0 + m00 - m11 - m22) * 2.0; w = (m21 - m12) / s; x = 0.25 * s; y = (m01 + m10) / s; z = (m02 + m20) / s; }
  else if (m11 > m22) { const double s = std::sqrt(1.0 + m11 - m00 - m22) * 2.0; w = (m02 - m20) / s; x = (m01 + m10) / s; y = 0.25 * s; z = (m12 + m21) / s; }
  else { const double s = std::sqrt(1.0 + m22 - m00 - m11) * 2.0; w = (m10 - m01) / s; x = (m02 + m20) / s; y = (m12 + m21) / s; z = 0.25 * s; }
  const double n = std::sqrt(x * x + y * y + z * z + w * w);
  q[0] = x / n; q[1] = y / n; q[2] = z / n; q[3] = w / n;
}
}  // namespace

icc_status icc_estimate_imu_to_camera_rotation(icc_handle* h, int n_views, const double* view_t, const double* q_cw, int n_imu, const double* imu_t,
                                               const double* gyro, const double* bias_in, double* q_out, double* td_out, double* bias_out, double* err_out, int32_t* iters_out) {
  if (!h || n_views < 2 || !view_t || !q_cw || n_imu < 2 || !imu_t || !gyro || !q_out || !td_out) return ICC_ERR_INVALID_ARGUMENT;
  if (h->device < 0) return fail(h, ICC_ERR_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
  CU(cudaSetDevice(h->device));
  // ---- host preparation (app :96-162): ordered maps, median frame interval, regular grid, common window ------------------
  // std::map semantics of the reference (time ordered, a repeated timestamp keeps the LAST sample); already-sorted input -- the
  // normal case -- skips the tree
  auto ordered = [](const double* t, int n) { std::vector<std::pair<double, int>> o; o.reserve(n);
    bool inc = true; for (int i = 1; i < n && inc; ++i) inc = t[i] > t[i - 1];
    if (inc) { for (int i = 0; i < n; ++i) o.emplace_back(t[i], i); return o; }
    std::map<double, int> m; for (int i = 0; i < n; ++i) m[t[i]] = i;
    for (const auto& kv : m) o.emplace_back(kv.first, kv.second);
    return o; };
  const std::vector<std::pair<double, int>> vmap = ordered(view_t, n_views), gmap = ordered(imu_t, n_imu);
  if (vmap.size() < 2 || gmap.size() < 2) return fail(h, ICC_ERR_INVALID_ARGUMENT, "need at least two distinct view and gyroscope timestamps");
  double imu_dt = 0.0;
  for (int i = 1; i < n_imu; ++i) imu_dt += imu_t[i] - imu_t[i - 1];                     // app :103-108 (file order)
  imu_dt /= (double)(n_imu - 1);
  std::vector<double> tv; std::vector<double4> qv;
  for (const auto& kv : vmap) { tv.push_back(kv.first); const double* q = q_cw + 4 * (size_t)kv.second; qv.push_back(make_double4(q[0], q[1], q[2], q[3])); }
  std::vector<double> diffs; for (size_t i = 1; i < tv.size(); ++i) diffs.push_back(tv[i] - tv[i - 1]);
  const double cam_dt = median_like_reference(diffs);
  if (!(cam_dt > 0.0)) return fail(h, ICC_ERR_INVALID_ARGUMENT, "non-positive median frame interval");
  std::vector<double> grid; for (double t = tv.front(); t < tv.back(); t += cam_dt) grid.push_back(t);   // app :139-144
  std::vector<double> tg, gg;    // gyroscope, time ordered, bias removed
  for (const auto& kv : gmap) { tg.push_back(kv.first); for (int d = 0; d < 3; ++d) gg.push_back(gyro[3 * (size_t)kv.second + d] - (bias_in ? bias_in[d] : 0.0)); }
  const double t0 = grid.front() >= tg.front() ? grid.front() : tg.front();               // :127-129
  const double tend = grid.back() >= tg.back() ? grid.back() : tg.back();                 // (the LATER end, as in the reference)
  std::vector<double> tI, wI; for (size_t i = 0; i < tg.size(); ++i) if (tg[i] >= t0 && tg[i] <= tend) { tI.push_back(tg[i] - t0); for (int d = 0; d < 3; ++d) wI.push_back(gg[3 * i + d]); }
  size_t g0 = 0; while (g0 < grid.size() && grid[g0] < t0) ++g0;
  std::vector<double> tV; for (size_t i = g0; i < grid.size(); ++i) if (grid[i] <= tend) tV.push_back(grid[i] - t0);
  const int N = (int)tI.size(), Mc = (int)tV.size(), M = (int)grid.size(), nv = (int)tv.size();
  if (N < 2 || Mc < 1) return fail(h, ICC_ERR_INVALID_ARGUMENT, "camera and gyroscope streams do not overlap");
  // ---- device pipeline --------------------------------------------------------------------------------------------------
  DevBuf<double> d_tv, d_grid, d_tV, d_tI, d_wI, d_wraw, d_wheld, d_wvis, d_wimu, d_shift; DevBuf<double4> d_qv, d_qgrid, d_qi; DevBuf<unsigned char> d_bad; DevBuf<RotInitState> d_state;
  CU(d_tv.upload(tv)); CU(d_qv.upload(qv)); CU(d_grid.upload(grid)); CU(d_tV.upload(tV)); CU(d_tI.upload(tI)); CU(d_wI.upload(wI));
  CU(d_qgrid.alloc(M)); CU(d_qi.alloc(N)); CU(d_wraw.alloc(3 * (size_t)N)); CU(d_wheld.alloc(3 * (size_t)N)); CU(d_wvis.alloc(3 * (size_t)N)); CU(d_wimu.alloc(3 * (size_t)N));
  CU(d_shift.alloc(6 * (size_t)N)); CU(d_bad.alloc(N)); CU(d_state.alloc(1));
  launch_interp_quat(nv, d_tv.p, d_qv.p, M, d_grid.p, d_qgrid.p, h->stream);              // views -> regular frame grid (app :150-156)
  launch_interp_quat(Mc, d_tV.p, d_qgrid.p + g0, N, d_tI.p, d_qi.p, h->stream);           // grid -> IMU rate (:172-173)
  launch_visual_angular_velocity(N, d_qi.p, imu_dt, d_wraw.p, d_bad.p, d_wheld.p, d_wvis.p, d_wI.p, d_wimu.p, h->stream);
  RotInitProblem Q; memset(&Q, 0, sizeof Q);
  Q.n = N; Q.t = d_tI.p; Q.vis = d_wvis.p; Q.imu = d_wimu.p; Q.vis_shift = d_shift.p; Q.state = d_state.p;
  Q.estimate_bias = bias_in ? 0 : 1; Q.tolerance = 1e-4;
  for (int d = 0; d < 3; ++d) Q.bias_in[d] = bias_in ? bias_in[d] : 0.0;
  // the bracket shrinks by the golden ratio per step whatever the data says, so the step count is known up to rounding
  int n_it = 0; { const double g = (1.0 + std::sqrt(5.0)) / 2.0; double a = -1.0, b = 1.0, c = b - (b - a) / g, d = a + (b - a) / g; while (std::fabs(c - d) > Q.tolerance && n_it < 200) { b = d; c = b - (b - a) / g; d = a + (b - a) / g; ++n_it; } }
  launch_golden_section(Q, 1.0, n_it + 2, h->sm_count > 0 ? h->sm_count : 148, h->stream);
  RotInitState S;
  CU(cudaMemcpyAsync(&S, d_state.p, sizeof S, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  if (cudaGetLastError() != cudaSuccess) return fail(h, ICC_ERR_CUDA, "rotation initialiser kernels failed");
  if (!S.done) return fail(h, ICC_ERR_NUMERIC, "golden-section search did not terminate");
  quat_from_rowmajor(S.R_best, q_out);
  *td_out = (S.b + S.a) / 2;                                                               // :259
  if (bias_out) for (int d = 0; d < 3; ++d) bias_out[d] = S.bias_best[d];
  if (err_out) *err_out = S.error;
  if (iters_out) *iters_out = S.iterations;
  return ICC_OK;
}

// ---- upstream row f2: spline error weighting -----------------------------------------------------------------------------
namespace {
// scipy.optimize.brentq (Brent 1973 as implemented in scipy/optimize/Zeros/brentq.c), xtol = 2e-12, rtol = 4 eps, 100 iterations
double brentq(const std::function<double(double)>& f, double xa, double xb, bool& ok) {
  const double xtol = 2e-12, rtol = 8.881784197001252e-16;
  double xpre = xa, xcur = xb, xblk = 0.0, fpre = f(xpre), fcur = f(xcur), fblk = 0.0, spre = 0.0, scur = 0.0;
  ok = true;
  if (fpre == 0.0) return xpre;
  if (fcur == 0.0) return xcur;
  if ((fpre > 0) == (fcur > 0)) { ok = false; return xcur; }
  for (int i = 0; i < 100; ++i) {
    if (fpre != 0.0 && fcur != 0.0 && ((fpre > 0) != (fcur > 0))) { xblk = xpre; fblk = fpre; spre = scur = xcur - xpre; }
    if (std::fabs(fblk) < std::fabs(fcur)) { xpre = xcur; xcur = xblk; xblk = xpre; fpre = fcur; fcur = fblk; fblk = fpre; }
    const double delta = (xtol + rtol * std::fabs(xcur)) / 2, sbis = (xblk - xcur) / 2;
    if (fcur == 0.0 || std::fabs(sbis) < delta) return xcur;
    if (std::fabs(spre) > delta && std::fabs(fcur) < std::fabs(fpre)) {
      double stry;
      if (xpre == xblk) stry = -fcur * (xcur - xpre) / (fcur - fpre);                       // secant
      else { const double dpre = (fpre - fcur) / (xpre - xcur), dblk = (fblk - fcur) / (xblk - xcur); stry = -fcur * (fblk * dblk - fpre * dpre) / (dblk * dpre * (fblk - fpre)); }   // inverse quadratic
      if (2 * std::fabs(stry) < std::min(std::fabs(spre), 3 * std::fabs(sbis) - delta)) { spre = scur; scur = stry; }
      else { spre = sbis; scur = sbis; }
    } else { spre = sbis; scur = sbis; }
    xpre = xcur; fpre = fcur;
    if (std::fabs(scur) > delta) xcur += scur; else xcur += (sbis > 0 ? delta : -delta);
    fcur = f(xcur);
  }
  ok = false;
  return xcur;
}
}  // namespace

icc_status icc_spline_error_weighting(icc_handle* h, int n, const double* times, const double* signal, double quality, double min_dt, double max_dt,
                                      double* dt_out, double* var_out, double* spectrum) {
  if (!h || n < 4 || !times || !signal || !dt_out || !var_out || !(quality > 0.0 && quality < 1.0)) return ICC_ERR_INVALID_ARGUMENT;
  if (h->device < 0) return fail(h, ICC_ERR_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
  CU(cudaSetDevice(h->device));
  double mean_dt = 0.0; for (int i = 1; i < n; ++i) mean_dt += times[i] - times[i - 1]; mean_dt /= (double)(n - 1);
  if (!(mean_dt > 0.0)) return fail(h, ICC_ERR_INVALID_ARGUMENT, "timestamps must increase on average");
  const double sample_rate = 1.0 / mean_dt, d = 1.0 / sample_rate, fscale = 1.0 / ((double)n * d);   // np.fft.fftfreq(n, d): k * (1 / (n d))
  if (!(min_dt > 0.0)) min_dt = 1.0 / sample_rate;                                                     // sew.py:156-160
  if (!(max_dt > 0.0)) max_dt = ((double)n / 4.0) / sample_rate;
  const int M = sew_fft_length(n);
  DevBuf<double> d_sig, d_xhat, d_scr, d_acc;
  CU(d_sig.alloc(3 * (size_t)n)); CU(d_xhat.alloc(n)); CU(d_scr.alloc(16 * (size_t)M)); CU(d_acc.alloc(2));
  CU(cudaMemcpyAsync(d_sig.p, signal, 3 * (size_t)n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  launch_sew_spectrum(n, d_sig.p, d_xhat.p, d_acc.p, d_scr.p, h->stream);
  double esum = 0.0;
  CU(cudaMemcpyAsync(&esum, d_acc.p, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (spectrum) CU(cudaMemcpyAsync(spectrum, d_xhat.p, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  if (cudaGetLastError() != cudaSuccess) return fail(h, ICC_ERR_CUDA, "spectrum kernels failed");
  const double max_remove = esum / (double)n * (1.0 - quality);                                        // signal_energy(Xhat) * (1 - quality)
  bool cuda_ok = true;
  auto removed = [&](double dt) -> double {      // signal_energy((1 - H) * Xhat)
    double e = 0.0;
    launch_sew_residual_energy(n, d_xhat.p, fscale, dt, d_acc.p + 1, h->sm_count > 0 ? h->sm_count : 148, h->stream);
    if (cudaMemcpyAsync(&e, d_acc.p + 1, sizeof(double), cudaMemcpyDeviceToHost, h->stream) != cudaSuccess || cudaStreamSynchronize(h->stream) != cudaSuccess) cuda_ok = false;
    return e / (double)n;
  };
  auto quality_func = [&](double dt) { return max_remove / removed(dt); };
  // find_max_quality_dt(quality_func, 1.0, min_dt, max_dt)   (sew.py:86-145)
  double dt = max_dt, found = 0.0; bool have = false;
  if (quality_func(dt) >= 1.0) { found = dt; have = true; }
  else {
    double step = max_dt * 0.5, max_quality = 0.0, max_quality_dt = dt; bool any = false;
    while (!have) {
      dt -= step; dt = std::max(dt, min_dt);
      const double q = quality_func(dt);
      if (q > 1.0) { bool ok; found = brentq([&](double x) { return quality_func(x) - 1.0; }, dt, max_dt, ok); if (!ok) return fail(h, ICC_ERR_NUMERIC, "Brent root search failed"); have = true; }
      else {
        step *= 0.5;
        if (q > max_quality) { max_quality = q; max_quality_dt = dt; any = true; }
        if (dt <= min_dt) { if (!any) return fail(h, ICC_ERR_NUMERIC, "no knot spacing satisfies the quality"); found = max_quality_dt; have = true; }
      }
      if (!cuda_ok) return fail(h, ICC_ERR_CUDA, "quality kernels failed");
    }
  }
  *dt_out = found;
  *var_out = removed(found) / (double)n;                                                               // dt_to_variance_spectrum (:196-199)
  if (!cuda_ok) return fail(h, ICC_ERR_CUDA, "quality kernels failed");
  return ICC_OK;
}

// ---- upstream row f4: camera intrinsic calibration (CameraCalibrator, src/core/camera_calibrator.cc) ----------------------
namespace {
// theia::CameraIntrinsicsModel::GetSubsetFromOptimizeIntrinsicsType per model, as bit masks over Theia's parameter order
struct IntrinsicSubsets { unsigned focal, aspect, principal, radial, tangential; };
IntrinsicSubsets intrinsic_subsets(int model) {
  auto bits = [](std::initializer_list<int> l) { unsigned m = 0; for (int i : l) m |= 1u << i; return m; };
  switch (model) {
    case CAM_PINHOLE: return {bits({0}), bits({1}), bits({3, 4}), bits({5, 6}), 0u};
    case CAM_PINHOLE_RADTAN: return {bits({0}), bits({1}), bits({3, 4}), bits({5, 6, 7}), bits({8, 9})};
    case CAM_FISHEYE: return {bits({0}), bits({1}), bits({3, 4}), bits({5, 6, 7, 8}), 0u};
    case CAM_FOV: return {bits({0}), bits({1}), bits({2, 3}), bits({4}), 0u};
    case CAM_DIVISION_UNDISTORTION: return {bits({0}), bits({1}), bits({2, 3}), bits({4}), 0u};
    case CAM_DOUBLE_SPHERE: return {bits({0}), bits({1}), bits({3, 4}), bits({5, 6}), 0u};
    case CAM_EXTENDED_UNIFIED: return {bits({0}), bits({1}), bits({3, 4}), bits({5, 6}), 0u};
    default: return {0u, 0u, 0u, 0u, 0u};
  }
}

// board points (the handle's), corner offsets, point ids and pixels of a camera calibration, on the device
struct CamCalInputs { DevBuf<double4> board; DevBuf<int> off, pid; DevBuf<double2> uv; };
icc_status upload_camcal_inputs(icc_handle* h, int nv, const int32_t* off, const int32_t* ids, const double* uv, CamCalInputs& in) {
  const int nc = off[nv], np = (int)(h->points.size() / 4);
  cudaStream_t st = h->stream;
  std::vector<double4> board(np);
  for (int i = 0; i < np; ++i) board[i] = make_double4(h->points[4 * i], h->points[4 * i + 1], h->points[4 * i + 2], h->points[4 * i + 3]);
  CU(in.board.upload(board));
  CU(in.off.alloc(nv + 1)); CU(in.pid.alloc(std::max(1, nc))); CU(in.uv.alloc(std::max(1, nc)));
  CU(cudaMemcpyAsync(in.off.p, off, (size_t)(nv + 1) * sizeof(int), cudaMemcpyHostToDevice, st));
  if (nc > 0) {
    CU(cudaMemcpyAsync(in.pid.p, ids, (size_t)nc * sizeof(int), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(in.uv.p, uv, (size_t)nc * sizeof(double2), cudaMemcpyHostToDevice, st));
  }
  return ICC_OK;
}

// device buffers of one bundle-adjustment iteration (sizes as in launch_camcal_accumulate / launch_camcal_step)
struct CamCalStepBufs { double *blocks, *sys, *red, *Y, *scale, *dk, *scal; };
// One iteration body of bundle_adjust: with `evaluate` the normal equations at `cur` (per-slot blocks, sys with the cost), then the
// damped step at `radius` into `cand` with its scalars, and the cost at `cand` into scal[CC_CAND_COST].
cudaError_t launch_camcal_iteration(const CamCalProblem& Q, const CamCalState& cur, const CamCalState& cand, const CamCalStepBufs& b,
                                    bool evaluate, bool compute_scale, double radius, cudaStream_t st) {
  cudaError_t e;
  if (evaluate) {
    if ((e = cudaMemsetAsync(b.sys, 0, (CC_PACK + 1) * sizeof(double), st)) != cudaSuccess) return e;
    launch_camcal_accumulate(Q, cur, true, b.blocks, b.sys, nullptr, nullptr, st);
  }
  if ((e = cudaMemsetAsync(b.red, 0, 66 * sizeof(double), st)) != cudaSuccess) return e;
  if ((e = cudaMemsetAsync(b.scal, 0, CC_SCAL_COUNT * sizeof(double), st)) != cudaSuccess) return e;
  launch_camcal_step(Q, cur, cand, b.blocks, b.sys, b.red, b.Y, b.scale, compute_scale ? 1 : 0, radius, 1e-6, 1e32, b.dk, b.scal, st);
  launch_camcal_accumulate(Q, cand, false, nullptr, nullptr, b.scal + CC_CAND_COST, nullptr, st);
  return cudaSuccess;
}
}  // namespace

icc_status icc_calibrate_camera(icc_handle* h, int model, int W, int H, int nv, const int32_t* off, const int32_t* ids, const double* uv,
                                const double* q_init, const double* p_init, const int32_t* init_valid, double focal_init, double distortion_init,
                                const icc_camcal_options* options, double* intr_out, double* q_out, double* p_out, double* err_out, int32_t* used_out,
                                icc_camcal_summary* summary) {
  using clk = std::chrono::steady_clock;
  const auto t_start = clk::now();
  if (!h || nv <= 0 || !off || !ids || !uv || !intr_out || !q_out || !p_out || !used_out || W <= 0 || H <= 0) return ICC_ERR_INVALID_ARGUMENT;
  if (h->device < 0) return fail(h, ICC_ERR_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
  if (camera_num_params(model) < 0) return fail(h, ICC_ERR_INVALID_ARGUMENT, "unknown camera model");
  if (h->points.empty()) return fail(h, ICC_ERR_STATE, "icc_set_board_points must be called first");
  if (off[0] != 0) return fail(h, ICC_ERR_INVALID_ARGUMENT, "corner offsets must start at 0");
  for (int i = 0; i < nv; ++i) if (off[i + 1] < off[i]) return fail(h, ICC_ERR_INVALID_ARGUMENT, "corner offsets must be non-decreasing");
  const int nc = off[nv], np = (int)(h->points.size() / 4);
  for (int i = 0; i < nc; ++i) if (ids[i] < 0 || ids[i] >= np) return fail(h, ICC_ERR_INVALID_ARGUMENT, "point id outside the board");
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
  const int launches0 = kernel_launch_count();
  CU(cudaSetDevice(h->device));
  cudaStream_t st = h->stream;
  // ---- inputs to the device ------------------------------------------------------------------------------------------------
  CamCalInputs in;
  { const icc_status r = upload_camcal_inputs(h, nv, off, ids, uv, in); if (r != ICC_OK) return r; }
  DevBuf<double4>& d_board = in.board; DevBuf<int>& d_off = in.off; DevBuf<int>& d_pid = in.pid; DevBuf<double2>& d_uv = in.uv;
  DevBuf<int> d_active;
  CU(d_active.alloc(nv));
  const double cx0 = W / 2.0, cy0 = H / 2.0;                       // AddView (:99)
  // ---- initial focal length and poses ----------------------------------------------------------------------------------------
  std::vector<double> q0(4 * (size_t)nv), p0(3 * (size_t)nv); std::vector<int> ok0(nv, 1);
  const bool need_focal = !(focal_init > 0.0), need_poses = !q_init || !p_init;
  double f0 = focal_init;
  if (need_focal || need_poses) {
    PoseProblem PQ; memset(&PQ, 0, sizeof PQ);
    PQ.model = CAM_PINHOLE; PQ.n_frames = nv; PQ.n_points = np; PQ.min_points = 6;
    PQ.board = d_board.p; PQ.f_off = d_off.p; PQ.pid = d_pid.p; PQ.thresh_sq = 1e300; PQ.max_err = 1e300;   // every corner takes part
    PQ.lm_rel_tol = 1e-6;                                                                                  // these poses only start the bundle adjustment
    DevBuf<double2> d_xy; DevBuf<unsigned char> d_use; DevBuf<double> d_f2, d_q, d_p, d_e; DevBuf<int> d_ok, d_valid;
    CU(d_xy.alloc(std::max(1, nc))); CU(d_use.alloc(std::max(1, nc))); CU(d_ok.alloc(std::max(1, nc)));
    if (need_focal) {
      CU(d_f2.alloc(nv));
      launch_board_focal(PQ, d_uv.p, cx0, cy0, d_xy.p, d_use.p, d_f2.p, st);
      std::vector<double> f2(nv);
      CU(cudaMemcpyAsync(f2.data(), d_f2.p, (size_t)nv * sizeof(double), cudaMemcpyDeviceToHost, st));
      CU(cudaStreamSynchronize(st));
      std::vector<double> fs; for (double v : f2) if (v > 0.0 && std::isfinite(v)) fs.push_back(std::sqrt(v));
      if (fs.empty()) return fail(h, ICC_ERR_NUMERIC, "no view yields a focal length estimate (fronto-parallel or degenerate views only)");
      f0 = median_like_reference(fs);
    }
    if (need_poses) {
      CU(d_q.alloc(4 * (size_t)nv)); CU(d_p.alloc(3 * (size_t)nv)); CU(d_e.alloc(nv)); CU(d_valid.alloc(nv));
      launch_pinhole_normalize(nc, d_uv.p, cx0, cy0, f0, d_xy.p, d_ok.p, st);
      launch_board_poses(PQ, d_xy.p, d_ok.p, d_use.p, d_q.p, d_p.p, d_e.p, d_valid.p, st);
      CU(cudaMemcpyAsync(q0.data(), d_q.p, 4 * (size_t)nv * sizeof(double), cudaMemcpyDeviceToHost, st));
      CU(cudaMemcpyAsync(p0.data(), d_p.p, 3 * (size_t)nv * sizeof(double), cudaMemcpyDeviceToHost, st));
      CU(cudaMemcpyAsync(ok0.data(), d_valid.p, (size_t)nv * sizeof(int), cudaMemcpyDeviceToHost, st));
      CU(cudaStreamSynchronize(st));
    }
  }
  if (!need_poses) {
    memcpy(q0.data(), q_init, 4 * (size_t)nv * sizeof(double)); memcpy(p0.data(), p_init, 3 * (size_t)nv * sizeof(double));
    if (init_valid) for (int i = 0; i < nv; ++i) ok0[i] = init_valid[i] != 0;
  }
  // ---- state: R_cw = conj(q_wc), camera centre, shared intrinsics ---------------------------------------------------------------
  std::vector<double> qs(4 * (size_t)nv), k0(10, 0.0);
  for (int v = 0; v < nv; ++v) { const Q4 q = qn(&q0[4 * v]); qs[4 * v] = -q.x; qs[4 * v + 1] = -q.y; qs[4 * v + 2] = -q.z; qs[4 * v + 3] = q.w; }
  // the internal initialiser refines (focal length, division distortion, poses) jointly before the target model takes over -- the
  // role of utils::initialize_radial_undistortion_camera (:283-306), which hands the reference a focal length and a division-model
  // distortion for every non-pinhole model
  const bool prestage = need_poses && need_focal && model != CAM_PINHOLE && model != CAM_PINHOLE_RADTAN;
  std::vector<int> active;
  for (int v = 0; v < nv; ++v) if (ok0[v]) active.push_back(v);
  S.n_views_initialized = (int)active.size();
  if (prestage) { k0[0] = f0; k0[1] = 1.0; k0[2] = cx0; k0[3] = cy0; k0[4] = -1e-2 / ((double)W * W + (double)H * H); }
  DevBuf<double> d_q[2], d_c[2], d_k[2], d_blocks, d_Y, d_scale, d_sys, d_red, d_dk, d_scal, d_verr;
  for (int i = 0; i < 2; ++i) { CU(d_q[i].upload(qs)); CU(d_c[i].upload(p0)); CU(d_k[i].upload(k0)); }
  const size_t na0 = std::max<size_t>(1, active.size());
  CU(d_blocks.alloc(na0 * CC_PACK)); CU(d_Y.alloc(na0 * CC_Y)); CU(d_scale.alloc(6 * na0 + 10)); CU(d_sys.alloc(CC_PACK + 1)); CU(d_red.alloc(66));
  CU(d_dk.alloc(10)); CU(d_scal.alloc(CC_SCAL_COUNT)); CU(d_verr.alloc(nv));
  const CamCalStepBufs bufs{d_blocks.p, d_sys.p, d_red.p, d_Y.p, d_scale.p, d_dk.p, d_scal.p};
  int cur = 0;
  CamCalProblem Q; memset(&Q, 0, sizeof Q);
  Q.model = model; Q.n_points = np; Q.huber = o.huber_width; Q.board = d_board.p; Q.f_off = d_off.p; Q.pid = d_pid.p; Q.uv = d_uv.p; Q.active = d_active.p;
  auto state = [&](int i) { CamCalState s; s.q = d_q[i].p; s.c = d_c[i].p; s.k = d_k[i].p; return s; };
  auto set_active = [&]() -> icc_status {
    Q.n_active = (int)active.size();
    if (!active.empty()) CU(cudaMemcpyAsync(d_active.p, active.data(), active.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));   // `active` may be modified by the caller right after
    return ICC_OK;
  };
  std::vector<double> verr(nv, 0.0);
  // GetReprojErrorOfView for every active view at the current state
  auto view_errors = [&]() -> icc_status {
    CU(cudaMemsetAsync(d_scal.p, 0, CC_SCAL_COUNT * sizeof(double), st));
    launch_camcal_accumulate(Q, state(cur), false, nullptr, nullptr, d_scal.p + CC_CAND_COST, d_verr.p, st);
    CU(cudaMemcpyAsync(verr.data(), d_verr.p, (size_t)nv * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return ICC_OK;
  };
  // RemoveViewsReprojError (:59-76)
  auto remove_views = [&](double max_err) -> icc_status {
    icc_status r = view_errors(); if (r != ICC_OK) return r;
    std::vector<int> keep; for (int v : active) if (!(verr[v] > max_err)) keep.push_back(v);
    active.swap(keep);
    return set_active();
  };
  // theia::BundleAdjustViews: Levenberg-Marquardt with Ceres' trust-region logic; one device->host read-back per iteration
  auto bundle_adjust = [&](unsigned mask, bool pose_free, int stage) -> icc_status {
    Q.intr_mask = mask; Q.pose_free = pose_free ? 1 : 0;
    double radius = 1e4, decrease_factor = 2.0, x_cost = 0.0, sc[CC_SCAL_COUNT];
    int invalid = 0; bool ne_valid = false, first = true;
    int term = 0, iters = 0;
    if (Q.n_active == 0 || (mask == 0u && !pose_free)) { if (stage >= 0) S.termination[stage] = 3; return ICC_OK; }
    for (int it = 0; it < o.max_num_iterations; ++it) {
      const bool fresh = !ne_valid;
      CU(launch_camcal_iteration(Q, state(cur), state(1 - cur), bufs, fresh, first, radius, st));
      ne_valid = true;
      CU(cudaMemcpyAsync(sc, d_scal.p, sizeof sc, cudaMemcpyDeviceToHost, st));
      CU(cudaStreamSynchronize(st));
      if (fresh) {
        x_cost = sc[CC_X_COST];
        if (first) { if (stage == 0) S.initial_cost = x_cost; if (!std::isfinite(x_cost)) return fail(h, ICC_ERR_NUMERIC, "non-finite initial cost"); }
        if (sc[CC_GRAD_MAX] <= o.gradient_tolerance) { term = 3; first = false; break; }
      }
      first = false;
      ++iters;
      const double model_change = 0.5 * (sc[CC_D_DELTA] - sc[CC_G_DELTA]);
      if (sc[CC_FAIL] != 0.0 || !(model_change > 0.0)) {
        if (++invalid >= 5) { term = 4; break; }
        radius /= decrease_factor; decrease_factor *= 2.0;
        continue;
      }
      invalid = 0;
      const double step_norm = std::sqrt(sc[CC_STEP_SQ]), x_norm = std::sqrt(sc[CC_X_SQ]);
      double cand_cost = sc[CC_CAND_COST];
      if (!std::isfinite(cand_cost)) cand_cost = 1.7976931348623157e308;
      if (step_norm <= o.parameter_tolerance * (x_norm + o.parameter_tolerance)) { term = 2; break; }
      const double cost_change = x_cost - cand_cost;
      if (std::fabs(cost_change) <= o.function_tolerance * x_cost) { term = 1; break; }   // Ceres returns before accepting this step
      const double rel = cost_change / model_change;
      if (rel > 1e-3) {
        cur = 1 - cur; x_cost = cand_cost; ne_valid = false;
        radius = std::min(1e16, radius / std::max(1.0 / 3.0, 1.0 - std::pow(2.0 * rel - 1.0, 3)));
        decrease_factor = 2.0;
      } else {
        radius /= decrease_factor; decrease_factor *= 2.0;
        if (radius < 1e-32) { term = 4; break; }
      }
    }
    // both state copies must agree on everything outside the last step (inactive views never move; the intrinsics / poses of
    // a rejected candidate are stale): bring the spare copy back to the current state
    CU(cudaMemcpyAsync(d_q[1 - cur].p, d_q[cur].p, 4 * (size_t)nv * sizeof(double), cudaMemcpyDeviceToDevice, st));
    CU(cudaMemcpyAsync(d_c[1 - cur].p, d_c[cur].p, 3 * (size_t)nv * sizeof(double), cudaMemcpyDeviceToDevice, st));
    CU(cudaMemcpyAsync(d_k[1 - cur].p, d_k[cur].p, 10 * sizeof(double), cudaMemcpyDeviceToDevice, st));
    if (stage >= 0) { S.final_cost[stage] = x_cost; S.iterations[stage] = iters; S.termination[stage] = term; } else S.init_iterations = iters;
    return ICC_OK;
  };
  auto finish = [&](bool success) -> icc_status {
    icc_status r = view_errors(); if (r != ICC_OK) return r;
    std::vector<double> qh(4 * (size_t)nv), ch(3 * (size_t)nv), kh(10);
    CU(cudaMemcpy(qh.data(), d_q[cur].p, qh.size() * sizeof(double), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(ch.data(), d_c[cur].p, ch.size() * sizeof(double), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(kh.data(), d_k[cur].p, 10 * sizeof(double), cudaMemcpyDeviceToHost));
    for (int v = 0; v < nv; ++v) {
      q_out[4 * v] = -qh[4 * v]; q_out[4 * v + 1] = -qh[4 * v + 1]; q_out[4 * v + 2] = -qh[4 * v + 2]; q_out[4 * v + 3] = qh[4 * v + 3];
      for (int d = 0; d < 3; ++d) p_out[3 * v + d] = ch[3 * v + d];
      used_out[v] = 0; if (err_out) err_out[v] = 0.0;
    }
    double tot = 0.0;
    for (int v : active) { used_out[v] = 1; if (err_out) err_out[v] = verr[v]; tot += verr[v]; }
    for (int i = 0; i < 10; ++i) intr_out[i] = kh[i];
    S.success = success ? 1 : 0; S.n_views_used = (int)active.size();
    S.final_reproj_error = active.empty() ? 0.0 : tot / (double)active.size();                 // :352-366
    S.gpu_launches = kernel_launch_count() - launches0;
    S.seconds_total = std::chrono::duration<double>(clk::now() - t_start).count();
    if (summary) *summary = S;
    if (!success) h->err = "Not enough views for proper calibration";
    return ICC_OK;
  };
  icc_status rc = set_active(); if (rc != ICC_OK) return rc;
  if (prestage) {
    Q.model = CAM_DIVISION_UNDISTORTION;
    rc = bundle_adjust((1u << 0) | (1u << 4), true, -1); if (rc != ICC_OK) return rc;
    Q.model = model;
    double kd[10];
    CU(cudaMemcpy(kd, d_k[cur].p, sizeof kd, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(p0.data(), d_c[cur].p, p0.size() * sizeof(double), cudaMemcpyDeviceToHost));
    if (kd[0] > 0.0 && std::isfinite(kd[0])) { f0 = kd[0]; if (model == CAM_DIVISION_UNDISTORTION) distortion_init = kd[4]; }
  }
  S.focal_length_init = f0;
  // ---- grid filter in file order (:313-325): a view is taken iff no accepted camera position lies within grid_size ---------------
  // (the reference scans all accepted positions; a hash grid with cells of grid_size visits only the 27 cells that can hold one
  // -- same decisions, linear time)
  if (o.grid_size > 0.0) {
    std::vector<int> sel;
    std::unordered_map<uint64_t, std::vector<int>> cells;
    const double inv = 1.0 / o.grid_size;
    bool hashable = true;
    for (int v : active) for (int d = 0; d < 3; ++d) if (!(std::fabs(p0[3 * v + d] * inv) < 1e6)) hashable = false;   // 21 bits per axis
    auto key = [](int64_t x, int64_t y, int64_t z) { return (uint64_t)((x + (1 << 20)) & 0x1fffff) << 42 | (uint64_t)((y + (1 << 20)) & 0x1fffff) << 21 | (uint64_t)((z + (1 << 20)) & 0x1fffff); };
    auto close_to = [&](int v, int a) { const double dx = p0[3 * v] - p0[3 * a], dy = p0[3 * v + 1] - p0[3 * a + 1], dz = p0[3 * v + 2] - p0[3 * a + 2]; return std::sqrt(dx * dx + dy * dy + dz * dz) < o.grid_size; };
    for (int v : active) {
      bool take = true;
      if (hashable) {
        const int64_t cx = (int64_t)std::floor(p0[3 * v] * inv), cy = (int64_t)std::floor(p0[3 * v + 1] * inv), cz = (int64_t)std::floor(p0[3 * v + 2] * inv);
        for (int64_t x = cx - 1; x <= cx + 1 && take; ++x) for (int64_t y = cy - 1; y <= cy + 1 && take; ++y) for (int64_t z = cz - 1; z <= cz + 1 && take; ++z) {
          auto it = cells.find(key(x, y, z));
          if (it != cells.end()) for (int a : it->second) if (close_to(v, a)) { take = false; break; }
        }
        if (take) cells[key(cx, cy, cz)].push_back(v);
      } else {
        for (int a : sel) if (close_to(v, a)) { take = false; break; }
      }
      if (take) sel.push_back(v);
    }
    active.swap(sel);
  }
  S.n_views_selected = (int)active.size();
  rc = set_active(); if (rc != ICC_OK) return rc;
  // ---- initial intrinsics of the target model (AddView :84-129) --------------------------------------------------------------------
  std::fill(k0.begin(), k0.end(), 0.0);
  k0[0] = f0; k0[1] = 1.0;
  switch (model) {
    case CAM_FOV: case CAM_DIVISION_UNDISTORTION: k0[2] = cx0; k0[3] = cy0; break;
    default: k0[3] = cx0; k0[4] = cy0; break;
  }
  if (model == CAM_DIVISION_UNDISTORTION) k0[4] = distortion_init;
  if (model == CAM_FOV) k0[4] = distortion_init != 0.0 ? distortion_init : 1e-3;   // theia's FOV model has no gradient at omega = 0
  if (model == CAM_DOUBLE_SPHERE) { k0[5] = -0.25; k0[6] = 0.5; }
  if (model == CAM_EXTENDED_UNIFIED) { k0[5] = 0.5; k0[6] = 1.0; }
  for (int i = 0; i < 2; ++i) CU(cudaMemcpy(d_k[i].p, k0.data(), 10 * sizeof(double), cudaMemcpyHostToDevice));
  if ((int)active.size() < o.min_num_views) return finish(false);                               // :132-135
  const IntrinsicSubsets sub = intrinsic_subsets(model);
  // 1. focal length and radial distortion, principal point fixed (:146-160)
  rc = bundle_adjust(sub.focal | (model != CAM_PINHOLE ? sub.radial : 0u), true, 0); if (rc != ICC_OK) return rc;
  rc = remove_views(o.max_view_error_stage1_px); if (rc != ICC_OK) return rc;                    // :162
  // 2. principal point, everything else fixed (:164-174)
  rc = bundle_adjust(sub.principal, false, 1); if (rc != ICC_OK) return rc;
  if ((int)active.size() < o.min_num_views) return finish(false);                               // :176-179
  // 3. full optimisation (:181-198)
  const unsigned stage3_mask = sub.principal | sub.focal | sub.aspect | (model == CAM_PINHOLE ? sub.radial : 0u) | (model == CAM_PINHOLE_RADTAN ? sub.tangential : 0u);
  rc = bundle_adjust(stage3_mask, true, 2);
  if (rc != ICC_OK) return rc;
  rc = remove_views(o.max_view_error_final_px); if (rc != ICC_OK) return rc;                     // :200
  if ((int)active.size() < o.min_num_views) return finish(false);                                // :202-205
  if (o.optimize_board_points) {                                                                 // :207-216
    // BundleAdjustTracks: every camera constant, one warp per board point over its observations in the remaining views ...
    std::vector<int> obs_view(std::max(1, nc), -1), pt_off, pt_obs;
    for (int v : active) for (int c = off[v]; c < off[v + 1]; ++c) obs_view[c] = v;
    build_point_adjacency(np, nc, ids, [&](int c) { return obs_view[c] >= 0; }, pt_off, pt_obs);
    DevBuf<int> d_view, d_pt_off, d_pt_obs, d_opt; DevBuf<double4> d_board2;
    CU(d_view.upload(obs_view)); CU(d_pt_off.upload(pt_off)); CU(d_pt_obs.alloc(std::max<size_t>(1, pt_obs.size()))); CU(d_opt.alloc(np)); CU(d_board2.alloc(np));
    if (!pt_obs.empty()) CU(cudaMemcpy(d_pt_obs.p, pt_obs.data(), pt_obs.size() * sizeof(int), cudaMemcpyHostToDevice));
    PointProblem PQ; memset(&PQ, 0, sizeof PQ);
    PQ.model = model; CU(cudaMemcpy(PQ.intr, d_k[cur].p, 10 * sizeof(double), cudaMemcpyDeviceToHost));
    PQ.normalized = 0; PQ.n_points = np; PQ.min_obs = 1; PQ.huber = o.huber_width;
    PQ.board_in = d_board.p; PQ.pt_off = d_pt_off.p; PQ.pt_obs = d_pt_obs.p; PQ.obs_view = d_view.p; PQ.meas = d_uv.p; PQ.q_cw = d_q[cur].p; PQ.cam_c = d_c[cur].p;
    launch_point_refine(PQ, d_board2.p, d_opt.p, st);
    std::vector<int> opt(np); std::vector<double4> board(np);
    CU(cudaMemcpyAsync(d_board.p, d_board2.p, (size_t)np * sizeof(double4), cudaMemcpyDeviceToDevice, st));
    CU(cudaMemcpyAsync(board.data(), d_board2.p, (size_t)np * sizeof(double4), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(opt.data(), d_opt.p, (size_t)np * sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (int i = 0; i < np; ++i) { h->points[4 * i] = board[i].x; h->points[4 * i + 1] = board[i].y; h->points[4 * i + 2] = board[i].z; h->points[4 * i + 3] = board[i].w; S.n_points_optimized += opt[i]; }
    // ... then BundleAdjustViews once more with the options of stage 3
    const int it3 = S.iterations[2];
    rc = bundle_adjust(stage3_mask, true, 2); if (rc != ICC_OK) return rc;
    S.iterations[2] += it3;
  }
  return finish(true);
}

icc_status icc_camcal_step(icc_handle* h, int model, int nv, const int32_t* off, const int32_t* ids, const double* uv,
                           const double* q_wc, const double* p_wc, const double* intrinsics, int n_active, const int32_t* active,
                           uint32_t intr_mask, int pose_free, double huber_width, double radius, const double* scale_in,
                           icc_camcal_step_out* out) {
  if (!h || nv <= 0 || !off || !ids || !uv || !q_wc || !p_wc || !intrinsics || n_active <= 0 || !active || !out) return ICC_ERR_INVALID_ARGUMENT;
  if (intr_mask >= (1u << 10) || !(huber_width > 0.0) || !(radius > 0.0)) return ICC_ERR_INVALID_ARGUMENT;
  NEED_DEVICE();
  if (camera_num_params(model) < 0) return fail(h, ICC_ERR_INVALID_ARGUMENT, "unknown camera model");
  if (h->points.empty()) return fail(h, ICC_ERR_STATE, "icc_set_board_points must be called first");
  if (off[0] != 0) return fail(h, ICC_ERR_INVALID_ARGUMENT, "corner offsets must start at 0");
  for (int i = 0; i < nv; ++i) if (off[i + 1] < off[i]) return fail(h, ICC_ERR_INVALID_ARGUMENT, "corner offsets must be non-decreasing");
  const int nc = off[nv], np = (int)(h->points.size() / 4);
  for (int i = 0; i < nc; ++i) if (ids[i] < 0 || ids[i] >= np) return fail(h, ICC_ERR_INVALID_ARGUMENT, "point id outside the board");
  std::vector<char> seen(nv, 0);
  for (int s = 0; s < n_active; ++s) {
    if (active[s] < 0 || active[s] >= nv || seen[active[s]]) return fail(h, ICC_ERR_INVALID_ARGUMENT, "active views must be distinct view indices");
    seen[active[s]] = 1;
  }
  CU(cudaSetDevice(h->device));
  cudaStream_t st = h->stream;
  CamCalInputs in;
  { const icc_status r = upload_camcal_inputs(h, nv, off, ids, uv, in); if (r != ICC_OK) return r; }
  std::vector<double> qs(4 * (size_t)nv), cs(p_wc, p_wc + 3 * (size_t)nv), ks(intrinsics, intrinsics + 10);
  for (int v = 0; v < nv; ++v) { const Q4 q = qn(&q_wc[4 * v]); qs[4 * v] = -q.x; qs[4 * v + 1] = -q.y; qs[4 * v + 2] = -q.z; qs[4 * v + 3] = q.w; }
  const size_t na = (size_t)n_active;
  DevBuf<int> d_active; DevBuf<double> d_q[2], d_c[2], d_k[2], d_blocks, d_Y, d_scale, d_sys, d_red, d_dk, d_scal, d_verr, d_vcost;
  CU(d_active.upload(std::vector<int>(active, active + n_active)));
  for (int i = 0; i < 2; ++i) { CU(d_q[i].upload(qs)); CU(d_c[i].upload(cs)); CU(d_k[i].upload(ks)); }
  CU(d_blocks.alloc(na * CC_PACK)); CU(d_Y.alloc(na * CC_Y)); CU(d_scale.alloc(6 * na + 10)); CU(d_sys.alloc(CC_PACK + 1)); CU(d_red.alloc(66));
  CU(d_dk.alloc(10)); CU(d_scal.alloc(CC_SCAL_COUNT)); CU(d_verr.alloc(nv)); CU(d_vcost.alloc(1));
  if (scale_in) CU(cudaMemcpyAsync(d_scale.p, scale_in, (6 * na + 10) * sizeof(double), cudaMemcpyHostToDevice, st));
  else CU(cudaMemsetAsync(d_scale.p, 0, (6 * na + 10) * sizeof(double), st));   // poses constant: the view part stays 0
  CamCalProblem Q; memset(&Q, 0, sizeof Q);
  Q.model = model; Q.n_points = np; Q.n_active = n_active; Q.pose_free = pose_free ? 1 : 0; Q.intr_mask = intr_mask; Q.huber = huber_width;
  Q.board = in.board.p; Q.f_off = in.off.p; Q.pid = in.pid.p; Q.uv = in.uv.p; Q.active = d_active.p;
  const CamCalState cur{d_q[0].p, d_c[0].p, d_k[0].p}, cand{d_q[1].p, d_c[1].p, d_k[1].p};
  const CamCalStepBufs bufs{d_blocks.p, d_sys.p, d_red.p, d_Y.p, d_scale.p, d_dk.p, d_scal.p};
  CU(launch_camcal_iteration(Q, cur, cand, bufs, true, scale_in == nullptr, radius, st));
  // GetReprojErrorOfView at the current state, as view_errors() of icc_calibrate_camera reads it
  CU(cudaMemsetAsync(d_verr.p, 0, (size_t)nv * sizeof(double), st)); CU(cudaMemsetAsync(d_vcost.p, 0, sizeof(double), st));
  launch_camcal_accumulate(Q, cur, false, nullptr, nullptr, d_vcost.p, d_verr.p, st);
  CU(cudaGetLastError());
  auto get = [&](double* dst, const double* src, size_t n) { return dst ? cudaMemcpyAsync(dst, src, n * sizeof(double), cudaMemcpyDeviceToHost, st) : cudaSuccess; };
  CU(get(out->blocks, d_blocks.p, na * CC_PACK)); CU(get(out->sys, d_sys.p, CC_PACK + 1)); CU(get(out->red, d_red.p, 66)); CU(get(out->Y, d_Y.p, na * CC_Y));
  CU(get(out->scale, d_scale.p, 6 * na + 10)); CU(get(out->dk, d_dk.p, 10)); CU(get(out->scalars, d_scal.p, CC_SCAL_COUNT));
  CU(get(out->intr_cand, d_k[1].p, 10)); CU(get(out->p_wc_cand, d_c[1].p, 3 * (size_t)nv)); CU(get(out->view_error_px, d_verr.p, nv));
  std::vector<double> qc(4 * (size_t)nv);
  CU(get(out->q_wc_cand ? qc.data() : nullptr, d_q[1].p, qc.size()));
  CU(cudaStreamSynchronize(st));
  if (out->q_wc_cand)
    for (int v = 0; v < nv; ++v) { out->q_wc_cand[4 * v] = -qc[4 * v]; out->q_wc_cand[4 * v + 1] = -qc[4 * v + 1]; out->q_wc_cand[4 * v + 2] = -qc[4 * v + 2]; out->q_wc_cand[4 * v + 3] = qc[4 * v + 3]; }
  return ICC_OK;
}

// ---- upstream: static IMU biases (python/get_imu_biases.py:36-53) -------------------------------------------------------------------
icc_status icc_estimate_imu_biases(icc_handle* h, int n, const double* acc, const double* gyr, double gravity_const, double accl_bias[3], double gyro_bias[3]) {
  if (!h || n <= 0 || !acc || !gyr || !accl_bias || !gyro_bias) return ICC_ERR_INVALID_ARGUMENT;
  if (h->device < 0) return fail(h, ICC_ERR_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
  CU(cudaSetDevice(h->device));
  DevBuf<double> d_a, d_g, d_s;
  CU(d_a.alloc(3 * (size_t)n)); CU(d_g.alloc(3 * (size_t)n)); CU(d_s.alloc(6));
  CU(cudaMemcpyAsync(d_a.p, acc, 3 * (size_t)n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(d_g.p, gyr, 3 * (size_t)n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  launch_imu_sums(n, d_a.p, d_g.p, d_s.p, h->sm_count, h->stream);
  double s[6];
  CU(cudaMemcpyAsync(s, d_s.p, sizeof s, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  if (cudaGetLastError() != cudaSuccess) return fail(h, ICC_ERR_CUDA, "bias kernel failed");
  double mean_a[3], mean_g[3];
  for (int d = 0; d < 3; ++d) { mean_a[d] = s[d] / n; mean_g[d] = s[3 + d] / n; }
  int ax = 0; for (int d = 1; d < 3; ++d) if (std::fabs(mean_a[d]) > std::fabs(mean_a[ax])) ax = d;          // :39-41 (first maximum)
  const double sgn = mean_a[ax] > 0.0 ? 1.0 : (mean_a[ax] < 0.0 ? -1.0 : 0.0);
  const double grav = (double)(float)(gravity_const * sgn);                                                     // float32 array (:43-44)
  for (int d = 0; d < 3; ++d) { accl_bias[d] = mean_a[d] - (d == ax ? grav : 0.0); gyro_bias[d] = mean_g[d]; }   // :46, :49-50
  return ICC_OK;
}

void icc_trim_device_cache(void) { block_cache().trim(); pinned_cache().trim(); }

}  // extern "C"
