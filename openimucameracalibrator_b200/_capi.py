"""ctypes binding of the C-ABI declared in include/icc_b200.h.

`CApi(lib, prefix)` binds every entry point of a loaded shared library; the product binds `libicc_b200.so` with prefix
`icc_`.  (tests/ bind the CPU oracle, which deliberately exports the same shapes under `icco_`, through the same class —
the product package itself never loads or references the oracle.)
"""
from __future__ import annotations

import ctypes as C

import numpy as np

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)
c_int64_p = C.POINTER(C.c_int64)

FLAG_POINTS, FLAG_T_I_C, FLAG_IMU_BIASES, FLAG_IMU_INTRINSICS = 1, 2, 4, 8
FLAG_GRAVITY_DIR, FLAG_CAM_LINE_DELAY, FLAG_SPLINE, FLAG_ACC_BIAS, FLAG_GYR_BIAS = 16, 32, 64, 128, 256
FLAG_CAM_INTRINSICS, FLAG_TIME_OFFSET = 512, 1024     # north-star extensions (the reference keeps both fixed)

STATUS_NAMES = {0: "ICC_OK", 1: "ICC_ERR_INVALID_ARGUMENT", 2: "ICC_ERR_NO_DEVICE", 3: "ICC_ERR_CUDA", 4: "ICC_ERR_STATE",
                5: "ICC_ERR_UNSUPPORTED", 6: "ICC_ERR_NUMERIC"}
TERMINATION = {0: "max_iterations", 1: "function_tolerance", 2: "parameter_tolerance", 3: "gradient_tolerance", 4: "failure"}
# icc_get_solver_plan's int32[16] (the last three are reserved)
PLAN_FIELDS = ("valid", "P", "w", "len", "rem", "L", "kd", "nb", "nk", "WS_A", "cl_global", "cs_global", "stage0")


class InitParams(C.Structure):
    _fields_ = [("T_i_c_init", C.c_double * 7), ("dt_so3_s", C.c_double), ("dt_r3_s", C.c_double), ("std_so3", C.c_double),
                ("std_r3", C.c_double), ("time_offset_imu_to_cam_s", C.c_double), ("init_line_delay_s", C.c_double),
                ("acc_intrinsics", C.c_double * 6), ("gyr_intrinsics", C.c_double * 9), ("acc_bias", C.c_double * 3),
                ("gyr_bias", C.c_double * 3), ("dispatch_fov", C.c_int32), ("reserved", C.c_int32)]


class SolverOptions(C.Structure):
    _fields_ = [("function_tolerance", C.c_double), ("parameter_tolerance", C.c_double), ("gradient_tolerance", C.c_double),
                ("initial_trust_region_radius", C.c_double), ("max_trust_region_radius", C.c_double),
                ("min_trust_region_radius", C.c_double), ("min_relative_decrease", C.c_double), ("min_lm_diagonal", C.c_double),
                ("max_lm_diagonal", C.c_double), ("jacobi_scaling", C.c_int32), ("max_consecutive_invalid_steps", C.c_int32)]


class Summary(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("successful_steps", C.c_int32), ("termination", C.c_int32), ("num_residuals", C.c_int32),
                ("num_tangent", C.c_int32), ("jacobian_evaluations", C.c_int32), ("cost_evaluations", C.c_int32),
                ("gpu_launches", C.c_int32), ("initial_cost", C.c_double), ("final_cost", C.c_double),
                ("mean_reproj_error", C.c_double), ("seconds_total", C.c_double), ("seconds_jacobian", C.c_double),
                ("seconds_linear_solve", C.c_double)]

    def as_dict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_}
        d["termination_name"] = TERMINATION.get(self.termination, "?")
        return d


class CamCalOptions(C.Structure):
    """icc_camcal_options (include/icc_b200.h): zero / negative fields select the reference's defaults."""
    _fields_ = [("grid_size", C.c_double), ("function_tolerance", C.c_double), ("parameter_tolerance", C.c_double), ("gradient_tolerance", C.c_double),
                ("huber_width", C.c_double), ("max_view_error_stage1_px", C.c_double), ("max_view_error_final_px", C.c_double),
                ("min_num_views", C.c_int32), ("max_num_iterations", C.c_int32), ("optimize_board_points", C.c_int32), ("reserved", C.c_int32)]


class CamCalSummary(C.Structure):
    _fields_ = [("success", C.c_int32), ("n_views_initialized", C.c_int32), ("n_views_selected", C.c_int32), ("n_views_used", C.c_int32),
                ("iterations", C.c_int32 * 3), ("termination", C.c_int32 * 3), ("gpu_launches", C.c_int32), ("init_iterations", C.c_int32), ("n_points_optimized", C.c_int32), ("reserved", C.c_int32),
                ("focal_length_init", C.c_double), ("initial_cost", C.c_double), ("final_cost", C.c_double * 3), ("final_reproj_error", C.c_double),
                ("seconds_total", C.c_double)]

    def as_dict(self):
        d = {}
        for k, _ in self._fields_:
            v = getattr(self, k)
            d[k] = list(v) if hasattr(v, "__len__") else v
        return d


class CamCalStepOut(C.Structure):
    """icc_camcal_step_out (include/icc_b200.h): caller-owned output arrays, each nullable."""
    _fields_ = [(k, c_double_p) for k in ("blocks", "sys", "red", "Y", "scale", "dk", "scalars", "q_wc_cand", "p_wc_cand", "intr_cand", "view_error_px")]


CC_PACK, CC_Y = 153, 66    # packed upper triangle of a view's 17 x 17 [J | r] block; A^-1 [H_pk | g_p] (6 x 11)
CAMCAL_SCALARS = ("cand_cost", "g_delta", "d_delta", "step_sq", "x_sq", "fail", "grad_max", "x_cost")


ALLREDUCE_FN =C.CFUNCTYPE(None, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p)


class IccError(RuntimeError):
    pass


def _dp(a):
    return None if a is None else a.ctypes.data_as(c_double_p)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


class CApi:
    """Thin object wrapper around one solver handle of a loaded library."""

    def __init__(self, lib: C.CDLL, prefix: str, create_arg: int = 0):
        self.lib, self.prefix = lib, prefix
        self._keepalive = []
        h = C.c_void_p()
        f = self._fn("create"); f.restype = C.c_int; f.argtypes = [C.POINTER(C.c_void_p), C.c_int]
        st = f(C.byref(h), create_arg)
        self.h = h
        if st != 0:
            msg = self.last_error() if h.value else ""
            self.h = None
            raise IccError(f"{prefix}create failed: {STATUS_NAMES.get(st, st)} {msg}")

    def _fn(self, name):
        return getattr(self.lib, self.prefix + name)

    def last_error(self) -> str:
        f = self._fn("last_error"); f.restype = C.c_char_p; f.argtypes = [C.c_void_p]
        return (f(self.h) or b"").decode()

    def _call(self, name, argtypes, *args):
        f = self._fn(name); f.restype = C.c_int; f.argtypes = [C.c_void_p] + list(argtypes)
        st = f(self.h, *args)
        if st != 0:
            raise IccError(f"{self.prefix}{name}: {STATUS_NAMES.get(st, st)}: {self.last_error()}")

    def close(self):
        if getattr(self, "h", None):
            f = self._fn("destroy"); f.restype = None; f.argtypes = [C.c_void_p]
            f(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- problem data --------------------------------------------------------------------------------------
    def set_solver_options(self, **kw):
        o = default_solver_options()
        for k, v in kw.items():
            setattr(o, k, v)
        self._call("set_solver_options", [C.POINTER(SolverOptions)], C.byref(o))

    def set_camera(self, model, intrinsics, width, height):
        k = _f64(intrinsics)
        self._call("set_camera", [C.c_int, c_double_p, C.c_int, C.c_int, C.c_int], int(model), _dp(k), k.size, int(width), int(height))

    def set_board_points(self, xyzw):
        p = _f64(xyzw).reshape(-1, 4)
        self._n_board = p.shape[0]
        self._call("set_board_points", [C.c_int, c_double_p], p.shape[0], _dp(p))

    def set_frames(self, t_s, corner_offsets, point_ids, uv, q_wc, p_wc):
        t = _f64(t_s); off = np.ascontiguousarray(corner_offsets, dtype=np.int32); ids = np.ascontiguousarray(point_ids, dtype=np.int32)
        uv = _f64(uv); q = _f64(q_wc); p = _f64(p_wc)
        assert off.size == t.size + 1 and ids.size == off[-1] and uv.size == 2 * ids.size and q.size == 4 * t.size and p.size == 3 * t.size
        self._call("set_frames", [C.c_int, c_double_p, c_int32_p, c_int32_p, c_double_p, c_double_p, c_double_p], t.size, _dp(t),
                   off.ctypes.data_as(c_int32_p), ids.ctypes.data_as(c_int32_p), _dp(uv), _dp(q), _dp(p))

    def set_imu(self, t_s, accel, gyro):
        t = _f64(t_s); a = _f64(accel); g = _f64(gyro)
        assert a.size == 3 * t.size and g.size == 3 * t.size
        self._call("set_imu", [C.c_int, c_double_p, c_double_p, c_double_p], t.size, _dp(t), _dp(a), _dp(g))

    # ---- upstream row f1: per-view board poses (PoseEstimator::EstimatePosesFromJson, src/core/pose_estimator.cc:92-191) ----
    def estimate_board_poses(self, corner_offsets, point_ids, uv, max_reproj_error=0.0, min_points=0):
        """-> (q_wc[n,4] x,y,z,w, p_wc[n,3], mean normalised reprojection error[n], valid[n]); camera + board points must be set."""
        off = np.ascontiguousarray(corner_offsets, dtype=np.int32); ids = np.ascontiguousarray(point_ids, dtype=np.int32); uv = _f64(uv)
        n = off.size - 1
        assert ids.size == off[-1] and uv.size == 2 * ids.size
        q = np.zeros((n, 4)); p = np.zeros((n, 3)); e = np.zeros(n); v = np.zeros(n, dtype=np.int32)
        self._call("estimate_board_poses", [C.c_int, c_int32_p, c_int32_p, c_double_p, C.c_double, C.c_int, c_double_p, c_double_p, c_double_p, c_int32_p],
                   n, off.ctypes.data_as(c_int32_p), ids.ctypes.data_as(c_int32_p), _dp(uv), float(max_reproj_error), int(min_points),
                   _dp(q), _dp(p), _dp(e), v.ctypes.data_as(c_int32_p))
        return q, p, e, v

    def filter_bad_poses(self, p_wc, valid):
        """PoseEstimator::FilterBadPoses (src/core/pose_estimator.cc:238-261): -> valid with the outlying camera heights cleared."""
        p = _f64(p_wc).reshape(-1, 3); v = np.array(valid, dtype=np.int32)
        self._call("filter_bad_poses", [C.c_int, c_double_p, c_int32_p], p.shape[0], _dp(p), v.ctypes.data_as(c_int32_p))
        return v

    def optimize_board_points(self, corner_offsets, point_ids, uv, q_wc, p_wc, valid, max_reproj_error=0.0, min_points=0, min_observations=0):
        """PoseEstimator::OptimizeBoardPoints + OptimizeAllPoses (pose_estimator.cc:193-236)
        -> (q_wc, p_wc, mean error, valid, board_xyzw, number of optimised points); the handle's board points are replaced."""
        off = np.ascontiguousarray(corner_offsets, dtype=np.int32); ids = np.ascontiguousarray(point_ids, dtype=np.int32); uv = _f64(uv)
        n = off.size - 1
        q = np.array(q_wc, dtype=np.float64).reshape(n, 4).copy(); p = np.array(p_wc, dtype=np.float64).reshape(n, 3).copy()
        v = np.array(valid, dtype=np.int32).copy(); e = np.zeros(n); nopt = C.c_int32()
        board = np.zeros((self.num_board_points(), 4))
        self._call("optimize_board_points", [C.c_int, c_int32_p, c_int32_p, c_double_p, C.c_double, C.c_int, C.c_int, c_double_p, c_double_p, c_double_p, c_int32_p, c_double_p, C.POINTER(C.c_int32)],
                   n, off.ctypes.data_as(c_int32_p), ids.ctypes.data_as(c_int32_p), _dp(uv), float(max_reproj_error), int(min_points), int(min_observations),
                   _dp(q), _dp(p), _dp(e), v.ctypes.data_as(c_int32_p), _dp(board), C.byref(nopt))
        return q, p, e, v, board, nopt.value

    def num_board_points(self):
        return getattr(self, "_n_board", 0)

    def get_board_points(self):
        b = np.zeros((self.num_board_points(), 4)); self._call("get_board_points", [c_double_p, C.c_int], _dp(b), b.shape[0]); return b

    def pixels_to_normalized(self, uv):
        """theia::Camera::PixelToNormalizedCoordinates / z for an (n, 2) pixel array -> (xy[n,2], ok[n])."""
        uv = _f64(uv).reshape(-1, 2); n = uv.shape[0]
        xy = np.zeros((n, 2)); ok = np.zeros(n, dtype=np.int32)
        self._call("pixels_to_normalized", [C.c_int, c_double_p, c_double_p, c_int32_p], n, _dp(uv), _dp(xy), ok.ctypes.data_as(c_int32_p))
        return xy, ok

    # ---- upstream row f4: CameraCalibrator::CalibrateCameraFromJson / RunCalibration (src/core/camera_calibrator.cc:131-389) ----
    def calibrate_camera(self, model, image_width, image_height, corner_offsets, point_ids, uv, q_wc_init=None, p_wc_init=None, init_valid=None,
                         focal_length_init=0.0, distortion_init=0.0, **options):
        """-> dict(intrinsics[n], q_wc[nv,4], p_wc[nv,3], view_error_px[nv], used[nv], summary); board points must be set.
        options: fields of icc_camcal_options (grid_size defaults to the reference's 0.04 m)."""
        off = np.ascontiguousarray(corner_offsets, dtype=np.int32); ids = np.ascontiguousarray(point_ids, dtype=np.int32); uv = _f64(uv)
        nv = off.size - 1
        assert ids.size == off[-1] and uv.size == 2 * ids.size
        o = CamCalOptions(); o.grid_size = -1.0
        for k, v in options.items():
            setattr(o, k, v)
        qi = None if q_wc_init is None else _f64(q_wc_init); pi = None if p_wc_init is None else _f64(p_wc_init)
        vi = None if init_valid is None else np.ascontiguousarray(init_valid, dtype=np.int32)
        intr = np.zeros(10); q = np.zeros((nv, 4)); p = np.zeros((nv, 3)); e = np.zeros(nv); used = np.zeros(nv, dtype=np.int32); s = CamCalSummary()
        self._call("calibrate_camera", [C.c_int, C.c_int, C.c_int, C.c_int, c_int32_p, c_int32_p, c_double_p, c_double_p, c_double_p, c_int32_p, C.c_double, C.c_double,
                                        C.POINTER(CamCalOptions), c_double_p, c_double_p, c_double_p, c_double_p, c_int32_p, C.POINTER(CamCalSummary)],
                   int(model), int(image_width), int(image_height), nv, off.ctypes.data_as(c_int32_p), ids.ctypes.data_as(c_int32_p), _dp(uv),
                   None if qi is None else _dp(qi), None if pi is None else _dp(pi), None if vi is None else vi.ctypes.data_as(c_int32_p),
                   float(focal_length_init), float(distortion_init), C.byref(o), _dp(intr), _dp(q), _dp(p), _dp(e), used.ctypes.data_as(c_int32_p), C.byref(s))
        from .camera_models import NUM_PARAMS
        return dict(intrinsics=intr[:NUM_PARAMS[int(model)]], q_wc=q, p_wc=p, view_error_px=e, used=used, summary=s.as_dict())

    def camcal_step(self, model, corner_offsets, point_ids, uv, q_wc, p_wc, intrinsics, active, intr_mask, pose_free, radius,
                    huber_width=1.345, scale_in=None):
        """One iteration body of the camera calibration's bundle adjustment at a given state (icc_camcal_step) -> dict of blocks
        (n_active, 153), sys (154), red (66), Y (n_active, 6, 11), scale (6 n_active + 10), dk (10), scalars (CAMCAL_SCALARS),
        q_wc_cand, p_wc_cand, intr_cand (10), view_error_px; board points must be set."""
        off = np.ascontiguousarray(corner_offsets, dtype=np.int32); ids = np.ascontiguousarray(point_ids, dtype=np.int32); uv = _f64(uv)
        act = np.ascontiguousarray(active, dtype=np.int32)
        nv, na = off.size - 1, act.size
        q, p, k = _f64(q_wc).reshape(nv, 4), _f64(p_wc).reshape(nv, 3), _f64(intrinsics)
        assert ids.size == off[-1] and uv.size == 2 * ids.size and k.size == 10
        si = None if scale_in is None else _f64(scale_in)
        assert si is None or si.size == 6 * na + 10
        r = dict(blocks=np.zeros((na, CC_PACK)), sys=np.zeros(CC_PACK + 1), red=np.zeros(66), Y=np.zeros((na, 6, 11)), scale=np.zeros(6 * na + 10),
                 dk=np.zeros(10), scalars=np.zeros(len(CAMCAL_SCALARS)), q_wc_cand=np.zeros((nv, 4)), p_wc_cand=np.zeros((nv, 3)),
                 intr_cand=np.zeros(10), view_error_px=np.zeros(nv))
        out = CamCalStepOut(*(_dp(r[f]) for f, _ in CamCalStepOut._fields_))
        self._call("camcal_step", [C.c_int, C.c_int, c_int32_p, c_int32_p, c_double_p, c_double_p, c_double_p, c_double_p, C.c_int, c_int32_p,
                                   C.c_uint32, C.c_int, C.c_double, C.c_double, c_double_p, C.POINTER(CamCalStepOut)],
                   int(model), nv, off.ctypes.data_as(c_int32_p), ids.ctypes.data_as(c_int32_p), _dp(uv), _dp(q), _dp(p), _dp(k), na,
                   act.ctypes.data_as(c_int32_p), int(intr_mask), int(pose_free), float(huber_width), float(radius), _dp(si), C.byref(out))
        r["scalars"] = dict(zip(CAMCAL_SCALARS, r["scalars"]))
        return r

    # ---- upstream row f3: ImuToCameraRotationEstimator (src/core/imu_to_camera_rotation_estimator.cc:116-274) -----------------
    def estimate_imu_to_camera_rotation(self, view_t_s, q_cw_xyzw, imu_t_s, gyro, gyro_bias=None):
        """-> dict(q_gyro_to_cam (x,y,z,w), time_offset_s, gyro_bias[3], error, iterations); gyro_bias=None estimates the bias."""
        vt = _f64(view_t_s); q = _f64(q_cw_xyzw); it = _f64(imu_t_s); g = _f64(gyro)
        assert q.size == 4 * vt.size and g.size == 3 * it.size
        qo = np.zeros(4); td = C.c_double(); bo = np.zeros(3); err = C.c_double(); iters = C.c_int32()
        b = None if gyro_bias is None else _f64(gyro_bias)
        self._call("estimate_imu_to_camera_rotation", [C.c_int, c_double_p, c_double_p, C.c_int, c_double_p, c_double_p, c_double_p, c_double_p,
                                                       C.POINTER(C.c_double), c_double_p, C.POINTER(C.c_double), C.POINTER(C.c_int32)],
                   vt.size, _dp(vt), _dp(q), it.size, _dp(it), _dp(g), None if b is None else _dp(b), _dp(qo), C.byref(td), _dp(bo), C.byref(err), C.byref(iters))
        return dict(q_gyro_to_cam=qo, time_offset_s=td.value, gyro_bias=bo, error=err.value, iterations=iters.value)

    # ---- upstream: static IMU biases (python/get_imu_biases.py:36-53) -----------------------------------------------------------------
    def estimate_imu_biases(self, accel, gyro, gravity_const=9.81):
        """-> (accl_bias[3], gyro_bias[3]) as written to the hot CLI's --imu_bias_file."""
        a = _f64(accel).reshape(-1, 3); g = _f64(gyro).reshape(-1, 3)
        assert a.shape == g.shape
        ba, bg = np.zeros(3), np.zeros(3)
        self._call("estimate_imu_biases", [C.c_int, c_double_p, c_double_p, C.c_double, c_double_p, c_double_p], a.shape[0], _dp(a), _dp(g), float(gravity_const), _dp(ba), _dp(bg))
        return ba, bg

    # ---- upstream row f2: spline error weighting (python/sew.py:knot_spacing_and_variance) ------------------------------------
    def spline_error_weighting(self, times_s, signal_xyz, quality, min_dt=0.0, max_dt=0.0, want_spectrum=False):
        """-> (knot_spacing, variance[, reference spectrum Xhat]); signal_xyz is (n, 3)."""
        t = _f64(times_s); x = _f64(signal_xyz).reshape(-1, 3)
        assert x.shape[0] == t.size
        dt = C.c_double(); var = C.c_double(); spec = np.zeros(t.size) if want_spectrum else None
        self._call("spline_error_weighting", [C.c_int, c_double_p, c_double_p, C.c_double, C.c_double, C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double), c_double_p],
                   t.size, _dp(t), _dp(x), float(quality), float(min_dt), float(max_dt), C.byref(dt), C.byref(var), None if spec is None else _dp(spec))
        return (dt.value, var.value, spec) if want_spectrum else (dt.value, var.value)

    def set_shard(self, rank, world):
        self._call("set_shard", [C.c_int, C.c_int], int(rank), int(world))

    def set_comm(self, comm):
        """Attach the library-owned NCCL communicator (Comm): sets the residual shard to its (rank, world) and routes every cross-rank
        sum through ncclAllReduce on the solver's stream.  None detaches."""
        self._call("set_comm", [C.c_void_p], comm.c if comm is not None else None)
        self._keepalive.append(comm)

    def set_allreduce(self, pyfunc):
        cb = ALLREDUCE_FN(pyfunc) if pyfunc is not None else C.cast(None, ALLREDUCE_FN)
        self._keepalive.append(cb)
        self._call("set_allreduce", [ALLREDUCE_FN, C.c_void_p], cb, None)

    def batch_init_spline(self, T_i_c_init, dt_so3_s, dt_r3_s, std_so3, std_r3, time_offset_imu_to_cam_s, init_line_delay_s,
                          acc_intrinsics=(0, 0, 0, 1, 1, 1), gyr_intrinsics=(0, 0, 0, 0, 0, 0, 1, 1, 1), acc_bias=(0, 0, 0),
                          gyr_bias=(0, 0, 0), dispatch_fov=False):
        p = InitParams()
        p.T_i_c_init[:] = list(map(float, T_i_c_init)); p.dt_so3_s = dt_so3_s; p.dt_r3_s = dt_r3_s; p.std_so3 = std_so3; p.std_r3 = std_r3
        p.time_offset_imu_to_cam_s = time_offset_imu_to_cam_s; p.init_line_delay_s = init_line_delay_s
        p.acc_intrinsics[:] = list(map(float, acc_intrinsics)); p.gyr_intrinsics[:] = list(map(float, gyr_intrinsics))
        p.acc_bias[:] = list(map(float, acc_bias)); p.gyr_bias[:] = list(map(float, gyr_bias)); p.dispatch_fov = int(bool(dispatch_fov))
        self._call("batch_init_spline", [C.POINTER(InitParams)], C.byref(p))

    def set_known_gravity_dir(self, g):
        g = _f64(g)
        self._call("set_known_gravity_dir", [c_double_p], _dp(g))

    # ---- solve ---------------------------------------------------------------------------------------------
    def optimize(self, max_iterations, flags) -> Summary:
        s = Summary()
        self._call("optimize", [C.c_int, C.c_int, C.POINTER(Summary)], int(max_iterations), int(flags), C.byref(s))
        return s

    def lm_iterations(self, n, flags) -> Summary:
        s = Summary()
        self._call("lm_iterations", [C.c_int, C.c_int, C.POINTER(Summary)], int(n), int(flags), C.byref(s))
        return s

    def time_evaluations(self, n, flags, with_jacobian=True) -> float:
        ms = C.c_double()
        self._call("time_evaluations", [C.c_int, C.c_int, C.c_int, c_double_p], int(n), int(flags), int(with_jacobian), C.byref(ms))
        return ms.value

    # ---- getters -------------------------------------------------------------------------------------------
    def get_T_i_c(self):
        T = np.zeros(7); self._call("get_T_i_c", [c_double_p], _dp(T)); return T

    def set_T_i_c(self, T):
        T = _f64(T); self._call("set_T_i_c", [c_double_p], _dp(T))

    def get_gravity(self):
        g = np.zeros(3); self._call("get_gravity", [c_double_p], _dp(g)); return g

    def get_line_delay(self):
        v = C.c_double(); self._call("get_line_delay", [c_double_p], C.byref(v)); return v.value

    def get_camera_intrinsics(self, n=10):
        k = np.zeros(n); self._call("get_camera_intrinsics", [c_double_p, C.c_int], _dp(k), n); return k

    def get_time_offset(self):
        v = C.c_double(); self._call("get_time_offset", [c_double_p], C.byref(v)); return v.value

    def set_line_delay(self, v):
        self._call("set_line_delay", [C.c_double], float(v))

    def num_knots(self):
        a, b, c, d = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        self._call("get_num_knots", [C.POINTER(C.c_int)] * 4, C.byref(a), C.byref(b), C.byref(c), C.byref(d))
        return a.value, b.value, c.value, d.value

    def get_knots(self):
        a, b, c, d = self.num_knots()
        so3, r3, ba, bg = np.zeros((a, 4)), np.zeros((b, 3)), np.zeros((c, 3)), np.zeros((d, 3))
        self._call("get_knots", [c_double_p] * 4, _dp(so3), _dp(r3), _dp(ba), _dp(bg))
        return so3, r3, ba, bg

    def set_knots(self, so3=None, r3=None, ba=None, bg=None):
        arrs = [None if x is None else _f64(x) for x in (so3, r3, ba, bg)]
        self._call("set_knots", [c_double_p] * 4, *[_dp(x) for x in arrs])

    def mean_reprojection_error(self):
        v = C.c_double(); self._call("get_mean_reprojection_error", [c_double_p], C.byref(v)); return v.value

    def imu_used(self):
        n = C.c_int(); self._call("get_num_imu_used", [C.POINTER(C.c_int)], C.byref(n))
        t, a, g = np.zeros(n.value), np.zeros((n.value, 3)), np.zeros((n.value, 3))
        self._call("get_imu_used", [c_double_p] * 3, _dp(t), _dp(a), _dp(g))
        return t, a, g

    def imu_cells(self):
        """Knot-interval cells of the kept IMU samples: rows (s_so3, s_r3, s_acc_bias, s_gyr_bias, i_begin, i_end)."""
        n = C.c_int(); self._call("get_num_imu_cells", [C.POINTER(C.c_int)], C.byref(n))
        c = np.zeros((n.value, 6), dtype=np.int32)
        self._call("get_imu_cells", [c_int32_p], c.ctypes.data_as(c_int32_p))
        return c

    def eval_trajectory(self, t_ns):
        t = np.ascontiguousarray(t_ns, dtype=np.int64); n = t.size
        out = dict(gyro=np.zeros((n, 3)), accel=np.zeros((n, 3)), gyro_bias=np.zeros((n, 3)), accel_bias=np.zeros((n, 3)),
                   pose_q=np.zeros((n, 4)), pose_p=np.zeros((n, 3)), valid=np.zeros(n, dtype=np.int32))
        self._call("eval_trajectory", [C.c_int, c_int64_p] + [c_double_p] * 6 + [c_int32_p], n, t.ctypes.data_as(c_int64_p), _dp(out["gyro"]),
                   _dp(out["accel"]), _dp(out["gyro_bias"]), _dp(out["accel_bias"]), _dp(out["pose_q"]), _dp(out["pose_p"]),
                   out["valid"].ctypes.data_as(c_int32_p))
        return out

    def get_stream(self) -> int:
        f = self._fn("get_stream"); f.restype = C.c_void_p; f.argtypes = [C.c_void_p]
        return int(f(self.h) or 0)

    # ---- test / measurement surface --------------------------------------------------------------------------
    def num_residuals(self):
        v, a, g = C.c_int(), C.c_int(), C.c_int()
        self._call("num_residuals", [C.POINTER(C.c_int)] * 3, C.byref(v), C.byref(a), C.byref(g))
        return v.value, a.value, g.value

    def num_tangent(self, flags):
        n = C.c_int(); self._call("num_tangent", [C.c_int, C.POINTER(C.c_int)], int(flags), C.byref(n)); return n.value

    def evaluate(self, flags, residuals=True, gradient=True, hessian=False):
        nres = sum(self.num_residuals()); n = self.num_tangent(flags)
        cost = C.c_double()
        r = np.zeros(nres) if residuals else None
        g = np.zeros(n) if gradient else None
        H = np.zeros((n, n)) if hessian else None
        self._call("evaluate", [C.c_int, c_double_p, c_double_p, c_double_p, c_double_p], int(flags), C.byref(cost), _dp(r), _dp(g), _dp(H))
        return cost.value, r, g, H

    def solver_plan(self, flags, chunks=0) -> dict:
        """Elimination plan of the damped solve (icc_get_solver_plan); chunks > 0 forces the level-0 chunk count."""
        p = np.zeros(16, dtype=np.int32)
        self._call("get_solver_plan", [C.c_int, C.c_int, c_int32_p], int(flags), int(chunks), p.ctypes.data_as(c_int32_p))
        return dict(zip(PLAN_FIELDS, (int(v) for v in p)))

    def solve_step(self, flags, radius, chunks=0, hessian=True) -> dict:
        """One damped solve at the current state (icc_solve_step): cost, gradient, hessian (None unless asked), scale, lm_diag,
        delta, model_change, all from the one evaluation the solve consumed, canonical tangent order."""
        n = self.num_tangent(flags)
        cost, mc = C.c_double(), C.c_double()
        g, s, d, x = np.zeros(n), np.zeros(n), np.zeros(n), np.zeros(n)
        H = np.zeros((n, n)) if hessian else None
        self._call("solve_step", [C.c_int, C.c_double, C.c_int] + [c_double_p] * 7, int(flags), float(radius), int(chunks),
                   C.byref(cost), _dp(g), _dp(H), _dp(s), _dp(d), _dp(x), C.byref(mc))
        return dict(cost=cost.value, gradient=g, hessian=H, scale=s, lm_diag=d, delta=x, model_change=mc.value)


def _normal_matvec(self, flags, V):
    """J^T J V from the packed normal equations of the current state (V: (nvec, n_tangent), canonical order)."""
    V = np.ascontiguousarray(V, dtype=np.float64)
    out = np.zeros_like(V)
    self._call("normal_matvec", [C.c_int, C.c_int, c_double_p, c_double_p], int(flags), int(V.shape[0]), _dp(V), _dp(out))
    return out


CApi.normal_matvec = _normal_matvec


class Comm:
    """icc_comm: the library's own NCCL communicator (include/icc_b200.h).  `unique_id()` on one rank, `Comm(lib, id, rank, world,
    device)` on every rank (collective)."""
    ID_BYTES = 128

    @staticmethod
    def unique_id(lib) -> bytes:
        buf = (C.c_ubyte * Comm.ID_BYTES)()
        f = lib.icc_comm_unique_id; f.restype = C.c_int; f.argtypes = [C.c_void_p]
        st = f(buf)
        if st != 0:
            e = lib.icc_comm_last_error; e.restype = C.c_char_p
            raise IccError(f"icc_comm_unique_id: {STATUS_NAMES.get(st, st)}: {(e() or b'').decode()}")
        return bytes(buf)

    def __init__(self, lib, uid: bytes, rank: int, world: int, device: int):
        self.lib, self.rank, self.world = lib, int(rank), int(world)
        out = C.c_void_p()
        buf = (C.c_ubyte * Comm.ID_BYTES).from_buffer_copy(uid)
        f = lib.icc_comm_create; f.restype = C.c_int; f.argtypes = [C.POINTER(C.c_void_p), C.c_void_p, C.c_int, C.c_int, C.c_int]
        st = f(C.byref(out), buf, int(rank), int(world), int(device))
        if st != 0:
            e = lib.icc_comm_last_error; e.restype = C.c_char_p
            raise IccError(f"icc_comm_create: {STATUS_NAMES.get(st, st)}: {(e() or b'').decode()}")
        self.c = out

    def close(self):
        if getattr(self, "c", None):
            f = self.lib.icc_comm_destroy; f.restype = None; f.argtypes = [C.c_void_p]
            f(self.c); self.c = None


def default_solver_options() -> SolverOptions:
    """ceres::Solver::Options of SplineTrajectoryEstimator::Optimize (impl.h:254-266) + Ceres 2.1 defaults."""
    return SolverOptions(1e-4, 1e-7, 1e-10, 1e4, 1e16, 1e-32, 1e-3, 1e-6, 1e32, 1, 5)


def load_dataset(api: CApi, ds: dict, known_gravity=True, dispatch_fov=None, shard=None, comm=None):
    """Feed a synthetic dataset (synthetic.make_dataset) through the boundary in the order the hot CLI does."""
    W, H = ds["image_size"]
    api.set_camera(ds["model"], ds["intrinsics"], W, H)
    api.set_board_points(ds["board_xyzw"])
    api.set_frames(ds["frame_t"], ds["corner_offsets"], ds["point_ids"], ds["uv"], ds["q_wc"], ds["p_wc"])
    api.set_imu(ds["imu_t"], ds["accel"], ds["gyro"])
    if shard is not None:
        api.set_shard(*shard)
    if comm is not None:
        api.set_comm(comm)
    if dispatch_fov is None:
        dispatch_fov = ds["model"] == 3
    api.batch_init_spline(ds["T_i_c_init"], ds["dt_so3_s"], ds["dt_r3_s"], ds["std_so3"], ds["std_r3"], ds["time_offset_imu_to_cam_s"],
                          ds["init_line_delay_s"], acc_bias=ds["acc_bias"], gyr_bias=ds["gyr_bias"], dispatch_fov=dispatch_fov)
    if known_gravity:
        api.set_known_gravity_dir(ds["gravity"])
