"""The C-ABI library loads, exports every symbol include/icc_b200.h declares, refuses to compute without a GPU, and its
host-side problem assembly (BatchInitSpline) agrees with the oracle's restatement of the reference."""
import ctypes
import os
import re

import numpy as np
import pytest

from openimucameracalibrator_b200 import _capi as capi
from openimucameracalibrator_b200 import calibrator
from openimucameracalibrator_b200 import synthetic as syn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "icc_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(icc_[a-z0-9_]+)\s*\(", text)) - {"icc_allreduce_fn"})


def test_library_exports_every_declared_symbol():
    lib = calibrator.load_library()
    syms = _declared_symbols()
    assert len(syms) >= 30
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/icc_b200.h but not exported"


def test_no_cpu_fallback_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present; the no-device path is exercised on the CPU box")
    with pytest.raises(capi.IccError, match="ICC_ERR_NO_DEVICE"):
        capi.CApi(calibrator.load_library(), "icc_", 0)
    # a host-only handle can assemble but must refuse every compute entry point
    h = capi.CApi(calibrator.load_library(), "icc_", -1)
    capi.load_dataset(h, syn.make_dataset(syn.tiny_config()))
    for call in (lambda: h.optimize(1, 66), lambda: h.evaluate(66), lambda: h.lm_iterations(1, 66), lambda: h.mean_reprojection_error(),
                 lambda: h.eval_trajectory([0]), lambda: h.time_evaluations(1, 66),
                 lambda: h.calibrate_camera(0, 960, 540, [0, 1], [0], [[1.0, 2.0]]), lambda: h.estimate_imu_biases(np.ones((4, 3)), np.ones((4, 3))),
                 lambda: h.camcal_step(0, [0, 1], [0], [[1.0, 2.0]], [[0, 0, 0, 1.0]], [[0, 0, 1.0]], np.ones(10), [0], 1, 1, 1e4),
                 lambda: h.optimize_board_points([0, 1], [0], [[1.0, 2.0]], [[0, 0, 0, 1.0]], [[0, 0, 1.0]], [1])):
        with pytest.raises(capi.IccError, match="ICC_ERR_NO_DEVICE"):
            call()


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    monkeypatch.setattr(calibrator, "_LIB", None)
    monkeypatch.setattr(calibrator, "library_path", lambda: str(tmp_path / "libicc_b200.so"))
    with pytest.raises(capi.IccError, match="no CPU fallback"):
        calibrator.load_library()


def test_product_package_never_references_the_oracle():
    pkg = os.path.join(ROOT, "openimucameracalibrator_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                text = open(os.path.join(dirpath, f)).read()
                assert "libicc_oracle" not in text and "icc_oracle" not in text and "oracle_api" not in text and "icco_" not in text.replace("`icco_`", ""), f


@pytest.mark.parametrize("cfg", [syn.tiny_config(), syn.tiny_config(dt_so3_s=0.04, dt_r3_s=0.07), syn.CONFIGS[1]], ids=["tiny", "tiny_uneven_dt", "cfg1"])
def test_host_assembly_matches_oracle(oracle_factory, cfg):
    """Knot counts, knot initialisation (slerp/lerp quirks), kept IMU samples, residual counts, gravity init."""
    ds = syn.make_dataset(cfg)
    o = oracle_factory(); capi.load_dataset(o, ds, known_gravity=False)
    h = capi.CApi(calibrator.load_library(), "icc_", -1); capi.load_dataset(h, ds, known_gravity=False)
    assert o.num_knots() == h.num_knots()
    assert o.num_residuals() == h.num_residuals()
    for a, b in zip(o.get_knots(), h.get_knots()):
        assert np.array_equal(a, b) or np.allclose(a, b, rtol=0, atol=1e-15)
    for a, b in zip(o.imu_used(), h.imu_used()):
        assert np.array_equal(a, b)
    assert np.allclose(o.get_gravity(), h.get_gravity(), rtol=0, atol=1e-14)
    assert np.allclose(o.get_T_i_c(), h.get_T_i_c(), rtol=0, atol=1e-15)
    for flags in (66, 66 | 16 | 32 | 4, 32, 66 | 8, 8, 66 | 1, 1):      # | 1 = POINTS: three tangent columns per board point
        assert o.num_tangent(flags) == h.num_tangent(flags)
    assert h.num_tangent(66 | 1) == h.num_tangent(66) + 3 * len(ds["board_xyzw"])
    with pytest.raises(capi.IccError, match="UNSUPPORTED"):
        h.num_tangent(66 | 1 | capi.FLAG_CAM_INTRINSICS)   # POINTS with this library's camera-intrinsics extension


def test_shards_partition_the_residuals(oracle_factory):
    ds = syn.make_dataset(syn.tiny_config())
    full = capi.CApi(calibrator.load_library(), "icc_", -1); capi.load_dataset(full, ds)
    tot = np.zeros(3, dtype=int)
    for r in range(3):
        h = capi.CApi(calibrator.load_library(), "icc_", -1); capi.load_dataset(h, ds, shard=(r, 3))
        o = oracle_factory(); capi.load_dataset(o, ds, shard=(r, 3))
        assert h.num_residuals() == o.num_residuals()
        tot += np.array(h.num_residuals())
    assert tuple(tot) == full.num_residuals()


def test_invalid_arguments_are_reported():
    h = capi.CApi(calibrator.load_library(), "icc_", -1)
    with pytest.raises(capi.IccError, match="INVALID_ARGUMENT"):
        h.set_camera(4, [1.0, 2.0], 10, 10)           # wrong intrinsic count
    with pytest.raises(capi.IccError, match="STATE"):
        h.batch_init_spline(np.array([0, 0, 0, 1, 0, 0, 0.0]), 0.05, 0.05, 1, 1, 0, 1e-5)
    with pytest.raises(capi.IccError, match="INVALID_ARGUMENT"):
        h.set_shard(3, 2)


@pytest.mark.parametrize("case", ["shuffled_imu", "imu_hole", "duplicate_view_time"])
def test_host_assembly_general_paths_match_oracle(oracle_factory, case):
    """The one-shard fast path of BatchInitSpline assumes a time-sorted, gap-free IMU stream and increasing view timestamps; anything
    else must fall back to the general path and still agree with the oracle."""
    ds = dict(syn.make_dataset(syn.tiny_config()))
    if case == "shuffled_imu":
        perm = np.random.default_rng(0).permutation(len(ds["imu_t"]))
        ds["imu_t"], ds["accel"], ds["gyro"] = ds["imu_t"][perm], ds["accel"][perm], ds["gyro"][perm]
    elif case == "imu_hole":
        t = ds["imu_t"].copy(); t[50] = 1e6; ds["imu_t"] = t            # one sample far outside the window, mid-stream
    else:
        t = ds["frame_t"].copy(); t[5] = t[4]; ds["frame_t"] = t
    o = oracle_factory(); capi.load_dataset(o, ds, known_gravity=False)
    h = capi.CApi(calibrator.load_library(), "icc_", -1); capi.load_dataset(h, ds, known_gravity=False)
    assert o.num_residuals() == h.num_residuals() and o.num_knots() == h.num_knots()
    for a, b in zip(o.imu_used(), h.imu_used()):
        assert np.array_equal(a, b)
    for a, b in zip(o.get_knots(), h.get_knots()):
        assert np.allclose(a, b, rtol=0, atol=1e-15)
    assert np.allclose(o.get_gravity(), h.get_gravity(), rtol=0, atol=1e-14)


@pytest.mark.parametrize("dts", [(0.05, 0.05), (0.04, 0.07), (0.09, 0.05)])
def test_imu_cells_by_bisection_equal_the_sample_by_sample_pass(dts, monkeypatch):
    """BatchInitSpline finds the knot-interval cells of a time-sorted IMU stream by galloping + bisection for the next interval boundary;
    the sample-by-sample pass (forced with ICC_NO_BISECTION) is the reference statement: same cells, same kept samples -- for irregular
    stamps, stamps exactly on knot boundaries of either spline and repeated stamps."""
    ds = dict(syn.make_dataset(syn.tiny_config(n_frames=40, dt_so3_s=dts[0], dt_r3_s=dts[1])))
    rng = np.random.default_rng(int(1000 * dts[0]))
    t0 = float(ds["frame_t"][0]) - ds["time_offset_imu_to_cam_s"]
    n = 4 * len(ds["imu_t"])
    t = np.sort(rng.uniform(ds["imu_t"][0] - 0.2, ds["imu_t"][-1] + 0.2, size=n))
    k = np.arange(0, n, 7); t[k] = t0 + dts[0] * np.round((t[k] - t0) / dts[0])
    k = np.arange(3, n, 11); t[k] = t0 + dts[1] * np.round((t[k] - t0) / dts[1])
    t = np.sort(t); t[5::13] = t[4::13][: len(t[5::13])]; t = np.sort(t)
    ds["imu_t"] = t; ds["accel"] = rng.normal(size=(n, 3)); ds["gyro"] = rng.normal(size=(n, 3))
    out = {}
    for mode in ("bisection", "sequential"):
        if mode == "sequential": monkeypatch.setenv("ICC_NO_BISECTION", "1")
        else: monkeypatch.delenv("ICC_NO_BISECTION", raising=False)
        h = capi.CApi(calibrator.load_library(), "icc_", -1); capi.load_dataset(h, ds, known_gravity=False)
        out[mode] = (h.imu_cells(), h.imu_used(), h.num_residuals()); h.close()
    cb, ub, rb = out["bisection"]; cs, us, rs = out["sequential"]
    assert rb == rs and len(cb) > 10
    assert np.array_equal(cb, cs)
    for a, b in zip(ub, us):
        assert np.array_equal(a, b)
    assert cb[0, 4] == 0 and cb[-1, 5] == len(ub[0]) and np.array_equal(cb[1:, 4], cb[:-1, 5])     # the cells tile the kept samples
