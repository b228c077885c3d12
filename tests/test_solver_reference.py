"""The damped normal-equation solve against a dense high-precision reference: the case table and the reference itself.

The GPU solve (icc_solver.cu) picks an elimination plan -- level-0 chunks, block cyclic reduction levels, shared-memory windows,
dense border blocks in global memory -- from a cost model and from shared-memory limits.  tests/test_gpu_solver_reference.py runs
one damped solve per (case, chunks, radius) of CASES and compares it with `damped_solve_reference`.  Here, without a GPU:
  * the plans of that table, read on host-only handles, reach every branch of the planner and the kernels at least once, so the
    GPU test cannot pass vacuously when some dataset's automatic plan moves;
  * the NumPy reference equals the oracle's independent statement of Ceres' step (icco_solve_step, the function lm_solve uses),
    so the GPU test cannot encode a misreading of the scaling, the damping or the model cost change."""
import numpy as np
import pytest

from helpers import F_ALL, F_STAGE1
from openimucameracalibrator_b200 import _capi as capi
from openimucameracalibrator_b200 import calibrator
from openimucameracalibrator_b200 import synthetic as syn

RADII = (1e-3, 1e4, 1e16)
F_WIDE = F_STAGE1 | capi.FLAG_IMU_BIASES | capi.FLAG_GRAVITY_DIR

# name -> (synthetic configuration, known gravity)
DATASETS = {
    "tiny": (lambda: syn.tiny_config(), True),
    "cfg2": (lambda: syn.CONFIGS[2], True),
    "uneven": (lambda: syn.tiny_config(n_frames=150, dt_so3_s=0.04, dt_r3_s=0.07), True),              # kd = 47
    "uneven_wide": (lambda: syn.tiny_config(n_frames=150, dt_so3_s=0.02, dt_r3_s=0.10), True),         # kd = 95
    "many": (lambda: syn.tiny_config(n_frames=400, fps=5.0, dt_so3_s=0.1, dt_r3_s=0.1, imu_rate_hz=50.0), True),   # nk = 4824
    # the 200 s sequence of test_very_wide_border_uses_hbm_border_blocks: 141 border columns with biases + gravity free
    "wide": (lambda: syn.tiny_config(n_frames=400, fps=2.0, dt_so3_s=0.5, dt_r3_s=0.5, imu_rate_hz=50.0, seed=41), False),
    "cfg4": (lambda: syn.CONFIGS[4], True),
}

# (case, dataset, flags, level-0 chunk counts; 0 = the library's own choice), all solved densely on the GPU box
CASES = [
    ("root_only_tic", "tiny", capi.FLAG_T_I_C, (0,)),
    ("root_only_line_delay", "tiny", capi.FLAG_CAM_LINE_DELAY, (0,)),
    ("empty_border", "tiny", capi.FLAG_SPLINE, (0, 1)),
    ("small", "tiny", F_STAGE1, (0, 1, 2, 3)),
    ("medium", "cfg2", F_STAGE1, (0, 1, 2, 3, 4, 5, 7, 16)),
    ("medium_border", "cfg2", F_ALL, (0, 4)),
    ("uneven", "uneven", F_STAGE1, (0, 2, 5)),
    ("uneven_wide", "uneven_wide", F_STAGE1, (0, 2, 5)),
    ("many_chunks", "many", F_STAGE1, (0, 64, 33)),
    ("wide_border", "wide", F_WIDE, (0, 1, 2)),
    ("widest_border", "cfg2", F_STAGE1 | capi.FLAG_POINTS, (0,)),
]
JACOBI_OFF = ("small", "medium")       # cases also solved without Jacobi scaling
# full size: no dense Hessian; the GPU test checks the residual through icc_normal_matvec
FULL_CASES = [("full_stage1", "cfg4", F_STAGE1, (0,)), ("full_all", "cfg4", F_ALL, (0,))]
# config 4's 144-point board with POINTS: 438 border columns, no plan fits the shared-memory limits
REFUSED = ("cfg4", F_STAGE1 | capi.FLAG_POINTS)


def load(api, name):
    cfg, known_gravity = DATASETS[name]
    capi.load_dataset(api, syn.make_dataset(cfg()), known_gravity=known_gravity)
    return api


def damped_solve_reference(H, g, radius, jacobi=True, min_diag=1e-6, max_diag=1e32, refinements=3, scale=None):
    """NumPy statement of one Levenberg-Marquardt step of Ceres (Jacobi scaling + clamped diagonal), solved densely in high precision:
    S = diag(1 / (1 + sqrt(H_ii))) (identity without Jacobi scaling; `scale` when given, e.g. the scale of a stage's first
    iteration reused on a later one), D = diag(clamp(diag(S H S), min, max) / radius),
    A = S H S + D, b = -S g; y from a float64 Cholesky plus `refinements` rounds of iterative refinement with the residual
    accumulated in long double.  -> dict(scale, lm_diag, A, b, y, delta = S y, model_change = 1/2 (y^T D y - y^T S g))."""
    from scipy.linalg import cho_factor, cho_solve
    H = np.asarray(H, dtype=np.float64); g = np.asarray(g, dtype=np.float64)
    if scale is not None:
        s = np.asarray(scale, dtype=np.float64)
    else:
        s = 1.0 / (1.0 + np.sqrt(np.diag(H))) if jacobi else np.ones(len(g))
    SHS = H * s[:, None] * s[None, :]
    D = np.minimum(np.maximum(np.diag(SHS), min_diag), max_diag) / radius
    A = SHS + np.diag(D)
    b = -s * g
    c = cho_factor(A, lower=True)
    y = cho_solve(c, b)
    Al, bl = A.astype(np.longdouble), b.astype(np.longdouble)
    for _ in range(refinements):
        y = y + cho_solve(c, (bl - Al @ y.astype(np.longdouble)).astype(np.float64))
    return dict(scale=s, lm_diag=D, A=A, b=b, y=y, delta=s * y, model_change=0.5 * float(y @ (D * y) - y @ (s * g)))


def backward_error(A, b, y):
    """Normwise backward error of y as a solution of A y = b, residual in long double: |A y - b|_inf / (|A|_inf |y|_inf + |b|_inf)."""
    r = A.astype(np.longdouble) @ np.asarray(y, dtype=np.longdouble) - np.asarray(b, dtype=np.longdouble)
    return float(np.abs(r).max() / (np.abs(A).sum(axis=1).max() * np.abs(y).max() + np.abs(b).max()))


def ulps(a, b):
    """Largest distance in units in the last place between two arrays of positive doubles."""
    return int(np.abs(np.asarray(a, dtype=np.float64).view(np.int64) - np.asarray(b, dtype=np.float64).view(np.int64)).max())


def odd_levels(P):
    """Cyclic-reduction levels whose block count is odd (the last block of such a level has no right neighbour)."""
    n, S = 0, P - 1
    while S > 1:
        n += S % 2; S //= 2
    return n


def test_case_table_covers_every_plan_branch():
    lib = calibrator.load_library()
    handles = {}
    plans = []
    for case, ds, flags, chunk_list in CASES + FULL_CASES:
        if ds not in handles:
            handles[ds] = load(capi.CApi(lib, "icc_", -1), ds)
        for chunks in chunk_list:
            p = handles[ds].solver_plan(flags, chunks)
            assert p["valid"] == 1, (case, chunks, p)
            plans.append((case, chunks, p))
    refused = handles[REFUSED[0]].solver_plan(REFUSED[1])
    assert refused["valid"] == 0 and refused["nb"] > 400, refused
    branches = {
        "nk = 0 (root only)": lambda p: p["nk"] == 0,
        "nb = 0 (no border)": lambda p: p["nb"] == 0 and p["nk"] > 0,
        "P = 1": lambda p: p["P"] == 1 and p["nk"] > 0,
        "P = 2": lambda p: p["P"] == 2,
        "P not a power of two": lambda p: p["P"] > 2 and p["P"] & (p["P"] - 1) != 0,
        "P >= 64": lambda p: p["P"] >= 64,
        "L >= 5": lambda p: p["L"] >= 5,
        "rem > 0": lambda p: p["rem"] > 0,
        "rem > 0 with odd block counts on two levels": lambda p: p["rem"] > 0 and odd_levels(p["P"]) >= 2,
        "kd > 35": lambda p: p["kd"] > 35 and p["P"] > 1,
        "kd > 35, one chunk": lambda p: p["kd"] > 35 and p["P"] == 1,
        "WS_A above its minimum": lambda p: p["WS_A"] > 1 << (p["kd"] + 16).bit_length(),
        "cl_global": lambda p: p["cl_global"] == 1,
        "cs_global": lambda p: p["cs_global"] == 1,
        "stage0 = 0": lambda p: p["stage0"] == 0,
        "chunked wide border (cl_global, P > 1)": lambda p: p["cl_global"] == 1 and p["P"] > 1,
    }
    missing = [name for name, hit in branches.items() if not any(hit(p) for _, _, p in plans)]
    assert not missing, f"no case of the table reaches: {missing}"
    # the automatic plans the GPU test's expectations rest on
    auto = {(case, chunks): p for case, chunks, p in plans}
    assert auto[("many_chunks", 0)]["P"] == 64 and auto[("full_stage1", 0)]["P"] == 128
    assert auto[("small", 3)]["P"] == 2                                   # forced chunks are clamped to leaves of >= kd + 1 columns


def test_forced_chunks_follow_the_planner():
    """chunks > 0 replaces only the chunk count: P = 1 is the sequential band factorisation, and an over-large request is halved /
    clamped exactly like the automatic choice (never a plan with leaves shorter than kd + 1)."""
    h = load(capi.CApi(calibrator.load_library(), "icc_", -1), "cfg2")
    p1 = h.solver_plan(F_STAGE1, 1)
    assert (p1["P"], p1["w"], p1["len"], p1["rem"], p1["L"]) == (1, 0, p1["nk"], 0, 0)
    for chunks in (2, 3, 7, 16, 31, 4096):
        p = h.solver_plan(F_STAGE1, chunks)
        assert p["valid"] == 1 and 1 <= p["P"] <= chunks
        assert p["len"] >= p["kd"] + 1 and p["P"] * p["len"] + p["rem"] + (p["P"] - 1) * p["w"] == p["nk"], (chunks, p)
        assert 0 <= p["rem"] < p["P"]
    assert h.solver_plan(F_STAGE1, 7)["P"] == 7


@pytest.mark.parametrize("ds", ["tiny", "cfg2"])
def test_numpy_reference_equals_the_oracle_step(oracle_factory, ds):
    """icco_solve_step (the step lm_solve takes: scale, clamped diagonal, sparse arrowhead Cholesky, model change) equals the dense
    NumPy reference on the oracle's own H and g, at small, default and huge radii, with and without Jacobi scaling."""
    o = load(oracle_factory(), ds)
    u = np.finfo(np.float64).eps
    for jacobi in (1, 0):
        o.set_solver_options(jacobi_scaling=jacobi)
        for radius in RADII:
            st = o.solve_step(F_STAGE1, radius)
            ref = damped_solve_reference(st["hessian"], st["gradient"], radius, jacobi=bool(jacobi))
            # the oracle forms diag(S H S) as H_ii (s_i s_i), the reference as (H_ii s_i) s_i: a few ulps apart
            assert ulps(st["scale"], ref["scale"]) <= 1 and ulps(st["lm_diag"], ref["lm_diag"]) <= 4
            kappa = float(np.linalg.cond(ref["A"]))
            bar = max(1e-12, 10 * u * kappa)
            fwd = np.linalg.norm(st["delta"] - ref["delta"]) / np.linalg.norm(ref["delta"])
            assert fwd <= bar, (jacobi, radius, fwd, kappa)
            assert abs(st["model_change"] - ref["model_change"]) <= bar * abs(ref["model_change"]), (jacobi, radius)
            assert backward_error(ref["A"], ref["b"], st["delta"] / st["scale"]) < 1e-14
            assert st["model_change"] > 0.0
