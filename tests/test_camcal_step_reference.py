"""One iteration of the camera calibration's bundle adjustment against a dense high-precision reference: the case table, the
reference itself, and the checks that need no GPU.

icc_camcal_step (icc_api.cu) runs the launches of one bundle_adjust iteration of icc_calibrate_camera at a given state: the
per-view normal-equation blocks (camcal_accumulate_kernel), the per-view Schur elimination (camcal_reduce_kernel), the reduced
intrinsics system (camcal_solve_kernel), the back-substitution and candidate state (camcal_update_kernel) and the cost at the
candidate.  tests/test_gpu_camcal_step_reference.py compares each stage with `camcal_reference`, `damped_solve_reference` and
`schur_reference` for every case of CASES and every radius of RADII.  Here, without a GPU:
  * icco_project_jacobian (the oracle's Jet<4> passes through its own project<T>) equals central differences of the NumPy camera
    models, and both flag the same points as outside a model's domain;
  * the reference gradient equals central differences of the reference cost along the right increment R_cw exp(eps d), the camera
    centre and the intrinsics, so the reference cannot encode a left / right increment mix-up;
  * the generated cases reach every branch the table claims (CTA edges of the three kernels, partial k-steps of the tile, the
    Huber tail, failed projections, empty views, gapped active lists, a stale scale), so the GPU test cannot pass vacuously.

Tangent of a view: [delta (right increment of R_cw = conj(q_wc)) | camera centre], then the free intrinsics in Theia order."""
import ctypes

import numpy as np
import pytest

from openimucameracalibrator_b200 import camera_models as cm
from openimucameracalibrator_b200 import synthetic as syn
from oracle_api import oracle_lib
from test_camera_calibration import scene
from test_camera_models import CASES as MODEL_CASES
from test_solver_reference import RADII, damped_solve_reference

HUBER = 1.345
COLS = 17
MODEL_K = {m: np.concatenate([k, np.zeros(10 - k.size)]) for m, k in MODEL_CASES}
ALL_MODELS = [m for m, _ in MODEL_CASES]


def intrinsic_subsets(model):
    """theia's GetSubsetFromOptimizeIntrinsicsType per model as bit masks (icc_api.cu: intrinsic_subsets)."""
    bits = lambda *l: sum(1 << i for i in l)  # noqa: E731
    noskew = model in (cm.FOV, cm.DIVISION_UNDISTORTION)
    radial = {cm.PINHOLE: bits(5, 6), cm.PINHOLE_RADIAL_TANGENTIAL: bits(5, 6, 7), cm.FISHEYE: bits(5, 6, 7, 8)}.get(model, bits(4) if noskew else bits(5, 6))
    return dict(focal=1, aspect=2, principal=bits(2, 3) if noskew else bits(3, 4), radial=radial,
                tangential=bits(8, 9) if model == cm.PINHOLE_RADIAL_TANGENTIAL else 0)


def stage_masks(model):
    """(mask, pose_free) of RunCalibration's three stages (icc_calibrate_camera)."""
    s = intrinsic_subsets(model)
    return [(s["focal"] | (s["radial"] if model != cm.PINHOLE else 0), True), (s["principal"], False),
            (s["principal"] | s["focal"] | s["aspect"] | (s["radial"] if model == cm.PINHOLE else 0) | s["tangential"], True)]


# ---- the case table ------------------------------------------------------------------------------------------------------------
# name -> spec.  n_views views of a 16 x 9 board; `active` picks n_active of them (gapped, shuffled) unless "all"; counts: corners
# per view (cycled; None = the whole board in order); repeat: point ids drawn with repetition; outside: extra board points behind
# every camera (outside the model's domain); stale: scale_in given, not the current diagonal's.
CASES = {}
for _m in ALL_MODELS:
    for _st, (_mask, _pf) in enumerate(stage_masks(_m)):
        CASES[f"{cm.MODEL_NAMES[_m]}-stage{_st + 1}"] = dict(model=_m, mask=_mask, pose_free=_pf, n_views=9, n_active=7, counts=(33, 5, 64, 1, 144, 3, 31, 4, 32))
CASES["DIVISION_UNDISTORTION-prestage"] = dict(model=cm.DIVISION_UNDISTORTION, mask=(1 << 0) | (1 << 4), pose_free=True, n_views=8, n_active=8)
CASES["PINHOLE_RADIAL_TANGENTIAL-all10"] = dict(model=cm.PINHOLE_RADIAL_TANGENTIAL, mask=(1 << 10) - 1, pose_free=True, n_views=9, n_active=9)
for _na in (1, 4, 5, 63, 64, 65, 129, 300):
    CASES[f"n_active{_na}"] = dict(model=cm.EXTENDED_UNIFIED, mask=stage_masks(cm.EXTENDED_UNIFIED)[2][0], pose_free=True, n_views=_na + _na // 8 + 1, n_active=_na,
                                   counts=(144, 65, 33, 0, 64, 5))
CASES["corner_counts"] = dict(model=cm.FISHEYE, mask=stage_masks(cm.FISHEYE)[0][0], pose_free=True, n_views=14, n_active=12,
                              counts=(0, 1, 3, 4, 5, 31, 32, 33, 64, 65, 144), repeat=True)
CASES["double_sphere_outside"] = dict(model=cm.DOUBLE_SPHERE, mask=stage_masks(cm.DOUBLE_SPHERE)[2][0], pose_free=True, n_views=10, n_active=8, outside=True)
CASES["stale_scale"] = dict(model=cm.PINHOLE_RADIAL_TANGENTIAL, mask=(1 << 10) - 1, pose_free=True, n_views=80, n_active=70, counts=(144, 33, 7), stale=True)
CASES["stale_scale_stage2"] = dict(model=cm.PINHOLE, mask=stage_masks(cm.PINHOLE)[1][0], pose_free=False, n_views=10, n_active=6, stale=True)
# full size (BASELINE config 4 sizes): checked blockwise, no dense factorisation
FULL = dict(model=cm.EXTENDED_UNIFIED, mask=stage_masks(cm.EXTENDED_UNIFIED)[2][0], pose_free=True, n_views=3000, n_active=3000)
W, H = 960, 540
_CACHE = {}


def make_case(name):
    """-> dict(model, board, off, ids, uv, q_wc, p_wc, k (10), active, mask, pose_free, scale_in or None): a scene of
    test_camera_calibration.scene at a perturbed state (about a fifth of the corners in the Huber tail)."""
    if name in _CACHE:
        return _CACHE[name]
    spec = FULL if name == "full" else CASES[name]
    model, nv, na = spec["model"], spec["n_views"], spec["n_active"]
    seed = sum(map(ord, name))
    rng = np.random.default_rng(seed)
    k_true = MODEL_K[model]
    B, off0, ids0, uv0, q, p = scene(model, k_true[:cm.NUM_PARAMS[model]], n_views=nv, seed=seed, grid=(16, 9))
    C = B.shape[0]
    counts = spec.get("counts")
    ids, uv, off = [], [], [0]
    for v in range(nv):
        if counts is None:
            sel = np.arange(C)
        else:
            n = counts[v % len(counts)]
            sel = rng.choice(C, n, replace=spec.get("repeat", False) and v % 2 == 0) if n else np.zeros(0, dtype=int)
        ids.append(sel); uv.append(uv0[off0[v] + sel]); off.append(off[-1] + sel.size)
    ids, uv = np.concatenate(ids).astype(np.int32), np.concatenate(uv)
    off = np.array(off, dtype=np.int32)
    if spec.get("outside"):
        # board points 1 m above the board: behind every camera (they look down onto z = 0 from 0.22 .. 0.45 m)
        extra = np.array([[0.02 * i, -0.01 * i, 1.0, 1.0] for i in range(3)])
        B = np.concatenate([B, extra])
        ids_l, uv_l, off_l = [], [], [0]
        for v in range(nv):
            e = np.arange(C, C + 3)[: 1 + v % 3]
            ids_l.append(np.concatenate([ids[off[v]:off[v + 1]], e])); uv_l.append(np.concatenate([uv[off[v]:off[v + 1]], rng.uniform(100, 400, (e.size, 2))]))
            off_l.append(off_l[-1] + ids_l[-1].size)
        ids, uv, off = np.concatenate(ids_l).astype(np.int32), np.concatenate(uv_l), np.array(off_l, dtype=np.int32)
    uv = uv + rng.normal(0, 0.3, uv.shape)
    tail = rng.random(uv.shape[0]) < 0.15
    uv[tail] += rng.normal(0, 6.0, (tail.sum(), 2))                                    # gross errors: Huber tail
    # perturbed state: rotations by ~3 mrad, centres by ~2 mm, focal length by 0.5 %, distortion slightly
    R = np.array([syn.quat_xyzw_to_matrix(qq) for qq in q]) @ syn.so3_exp(rng.normal(0, 3e-3, (nv, 3)))
    q_wc = syn.matrix_to_quat_xyzw(R) * (1.0 + rng.uniform(-1e-3, 1e-3, (nv, 1)))       # not quite unit: the library normalises
    p_wc = p + rng.normal(0, 2e-3, p.shape)
    k = k_true.copy()
    k[0] *= 1.005
    k[1] = 1.0 + 0.002
    n = cm.NUM_PARAMS[model]
    k[5:n] *= 1.02
    if model == cm.PINHOLE_RADIAL_TANGENTIAL:
        k[2] = 0.1
    active = np.sort(rng.choice(nv, na, replace=False)) if na < nv else np.arange(nv)
    active = rng.permutation(active).astype(np.int32)
    case = dict(model=model, board=B, off=off, ids=ids, uv=uv, q_wc=q_wc, p_wc=p_wc, k=k, active=active, mask=spec["mask"], pose_free=spec["pose_free"],
                scale_in=None)
    if spec.get("stale"):
        ref = camcal_reference(case)
        H, g, _ = assemble(ref["M"], None, case["mask"], case["pose_free"])
        s = np.zeros(6 * na + 10)
        s_cur = 1.0 / (1.0 + np.sqrt(np.diag(H)))
        free = free_intrinsics(case["mask"])
        if case["pose_free"]:
            s[: 6 * na] = s_cur[: 6 * na]
        s[6 * na + free] = s_cur[-free.size:]
        s = s * rng.uniform(0.5, 2.0, s.shape)
        s[: 6 * na].reshape(na, 6)[::3] *= 1e-4     # clamped at min_diag: the damping of these views depends on their scale
        case["scale_in"] = s
    _CACHE[name] = case
    return case


def radii_for(case):
    """RADII, without 1e16 when an active view has 1 or 2 corners: its pose block then has rank <= 4 and a damping of 1e-22 leaves
    the system singular to working precision (a calibration never keeps such a view)."""
    cnt = np.diff(case["off"])[case["active"]]
    return RADII if not ((cnt > 0) & (cnt < 3)).any() else tuple(r for r in RADII if r < 1e10)


# ---- the reference ------------------------------------------------------------------------------------------------------------
def project_jacobian(model, k, pts):
    """icco_project_jacobian: pixel (n, 2), point Jacobian (n, 2, 3), intrinsic Jacobian (n, 2, 10), ok (n,)."""
    lib = oracle_lib()
    dp = ctypes.POINTER(ctypes.c_double)
    pts = np.ascontiguousarray(pts, dtype=np.float64).reshape(-1, 3)
    k = np.ascontiguousarray(k, dtype=np.float64)
    n = pts.shape[0]
    px, Jp, Jk, ok = np.zeros((n, 2)), np.zeros((n, 2, 3)), np.zeros((n, 2, 10)), np.zeros(n, dtype=np.int32)
    lib.icco_project_jacobian(ctypes.c_int(model), k.ctypes.data_as(dp), ctypes.c_int(n), pts.ctypes.data_as(dp), px.ctypes.data_as(dp),
                              Jp.ctypes.data_as(dp), Jk.ctypes.data_as(dp), ok.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)))
    return px, Jp, Jk, ok.astype(bool)


def hat(v):
    z = np.zeros(v.shape[:-1])
    return np.stack([np.stack([z, -v[..., 2], v[..., 1]], -1), np.stack([v[..., 2], z, -v[..., 0]], -1), np.stack([-v[..., 1], v[..., 0], z], -1)], -2)


def free_intrinsics(mask):
    return np.array([a for a in range(10) if (mask >> a) & 1], dtype=int)


def rotations_cw(q_wc):
    q = np.asarray(q_wc, dtype=np.float64)
    q = q / np.linalg.norm(q, axis=-1, keepdims=True)
    return np.array([syn.quat_xyzw_to_matrix(qq).T for qq in q])


def camcal_reference(case, q_wc=None, p_wc=None, k=None, jacobian=True):
    """Residuals and Jacobians of the active views from icco_project_jacobian, the chain rule to the right-increment tangent in NumPy
    (d pc / d delta = -R [d]x, d pc / d c = -R with pc = R (X - c), R = R_cw), Huber weights sqrt(rho'), 1e10 for a failed corner
    (zero rows).  -> dict(M (n_active, 17, 17) long double: per slot [J | r]^T [J | r] of the weighted rows (columns pose 6 |
    intrinsics 10 | residual), mag: (|J|^T |J|) of the same rows, cost, n_fail, n_tail, view_err (n_views), x_sq as the GPU states
    it: sum k^2 + sum over active views (1 + |c|^2))."""
    q_wc = case["q_wc"] if q_wc is None else q_wc
    p_wc = case["p_wc"] if p_wc is None else p_wc
    k = case["k"] if k is None else k
    model, off, ids, uv, active = case["model"], case["off"], case["ids"], case["uv"], case["active"]
    B = case["board"]
    X = B[:, :3] / B[:, 3:]
    Rcw = rotations_cw(q_wc)
    corner = np.concatenate([np.arange(off[v], off[v + 1]) for v in active]).astype(int) if len(active) else np.zeros(0, int)
    slot = np.concatenate([np.full(off[v + 1] - off[v], s) for s, v in enumerate(active)]).astype(int)
    view = active[slot]
    d = X[ids[corner]] - p_wc[view]
    R = Rcw[view]
    pc = np.einsum("nij,nj->ni", R, d)
    px, Jp, Jk, ok = project_jacobian(model, k, pc)
    r = px - uv[corner]
    rn = np.sqrt((r * r).sum(-1))
    inside = rn <= HUBER
    per = np.where(ok, np.where(inside, 0.5 * rn * rn, HUBER * rn - 0.5 * HUBER * HUBER), 1e10)
    err = np.where(ok, rn, 1e10)
    na, nv = len(active), off.size - 1
    view_err = np.zeros(nv)
    for s, v in enumerate(active):
        m = slot == s
        view_err[v] = err[m].sum() / m.sum() if m.any() else 0.0
    out = dict(cost=float(per.sum()), n_fail=int((~ok).sum()), n_tail=int((ok & ~inside).sum()), view_err=view_err,
               x_sq=float((k * k).sum() + sum(1.0 + p_wc[v] @ p_wc[v] for v in active)), slot=slot, ok=ok)
    if not jacobian:
        return out
    sw = np.where(inside, 1.0, np.sqrt(HUBER / np.where(inside, 1.0, rn)))
    rows = np.zeros((corner.size, 2, COLS))
    if case["pose_free"]:
        rows[:, :, 0:3] = np.einsum("nrj,njk->nrk", Jp, -R @ hat(d))
        rows[:, :, 3:6] = np.einsum("nrj,njk->nrk", Jp, -R)
    free = free_intrinsics(case["mask"])
    rows[:, :, 6 + free] = Jk[:, :, free]
    rows[:, :, 16] = r
    rows *= (sw * ok)[:, None, None]
    M = np.zeros((na, COLS, COLS), dtype=np.longdouble)
    mag = np.zeros((na, COLS, COLS))
    bounds = np.searchsorted(slot, np.arange(na + 1))
    for s in range(na):
        J = rows[bounds[s]:bounds[s + 1]].reshape(-1, COLS)
        Jl = J.astype(np.longdouble)
        M[s] = Jl.T @ Jl
        mag[s] = np.abs(J).T @ np.abs(J)
    out.update(M=M, mag=mag)
    return out


def assemble(M, M_sys, mask, pose_free):
    """Dense H, g (float64) over the free columns [6 per slot if pose_free | free intrinsics] from per-slot 17 x 17 blocks M; the
    intrinsics part from M_sys (17 x 17, rows / columns >= 6 used) when given, else summed over the slots.  -> (H, g, columns)."""
    M = np.asarray(M, dtype=np.longdouble)
    na = M.shape[0]
    free = free_intrinsics(mask)
    npose = 6 * na if pose_free else 0
    n = npose + free.size
    H = np.zeros((n, n), dtype=np.longdouble); g = np.zeros(n, dtype=np.longdouble)
    kc = npose + np.arange(free.size)
    if pose_free:
        for s in range(na):
            sl = slice(6 * s, 6 * s + 6)
            H[sl, sl] = M[s, :6, :6]
            H[sl, kc] = M[s][:6, 6 + free]; H[kc, sl] = M[s][6 + free, :6]
            g[sl] = M[s, :6, 16]
    S = M.sum(0) if M_sys is None else np.asarray(M_sys, dtype=np.longdouble)
    H[np.ix_(kc, kc)] = S[np.ix_(6 + free, 6 + free)]
    g[kc] = S[6 + free, 16]
    return H.astype(np.float64), g.astype(np.float64), kc


def schur_reference(App, Hpk, gp, Dp):
    """Per slot Y = (A_pp + diag(Dp))^-1 [H_pk | g_p] (6 x 11) and the reduced system -sum H_pk^T Y (10 x 11: matrix | gradient)."""
    Y = np.linalg.solve(App.astype(np.longdouble).astype(np.float64) + Dp[:, :, None] * np.eye(6), np.concatenate([Hpk, gp[..., None]], -1))
    return Y, -np.einsum("sia,sib->ab", Hpk.astype(np.longdouble), Y.astype(np.longdouble)).astype(np.float64)


def lm_damping(hii, s, radius, min_diag=1e-6, max_diag=1e32):
    """The unscaled LM diagonal of a column with Jacobi scale s (icc_camcal.cu: lm_damping)."""
    return np.minimum(np.maximum(s * s * hii, min_diag), max_diag) / (radius * s * s)


def quat_mul(a, b):
    ax, ay, az, aw = np.moveaxis(a, -1, 0); bx, by, bz, bw = np.moveaxis(b, -1, 0)
    return np.stack([aw * bx + ax * bw + ay * bz - az * by, aw * by + ay * bw + az * bx - ax * bz, aw * bz + az * bw + ax * by - ay * bx,
                     aw * bw - ax * bx - ay * by - az * bz], -1)


def quat_exp(w):
    th = np.linalg.norm(w, axis=-1, keepdims=True)
    s = np.where(th < 1e-8, 0.5 - th * th / 48.0, np.sin(0.5 * th) / np.where(th < 1e-8, 1.0, th))
    return np.concatenate([s * w, np.cos(0.5 * th)], -1)


def plus(case, q_wc, p_wc, k, dpose, dk):
    """Plus(cur, delta) of the right-increment tangent: R_cw <- R_cw exp(delta), c <- c + dc, k <- k + dk; -> q_wc, p_wc, k."""
    q = np.asarray(q_wc, dtype=np.float64)
    q = q / np.linalg.norm(q, axis=-1, keepdims=True)
    q_cw = q * np.array([-1.0, -1.0, -1.0, 1.0])
    qn, pn = q.copy(), np.array(p_wc, dtype=np.float64)
    a = case["active"]
    qc = quat_mul(q_cw[a], quat_exp(dpose[:, :3]))
    qc /= np.linalg.norm(qc, axis=-1, keepdims=True)
    qn[a] = qc * np.array([-1.0, -1.0, -1.0, 1.0])
    pn[a] = pn[a] + dpose[:, 3:]
    return qn, pn, k + dk


# ---- CPU checks --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model,k", MODEL_CASES, ids=[cm.MODEL_NAMES[m] for m, _ in MODEL_CASES])
def test_project_jacobian_matches_numpy_central_differences(model, k):
    rng = np.random.default_rng(100 + model)
    pts = np.concatenate([rng.uniform(-0.3, 0.3, (150, 2)), rng.uniform(0.3, 1.0, (150, 1))], axis=1)
    if model in (cm.DOUBLE_SPHERE, cm.EXTENDED_UNIFIED):
        pts = np.concatenate([pts, [[0.1, 0.0, -5.0], [0.0, 0.2, -3.0]]])          # outside the unified models' domain
    k10 = np.concatenate([k, np.zeros(10 - k.size)])
    n = cm.NUM_PARAMS[model]
    px, Jp, Jk, ok = project_jacobian(model, k10, pts)
    uv, valid = cm.project(model, k, pts)
    assert (ok == valid).all()
    if model in (cm.DOUBLE_SPHERE, cm.EXTENDED_UNIFIED):
        assert not ok[-2:].any() and ok[:-2].all()
    assert np.allclose(px[ok], uv[ok], rtol=1e-13, atol=1e-10)
    for j in range(3):
        e = np.zeros(3); e[j] = 1e-6
        fd = (cm.project(model, k, pts + e)[0] - cm.project(model, k, pts - e)[0]) / 2e-6
        assert np.allclose(Jp[ok, :, j], fd[ok], rtol=1e-6, atol=1e-6 * np.abs(fd[ok]).max()), j
    for j in range(10):
        if j >= n:
            assert (Jk[:, :, j] == 0.0).all()
            continue
        h = 1e-6 * abs(k[j]) if k[j] != 0.0 else 1e-7
        kp, km = k.copy(), k.copy(); kp[j] += h; km[j] -= h
        fd = (cm.project(model, kp, pts)[0] - cm.project(model, km, pts)[0]) / (2 * h)
        assert np.allclose(Jk[ok, :, j], fd[ok], rtol=1e-6, atol=1e-6 * max(np.abs(fd[ok]).max(), 1.0)), j


@pytest.mark.parametrize("name", ["PINHOLE_RADIAL_TANGENTIAL-all10", "FOV-stage3", "DOUBLE_SPHERE-stage1"])
def test_reference_gradient_matches_central_differences(name):
    """g = sum rho' J^T r equals d cost / d x along R_cw exp(eps d), c + eps d and k + eps d (second view of the active list)."""
    case = make_case(name)
    ref = camcal_reference(case)
    H, g, kc = assemble(ref["M"], None, case["mask"], case["pose_free"])
    s = 1
    v = case["active"][s]
    cost = lambda q, p, k: camcal_reference(case, q, p, k, jacobian=False)["cost"]  # noqa: E731
    Rcw = rotations_cw(case["q_wc"])
    for j in range(6):
        e = np.zeros(3); e[j % 3] = 1.0
        vals = []
        for sgn in (1.0, -1.0):
            q, p = case["q_wc"].copy(), case["p_wc"].copy()
            if j < 3:
                q[v] = syn.matrix_to_quat_xyzw((Rcw[v] @ syn.so3_exp(sgn * 1e-6 * e)).T[None])[0]
            else:
                p[v] = p[v] + sgn * 1e-6 * e
            vals.append(cost(q, p, case["k"]))
        fd = (vals[0] - vals[1]) / 2e-6
        assert abs(fd - g[6 * s + j]) <= 1e-5 * max(abs(g[6 * s + j]), 1.0), (j, fd, g[6 * s + j])
    for i, a in enumerate(free_intrinsics(case["mask"])):
        h = 1e-6 * abs(case["k"][a]) if case["k"][a] != 0.0 else 1e-7
        kp, km = case["k"].copy(), case["k"].copy(); kp[a] += h; km[a] -= h
        fd = (cost(case["q_wc"], case["p_wc"], kp) - cost(case["q_wc"], case["p_wc"], km)) / (2 * h)
        assert abs(fd - g[kc[i]]) <= 1e-5 * abs(g[kc[i]]) + 1e-6 * abs(cost(case["q_wc"], case["p_wc"], case["k"])) / max(h, 1e-300) * 1e-9, (a, fd, g[kc[i]])


def _partial_k_steps(counts):
    return [c for c in counts if c % 32 and (c % 32) % 4]


def test_case_table_covers_every_branch():
    """Asserted on the generated data: each claimed kernel edge and each branch of the per-corner code is reached."""
    seen_models_stages, n_active, counts, hits = set(), set(), set(), dict.fromkeys(
        ["repeated ids", "shuffled ids", "gapped unsorted active", "failed projections", "Huber tail", "empty active view", "stale scale",
         "stale scale with gapped active", "prestage mask", "all 10 intrinsics", "partial k-step", "poses constant"], False)
    for name, spec in CASES.items():
        case = make_case(name)
        model, mask, pf, act, off, ids = case["model"], case["mask"], case["pose_free"], case["active"], case["off"], case["ids"]
        for st, (m, p) in enumerate(stage_masks(model)):
            if (m, p) == (mask, pf):
                seen_models_stages.add((model, st))
        n_active.add(act.size)
        cnt = np.diff(off)[act]
        counts.update(cnt.tolist())
        ref = camcal_reference(case, jacobian=False)
        for v in act:
            vi = ids[off[v]:off[v + 1]]
            hits["repeated ids"] |= np.unique(vi).size < vi.size
            hits["shuffled ids"] |= vi.size > 1 and (np.diff(vi) < 0).any()
        hits["gapped unsorted active"] |= (np.diff(act) < 0).any() and act.max() + 1 > act.size
        hits["failed projections"] |= ref["n_fail"] > 0
        hits["Huber tail"] |= ref["n_tail"] > 0
        hits["empty active view"] |= (cnt == 0).any()
        if case["scale_in"] is not None:
            full = camcal_reference(case)
            H, _, kc = assemble(full["M"], None, mask, pf)
            s_cur = 1.0 / (1.0 + np.sqrt(np.diag(H)))
            used = np.concatenate([np.arange(6 * act.size) if pf else np.zeros(0, int), 6 * act.size + free_intrinsics(mask)])
            assert not np.allclose(case["scale_in"][used], s_cur)
            hits["stale scale"] = True
            hits["stale scale with gapped active"] |= pf and act.max() + 1 > act.size and (np.diff(act) < 0).any()
        hits["prestage mask"] |= model == cm.DIVISION_UNDISTORTION and mask == 0b10001 and pf
        hits["all 10 intrinsics"] |= mask == (1 << 10) - 1
        hits["partial k-step"] |= bool(_partial_k_steps(cnt))
        hits["poses constant"] |= not pf
        assert ref["n_tail"] > 0 or cnt.sum() < 10, name
    assert seen_models_stages == {(m, s) for m in ALL_MODELS for s in range(3)}
    assert {1, 4, 5, 63, 64, 65, 129, 300} <= n_active                        # accumulate (4), reduce (64) and update (128) CTA edges
    assert {0, 1, 3, 4, 5, 31, 32, 33, 64, 65, 144} <= counts
    missing = [k for k, v in hits.items() if not v]
    assert not missing, f"no case of the table reaches: {missing}"
    assert len(RADII) == 3 and min(RADII) == 1e-3 and max(RADII) == 1e16
    huge = [name for name in CASES if 1e16 in radii_for(make_case(name))]
    assert {f"n_active{n}" for n in (1, 4, 5, 63, 64, 65, 129, 300)} | {"double_sphere_outside", "stale_scale"} <= set(huge), huge


@pytest.mark.parametrize("name", ["FISHEYE-stage1", "stale_scale_stage2"])
def test_schur_reference_equals_the_dense_solve(name):
    """Eliminating the poses with schur_reference and back-substituting gives the dense damped step of damped_solve_reference."""
    case = make_case(name)
    ref = camcal_reference(case)
    H, g, kc = assemble(ref["M"], None, case["mask"], case["pose_free"])
    na = case["active"].size
    free = free_intrinsics(case["mask"])
    for radius in radii_for(case):
        d = damped_solve_reference(H, g, radius)
        s = d["scale"]
        Dfull = d["lm_diag"] / (s * s)                                          # unscaled damping
        M = np.asarray(ref["M"], dtype=np.float64)
        if case["pose_free"]:
            Y, red = schur_reference(M[:, :6, :6], M[:, :6, 6:16], M[:, :6, 16], Dfull[: 6 * na].reshape(na, 6))
        else:
            Y, red = np.zeros((na, 6, 11)), np.zeros((10, 11))
        A = H[np.ix_(kc, kc)] + np.diag(Dfull[kc]) + red[np.ix_(free, free)]
        dk = np.linalg.solve(A, -(g[kc] + red[free, 10]))
        dkk = np.zeros(10); dkk[free] = dk
        dp = -(Y[:, :, 10] + Y[:, :, :10] @ dkk)
        delta = np.concatenate([dp.ravel() if case["pose_free"] else np.zeros(0), dk])
        assert np.linalg.norm(delta - d["delta"]) <= 1e-8 * np.linalg.norm(d["delta"]), radius
