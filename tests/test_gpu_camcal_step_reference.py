"""One bundle-adjustment iteration of the camera calibration on the GPU, stage by stage, against the dense high-precision reference.

For every case of test_camcal_step_reference.CASES and every radius of radii_for(case), icc_camcal_step runs the launches of one
iteration of icc_calibrate_camera's bundle_adjust and returns what each kernel produced.  Three checks, each isolating one stage:
  * evaluation (camcal_accumulate_kernel): the per-slot 17 x 17 blocks and the summed intrinsics system against camcal_reference,
    built from the oracle's Jet Jacobians, entrywise |dM_ab| <= C_H u (|J|^T |J|)_ab; the cost to relative COST_BAR;
  * solve (camcal_reduce_kernel, camcal_solve_kernel), on the GPU's own H and g assembled from the returned blocks: the scale to
    1 ulp (or equal to scale_in), the normwise backward error of y = delta / S <= ETA_BAR, delta and the model change to
    max(1e-12, FWD_C u kappa_2(A)) against damped_solve_reference, Y per slot against schur_reference and the reduced system
    against -sum H_pk^T Y of the GPU's own Y (entrywise, RED_C u sum |H_pk|^T |Y|);
  * update and cost (camcal_update_kernel, cost-only accumulate): the candidate state equals Plus(cur, delta) in NumPy, the
    scalars g.delta, delta^T D delta, |delta|^2 and x^2 match to relative 1e-13, and the candidate cost and the per-view errors
    match a NumPy evaluation through camera_models.project (a third statement of the models) at the GPU's states.
Full size (3000 views x 144 corners, EUCM; 47 reduce CTAs, 24 update CTAs): the blocks entrywise, Y and the reduced system as
above, and the componentwise relative residual of the arrow system (A_pp + D) delta_p + H_pk delta_k = -g_p,
sum H_pk^T delta_p + (H_kk + D_k) delta_k = -g_k, formed in long double, at the three radii.

Bars, measured on an NVIDIA B200 (1000 W power limit, read in the same run and printed), one decade of margin:
  C_H = 6e4            max |dM| / (u (|J|^T |J|)) <= 6.0e3 (PINHOLE_RADIAL_TANGENTIAL stage 2: closed-form vs autodiff Jacobians)
  COST_BAR = 1e-13     relative cost difference <= 1.1e-14
  ETA_BAR = 5e-15      backward error of y = delta / S <= 2.9e-16
  FWD_C = 3            forward error / (u kappa_2) <= 1.7 (the 1e-12 floor decides there)
  RED_C = 32           reduced system vs -sum H_pk^T Y <= 3.0 u sum |H_pk|^T |Y|
  FULL_ETA_BAR = 5e-15 full-size arrow residual <= 4.2e-16
Each of these value-only mutations of icc_camcal.cu fails this test: the CTA sum of camcal_reduce_kernel over RED_THREADS - 1
threads (n_active >= 64 and full size), nsteps = nact >> 2 (every case with a partial k-step), the tail residual column left
unweighted, the view's Jacobi scale read by view instead of slot (the stale scale with a gapped list), the last intrinsic dropped
from the back-substitution (10-parameter masks), and one Schur entry scaled by 1 + 1e-9.
"""
import subprocess

import numpy as np
import pytest

from openimucameracalibrator_b200 import _capi as capi
from openimucameracalibrator_b200 import camera_models as cm
from openimucameracalibrator_b200 import synthetic as syn
from test_camcal_step_reference import (CASES, HUBER, assemble, camcal_reference, free_intrinsics, lm_damping, make_case, plus, radii_for,
                                        schur_reference)
from test_solver_reference import RADII, backward_error, damped_solve_reference, ulps

pytestmark = pytest.mark.gpu
U = np.finfo(np.float64).eps
C_H = 6e4
COST_BAR = 1e-13
ETA_BAR = 5e-15
FWD_C = 3.0
RED_C = 32.0
FULL_ETA_BAR = 5e-15
IU = np.triu_indices(17)
_MEASURED = {}


def _card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # noqa: BLE001
        return f"unknown ({e})"


@pytest.fixture(scope="module")
def card():
    name = _card()
    print(f"\n[camcal-step] device: {name}")
    yield name
    print(f"\n[camcal-step] device: {name}; largest measured: " + ", ".join(f"{k}={v:.3g}" for k, v in sorted(_MEASURED.items())))


def _note(key, value):
    _MEASURED[key] = max(_MEASURED.get(key, 0.0), float(value))


def unpack(packed):
    """Packed upper triangles (..., 153) -> symmetric (..., 17, 17)."""
    packed = np.asarray(packed)
    M = np.zeros(packed.shape[:-1] + (17, 17))
    M[..., IU[0], IU[1]] = packed
    M[..., IU[1], IU[0]] = packed
    return M


def run_step(cuda_lib, case, radius):
    api = capi.CApi(cuda_lib, "icc_", 0)
    try:
        api.set_board_points(case["board"])
        return api.camcal_step(case["model"], case["off"], case["ids"], case["uv"], case["q_wc"], case["p_wc"], case["k"], case["active"],
                               case["mask"], case["pose_free"], radius, huber_width=HUBER, scale_in=case["scale_in"])
    finally:
        api.close()


def check_blocks(tag, Mg, ref, bar_c):
    """Entrywise |M_gpu - M_ref| <= bar_c u mag; entries whose magnitude is 0 must be exactly 0."""
    dM = np.abs(Mg - np.asarray(ref["M"], dtype=np.float64))
    mag = ref["mag"]
    assert (dM[mag == 0] == 0).all(), tag
    ratio = float((dM[mag > 0] / (U * mag[mag > 0])).max()) if (mag > 0).any() else 0.0
    _note("C_H", ratio)
    assert ratio <= bar_c, (tag, ratio)
    return ratio


def pose_step(Y, dk):
    """Back-substitution of the pose steps: dp = -(Y[:, :, 10] + Y[:, :, :10] dk) per slot."""
    return -(Y[:, :, 10] + Y[:, :, :10] @ dk)


def numpy_costs(case, q_wc, p_wc, k):
    """Cost and per-view mean errors at a state through camera_models.project (1e10 per failed corner)."""
    model, off, ids, uv, B = case["model"], case["off"], case["ids"], case["uv"], case["board"]
    X = B[:, :3] / B[:, 3:]
    q = q_wc / np.linalg.norm(q_wc, axis=-1, keepdims=True)
    cost, errs = 0.0, np.zeros(off.size - 1)
    for v in case["active"]:
        if off[v + 1] == off[v]:
            continue
        R_cw = syn.quat_xyzw_to_matrix(q[v]).T
        pc = (X[ids[off[v]:off[v + 1]]] - p_wc[v]) @ R_cw.T
        px, ok = cm.project(model, k[: cm.NUM_PARAMS[model]], pc)
        rn = np.linalg.norm(px - uv[off[v]:off[v + 1]], axis=-1)
        cost += np.where(ok, np.where(rn <= HUBER, 0.5 * rn * rn, HUBER * rn - 0.5 * HUBER * HUBER), 1e10).sum()
        errs[v] = np.where(ok, rn, 1e10).mean()
    return cost, errs


def check_schur(tag, Mg, scale_pose, radius, Y, red, free):
    """Y against schur_reference of the GPU's blocks; red against -sum H_pk^T Y of the GPU's own Y."""
    App, Hpk, gp = Mg[:, :6, :6], Mg[:, :6, 6:16], Mg[:, :6, 16]
    Dp = lm_damping(np.diagonal(App, axis1=1, axis2=2), scale_pose, radius)
    Yr, _ = schur_reference(App, Hpk, gp, Dp)
    A = App + Dp[:, :, None] * np.eye(6)
    Bm = np.concatenate([Hpk, gp[..., None]], -1)
    nA, nAi = np.linalg.norm(A, 2, axis=(1, 2)), np.linalg.norm(np.linalg.inv(A), 2, axis=(1, 2))
    bound = 6 * 10 * U * nAi * (nA * np.linalg.norm(Y, 2, axis=(1, 2)) + np.linalg.norm(Bm, 2, axis=(1, 2)))
    err = np.linalg.norm(Y - Yr, 2, axis=(1, 2))
    _note("Y/bound", float((err / np.maximum(bound, 1e-300)).max()))
    assert (err <= bound).all(), (tag, float((err / bound).max()))
    R = -np.einsum("sia,sib->ab", Hpk.astype(np.longdouble), Y.astype(np.longdouble))
    mag = np.einsum("sia,sib->ab", np.abs(Hpk), np.abs(Y))
    red_full = np.zeros((10, 11))
    red_full[IU10[0], IU10[1]] = red[:55]
    red_full[:, 10] = red[55:65]
    upper = np.zeros((10, 11), dtype=bool); upper[IU10[0], IU10[1]] = True; upper[:, 10] = True
    d = np.abs(red_full - R.astype(np.float64))[upper]
    m = mag[upper]
    assert (d[m == 0] == 0).all(), tag
    ratio = float((d[m > 0] / (U * m[m > 0])).max()) if (m > 0).any() else 0.0
    _note("RED_C", ratio)
    assert ratio <= RED_C, (tag, ratio)


IU10 = np.triu_indices(10)


@pytest.mark.parametrize("name", list(CASES))
def test_camcal_step_matches_reference(cuda_lib, card, name):
    case = make_case(name)
    ref = camcal_reference(case)
    mask, pf, act = case["mask"], case["pose_free"], case["active"]
    na, free = act.size, free_intrinsics(mask)
    for radius in radii_for(case):
        tag = (name, radius)
        st = run_step(cuda_lib, case, radius)
        # ---- evaluation --------------------------------------------------------------------------------------------------
        Mg = unpack(st["blocks"])
        ch = check_blocks(tag, Mg, ref, C_H)
        Sg = unpack(st["sys"][:153])
        S_ref = dict(M=np.asarray(ref["M"], dtype=np.longdouble).sum(0)[None], mag=ref["mag"].sum(0)[None])
        S_ref["M"][:, :6, :] = 0; S_ref["M"][:, :, :6] = 0; S_ref["mag"][:, :6, :] = 0; S_ref["mag"][:, :, :6] = 0
        check_blocks(tag + ("sys",), Sg[None], S_ref, C_H)
        dcost = abs(st["sys"][153] - ref["cost"]) / ref["cost"]
        _note("COST", dcost)
        assert dcost <= COST_BAR, (tag, dcost)
        # ---- solve on the GPU's own H and g --------------------------------------------------------------------------------
        H, g, kc = assemble(Mg, Sg, mask, pf)
        used = np.concatenate([np.arange(6 * na) if pf else np.zeros(0, int), 6 * na + free])
        s_in = None if case["scale_in"] is None else case["scale_in"][used]
        d = damped_solve_reference(H, g, radius, scale=s_in)
        s_gpu = st["scale"][used]
        if s_in is None:
            assert ulps(s_gpu, d["scale"]) <= 1, tag
        else:
            assert (s_gpu == s_in).all(), tag
        dk = st["dk"]
        assert (dk[np.setdiff1d(np.arange(10), free)] == 0).all() and st["scalars"]["fail"] == 0.0, tag
        Y = st["Y"]
        dp = pose_step(Y, dk) if pf else np.zeros((na, 6))
        delta = np.concatenate([dp.ravel() if pf else np.zeros(0), dk[free]])
        eta = backward_error(d["A"], d["b"], delta / d["scale"])
        ev = np.linalg.eigvalsh(d["A"])
        kappa = float(ev[-1] / ev[0]) if ev[0] > 0 else np.inf
        fwd = float(np.linalg.norm(delta - d["delta"]) / np.linalg.norm(d["delta"]))
        mc_gpu = 0.5 * (st["scalars"]["d_delta"] - st["scalars"]["g_delta"])
        mc = abs(mc_gpu - d["model_change"]) / abs(d["model_change"])
        _note("ETA", eta); _note("FWD/(u kappa)", max(fwd, mc) / (U * kappa))
        print(f"[camcal-step] {name} radius={radius:.0e} n_active={na} C_H={ch:.2f} eta={eta:.2e} fwd={fwd:.2e} mc={mc:.2e} kappa={kappa:.2e}")
        assert eta <= ETA_BAR, (tag, eta)
        bar = max(1e-12, FWD_C * U * kappa)
        assert fwd <= bar and mc <= bar, (tag, fwd, mc, kappa)
        if pf:
            check_schur(tag, Mg, st["scale"][: 6 * na].reshape(na, 6), radius, Y, st["red"], free)
            assert st["scalars"]["grad_max"] == np.abs(g).max(), tag
        else:
            assert (st["red"] == 0).all() and (Y == 0).all(), tag
        # ---- update and cost-only kernels -----------------------------------------------------------------------------------
        qn, pn, kn = plus(case, case["q_wc"], case["p_wc"], case["k"], dp, dk)
        qg, pg = st["q_wc_cand"], st["p_wc_cand"]
        qd = np.minimum(np.abs(qg - qn).max(-1), np.abs(qg + qn).max(-1))
        bt = 16 * U * (np.abs(Y[:, :, 10]) + np.abs(Y[:, :, :10]) @ np.abs(dk))          # rounding of the back-substitution itself
        assert (qd[act] <= 8 * U + 2 * bt[:, :3].max(-1)).all(), (tag, float(qd.max()))
        cbar = 4 * U * np.maximum(np.abs(case["p_wc"][act]), np.abs(dp[:, 3:])) + bt[:, 3:]
        assert (np.abs(pg[act] - pn[act]) <= cbar).all(), tag
        others = np.setdiff1d(np.arange(case["off"].size - 1), act)
        assert (pg[others] == case["p_wc"][others]).all() and (st["intr_cand"] == case["k"] + dk).all(), tag
        gd_terms = g * delta
        sc = st["scalars"]
        Dfull = d["lm_diag"] / (d["scale"] ** 2)
        for key, val, scale in (("g_delta", gd_terms.sum(), np.abs(gd_terms).sum()), ("d_delta", (Dfull * delta * delta).sum(), (Dfull * delta * delta).sum()),
                                ("step_sq", (delta * delta).sum(), (delta * delta).sum()), ("x_sq", ref["x_sq"], ref["x_sq"])):
            assert abs(sc[key] - val) <= 1e-13 * scale, (tag, key, sc[key], val)
        cand_cost, _ = numpy_costs(case, qg, pg, st["intr_cand"])
        _, errs = numpy_costs(case, case["q_wc"], case["p_wc"], case["k"])
        n_c = int(np.diff(case["off"])[act].sum())
        assert abs(sc["cand_cost"] - cand_cost) <= 1e-12 * cand_cost + 1e-9 * n_c, (tag, sc["cand_cost"], cand_cost)
        assert np.allclose(st["view_error_px"], errs, rtol=1e-11, atol=1e-9), tag
        assert (st["view_error_px"][others] == 0).all()


def test_full_size_step(cuda_lib, card):
    """3000 views x 144 corners: blocks entrywise, Y and the reduced system, and the residual of the arrow system at three radii."""
    case = make_case("full")
    ref = camcal_reference(case)
    mask, act = case["mask"], case["active"]
    na, free = act.size, free_intrinsics(mask)
    for radius in RADII:
        st = run_step(cuda_lib, case, radius)
        Mg = unpack(st["blocks"])
        check_blocks(("full", radius), Mg, ref, C_H)
        Sg = unpack(st["sys"][:153])
        assert abs(st["sys"][153] - ref["cost"]) <= COST_BAR * ref["cost"]
        s_pose = st["scale"][: 6 * na].reshape(na, 6)
        assert ulps(s_pose, 1.0 / (1.0 + np.sqrt(np.diagonal(Mg[:, :6, :6], axis1=1, axis2=2)))) <= 1
        check_schur(("full", radius), Mg, s_pose, radius, st["Y"], st["red"], free)
        dk = st["dk"]
        dp = pose_step(st["Y"], dk)
        sk = st["scale"][6 * na + free]
        L = np.longdouble
        App, Hpk, gp = Mg[:, :6, :6].astype(L), Mg[:, :6, 6 + free].astype(L), Mg[:, :6, 16].astype(L)
        Dp = lm_damping(np.diagonal(Mg[:, :6, :6], axis1=1, axis2=2), s_pose, radius).astype(L)
        Hkk = Sg[np.ix_(6 + free, 6 + free)].astype(L)
        Dk = lm_damping(np.diag(Sg)[6 + free], sk, radius).astype(L)
        gk = Sg[6 + free, 16].astype(L)
        dpl, dkl = dp.astype(L), dk[free].astype(L)
        rp = np.einsum("sij,sj->si", App, dpl) + Dp * dpl + Hpk @ dkl + gp
        dp_den = np.einsum("sij,sj->si", np.abs(App), np.abs(dpl)) + Dp * np.abs(dpl) + np.abs(Hpk) @ np.abs(dkl) + np.abs(gp)
        rk = np.einsum("sia,si->a", Hpk, dpl) + Hkk @ dkl + Dk * dkl + gk
        dk_den = np.einsum("sia,si->a", np.abs(Hpk), np.abs(dpl)) + np.abs(Hkk) @ np.abs(dkl) + Dk * np.abs(dkl) + np.abs(gk)
        eta = float(max((np.abs(rp) / dp_den).max(), (np.abs(rk) / dk_den).max()))
        _note("FULL_ETA", eta)
        print(f"[camcal-step] full radius={radius:.0e} arrow residual={eta:.2e}")
        assert eta <= FULL_ETA_BAR, (radius, eta)
        assert st["scalars"]["fail"] == 0.0 and 0.5 * (st["scalars"]["d_delta"] - st["scalars"]["g_delta"]) > 0.0
