"""One damped normal-equation solve on the GPU against the same system solved densely on the host in high precision.

For every (case, chunks) of test_solver_reference.CASES and every radius in RADII, icc_solve_step returns the cost, g and H of one
evaluation together with the scale S, the LM diagonal D, the step delta and the model cost change of the solve that consumed that
evaluation.  The reference (test_solver_reference.damped_solve_reference) rebuilds A = S H S + D, b = -S g from the returned H and g:
  * S and D equal the formula evaluated on H to 1 ulp (sqrt and division are correctly rounded);
  * the normwise backward error eta = |A y - b|_inf / (|A|_inf |y|_inf + |b|_inf) of y = delta / S is the main bar: it does not
    depend on the conditioning, and a structural error of the elimination (a wrong remainder column, a wrong border entry) lifts
    it from ~1e-16 to 1e-4 or more;
  * delta and the model cost change agree with the reference to max(1e-12, FWD_C u kappa_2(A)); where A is singular to working
    precision (eigvalsh finds a non-positive eigenvalue: some radius-1e16 systems) only the backward error can be held.
Full-size config 4 has no dense H: the residual A y - b is formed from icc_normal_matvec applied to delta (a second evaluation,
so this bar also absorbs the run-to-run scatter of the atomic sums).

Bars, measured on an NVIDIA B200 (1000 W power limit), one decade of margin over the P = 1 plans:
  ETA_BAR = 5e-15        eta of the P = 1 plans <= 4.8e-16 (all plans <= 6.8e-16, the P = 16 plan with 294 border columns)
  FWD_C = 3              forward error / (u kappa_2) of the P = 1 plans <= 0.21 (kd = 95, radius 1e16), all plans <= 0.21
  FULL_ETA_BAR = 5e-14   config 4 (P = 128) relative residual <= 4.5e-15 (radius 1e16)
One Schur piece of reduce_kernel scaled by 1 + 1e-9 already lifts eta to 5.7e-15 .. 2.4e-12 on the chunked plans.
"""
import numpy as np
import pytest

from openimucameracalibrator_b200 import _capi as capi
from test_solver_reference import CASES, FULL_CASES, JACOBI_OFF, RADII, REFUSED, backward_error, damped_solve_reference, load, ulps

pytestmark = pytest.mark.gpu
U = np.finfo(np.float64).eps
ETA_BAR = 5e-15
FWD_C = 3.0
FULL_ETA_BAR = 5e-14
_KAPPA = {}        # case -> {(jacobi, radius): kappa_2(A)}, shared by the chunk counts of a case


@pytest.fixture(scope="module")
def handles(cuda_lib):
    """One GPU handle per dataset, shared by the module's tests."""
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = load(capi.CApi(cuda_lib, "icc_", 0), name)
        return cache[name]
    yield get
    for h in cache.values():
        h.close()


def _plan_str(p):
    return " ".join(f"{k}={p[k]}" for k in ("P", "w", "len", "rem", "L", "kd", "nb", "nk", "WS_A", "cl_global", "cs_global", "stage0"))


@pytest.mark.parametrize("case,ds,flags,chunks", [(c, d, f, k) for c, d, f, ks in CASES for k in ks],
                         ids=[f"{c}-chunks{k}" for c, _, _, ks in CASES for k in ks])
def test_damped_solve_matches_dense_reference(handles, case, ds, flags, chunks):
    h = handles(ds)
    plan = h.solver_plan(flags, chunks)
    kappa = _KAPPA.setdefault(case, {})
    for jacobi in ((1, 0) if case in JACOBI_OFF else (1,)):
        h.set_solver_options(jacobi_scaling=jacobi)
        try:
            for radius in RADII:
                st = h.solve_step(flags, radius, chunks)
                ref = damped_solve_reference(st["hessian"], st["gradient"], radius, jacobi=bool(jacobi))
                assert ulps(st["scale"], ref["scale"]) <= 1 and ulps(st["lm_diag"], ref["lm_diag"]) <= 1
                eta = backward_error(ref["A"], ref["b"], st["delta"] / st["scale"])
                if (jacobi, radius) not in kappa:     # A moves only at rounding level from one evaluation to the next
                    ev = np.linalg.eigvalsh(ref["A"])
                    kappa[(jacobi, radius)] = float(ev[-1] / ev[0]) if ev[0] > 0 else np.inf
                k2 = kappa[(jacobi, radius)]
                fwd = float(np.linalg.norm(st["delta"] - ref["delta"]) / np.linalg.norm(ref["delta"]))
                mc = abs(st["model_change"] - ref["model_change"]) / abs(ref["model_change"])
                print(f"[solve] {case} chunks={chunks} jacobi={jacobi} radius={radius:.0e} | {_plan_str(plan)} | eta={eta:.2e} "
                      f"fwd={fwd:.2e} mc={mc:.2e} kappa={k2:.2e} fwd/(u kappa)={fwd / (U * k2):.2e}")
                assert eta <= ETA_BAR, (case, chunks, jacobi, radius, eta)
                bar = max(1e-12, FWD_C * U * k2)
                assert fwd <= bar and mc <= bar, (case, chunks, jacobi, radius, fwd, mc, k2)
                assert st["model_change"] > 0.0
        finally:
            h.set_solver_options(jacobi_scaling=1)


@pytest.mark.parametrize("case,ds,flags", [(c, d, f) for c, d, f, _ in FULL_CASES], ids=[c for c, _, _, _ in FULL_CASES])
def test_full_size_solve_residual(handles, case, ds, flags):
    """Config 4 (automatic plan P = 128, six reduction levels): relative residual of A y = b with A y = S (H delta) + D y."""
    h = handles(ds)
    plan = h.solver_plan(flags)
    for radius in RADII:
        st = h.solve_step(flags, radius, hessian=False)
        s, D = st["scale"], st["lm_diag"]
        y = st["delta"] / s
        SHd = s * h.normal_matvec(flags, st["delta"][None, :])[0]
        b = -s * st["gradient"]
        r = SHd + D * y - b
        eta = float(np.abs(r).max() / (np.abs(SHd).max() + np.abs(D * y).max() + np.abs(b).max()))
        print(f"[solve] {case} radius={radius:.0e} | {_plan_str(plan)} | full-size eta={eta:.2e}")
        assert eta <= FULL_ETA_BAR, (case, radius, eta)
        assert st["model_change"] > 0.0


def test_too_wide_border_is_refused(handles):
    """Config 4's board with POINTS: no plan fits, the solve reports ICC_ERR_UNSUPPORTED and never returns a result."""
    h = handles(REFUSED[0])
    assert h.solver_plan(REFUSED[1])["valid"] == 0
    with pytest.raises(capi.IccError, match="UNSUPPORTED"):
        h.solve_step(REFUSED[1], 1e4, hessian=False)
