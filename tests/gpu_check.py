"""Ad-hoc GPU vs oracle comparison (developer tool; the real parity tests live in test_*.py)."""
import os, sys, time, numpy as np
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE)); sys.path.insert(0, HERE)
from oracle_api import new_oracle
from openimucameracalibrator_b200 import synthetic as syn, _capi as capi, calibrator
from openimucameracalibrator_b200 import camera_models as cm

def compare(ds, flags, known_gravity=True, label=""):
    o = new_oracle(); capi.load_dataset(o, ds, known_gravity=known_gravity)
    g = capi.CApi(calibrator.load_library(), "icc_", 0); capi.load_dataset(g, ds, known_gravity=known_gravity)
    co, ro, go, Ho = o.evaluate(flags, hessian=True)
    cg, rg, gg, Hg = g.evaluate(flags, hessian=True)
    def rel(a, b): return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)
    print(f"[{label}] n={go.size} cost rel {abs(co-cg)/co:.2e} res rel {rel(rg, ro):.2e} grad rel {rel(gg, go):.2e} H rel {rel(Hg, Ho):.2e}")
    # per-block breakdown of worst gradient mismatch
    bad = np.argmax(np.abs(gg - go)); print("   worst grad idx", bad, gg[bad], go[bad])
    c2, _, _, _ = g.evaluate(flags, residuals=False, gradient=False); print("   cost-only rel", abs(c2 - co) / co)
    return o, g

F = capi.FLAG_SPLINE | capi.FLAG_T_I_C
FALL = F | capi.FLAG_GRAVITY_DIR | capi.FLAG_CAM_LINE_DELAY | capi.FLAG_IMU_BIASES
ds = syn.make_dataset(syn.tiny_config())
compare(ds, F, label="tiny divundist default")
compare(ds, FALL, known_gravity=False, label="tiny divundist all")
compare(ds, capi.FLAG_CAM_LINE_DELAY, label="tiny ld only")
for k in range(8):
    c = syn.config5(k); c.n_frames = 20
    d = syn.make_dataset(c)
    compare(d, FALL, known_gravity=False, label=c.name)
# LM parity on config 1
ds = syn.make_dataset(syn.CONFIGS[1])
o, g = compare(ds, F, label="cfg1")
t = time.time(); so = o.optimize(50, F); to = time.time() - t
t = time.time(); sg = g.optimize(50, F); tg = time.time() - t
print("oracle", so.as_dict()); print("gpu", sg.as_dict())
print("T_ic oracle", o.get_T_i_c()); print("T_ic gpu   ", g.get_T_i_c())
print("times", to, tg)
s2o = o.optimize(10, capi.FLAG_CAM_LINE_DELAY); s2g = g.optimize(10, capi.FLAG_CAM_LINE_DELAY)
print("ld", o.get_line_delay(), g.get_line_delay(), s2o.iterations, s2g.iterations)
tt = (np.asarray(g.imu_used()[0][:5]) * 1e9).astype(np.int64)
print("traj gpu", g.eval_trajectory(tt)["gyro"][:2], "oracle", o.eval_trajectory(tt)["gyro"][:2])
