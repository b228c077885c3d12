"""Residual sharding on real GPUs: 2 ranks over NCCL evaluate their time slices, all-reduce the packed normal equations on
the solver stream and must follow exactly the single-GPU LM path.  Needs >= 2 visible GPUs; skips on fewer."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, out_dir, native):
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch
    import torch.distributed as dist
    from helpers import F_STAGE1
    from openimucameracalibrator_b200 import _capi as capi, calibrator, synthetic as syn
    from openimucameracalibrator_b200.distributed import make_allreduce_hook, make_comm
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    ds = syn.make_dataset(syn.CONFIGS[2])
    g = capi.CApi(calibrator.load_library(), "icc_", rank)
    if native:   # the library's own NCCL communicator: no Python in the collective path
        capi.load_dataset(g, ds, comm=make_comm(calibrator.load_library(), rank))
    else:        # caller-supplied hook (torch.distributed)
        capi.load_dataset(g, ds, shard=(rank, world))
        g.set_allreduce(make_allreduce_hook(g.get_stream(), rank))
    s = g.optimize(50, F_STAGE1)
    if rank == 0:
        np.save(os.path.join(out_dir, "T.npy"), g.get_T_i_c())
        np.save(os.path.join(out_dir, "it.npy"), np.array([s.iterations, s.termination, s.num_residuals]))
        np.save(os.path.join(out_dir, "reproj.npy"), np.array([s.mean_reproj_error, s.final_cost]))
    dist.destroy_process_group()


@pytest.mark.parametrize("native", [True, False], ids=["library_nccl", "torch_hook"])
def test_two_gpu_sharded_lm_matches_single_gpu(tmp_path, gpu_factory, native):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from helpers import F_STAGE1, rel
    from openimucameracalibrator_b200 import _capi as capi, synthetic as syn
    port = 29600 + (os.getpid() % 2000)
    mp.spawn(_worker, args=(2, port + int(native), str(tmp_path), native), nprocs=2, join=True)
    ds = syn.make_dataset(syn.CONFIGS[2])
    g = gpu_factory(); capi.load_dataset(g, ds)
    s = g.optimize(50, F_STAGE1)
    it = np.load(tmp_path / "it.npy"); T = np.load(tmp_path / "T.npy"); rp = np.load(tmp_path / "reproj.npy")
    assert it[0] == s.iterations and it[1] == s.termination
    assert rel(T, g.get_T_i_c()) < 1e-8
    assert abs(rp[0] - s.mean_reproj_error) < 1e-8 and abs(rp[1] - s.final_cost) <= 1e-9 * s.final_cost


def test_cli_gpus_flag_matches_single_gpu(tmp_path):
    """The drop-in binary's sharded mode (--gpus 2: one rank process per device spawned by the binary itself, the NCCL id handed over on
    the command line, ncclAllReduce inside libicc_b200.so) must write the same calibration as the single-GPU run of the same files."""
    import subprocess
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
    from openimucameracalibrator_b200 import camera_models as cm, io_formats as iof, synthetic as syn
    from test_cli_formats import _args
    cfg = syn.tiny_config(cm.DOUBLE_SPHERE, (342.4, 1.0, 0.0, 472.6, 273.9, -0.215, 0.513), n_frames=60, imu_rate_hz=200.0, seed=22, line_delay_init_scale=1.1)
    ds = syn.make_dataset(cfg)
    res = []
    for gpus in (1, 2):
        d = tmp_path / f"g{gpus}"; d.mkdir()
        paths = iof.write_dataset_files(ds, str(d))
        env = dict(os.environ); env["NCCL_DEBUG"] = "WARN"
        proc = subprocess.Popen(_args(paths, str(d), ["--calibrate_cam_line_delay", f"--gpus={gpus}"]), stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env, start_new_session=True)
        try:
            so, se = proc.communicate(timeout=90)
        except subprocess.TimeoutExpired:
            import signal
            os.killpg(proc.pid, signal.SIGKILL)          # the launcher and the rank processes it spawned
            so, se = proc.communicate()
            pytest.fail(f"--gpus={gpus} did not finish in 90 s\nstdout:\n{so[-3000:]}\nstderr:\n{se[-3000:]}")
        out = subprocess.CompletedProcess(proc.args, proc.returncode, so, se)
        assert out.returncode == 0, out.stderr + out.stdout
        if gpus == 2:
            assert "sharded over 2 GPUs" in out.stdout
        res.append(iof.read_result_json(str(d / "result.json")))
    a, b = res
    for k in ("x", "y", "z", "w"):
        assert abs(a["q_i_c"][k] - b["q_i_c"][k]) < 1e-9
    for k in ("x", "y", "z"):
        assert abs(a["t_i_c"][k] - b["t_i_c"][k]) < 1e-8
    assert abs(a["final_reproj_error"] - b["final_reproj_error"]) < 1e-9 and abs(a["calib_line_delay_us"] - b["calib_line_delay_us"]) < 1e-8
