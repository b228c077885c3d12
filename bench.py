#!/usr/bin/env python
"""bench.py — residuals/sec per Levenberg-Marquardt iteration of the continuous-time IMU-camera calibration solve.

Contract (see DESIGN.md "Measurement"):
  python bench.py --gpus N --steps K --warmup W [--impl reference] [--config 4] [--dump-outputs DIR]
  * workload  = BASELINE.json configs[3]: ExtendedUnified, 3000 frames x 144 corners, 1 kHz IMU (the config the metric's
                target is quoted on; fits one B200).  N > 1 shards the residuals by time slice, NCCL all-reduce of the
                packed J^T J / J^T r buffer (strong scaling).
  * step      = ONE full LM iteration from the same initial state: residual + analytic Jacobian evaluation fused with the
                J^T J / J^T r reduction, Jacobi scaling, damped banded+bordered LDL^T solve, manifold update, candidate
                cost evaluation, accept/reject.  Inputs resident in HBM.  `value` = scalar residuals / step time.
  * e2e       = the whole user job through the C-ABI with HOST buffers: set_* + BatchInitSpline (problem assembly + H2D) +
                Optimize(50) to convergence + result read-back; value = residuals x LM iterations / wall time.
  * roofline  = the dominant kernel (vision residual/Jacobian kernel) timed alone with CUDA events on its stream.
  * cpu_baseline / --impl reference = the CPU restatement of the reference Ceres path (oracle/), all host threads, on a
                bounded sample of the same workload (the real reference cannot be built offline: Ceres/Theia/Eigen absent).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from openimucameracalibrator_b200 import _capi as capi  # noqa: E402
from openimucameracalibrator_b200 import synthetic as syn  # noqa: E402

FLAGS = capi.FLAG_SPLINE | capi.FLAG_T_I_C      # the hot CLI's stage-1 flags with a known gravity axis (app :200-215)
METRIC = "residuals/sec per LM iter"
UNIT = "residuals/s"
# summary fields that depend only on the computation (timings and launch counts are left out)
DUMP_SUMMARY_FIELDS = ("iterations", "successful_steps", "termination", "num_residuals", "num_tangent", "initial_cost", "final_cost", "mean_reproj_error")


def dump_outputs(out_dir, api, summ, prefix=""):
    """--dump-outputs: what one LM-iteration step hands its caller, as float64 DIR/<prefix><name>.npy -- the updated spline knots,
    T_i_c and line delay read back from the handle, and the returned summary.  Every step starts from the same state and the
    inputs are seeded, so two builds run with the same arguments can be compared file for file."""
    os.makedirs(out_dir, exist_ok=True)
    so3, r3, ba, bg = api.get_knots()
    arrays = {"so3_knots": so3, "r3_knots": r3, "accel_bias_knots": ba, "gyro_bias_knots": bg, "T_i_c": api.get_T_i_c(),
              "line_delay": [api.get_line_delay()]}
    arrays.update({"summary_" + k: [getattr(summ, k)] for k in DUMP_SUMMARY_FIELDS})
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), np.asarray(a, dtype=np.float64))


def workload_name(cfg):
    return f"{cfg.name} (frames={cfg.n_frames}, corners={cfg.grid[0] * cfg.grid[1]}, imu={cfg.imu_rate_hz:g}Hz, flags=SPLINE|T_I_C)"


def algorithmic_bytes(ds, n_frames, n_corners, n_imu, n_cells):
    """SURVEY.md §8(d): per corner 20 B; per frame 336 (knots) + 32 (s,u) + 7920 (43-col tile + J^T r + cost);
    per IMU sample pair 56 B; per knot-interval cell 336 + 144 (bias knots) + tile (36+1 cols, no bias: (37*38/2+... ) ) B."""
    vis = 20 * n_corners + (336 + 32 + (43 * 44 // 2 + 43 + 1) * 8) * n_frames
    d_imu = 36  # stage-1 active columns of an IMU tile (so3 18 + r3 18)
    imu = 56 * n_imu + (336 + 144 + (d_imu * (d_imu + 1) // 2 + d_imu + 1) * 8) * n_cells
    return vis, imu


class ClockSampler:
    """SM clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe: the same fields as the nvidia-smi clocks line).
    Read through NVML inside this process (nvidia_ml_py, one handle opened before the timed region), ONE sample per step taken by the
    timing loop itself between two steps -- while the L2-flush fill of the next step keeps the GPU under load, outside the CUDA-event
    bracket of either step.  Every out-of-band sampler perturbed the number it was meant to vouch for: a freshly started `nvidia-smi -lms`
    stalls the driver for a few milliseconds per sample (at N = 8 a 5 ms step on every rank: the peers wait inside the all-reduce), an
    NVML polling thread still cost one 0.5 ms step in twenty (N = 4).  Falls back to the nvidia-smi subprocess when NVML cannot be loaded."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.p, self.thread, self.samples, self.stop_flag, self.index = None, None, [], False, index
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[index]) if visible and all(x.strip().isdigit() for x in visible.split(",")) else index
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.thread = True          # NVML mode: sample() is called by the timing loop
        except Exception:
            self.thread = None
            try:
                self.p = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                          stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            except Exception:
                self.p = None

    def sample(self):
        if self.thread is None:
            return
        nv = self.nv
        try:
            try:
                reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:
                reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            self.samples.append((float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)), int(reasons)))
        except Exception:
            pass

    def stop(self):
        if self.thread is not None:
            nv = self.nv
            names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                     "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
            sm = [s for s, _ in self.samples]
            reasons = sorted(k for k, bit in names.items() if any(r & bit for _, r in self.samples))
            hot = sorted(sm)[len(sm) // 2:] if sm else []
            return {"sm_mhz": float(np.median(hot)) if hot else None, "sm_max_mhz": self.sm_max, "reasons": reasons, "samples": len(sm), "source": "nvml (in-process, one sample per step between the event brackets, GPU busy with the L2 flush)"}
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            out = ""
        sm, mx, reasons = [], [], set()
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        hot = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": float(np.median(hot)) if hot else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 200"}


def run_reference(args, cfg):
    """CPU arm: the oracle restatement of the reference Ceres path on the FULL workload (same config as the GPU arm), on the host
    threads the box grants (persistent pool; the count that evaluates fastest among 8 / 32 / all is used and all three are reported)."""
    from oracle_api import new_oracle
    import copy
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    c = copy.copy(cfg)
    c.n_frames = min(cfg.n_frames, args.sample_frames) if args.sample_frames > 0 else cfg.n_frames
    c.name = cfg.name
    ds = syn.make_dataset(c)
    budget = new_oracle(0); capi.load_dataset(budget, ds)
    all_threads = int(budget.lib.icco_num_threads(budget.h)); nres = sum(budget.num_residuals()); budget.close()
    scaling, best = {}, None
    for nt in sorted({min(8, all_threads), min(32, all_threads), all_threads}):
        o = new_oracle(nt); capi.load_dataset(o, ds)
        o.time_evaluations(1, FLAGS, 1)
        ms_eval = o.time_evaluations(2, FLAGS, 1)
        scaling[str(nt)] = {"jacobian_eval_ms": ms_eval, "residuals_per_s": nres / (ms_eval * 1e-3), "residuals_per_s_per_thread": nres / (ms_eval * 1e-3) / nt}
        if best is None or ms_eval < best[1]:
            best = (nt, ms_eval)
        o.close()
    cores = best[0]
    o = new_oracle(cores); capi.load_dataset(o, ds)
    so3, r3, ba, bg = o.get_knots(); T0 = o.get_T_i_c(); ld0 = o.get_line_delay()
    times = []
    for i in range(args.warmup + args.steps):
        o.set_knots(so3, r3, ba, bg); o.set_T_i_c(T0); o.set_line_delay(ld0)
        t = time.perf_counter(); summ = o.lm_iterations(1, FLAGS); dt = time.perf_counter() - t
        if i >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, o, summ)
    ms = 1e3 * float(np.mean(times))
    value = nres / (ms * 1e-3)
    full = c.n_frames == cfg.n_frames
    sample = (f"the full workload ({nres} scalar residuals/step)" if full else f"first {c.n_frames} of {cfg.n_frames} frames ({nres} scalar residuals/step)") + ", 1 LM iteration/step"
    return {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "reference",
            "config": {"workload": workload_name(cfg), "scalar_residuals": nres, "sample": sample, "parallelism": f"cpu{cores}", "same_config": full},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": int(cores), "kind": "port", "sample": sample, "host_thread_budget": all_threads,
                             "thread_scaling": scaling, "per_core_residuals_per_s": value / cores,
                             "what": "CPU restatement of the reference Ceres path (oracle/: Jet<4> autodiff passes x local parameterisations, banded+bordered Cholesky, persistent thread pool)"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}


def run_batch_of_eight(args):
    """BASELINE configs[4]: 8 independent calibration sequences (mixed camera models), replicas only — rank r owns sequences
    r, r+N, ...; no data-path collective.  step = one LM iteration on every owned sequence; value = all residuals / max-rank time."""
    import torch
    import torch.distributed as dist
    from openimucameracalibrator_b200 import calibrator
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": "config 5 is measured on the GPU arm only; use --config 4 for the CPU arm"}), flush=True)
        return 0
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    mine = list(range(rank, 8, world))
    handles, inits, nres = [], [], 0
    for k in mine:
        ds = syn.make_dataset(syn.config5(k))
        a = capi.CApi(calibrator.load_library(), "icc_", local); capi.load_dataset(a, ds)
        handles.append(a); inits.append((a.get_knots(), a.get_T_i_c(), a.get_line_delay())); nres += sum(a.num_residuals())
    def reset():
        for a, (kn, T0, ld0) in zip(handles, inits):
            a.set_knots(*kn); a.set_T_i_c(T0); a.set_line_delay(ld0)
    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(); torch.cuda.synchronize()
    sampler = ClockSampler(local) if rank == 0 else None
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=f"cuda:{local}")   # > L2 (126 MB): every round starts cold
    total_ms, launches = 0.0, 0
    for i in range(args.warmup + args.steps):       # warm-up rounds run exactly like timed ones, they are just not recorded
        if i == args.warmup and sampler: sampler.samples.clear()
        reset(); flush.fill_(float(i))
        if sampler: sampler.sample()                # under load (the fill is running), outside the wall-clock bracket of any round
        sync()
        t0 = time.perf_counter()
        summs = [a.lm_iterations(1, FLAGS) for a in handles]     # each call ends with a stream synchronisation
        torch.cuda.synchronize()
        if i >= args.warmup:
            total_ms += 1e3 * (time.perf_counter() - t0); launches += sum(s.gpu_launches for s in summs)
    sync()
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs:
        for k, a, s in zip(mine, handles, summs):
            dump_outputs(args.dump_outputs, a, s, prefix=f"seq{k}_")
    tot_res = nres
    if world > 1:
        t = torch.tensor([total_ms, float(nres)], dtype=torch.float64, device=f"cuda:{local}")
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX); dist.all_reduce(t); total_ms = float(tmax[0]); tot_res = int(t[1])
    ms = total_ms / args.steps
    if rank == 0:
        print(json.dumps({"metric": METRIC, "value": tot_res / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
                          "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                          "config": {"workload": "cfg5: 8 independent 300x96 sequences, models Pinhole/Fisheye/DivUndist/DoubleSphere/EUCM/FOV/Fisheye/EUCM", "scalar_residuals": tot_res,
                                     "parallelism": f"replicas x{world} (no collective)", "timing": "host clock around per-sequence LM iterations (each ends in a stream sync)", "l2": "flushed between rounds (256 MiB fill)"},
                          "clocks": clocks, "gpu_launches": launches, "e2e": None, "roofline": None, "cpu_baseline": None}), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=4, help="BASELINE config index 1-4; 5 = batch of 8 independent sequences (replicas, one handle each)")
    ap.add_argument("--sample-frames", type=int, default=0, help="frames of the workload used per CPU-arm step (0 = the full workload)")
    ap.add_argument("--cpu-baseline-steps", type=int, default=3)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.config == 5:
        return run_batch_of_eight(args)
    cfg = syn.CONFIGS[args.config]

    if args.impl == "reference":
        line = run_reference(args, cfg)
        if line is not None:
            print(json.dumps(line), flush=True)
        return 0

    import torch
    import torch.distributed as dist
    from openimucameracalibrator_b200 import calibrator

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device: the solver has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ds = syn.make_dataset(cfg)

    api = capi.CApi(calibrator.load_library(), "icc_", local)
    # N > 1: the library's own NCCL communicator (one per process, created once like the CUDA context; handles borrow it).  The
    # collectives of the solve are ncclAllReduce calls inside libicc_b200.so on the solver's stream -- no Python in that path.
    comm = None
    if world > 1:
        from openimucameracalibrator_b200.distributed import make_comm
        os.environ.setdefault("NCCL_DEBUG", "WARN")      # keep NCCL's version banner off stdout: the contract is ONE JSON line
        comm = make_comm(calibrator.load_library(), local)

    t_load0 = time.perf_counter()
    capi.load_dataset(api, ds, comm=comm)
    t_load = time.perf_counter() - t_load0
    ext_stream = torch.cuda.ExternalStream(api.get_stream(), device=f"cuda:{local}")
    nres_local = sum(api.num_residuals())
    nres = nres_local
    if world > 1:
        t = torch.tensor([nres_local], dtype=torch.int64, device=f"cuda:{local}"); dist.all_reduce(t); nres = int(t.item())
    so3, r3, ba, bg = api.get_knots(); T0 = api.get_T_i_c(); ld0 = api.get_line_delay()
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=f"cuda:{local}")   # 256 MiB > 126 MB L2

    def reset():
        api.set_knots(so3, r3, ba, bg); api.set_T_i_c(T0); api.set_line_delay(ld0)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    launches = 0
    step_ms = []
    summ = None
    sampler = ClockSampler(local) if rank == 0 else None   # NVML is initialised (and queried once per warm-up step) before the timed region
    import gc
    gc.collect(); gc.disable()                      # no collector pause inside a timed step (at N > 1 every rank waits for the slowest)
    barrier()
    # Warm-up steps run EXACTLY like timed ones (state reset, L2 flush, clock sample, rank barrier, event bracket) and are simply not recorded:
    # with a plain warm-up loop the first timed step was the first to see a cold L2 and a rank barrier and came out 5 % (N = 1) to 60 % (N = 8) slow.
    for i in range(args.warmup + args.steps):
        timed = i >= args.warmup
        if i == args.warmup and sampler: sampler.samples.clear()
        reset()
        flush.fill_(float(i))
        if sampler: sampler.sample()                # under load (the fill is running), outside the event bracket of any step
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(ext_stream)
        summ = api.lm_iterations(1, FLAGS)
        e1.record(ext_stream)
        e1.synchronize()
        if timed:
            step_ms.append(e0.elapsed_time(e1)); launches += summ.gpu_launches
    barrier()
    clocks = sampler.stop() if sampler else None
    gc.enable()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, api, summ)
    total_ms = float(np.sum(step_ms))
    if world > 1:
        t = torch.tensor([total_ms], dtype=torch.float64, device=f"cuda:{local}"); dist.all_reduce(t, op=dist.ReduceOp.MAX); total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = nres / (ms_per_step * 1e-3)

    # ---- kernel-level numbers (rank 0, N = 1 semantics: this rank's shard) ----------------------------------------
    reset()
    ms_vis = api.time_evaluations(20, FLAGS, 2)
    ms_imu = api.time_evaluations(20, FLAGS, 3)
    ms_cost = api.time_evaluations(20, FLAGS, 0)
    nv, na, ng = api.num_residuals()
    n_frames_local = len(ds["frame_t"]) if world == 1 else None
    jac_s, lin_s = summ.seconds_jacobian, summ.seconds_linear_solve
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0)); peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback"
    roof = None
    if world == 1:
        ncells = len({(int(s // int(cfg.dt_so3_s * 1e9))) for s in ((api.imu_used()[0] * 1e9).astype(np.int64) - int(ds["frame_t"].min() * 1e9))})
        b_vis, b_imu = algorithmic_bytes(ds, len(ds["frame_t"]), nv // 2, na // 3, ncells)
        ach = b_vis / (ms_vis * 1e-3) / 1e9
        # FP64 work of the vision kernel against the MEASURED FP64 ceilings of this chip (tools/fp64_peaks.cu -> profiles/r2_fp64_peaks.json):
        # DMMA (mma.sync m8n8k4 f64) and DFMA share ONE FP64 pipe on B200 (mixed microbenchmark: DMMA 32.3 + DFMA 4.0 TF concurrently
        # vs 37.1 / 33.9 alone), so the floor is the SUM of both instruction streams' pipe time, not the max.
        rows = nv
        dmma_flops = (rows / 4.0) * 21 * 512                      # 21 block products per 4 tile rows, 512 flop each
        simt_instr_per_corner = 1170.0                            # FP64 SIMT warp-instructions per 32 corners (ncu: 15.8 M per 13 500 chunks)
        simt_flops = (rows / 2.0) * simt_instr_per_corner * 2     # counted as FMAs
        fp = {}
        try:
            fp = json.load(open(os.path.join(ROOT, "profiles", "r2_fp64_peaks.json")))
        except Exception:
            pass
        dmma_peak = float(fp.get("dmma_m8n8k4_tflops_21acc", 37.0)); dfma_peak = float(fp.get("dfma_tflops", 34.0))
        pipe_floor_ms = 1e3 * (dmma_flops / (dmma_peak * 1e12) + simt_flops / (dfma_peak * 1e12))
        traffic, traffic_src = None, None
        try:   # dram__bytes_read.sum + dram__bytes_write.sum of this kernel from the committed ncu --set full capture (config 4 only)
            if args.config == 4:
                nc = json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_summary.json")))["eval_tmem_kernel<6>"]
                traffic = nc["dram_bytes_read"] + nc["dram_bytes_write"]; traffic_src = "profiles/r2_ncu_summary.json (ncu --set full, one launch)"
        except Exception:
            pass
        roof = {"kernel": "vision_tmem_kernel<MODEL> (residual + analytic Jacobian + J^T J tile: persistent 12-warp CTAs, accumulators parked in TMEM)", "bound": "hbm", "achieved": ach,
                "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": b_vis, "launch_ms": ms_vis,
                "note": "arithmetic intensity >> FP64 ridge: the kernel is bound by the FP64 pipe (DMMA + DFMA share it), not by HBM (DESIGN.md); see fp64",
                "fp64": {"tensor_tflops_issued": dmma_flops / (ms_vis * 1e-3) / 1e12, "simt_tflops_issued": simt_flops / (ms_vis * 1e-3) / 1e12,
                         "measured_peak_dmma_tflops": dmma_peak, "measured_peak_dfma_tflops": dfma_peak, "peak_source": "profiles/r2_fp64_peaks.json (tools/fp64_peaks.cu on B200)" if fp else "nominal",
                         "fp64_pipe_floor_ms": pipe_floor_ms, "frac_of_fp64_pipe": pipe_floor_ms / ms_vis},
                "imu_kernel": {"launch_ms": ms_imu, "algorithmic_bytes_per_launch": b_imu, "achieved": b_imu / (ms_imu * 1e-3) / 1e9},
                "cost_only_eval_ms": ms_cost, "jacobian_eval_ms_in_step": 1e3 * jac_s / max(1, summ.jacobian_evaluations),
                "linear_solve_ms_in_step": 1e3 * lin_s / max(1, summ.iterations)}

    # ---- e2e: whole job from host buffers through the C-ABI ------------------------------------------------------
    e2e = None
    h2d = sum(int(np.asarray(ds[k]).nbytes) for k in ("uv", "point_ids", "corner_offsets", "frame_t", "q_wc", "p_wc", "imu_t", "accel", "gyro", "board_xyzw"))
    e2e_vals, e2e_wall, e2e_iters = [], [], []
    # the job's inputs live in page-locked host memory (the contract's "from pinned host memory"): the library then sends the large arrays
    # straight to the device by DMA inside icc_set_frames / icc_set_imu and waits for it there (no staging copy, nothing borrowed after return)
    ds_host, _pins = dict(ds), []
    for k in ("uv", "point_ids", "accel", "gyro", "imu_t"):
        tpin = torch.from_numpy(np.ascontiguousarray(ds[k])).pin_memory(); _pins.append(tpin); ds_host[k] = tpin.numpy()
    for i in range(max(1, args.e2e_steps)):
        barrier()
        t0 = time.perf_counter()
        a2 = capi.CApi(calibrator.load_library(), "icc_", local)
        capi.load_dataset(a2, ds_host, comm=comm)
        s2 = a2.optimize(50, FLAGS)
        T = a2.get_T_i_c(); ld = a2.get_line_delay()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([wall], dtype=torch.float64, device=f"cuda:{local}"); dist.all_reduce(t, op=dist.ReduceOp.MAX); wall = float(t.item())
        e2e_wall.append(wall); e2e_iters.append(s2.iterations); e2e_vals.append(nres * s2.iterations / wall)
        a2.close()
    e2e = {"value": float(np.median(e2e_vals)), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 8 * 8 + 8 * 8 * int(np.median(e2e_iters)),
           "wall_clock_to_convergence_s": float(np.median(e2e_wall)), "lm_iterations": int(np.median(e2e_iters)),
           "final_T_i_c": [float(x) for x in T], "final_reproj_error_px": float(s2.mean_reproj_error),
           "what": "set_* (H2D of the corner / IMU arrays from page-locked host buffers) + BatchInitSpline (host assembly + H2D of the tables) + Optimize(50) to Ceres-style convergence + getters, host buffers in, results out"}

    # ---- CPU baseline (rank 0, N == 1) ---------------------------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        import copy
        ns = copy.copy(args); ns.steps = args.cpu_baseline_steps; ns.warmup = 0; ns.dump_outputs = None
        ref = run_reference(ns, cfg)
        cpu = ref["cpu_baseline"]

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": workload_name(cfg), "scalar_residuals": nres, "tangent_params": summ.num_tangent,
                           "parallelism": f"residual-sharded x{world}" if world > 1 else "single",
                           "l2": "flushed between steps (256 MiB fill); step time = per-step CUDA events on the solver stream, summed",
                           "step": "1 LM iteration: J eval + J^T J reduce + scale + banded/bordered LDL^T + update + cost eval"},
                "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roof, "cpu_baseline": cpu,
                "problem_load_s": t_load, "step_ms": [round(x, 4) for x in step_ms]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
