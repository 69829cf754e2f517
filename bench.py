#!/usr/bin/env python
"""Benchmark of the GP slip-prediction hot path (BASELINE.json: "GP slip predictions/sec").

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, through libcngp)
    python bench.py --impl reference --gpus N ...            # reference arm: the CPU port (oracle/) on the host cores

Workload (config.workload): BASELINE.json configs[1] - 4096 independent slip windows per GPU, N = 256 training
samples, SE + periodic kernel at fixed hyper-parameters, M = 600 predicted points (gp_slip_node.py:45), predict-only.
One step = one pass of the hot path over that batch: kernel-matrix assembly, Cholesky, z = L^-1 y, LML, predictive
mean and variance at 600 points, for every window.  Unit: windows/s (1 prediction = 1 window); N>1 is weak scaling
(4096 windows per GPU, no data-path collective; one all_gather of per-window LML after the timed region).

value    : whole-job windows/s with inputs resident in HBM, timed per step with CUDA events on the launching stream
           (L2 flushed between steps), max over ranks.
e2e      : the same metric through GpContext.predict with pinned HOST buffers (H2D of x, y, x*, theta and D2H of mean,
           var, lml, status inside the timed region).
roofline : dominant kernel (gp_var_kernel) algorithmic FP64 flop / its CUDA-event duration, against cuBLAS DGEMM
           measured live in this run on the same GPU (MEASURED_PEAKS.json holds no FP64 figure; SURVEY.md section 6).
cpu_baseline : the oracle port (vectorised predict, one window per process, 1 BLAS thread each) on a bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark writes nothing into the tree it runs from (it may be read-only)

KERNEL = "rbf+stdperiodic"
B_PER_GPU = 4096
N_TRAIN = 256
M_TEST = 600
METRIC = "GP slip predictions/sec (windows/s; N=256 windows, SE+periodic, M=600 predicted points, predict-only)"
UNIT = "windows/s"


def flops_per_window(N=N_TRAIN, M=M_TEST):
    """SURVEY.md 8d: F_chol + F_alpha + F_mean + F_var (FP64, mul+add = 2)."""
    return dict(chol=N ** 3 / 3.0, alpha=2.0 * N * N, mean=2.0 * N * M, var=float(N) * N * M + 2.0 * N * M)


# ----------------------------------------------------------------------------------------------------------------
# CPU port (oracle) legs
# ----------------------------------------------------------------------------------------------------------------
def _cpu_worker_pointwise(args):
    """The reference's own loop shape (gp_slip_node.py:47-50): one m.predict([[x]]) per test point."""
    first, count = args
    from threadpoolctl import threadpool_limits
    from corenav_gp_b200 import synthetic as syn
    from oracle import gp_oracle as go
    with threadpool_limits(limits=1):
        x, y = syn.slip_windows(first, count, N_TRAIN)
        th = syn.theta_for(KERNEL)
        e = go.KernelExpr(KERNEL)
        acc = 0.0
        for b in range(count):
            xs = syn.test_grid(x[b], M_TEST)
            mu, var = go.predict_pointwise(e, th[:-1], th[-1], x[b], y[b], xs)
            acc += float(mu[0] + var[0])
    return acc


def _cpu_worker(args):
    first, count = args
    from threadpoolctl import threadpool_limits
    from corenav_gp_b200 import synthetic as syn
    from oracle import gp_oracle as go
    with threadpool_limits(limits=1):
        x, y = syn.slip_windows(first, count, N_TRAIN)
        th = syn.theta_for(KERNEL)
        e = go.KernelExpr(KERNEL)
        acc = 0.0
        for b in range(count):
            xs = syn.test_grid(x[b], M_TEST)
            mu, var = go.predict(e, th[:-1], th[-1], x[b], y[b], xs)
            acc += float(mu[0] + var[0])
    return acc


def cpu_port_throughput(windows_per_core: int, cores: int, worker=None):
    """Windows/s of the oracle port with `cores` worker processes (1 BLAS thread each)."""
    import multiprocessing as mp
    worker = worker or _cpu_worker
    ctx = mp.get_context("fork")
    jobs = [(10_000_000 + i * windows_per_core, windows_per_core) for i in range(cores)]
    with ctx.Pool(cores) as pool:
        pool.map(worker, [(0, 1)] * cores)                # warm the workers (imports, first BLAS call)
        t0 = time.perf_counter()
        pool.map(worker, jobs, chunksize=1)
        dt = time.perf_counter() - t0
    return windows_per_core * cores / dt, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    per_core = 8
    thr, _ = cpu_port_throughput(1, cores)                # calibrate so each step is a few seconds
    per_core = int(max(1, min(64, round(3.0 * thr / cores))))
    for _ in range(args.warmup):
        cpu_port_throughput(1, cores)
    t_all, n_all = 0.0, 0
    for _ in range(args.steps):
        v, dt = cpu_port_throughput(per_core, cores)
        t_all += dt
        n_all += per_core * cores
    value = n_all / t_all
    sample = (f"{per_core * cores} windows per step of the same workload (oracle/gp_oracle.py predict: numpy kernel "
              f"assembly + LAPACK dpotrf/dpotrs/dtrtrs with all {M_TEST} points as one RHS block), "
              f"{cores} processes x 1 BLAS thread")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_all / max(1, args.steps), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)
    return 0


def workload_config(n_gpus):
    return {"workload": "BASELINE.json configs[1]: batched 4096 independent slip windows per GPU, N=256, "
                        "SE+periodic kernel (rbf+stdperiodic, fixed hypers), predict-only, M=600",
            "windows_per_gpu": B_PER_GPU, "N": N_TRAIN, "M": M_TEST, "kernel": KERNEL,
            "parallelism": f"window sharding x{n_gpus} (no data-path collective)",
            "l2": "flushed between timed steps (256 MiB memset); factor scratch 1.1 GB > L2"}


# ----------------------------------------------------------------------------------------------------------------
# clocks sampling
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        for r in self.rows:
            f = [t.strip() for t in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


# ----------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------
def measure_dgemm_peak(torch, n=4096, reps=6):
    a = torch.randn(n, n, device="cuda", dtype=torch.float64)
    b = torch.randn(n, n, device="cuda", dtype=torch.float64)
    for _ in range(2):
        torch.matmul(a, b)
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(a, b); e1.record(); e1.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    return 2.0 * n ** 3 / best * 1e-9   # TFLOP/s


def run_ours(args):
    import torch
    import torch.distributed as dist
    from corenav_gp_b200 import _lib as L
    from corenav_gp_b200 import synthetic as syn
    from corenav_gp_b200.api import GpContext

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - this framework has no CPU fallback (use --impl reference for the CPU port)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    ctx = GpContext(device=local)

    # this rank's shard of the global batch: windows [rank*B, (rank+1)*B)
    x, y = syn.slip_windows(rank * B_PER_GPU, B_PER_GPU, N_TRAIN)
    xs = syn.test_grid(x[0], M_TEST)
    th = syn.theta_for(KERNEL)
    dx, dy, dxs, dth = (torch.from_numpy(a).cuda() for a in (x, y, xs, th))
    d_mean = torch.empty(B_PER_GPU, M_TEST, dtype=torch.float64, device="cuda")
    d_var = torch.empty_like(d_mean)
    d_lml = torch.empty(B_PER_GPU, dtype=torch.float64, device="cuda")
    d_status = torch.empty(B_PER_GPU, dtype=torch.int32, device="cuda")
    out_dev = (d_mean, d_var, d_lml, d_status)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def step_device():
        ctx.predict(KERNEL, dth, dx, dy, dxs, out=out_dev)

    peak_tflops = measure_dgemm_peak(torch)

    for _ in range(max(3, args.warmup)):
        step_device()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ctx.set_profiling(True)
    for kid in range(6):
        ctx.profile_read(kid, reset=True)
    launches0 = ctx.launch_count()
    torch.cuda.synchronize()
    t_wall0 = time.perf_counter()
    evs = []
    for _ in range(args.steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step_device()
        e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_wall0
    launches = ctx.launch_count() - launches0
    step_ms = [a.elapsed_time(b) for a, b in evs]
    total_ms = float(sum(step_ms))
    fit_ms, fit_n = ctx.profile_read(L.PROF_FIT)
    var_ms, var_n = ctx.profile_read(L.PROF_VAR)
    ctx.set_profiling(False)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out_dev)

    # ---- e2e: public API, pinned host buffers, copies inside the timed region ----
    hx, hy = torch.from_numpy(x).pin_memory(), torch.from_numpy(y).pin_memory()
    hxs, hth = torch.from_numpy(xs).pin_memory(), torch.from_numpy(th).pin_memory()
    h_out = (torch.empty(B_PER_GPU, M_TEST, dtype=torch.float64).pin_memory(),
             torch.empty(B_PER_GPU, M_TEST, dtype=torch.float64).pin_memory(),
             torch.empty(B_PER_GPU, dtype=torch.float64).pin_memory(),
             torch.empty(B_PER_GPU, dtype=torch.int32).pin_memory())
    for _ in range(2):
        ctx.predict(KERNEL, hth, hx, hy, hxs, out=h_out)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ctx.predict(KERNEL, hth, hx, hy, hxs, out=h_out)      # returns with the results in host memory
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    h2d = int(hx.numel() * 8 + hy.numel() * 8 + hxs.numel() * 8 + hth.numel() * 8)
    d2h = int(h_out[0].numel() * 8 + h_out[1].numel() * 8 + h_out[2].numel() * 8 + h_out[3].numel() * 4)
    # the e2e results must equal the device-resident path bit for bit
    same = bool(torch.equal(h_out[0], d_mean.cpu()) and torch.equal(h_out[1], d_var.cpu()))
    ok = bool((d_status == 0).all().item()) and bool(torch.isfinite(d_mean).all().item())

    # ---- max over ranks; C1: gather per-window LML once, after the timed region ----
    if world > 1:
        t = torch.tensor([total_ms, e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_s = float(t[0]), float(t[1])
        gathered = [torch.empty_like(d_lml) for _ in range(world)]
        dist.all_gather(gathered, d_lml)
        lml_checksum = float(torch.stack(gathered).sum().item())
    else:
        lml_checksum = float(d_lml.sum().item())

    if rank == 0:
        fl = flops_per_window()
        windows_total = B_PER_GPU * world
        value = windows_total * args.steps / (total_ms * 1e-3)
        # per predict call: the variance phase may be two launches (full rounds of 12 test tiles + the last 1..3 tiles)
        var_avg_ms = var_ms / max(1, args.steps)
        fit_avg_ms = fit_ms / max(1, args.steps)
        var_flops = (fl["var"] + fl["mean"]) * B_PER_GPU
        fit_flops = (fl["chol"] + fl["alpha"]) * B_PER_GPU
        achieved = var_flops / (var_avg_ms * 1e-3) * 1e-12
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            try:
                tj = json.load(open(tpath))
                traffic = tj.get("gp_var_kernel_dram_bytes_per_launch")
                traffic_src = tj.get("source")
            except Exception:
                traffic = None
        dmma_peak = None
        try:                                   # DMMA / DFMA issue micro-benchmark (tools/fp64_peak.cu), a second anchor
            r = subprocess.run([os.path.join(ROOT, "tools", "fp64_peak")], capture_output=True, text=True, timeout=60)
            dmma_peak = json.loads(r.stdout.strip().splitlines()[-1])
        except Exception:
            dmma_peak = None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(world),
            "e2e": {"value": windows_total * args.steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "matches_device_path": same},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {
                "bound": "fp64", "kernel": "gp_var_kernel", "achieved": achieved, "peak": peak_tflops,
                "unit": "TFLOP/s", "frac": achieved / peak_tflops, "traffic": traffic,
                "traffic_source": traffic_src, "fp64_issue_peaks": dmma_peak,
                "peak_source": "cuBLAS DGEMM 4096^3 (torch.matmul float64) measured live in this run, burst best-of-6; "
                               "MEASURED_PEAKS.json has no FP64 figure (profiles/fp64_peak_r01.json: DMMA issue peak 37.2)",
                "algorithmic_flop_per_launch": var_flops, "avg_launch_ms": var_avg_ms,
                "launches_per_step": {"gp_var_kernel": var_n / max(1, args.steps), "gp_fit_kernel": fit_n / max(1, args.steps)},
                "share_of_step": var_ms / max(1e-9, total_ms),
                "whole_step": {"flop": (fl["chol"] + fl["alpha"] + fl["mean"] + fl["var"]) * B_PER_GPU,
                               "tflops": (fl["chol"] + fl["alpha"] + fl["mean"] + fl["var"]) * B_PER_GPU /
                                         (total_ms / args.steps * 1e-3) * 1e-12,
                               "frac": (fl["chol"] + fl["alpha"] + fl["mean"] + fl["var"]) * B_PER_GPU /
                                       (total_ms / args.steps * 1e-3) * 1e-12 / peak_tflops},
                "gp_fit_kernel": {"avg_launch_ms": fit_avg_ms, "tflops": fit_flops / (fit_avg_ms * 1e-3) * 1e-12,
                                  "share_of_step": fit_ms / max(1e-9, total_ms)},
                "hbm": {"algorithmic_bytes_per_window": 16 * N_TRAIN + 16 * M_TEST,
                        "note": "arithmetic intensity > 3000 flop/B: HBM is not the bound (SURVEY.md 8d)"},
            },
            "checks": {"all_status_ok_and_finite": ok, "lml_checksum": lml_checksum,
                       "host_wall_s_timed_region": t_wall},
        }
        # ---- CPU baseline: bounded sample on this box's host cores ----
        if not args.no_cpu_baseline:
            # run in a fresh process: forking a CUDA-initialised parent is not safe
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "cpu_probe"],
                               capture_output=True, text=True, timeout=600)
            try:
                line["cpu_baseline"] = json.loads(r.stdout.strip().splitlines()[-1])
            except Exception:
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
                                        "sample": "failed: " + (r.stderr or r.stdout)[-200:]}
    # ---- extra: the other BASELINE configs and the FP32 mode, device-timed, outside the headline's timed region ----
    extra = None
    if not args.no_extra:
        extra = run_extra(ctx, torch, rank, world, (dx, dy, dxs, dth), out_dev)
    if rank == 0:
        if extra is not None:
            line["extra"] = extra
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()
    return 0


def dump_outputs(path, out_dev):
    """What the last timed step returned to its caller - predictive mean and variance [B, M], LML [B] and status [B] of
    rank 0's windows - as float64 .npy files (8 * (2 * B * M + 2 * B) bytes), so that two builds can be compared output
    for output."""
    os.makedirs(path, exist_ok=True)
    for name, t in zip(("mean", "var", "lml", "status"), out_dev):
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy().astype(np.float64))


def run_extra(ctx, torch, rank, world, dev_in, out_dev):
    """Numbers for the configs the headline does not carry, so that the driver's records hold them (every rank takes
    part: configs[3] is sharded over the ranks, configs[4] is factored block-cyclically over them):
      configs[0]  one N=100 window, host buffers: ms per predict + look-ahead callback                 (rank 0)
      configs[2]  Kernel Selection sweep, 64 candidates x 4096 windows, N=256: LML+gradient per second   (rank 0)
      configs[3]  Monte-Carlo shard of 131072 windows per GPU, N=128: windows/s over all ranks
      configs[4]  one N=32768 window, blocked Cholesky over all ranks: ms
      fp32_mode   the headline workload in FP32 mode (3xTF32 variance phase): windows/s per GPU        (rank 0)."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import bench_configs as bc
    import bench_large as bl
    ex = {"configs": {}}
    try:
        if rank == 0:
            ex["configs"]["configs[0]"] = bc.single(ctx)
            ex["configs"]["configs[2]"] = bc.sweep(ctx, 1.0)
            # FP32 mode on the headline workload
            dx, dy, dxs, dth = dev_in
            ctx.set_precision("f32")
            for _ in range(2):
                ctx.predict(KERNEL, dth, dx, dy, dxs, out=out_dev)
            torch.cuda.synchronize()
            ctx.set_profiling(True)
            for kid in range(6):
                ctx.profile_read(kid, reset=True)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 5
            e0.record()
            for _ in range(reps):
                ctx.predict(KERNEL, dth, dx, dy, dxs, out=out_dev)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / reps
            var_ms, _ = ctx.profile_read(1)
            fit_ms, _ = ctx.profile_read(0)
            ctx.set_profiling(False)
            ctx.set_precision("f64")
            ex["fp32_mode"] = {"windows_per_s_per_gpu": B_PER_GPU / (ms * 1e-3), "ms_per_step": ms,
                               "var_phase_ms": var_ms / reps, "fit_phase_ms": fit_ms / reps,
                               "what": "cngp_config.precision = F32: FP64 factorisation + 3xTF32 mma.sync variance phase, "
                                       "1e-4 normwise (tests/test_gpu_fp32_mode.py)"}
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        r = bc.mc(ctx, 1.0, rank, world)
        if rank == 0:
            ex["configs"]["configs[3]"] = r
        r = bl.run(ctx, 32768, 2, rank, world)
        if rank == 0:
            ex["configs"]["configs[4]"] = r
    except Exception as e:      # the headline must survive a failing extra leg
        ex["error"] = repr(e)[:300]
    return ex


_RESULT_FD = None


def _claim_stdout():
    """The driver reads ONE JSON line from stdout.  Libraries write there too (NCCL prints its version banner on
    stdout at communicator creation), so file descriptor 1 is pointed at stderr for the run and the result line is
    written to the original stdout."""
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_RESULT_FD, data)


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "cpu_probe"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra.configs legs (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (float64; --impl ours only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path: it needs --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    if args.impl == "cpu_probe":      # bounded CPU-port sample for the cpu_baseline object of our arm
        cores = os.cpu_count() or 1
        thr, _ = cpu_port_throughput(1, cores)
        per_core = int(max(1, min(64, round(12.0 * thr / cores))))
        v, dt = cpu_port_throughput(per_core, cores)
        # the reference's own loop shape beside it: one predict call per test point (gp_slip_node.py:47-50)
        vp, dtp = cpu_port_throughput(2, cores, worker=_cpu_worker_pointwise)
        emit({"value": v, "unit": UNIT, "cores": cores, "kind": "port",
              "sample": f"{per_core * cores} windows of the same workload in {dt:.1f} s "
                        f"(oracle/gp_oracle.py, vectorised {M_TEST}-RHS dtrtrs), {cores} processes x 1 BLAS thread",
              "faithful_loop": {"value": vp, "unit": UNIT,
                                "sample": f"{2 * cores} windows in {dtp:.1f} s with the reference's per-point loop "
                                          f"(one predict call per test point, gp_slip_node.py:47-50), same processes"}})
        return 0
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
