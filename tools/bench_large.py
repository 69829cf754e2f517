#!/usr/bin/env python
"""Time the large-window factorisation (BASELINE.json configs[4]) on one GPU or, under torchrun, block-cyclic over N GPUs.

    python tools/bench_large.py [N=32768] [reps=3]
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 tools/bench_large.py 32768 3

Prints one JSON line: seconds per factorisation (CUDA events, max over ranks), FP64 TFLOP/s on N^3/3, and the residual
||Ky alpha - y|| / ||y|| evaluated with cngp_large_matvec.

    python tools/bench_large.py [N [reps [lookahead]]] --predict [M=600]

adds the predict pass at M test points (the callback's horizon by default) from the same factor, timed apart from the
factorisation: ms per pass, the update GEMM alone and its FP64 TFLOP/s, and the payload bytes each pass broadcasts.

    python tools/bench_large.py [N [reps [lookahead]]] --grad

times the LML gradient pass instead, alternated with the factorisation on the same GPU: ms per pass and per
factorisation (best and median), the sweep GEMM and the SYRK launches alone with their FP64 TFLOP/s, the contraction,
and the payload bytes per pass."""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from corenav_gp_b200 import large, synthetic as syn  # noqa: E402
from corenav_gp_b200.api import GpContext  # noqa: E402


def run(ctx, N, reps, rank, world, lookahead=True):
    """Factor one N-point window `reps` + 1 times (first one untimed) on `world` ranks; returns the result dict on every
    rank (timings are the max over ranks)."""
    if world > 1:
        import torch.distributed as dist
    kname = "rbf+stdperiodic"
    th = np.array([0.01, 10.0, 0.0025, 37.0, 1.0, 1e-2])
    x, y = syn.slip_windows(5, 1, N)
    win = large.LargeWindow(ctx, kname, th, x[0], y[0], rank=rank, world=world)
    times = []
    host_ms = []
    out = None
    for it in range(reps + 1):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctx.set_profiling(it == reps)
        e0.record()
        out = large.chol_large_distributed(win, rank, world, want_alpha=True, lookahead=lookahead,
                                           profile=(it == reps and bool(os.environ.get("CNGP_LARGE_PHASES"))))
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if it > 0:
            times.append(float(t[0]))
            host_ms.append(out.get("host_enqueue_ms"))
    prof_ms, prof_n = ctx.profile_read(4)
    ctx.set_profiling(False)
    r = ctx.large_matvec(kname, th, win.x, out["alpha"].contiguous())
    res = float(torch.linalg.norm(r - win.y) / torch.linalg.norm(win.y))
    best = min(times)
    del win
    return {"N": N, "n_gpus": world, "lookahead": lookahead, "ms": times, "best_ms": best,
            "median_ms": float(np.median(times)), "chunk_rows": int(os.environ.get("CNGP_LARGE_CHUNK_ROWS", "0")),
            "tflops_n3_over_3": N ** 3 / 3.0 / (best * 1e-3) * 1e-12, "lml": out["lml"],
            "logdet": out["logdet"], "quad": out["quad"], "residual": res,
            "rank0_kernel_ms_last_rep": prof_ms, "rank0_launches_last_rep": prof_n,
            "host_enqueue_ms_per_rep": host_ms,
            "phase_ms_rank": {"rank": rank, **(out.get("phase_ms") or {})}}


def run_predict(ctx, N, M, reps, rank, world, lookahead=True):
    """Factor one N-point window once, then run the predict pass at M test points `reps` + 1 times (first one untimed)
    and the update GEMM of the pass on its own; times are the max over ranks."""
    if world > 1:
        import torch.distributed as dist
    kname = "rbf+stdperiodic"
    th = np.array([0.01, 10.0, 0.0025, 37.0, 1.0, 1e-2])
    x, y = syn.slip_windows(5, 1, N)
    xs = syn.test_grid(x[0], M)
    win = large.LargeWindow(ctx, kname, th, x[0], y[0], rank=rank, world=world)
    large.chol_large_distributed(win, rank, world, want_alpha=True, lookahead=lookahead)

    def timed(fn):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), r

    times, out = [], None
    for it in range(reps + 1):
        ctx.set_profiling(it == reps)
        t, out = timed(lambda: large.predict_large_distributed(win, xs, rank, world, lookahead=lookahead))
        if it > 0:
            times.append(t)
    prof_ms, prof_n = ctx.profile_read(4)
    ctx.set_profiling(False)
    nblk = win.n_blockcols
    # the update GEMM alone, on whatever R holds (its time does not depend on the values): every rank's own columns
    upd = []
    for _ in range(reps):
        t, _ = timed(lambda: [win.predict_update(k, k + 1, nblk) for k in range(nblk)])
        upd.append(t)
    m_rows = -(-M // 128) * 128                                                           # R rows, padded
    n_pad = win.n_pad
    upd_flop = sum(2.0 * m_rows * 256 * 256 * (nblk - k - 1) for k in range(nblk))      # executed, padded rows
    useful_flop = float(N) * N * M                                                         # 2 M sum_k 256 (N - 256 (k+1))
    payload_bytes = sum(win._pred_sizes(M, k)[1] * 8 for k in range(nblk))
    best = min(times)
    mean = out["mean"]
    del win
    return {"N": N, "M": M, "n_gpus": world, "lookahead": lookahead, "predict_ms": times, "predict_best_ms": best,
            "predict_median_ms": float(np.median(times)), "update_gemm_ms": upd, "update_gemm_best_ms": min(upd),
            "update_gemm_tflops": upd_flop / (min(upd) * 1e-3) * 1e-12, "update_gemm_flop": upd_flop,
            "useful_tflops_n2m_over_pass": useful_flop / (best * 1e-3) * 1e-12, "rows_padded_to": m_rows,
            "payload_bytes_per_pass": payload_bytes, "n_pad": n_pad,
            "rank0_kernel_ms_last_rep": prof_ms, "rank0_launches_last_rep": prof_n,
            "mean_finite": bool(torch.isfinite(mean).all())}


def run_grad(ctx, N, reps, rank, world, lookahead=True):
    """The LML gradient pass from the stored factor, alternated with the factorisation on the same GPU `reps` times
    (after one untimed round of each), then the pass's sweep GEMM, its accumulation (SYRK) launches and the contraction
    timed on their own; times are the max over ranks."""
    if world > 1:
        import torch.distributed as dist
    kname = "rbf+stdperiodic"
    th = np.array([0.01, 10.0, 0.0025, 37.0, 1.0, 1e-2])
    x, y = syn.slip_windows(5, 1, N)
    win = large.LargeWindow(ctx, kname, th, x[0], y[0], rank=rank, world=world)

    def timed(fn):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), r

    fac_ms, grad_ms, out, g = [], [], None, None
    for it in range(reps + 1):
        tf, out = timed(lambda: large.chol_large_distributed(win, rank, world, want_alpha=True, lookahead=lookahead))
        tg, g = timed(lambda: large.lml_grad_large_distributed(win, rank, world, lookahead=lookahead))
        if it > 0:
            fac_ms.append(tf)
            grad_ms.append(tg)
    nblk = win.n_blockcols
    # the pass's pieces on their own, on whatever RG and the payloads hold (their time does not depend on the values)
    sweep, syrk, contract = [], [], []
    for _ in range(reps):
        sweep.append(timed(lambda: [win.grad_update(k, k + 1, nblk) for k in range(nblk)])[0])
        syrk.append(timed(lambda: [win.grad_update(k, 0, k + 1) for k in range(nblk)])[0])
        contract.append(timed(win.grad_contract)[0])
    # executed flop (one rank's share is 1/world of it): sweep 2 x 256(k+1) x 256 x 256 per column c > k; SYRK one
    # 128 x 128 x 256 block product per lower 128-block of the (k+1) x (k+1) block triangle
    sweep_flop = sum(2.0 * 256 * (k + 1) * 256 * 256 * (nblk - k - 1) for k in range(nblk))
    syrk_flop = sum(2.0 * 128 * 128 * 256 * (2 * (k + 1)) * (2 * (k + 1) + 1) / 2 for k in range(nblk))
    payload_bytes = nblk * win.grad_payload(0).numel() * 8
    best, fbest = min(grad_ms), min(fac_ms)
    grad = g["grad"].cpu().numpy()
    del win
    return {"N": N, "n_gpus": world, "lookahead": lookahead, "kernel": kname, "theta": th.tolist(),
            "grad_ms": grad_ms, "grad_best_ms": best, "grad_median_ms": float(np.median(grad_ms)),
            "factor_ms_alternated": fac_ms, "factor_best_ms": fbest, "factor_median_ms": float(np.median(fac_ms)),
            "grad_over_factor_best": best / fbest,
            "grad_over_factor_median": float(np.median(grad_ms)) / float(np.median(fac_ms)),
            "sweep_gemm_ms": sweep, "sweep_gemm_tflops": sweep_flop / world / (min(sweep) * 1e-3) * 1e-12,
            "syrk_ms": syrk, "syrk_tflops": syrk_flop / world / (min(syrk) * 1e-3) * 1e-12,
            "sweep_flop": sweep_flop, "syrk_flop": syrk_flop, "contract_ms": contract,
            "payload_bytes_per_pass": payload_bytes, "lml": out["lml"], "grad": grad.tolist(),
            "grad_finite": bool(np.all(np.isfinite(grad)))}


def main():
    argv = list(sys.argv[1:])
    grad = "--grad" in argv
    if grad:
        argv.remove("--grad")
    M = None
    if "--predict" in argv:
        i = argv.index("--predict")
        M = 600
        if i + 1 < len(argv) and argv[i + 1].isdigit():
            M = int(argv.pop(i + 1))
        argv.pop(i)
    N = int(argv[0]) if len(argv) > 0 else 32768
    reps = int(argv[1]) if len(argv) > 1 else 3
    lookahead = (argv[2] != "0") if len(argv) > 2 else True
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    ctx = GpContext(device=local)
    if grad:
        line = run_grad(ctx, N, reps, rank, world, lookahead)
        line["device"] = torch.cuda.get_device_properties(local).name
        if rank == 0:
            print(json.dumps(line))
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        ctx.close()
        return
    line = run(ctx, N, reps, rank, world, lookahead)
    if M is not None:
        line["predict"] = run_predict(ctx, N, M, reps, rank, world, lookahead)
        line["predict"]["predict_over_factor"] = line["predict"]["predict_best_ms"] / line["best_ms"]
        props = torch.cuda.get_device_properties(local)
        line["device"] = props.name
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()


if __name__ == "__main__":
    main()
