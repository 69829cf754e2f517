#!/usr/bin/env python
"""Time the large-window factorisation (BASELINE.json configs[4]) on one GPU or, under torchrun, block-cyclic over N GPUs.

    python tools/bench_large.py [N=32768] [reps=3]
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 tools/bench_large.py 32768 3

Prints one JSON line: seconds per factorisation (CUDA events, max over ranks), FP64 TFLOP/s on N^3/3, and the residual
||Ky alpha - y|| / ||y|| evaluated with cngp_large_matvec.

    python tools/bench_large.py [N [reps [lookahead]]] --predict [M=600]

adds the predict pass at M test points (the callback's horizon by default) from the same factor, timed apart from the
factorisation: ms per pass, the update GEMM alone and its FP64 TFLOP/s, and the payload bytes each pass broadcasts."""
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


def main():
    argv = list(sys.argv[1:])
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
