"""Ragged recorder windows through the GP callback and the stop look-ahead on one GPU (cngp_*_ragged).

Workload: 4096 rows of cngp_slip_record_batch output (2048 synthetic drives with paused drive commands x 2 windows,
cap 150), every published window kept at its own length.  Timed with CUDA events around the calls, after one warm-up of every shape:
  * gp_slip_ragged with fixed theta, with the fit (theta = None), and the look-ahead on its output;
  * the same windows through the fixed-shape path available before: grouped by exact (n, span), one
    cngp_gp_slip_batch per group (host memory, as that entry point takes);
  * a batch in which every window has n = 149: gp_slip_ragged and cngp_gp_slip_batch alternated in one process.
Algorithmic flop per window (SURVEY.md 8d, as tools/bench_configs.py counts configs[3]): N^3/3 + 2N^2 + 2NM + N^2 M + 2NM
with N = int(0.9 n_b), M = m_b of each window; the fit's optimiser iterations are not counted.  The look-ahead counts
2 x 2 x 15^3 flop per executed step (P = F P F' + Q).  Writes profiles/bench_ragged_<rev>.json.

Usage: python tools/bench_ragged.py [--reps 5] [--out profiles]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from corenav_gp_b200 import synthetic as syn  # noqa: E402
from corenav_gp_b200.api import GpContext  # noqa: E402

KERNEL = "rbf*brownian"
CAP, W = 150, 2


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def revision():
    try:
        return subprocess.run(["git", "rev-parse", "--short", "HEAD"], capture_output=True, text=True, cwd=ROOT).stdout.strip() or "worktree"
    except Exception:
        return "worktree"


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), [float(t) for t in ts]


def gp_flop(ntr, m):
    N, M = ntr.astype(np.float64), m.astype(np.float64)
    return float(np.sum(N ** 3 / 3 + 2 * N * N + 2 * N * M + N * N * M + 2 * N * M))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--rev", default=None, help="git revision to record (default: git rev-parse of the tree)")
    args = ap.parse_args()
    card = gpu_info()
    ctx = GpContext(0)
    th = syn.theta_for(KERNEL)
    th_d = torch.from_numpy(th).cuda()
    d = syn.drives(0, 2048, T=420, pauses=True)
    dev = {k: torch.from_numpy(v).cuda() for k, v in d.items()}
    rec = ctx.slip_record(dev["joint"], dev["att"], dev["vel"], dev["cmd"], dev["stop_cmd"], max_windows=W, cap=CAP)
    if int(rec["n_samples"].max()) > CAP:
        raise SystemExit("a window exceeded cap: it would be cut, not measured")
    n = torch.where(rec["published"] != 0, rec["n_samples"], torch.zeros_like(rec["n_samples"])).reshape(-1).to(torch.int32)
    t, s = rec["time_array"].reshape(-1, CAP).contiguous(), rec["slip_array"].reshape(-1, CAP).contiguous()
    B = n.numel()
    mc = syn.monte_carlo_contexts(0, B)
    cdev = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in mc.items()}
    nh = n.cpu().numpy()
    live = nh > 0
    res = {"card": card, "revision": args.rev or revision(), "kernel": KERNEL, "rows": B, "published": int(live.sum()),
           "n_min": int(nh[live].min()), "n_max": int(nh[live].max()), "distinct_n": int(len(set(nh[live].tolist())))}

    out = {}

    def fixed():
        out["r"] = ctx.gp_slip_ragged(KERNEL, t, s, n, theta=th_d)

    def fitted():
        out["f"] = ctx.gp_slip_ragged(KERNEL, t, s, n)

    ms, all_ms = timed(fixed, args.reps)
    mean, sigma, m_out, _ = out["r"]
    mh = m_out.cpu().numpy()
    ntr = (0.9 * nh[live]).astype(np.int64)
    fl = gp_flop(ntr, mh[live])
    res["gp_slip_ragged_fixed_theta"] = {"ms": ms, "all_ms": all_ms, "windows_per_s": live.sum() / (ms * 1e-3),
                                         "gflop": fl * 1e-9, "tflops_fp64": fl / (ms * 1e-3) * 1e-12}
    ms, all_ms = timed(fitted, max(1, args.reps // 2))
    res["gp_slip_ragged_with_fit"] = {"ms": ms, "all_ms": all_ms, "windows_per_s": live.sum() / (ms * 1e-3),
                                      "prediction_tflops_fp64": fl / (ms * 1e-3) * 1e-12}

    def look():
        out["la"] = ctx.zupt_lookahead(mean, sigma, cdev["P"], cdev["Q"], cdev["STM"], cdev["Hvec"], cdev["pos"], m=m_out)

    ms, all_ms = timed(look, args.reps)
    steps = int(out["la"]["step_stop"].sum().item())
    lf = 4.0 * 15 ** 3 * steps
    res["lookahead_ragged"] = {"ms": ms, "all_ms": all_ms, "windows_per_s": B / (ms * 1e-3), "steps": steps,
                               "tflops_fp64": lf / (ms * 1e-3) * 1e-12,
                               "triggered": int(out["la"]["triggered"].sum().item())}

    # the path available before: group by exact (n, span), one cngp_gp_slip_batch per group (host arrays)
    th_np, sh_np = t.cpu().numpy(), s.cpu().numpy()
    groups = {}
    for b in np.nonzero(live)[0]:
        k = nh[b]
        span = int(np.ceil(th_np[b, :k].max() + 600 - th_np[b, :k].min()))
        groups.setdefault((int(k), span), []).append(b)
    packed = [(np.ascontiguousarray(th_np[idx, :k]), np.ascontiguousarray(sh_np[idx, :k])) for (k, _), idx in
              ((key, np.array(v)) for key, v in groups.items())]

    def grouped():
        for tt, ss in packed:
            ctx.gp_slip(KERNEL, tt, ss, theta=th)

    t0 = time.perf_counter()
    grouped()
    ms_g = (time.perf_counter() - t0) * 1e3
    res["grouped_gp_slip_batch_fixed_theta"] = {"groups": len(packed), "ms": ms_g,
                                                "windows_per_s": live.sum() / (ms_g * 1e-3),
                                                "tflops_fp64": fl / (ms_g * 1e-3) * 1e-12}

    # every window n = 149: ragged vs the fixed-shape call, alternated
    xb, yb = syn.slip_windows(0, 4096, 149)
    xb = xb + 10.0 * (np.arange(4096) % 7)[:, None]
    nb = np.full(4096, 149, np.int32)
    rag, bat = [], []
    for _ in range(args.reps):
        t0 = time.perf_counter()
        ctx.gp_slip(KERNEL, xb, yb, theta=th)
        bat.append((time.perf_counter() - t0) * 1e3)
        t0 = time.perf_counter()
        ctx.gp_slip_ragged(KERNEL, xb, yb, nb, theta=th)
        rag.append((time.perf_counter() - t0) * 1e3)
    res["equal_n149_B4096"] = {"gp_slip_batch_ms": bat, "gp_slip_ragged_ms": rag,
                               "note": "host arrays on both sides; host clock around each call (both return after "
                                       "their copy-out)"}
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, f"bench_ragged_{res['revision']}.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
