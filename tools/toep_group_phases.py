"""Where the time of the shared-covariance predict goes on the bench workload (4096 windows, N = 256, M = 600,
rbf+stdperiodic, one theta).

Default: per-launch times from torch.profiler with CUDA activities; writes a JSON of the mean us per step of every
kernel, and prints them.
--lib LIB: run a timing build of the library instead, whose group kernels stamp %globaltimer at their phase boundaries
(csrc/gp_toep_group.cuh, CNGP_TG_TIMING) and print, per call, the group fit's phases (from its start) and the member
kernel's (from the start of its CTA 0: the variance row's end, the first member CTA's start, the last z and alpha
ends and the last member's end).  Built next to the product objects:
  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -DCNGP_TG_TIMING \
       -c corenav_gp_b200/csrc/cngp_api.cu -o build/timing/cngp_api.o
  nvcc -gencode arch=compute_100a,code=sm_100a -shared -o build/timing/libcngp.so build/timing/cngp_api.o \
       $(ls corenav_gp_b200/csrc/_obj/*.o | grep -v cngp_api) -lcudart
usage: python tools/toep_group_phases.py [--lib LIB] [out.json] [steps=20] [B=4096] [N=256]"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from torch.profiler import ProfilerActivity, profile

from corenav_gp_b200 import _lib

args = sys.argv[1:]
timing_lib = None
if args[:1] == ["--lib"]:
    timing_lib, args = os.path.abspath(args[1]), args[2:]
    _lib.LIB_PATH = timing_lib
from corenav_gp_b200 import synthetic as syn  # noqa: E402
from corenav_gp_b200.api import GpContext  # noqa: E402

out_path = args[0] if len(args) > 0 else None
steps = int(args[1]) if len(args) > 1 else 20
B = int(args[2]) if len(args) > 2 else 4096
N = int(args[3]) if len(args) > 3 else 256
M, kern = 600, "rbf+stdperiodic"

ctx = GpContext(0)
x, y = syn.slip_windows(0, B, N)
xs = syn.test_grid(x[0], M)
th = syn.theta_for(kern)
dx, dy, dxs, dth = (torch.from_numpy(a).cuda() for a in (x, y, xs, th))
out = (torch.empty(B, M, dtype=torch.float64, device="cuda"), torch.empty(B, M, dtype=torch.float64, device="cuda"),
       torch.empty(B, dtype=torch.float64, device="cuda"), torch.empty(B, dtype=torch.int32, device="cuda"))
for _ in range(5):
    ctx.predict(kern, dth, dx, dy, dxs, out=out)
torch.cuda.synchronize()
if timing_lib:
    for _ in range(steps):
        ctx.predict(kern, dth, dx, dy, dxs, out=out)
    torch.cuda.synchronize()
    ctx.close()
    sys.exit(0)
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(steps):
        ctx.predict(kern, dth, dx, dy, dxs, out=out)
    torch.cuda.synchronize()
rows = {}
for ev in prof.key_averages():
    t = getattr(ev, "device_time_total", None)
    if t is None:
        t = ev.cuda_time_total
    if t <= 0:
        continue
    rows[ev.key] = {"us_per_step": t / steps, "calls_per_step": ev.count / steps}
rows = dict(sorted(rows.items(), key=lambda kv: -kv[1]["us_per_step"]))
gpu = torch.cuda.get_device_name(0)
res = {"gpu": gpu, "B": B, "N": N, "M": M, "kernel": kern, "steps": steps,
       "sum_us_per_step": sum(r["us_per_step"] for r in rows.values()), "launches": rows}
for k, r in rows.items():
    print(f"{r['us_per_step']:9.1f} us  x{r['calls_per_step']:.0f}  {k[:110]}")
print(f"{res['sum_us_per_step']:9.1f} us  kernel time per step ({gpu})")
if out_path:
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
ctx.close()
