"""GPU tests of the predict pass on the large window (cngp_large_predict_*, cngp_chol_large_predict, large.py
predict_large_distributed): mean and variance against the CPU oracle (GPy m.predict restated with scipy LAPACK in
oracle/gp_oracle.py), the same bits on every world size (ranks emulated as threads on one GPU), the factorisation left as
it was, and the full N = 32768 size through size-independent properties.

Tolerance: 1e-9 relative (north_star, FP64): |got - ref| / max(1, |ref|)."""
import threading

import numpy as np
import pytest
import torch

from corenav_gp_b200 import large
from corenav_gp_b200 import synthetic as syn
from oracle import gp_oracle as go

pytestmark = pytest.mark.gpu
TOL = 1e-9

KERNELS = [
    ("rbf*brownian", [0.01, 10.0, 0.05, 1e-2]),                   # deployed (gp_slip_node.py:31), non-stationary
    ("se+periodic", [0.01, 10.0, 0.0025, 37.0, 1.0, 1e-3]),       # the benchmark's kernel
    ("matern32+linear", [0.02, 7.0, 1e-7, 5e-3]),
]


def series(N, seed=5):
    x, y = syn.slip_windows(seed, 1, N)
    return x[0], y[0]


def xstar_points(x, target=900):
    """Before the first stamp, the node's grid arange(min, max + horizon) (thinned to about `target` points), between
    stamps and on them."""
    grid = go.prediction_grid(x)
    step = max(1, len(grid) // target)
    return np.concatenate([x.min() - np.array([7.5, 1.0]), grid[::step], x[::97] + 0.5, x[::61]])


def relmax(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.max(np.abs(a - b) / np.maximum(1.0, np.abs(b))))


def oracle(kname, th, x, y, xs):
    return go.predict(go.KernelExpr(kname), th[:-1], th[-1], x, y, xs)


@pytest.mark.parametrize("N", [200, 300, 1500, 4096])
@pytest.mark.parametrize("kname,theta", KERNELS)
def test_predict_matches_oracle(gp_ctx, kname, theta, N):
    x, y = series(N)
    th = np.array(theta)
    xs = xstar_points(x)
    out = gp_ctx.chol_large_predict(kname, th, x, y, xs)
    assert out["pivot"] == 0
    mu, var = oracle(kname, th, x, y, xs)
    assert relmax(out["mean"], mu) < TOL
    assert relmax(out["var"], var) < TOL


@pytest.mark.parametrize("M", [1, 7, 8, 600, 1000])
def test_predict_test_point_counts(gp_ctx, M):
    kname, theta = KERNELS[0]
    x, y = series(1500)
    th = np.array(theta)
    xs = np.linspace(x[0] - 3.0, x[-1] + 600.0, M)
    out = gp_ctx.chol_large_predict(kname, th, x, y, xs)
    mu, var = oracle(kname, th, x, y, xs)
    assert out["mean"].shape == (M,) and relmax(out["mean"], mu) < TOL and relmax(out["var"], var) < TOL


def test_variance_floor(gp_ctx):
    """Test points on the training stamps with a tiny signal and tiny noise: k** - sum W^2 falls under 1e-15 and is
    clipped there before the noise is added (GPy posterior.py)."""
    x, y = series(300)
    th = np.array([1e-18, 10.0, 1e-12])
    xs = np.concatenate([x, x[:50] + 0.5])
    out = gp_ctx.chol_large_predict("rbf", th, x, y, xs)
    mu, var = oracle("rbf", th, x, y, xs)
    assert np.all(out["var"] == 1e-15 + 1e-12) and np.all(var == out["var"])
    assert np.max(np.abs(out["mean"] - mu)) < TOL * max(1e-30, np.max(np.abs(mu)))


def test_factor_once_predict_many(gp_ctx):
    """The factorisation is the same with and without predict passes after it, and two passes on one factored window
    give exactly what two one-call predicts give."""
    kname, theta = KERNELS[1]
    th = np.array(theta)
    x, y = series(1800)
    xs1, xs2 = xstar_points(x), x[-1] + 1.0 + np.arange(600.0)
    ref = gp_ctx.chol_large(kname, th, x, y, want_alpha=True)
    one1 = gp_ctx.chol_large_predict(kname, th, x, y, xs1)
    one2 = gp_ctx.chol_large_predict(kname, th, x, y, xs2)
    for key in ("logdet", "quad", "lml"):
        assert one1[key] == ref[key] and one2[key] == ref[key]
    out = large.chol_large(gp_ctx, kname, th, x, y)
    win = out["window"]
    alpha0 = win.alpha.clone()
    assert out["logdet"] == ref["logdet"] and out["quad"] == ref["quad"]
    p1 = large.predict_large_distributed(win, xs1, 0, 1)
    p2 = large.predict_large_distributed(win, xs2, 0, 1)
    torch.cuda.synchronize()
    assert torch.equal(win.alpha, alpha0) and np.array_equal(alpha0[: len(x)].cpu().numpy(), ref["alpha"])
    assert np.array_equal(p1["mean"].cpu().numpy(), one1["mean"]) and np.array_equal(p1["var"].cpu().numpy(), one1["var"])
    assert np.array_equal(p2["mean"].cpu().numpy(), one2["mean"]) and np.array_equal(p2["var"].cpu().numpy(), one2["var"])


def test_host_and_device_pointers(gp_ctx):
    kname, theta = KERNELS[2]
    th = np.array(theta)
    x, y = series(1000)
    xs = xstar_points(x)
    host = gp_ctx.chol_large_predict(kname, th, x, y, xs)
    dev = gp_ctx.chol_large_predict(kname, th, torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(),
                                    torch.from_numpy(xs).cuda())
    assert host["lml"] == dev["lml"]
    assert np.array_equal(host["mean"], dev["mean"].cpu().numpy()) and np.array_equal(host["var"], dev["var"].cpu().numpy())


def test_not_positive_definite(gp_ctx):
    from corenav_gp_b200.api import CngpError
    x, y = series(600)
    th = np.array([1.0, 50.0, -0.5])                    # negative noise: Ky indefinite
    xs = x[-1] + 1.0 + np.arange(20.0)
    with pytest.raises(CngpError, match="positive definite at pivot") as e:
        gp_ctx.chol_large("rbf", th, x, y)
    pivot = int(str(e.value).rsplit(" ", 1)[1])
    out = gp_ctx.chol_large_predict("rbf", th, x, y, xs)
    assert out["pivot"] == pivot and np.all(np.isnan(out["mean"])) and np.all(np.isnan(out["var"]))
    assert np.isnan(out["lml"])
    fac = large.chol_large(gp_ctx, "rbf", th, x, y)
    p = large.predict_large_distributed(fac["window"], xs, 0, 1)
    assert fac["pivot"] == pivot and p["pivot"] == pivot
    assert torch.isnan(p["mean"]).all() and torch.isnan(p["var"]).all() and p["mean"].shape == (20,)


class ThreadCollectives:
    """In-process stand-in for the NCCL broadcast / all-reduce: `world` ranks are threads sharing one GPU."""

    class _Done:
        def wait(self):
            return True

    def __init__(self, world):
        self.world = world
        self.bar = threading.Barrier(world)
        self.slot = {}
        self.lock = threading.Lock()

    def for_rank(self, rank):
        parent = self

        class C:
            def broadcast_async(self, t, src):
                torch.cuda.synchronize()
                if rank == src:
                    parent.slot["b"] = t
                parent.bar.wait()
                if rank != src:
                    t.copy_(parent.slot["b"])
                torch.cuda.synchronize()
                parent.bar.wait()
                return ThreadCollectives._Done()

            def _reduce(self, t, op):
                torch.cuda.synchronize()
                with parent.lock:
                    parent.slot.setdefault("r", []).append(t.clone())
                parent.bar.wait()
                parts = torch.stack(parent.slot["r"])
                res = parts.sum(0) if op == "sum" else parts.max(0).values
                parent.bar.wait()
                if rank == 0:
                    parent.slot["r"] = []
                parent.bar.wait()
                t.copy_(res)

            def all_reduce_sum(self, t):
                self._reduce(t, "sum")

            def all_reduce_max(self, t):
                self._reduce(t, "max")

        return C()


def run_ranks(world, kname, th, x, y, xs, lookahead):
    from corenav_gp_b200.api import GpContext
    coll = ThreadCollectives(world)
    outs, errs = [None] * world, []

    def body(rank):
        try:
            torch.cuda.set_device(0)
            ctx = GpContext(device=0)
            with torch.cuda.stream(torch.cuda.Stream()):
                c = coll.for_rank(rank)
                fac = large.chol_large(ctx, kname, th, x, y, rank=rank, world=world, coll=c, lookahead=lookahead)
                o = large.predict_large_distributed(fac["window"], xs, rank, world, coll=c, lookahead=lookahead)
                torch.cuda.synchronize()
            outs[rank] = dict(mean=o["mean"].cpu().numpy(), var=o["var"].cpu().numpy(), pivot=o["pivot"])
            del fac
            ctx.close()
        except Exception as e:  # pragma: no cover
            errs.append(e)
            coll.bar.abort()

    ts = [threading.Thread(target=body, args=(r,)) for r in range(world)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    if errs:
        raise errs[0]
    return outs


@pytest.mark.parametrize("world,N", [(2, 1500), (3, 2048), (8, 1300)])
def test_block_cyclic_ranks_equal_single_gpu(gp_ctx, world, N):
    """Every R(:, c) is written by one rank in increasing k, so every rank's mean and var equal the one-GPU entry point
    bit for bit, with and without the look-ahead.  (8 ranks at N = 1300: ranks 6 and 7 own no block column.)"""
    kname, theta = KERNELS[0]
    th = np.array(theta)
    x, y = series(N)
    xs = xstar_points(x, 500)
    single = gp_ctx.chol_large_predict(kname, th, x, y, xs)
    for look in (True, False):
        for o in run_ranks(world, kname, th, x, y, xs, look):
            assert o["pivot"] == 0
            assert np.array_equal(o["mean"], single["mean"]) and np.array_equal(o["var"], single["var"])


def test_full_size_properties(gp_ctx):
    """N = 32768 (configs[4]), M = 600: at training stamps K(x*, x) alpha = y - (noise + 1e-8) alpha, with alpha checked
    through the residual of Ky alpha = y; everywhere var >= noise."""
    N, M = 32768, 600
    kname, theta = KERNELS[1]
    th = np.array(theta)
    x, y = series(N)
    dx, dy = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    fac = large.chol_large(gp_ctx, kname, th, dx, dy)
    alpha = fac["alpha"].contiguous()
    r = gp_ctx.large_matvec(kname, th, dx, alpha)
    assert float(torch.linalg.norm(r - dy) / torch.linalg.norm(dy)) < 1e-9
    idx = np.linspace(0, N - 1, M // 2).astype(np.int64)
    xs = np.concatenate([x[idx], x[-1] + 1.0 + np.arange(M - M // 2)])
    out = large.predict_large_distributed(fac["window"], xs, 0, 1)
    mean, var = out["mean"].cpu().numpy(), out["var"].cpu().numpy()
    al = alpha.cpu().numpy()
    expect = y[idx] - (th[-1] + 1e-8) * al[idx]
    assert relmax(mean[: M // 2], expect) < TOL
    assert np.all(var >= th[-1]) and np.all(np.isfinite(mean))
