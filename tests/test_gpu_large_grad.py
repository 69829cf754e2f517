"""GPU tests of the LML gradient pass on the large window (cngp_large_grad_*, cngp_chol_large_grad, large.py
lml_grad_large_distributed): the gradient and the LML against the CPU oracles, the same bits on every world size (ranks
emulated as threads on one GPU), the factorisation left as it was, and the full N = 32768 size against a central
difference of the factorisation's own LML.

Tolerance: 1e-9 relative (north_star, FP64): |got - ref| / max(1, |ref|).  Up to N = 1000 the reference is the
extended-precision oracle (oracle/xp_oracle.py); beyond, float64 gp_oracle.  Measured on CPU on these fixtures, float64
gp_oracle is within 5e-15 of xp_oracle for rbf*brownian and matern32+linear at N <= 1000; for se+periodic the gap is
4.8e-13 at N = 600, 3.6e-12 at N = 1000 and 1.5e-12 at N = 1500 (1.0e-13 for matern32+linear) - far inside
the tolerance."""
import threading

import numpy as np
import pytest
import torch

from corenav_gp_b200 import large
from oracle import gp_oracle as go
from test_gpu_large_predict import KERNELS, ThreadCollectives, relmax, series, xstar_points

pytestmark = pytest.mark.gpu
TOL = 1e-9


def oracle(kname, th, x, y, xp=False):
    if xp:
        from oracle import xp_oracle
        inf = xp_oracle.inference(go.KernelExpr(kname), th[:-1], th[-1], x, y, want_grad=True)
        return float(inf.lml), np.asarray(inf.grad, dtype=np.float64)
    inf = go.inference(go.KernelExpr(kname), th[:-1], th[-1], x, y, want_grad=True)
    return inf.lml, inf.grad


@pytest.mark.parametrize("N", [200, 300, 1000, 1500, 4096])
@pytest.mark.parametrize("kname,theta", KERNELS)
def test_grad_matches_oracle(gp_ctx, kname, theta, N):
    x, y = series(N)
    th = np.array(theta)
    out = gp_ctx.chol_large_grad(kname, th, x, y)
    assert out["pivot"] == 0 and out["grad"].shape == (len(th),)
    lml, grad = oracle(kname, th, x, y, xp=N <= 1000)
    assert relmax(out["grad"], grad) < TOL
    assert relmax([out["lml"]], [lml]) < TOL


def run_ranks(world, kname, th, x, y, lookahead):
    """Factor and run the gradient pass on `world` thread ranks; returns every rank's results."""
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
                g = large.lml_grad_large_distributed(fac["window"], rank, world, coll=c, lookahead=lookahead)
                torch.cuda.synchronize()
            outs[rank] = dict(grad=g["grad"].cpu().numpy(), pivot=g["pivot"])
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


@pytest.mark.parametrize("world,N", [(1, 1500), (2, 1500), (3, 2048), (8, 1300)])
def test_block_cyclic_ranks_equal_single_gpu(gp_ctx, world, N):
    """Every R(:, c) and G(:, c) is written by one rank in increasing k and the parts are added in increasing block
    column, so every rank's gradient equals the one-GPU entry point bit for bit, with and without the look-ahead.
    (8 ranks at N = 1300: ranks 6 and 7 own no block column.)"""
    kname, theta = KERNELS[0]
    th = np.array(theta)
    x, y = series(N)
    single = gp_ctx.chol_large_grad(kname, th, x, y)
    for look in (True, False):
        for o in run_ranks(world, kname, th, x, y, look):
            assert o["pivot"] == 0 and np.array_equal(o["grad"], single["grad"])


def test_factor_reuse_predict_and_grad(gp_ctx):
    """A gradient pass leaves the factorisation as it was: predict before and after it gives the same bits, two gradient
    passes are bit-equal and equal the one-call entry point."""
    kname, theta = KERNELS[1]
    th = np.array(theta)
    x, y = series(1800)
    xs = xstar_points(x)
    one = gp_ctx.chol_large_grad(kname, th, x, y)
    out = large.chol_large(gp_ctx, kname, th, x, y)
    win = out["window"]
    assert out["lml"] == one["lml"] and out["logdet"] == one["logdet"] and out["quad"] == one["quad"]
    A0, winv0, alpha0 = win.A.clone(), win.winv.clone(), win.alpha.clone()
    p1 = large.predict_large_distributed(win, xs, 0, 1)
    g1 = large.lml_grad_large_distributed(win, 0, 1)
    p2 = large.predict_large_distributed(win, xs, 0, 1)
    g2 = large.lml_grad_large_distributed(win, 0, 1, lookahead=False)
    torch.cuda.synchronize()
    assert torch.equal(win.A, A0) and torch.equal(win.winv, winv0) and torch.equal(win.alpha, alpha0)
    assert torch.equal(p1["mean"], p2["mean"]) and torch.equal(p1["var"], p2["var"])
    assert torch.equal(g1["grad"], g2["grad"]) and np.array_equal(g1["grad"].cpu().numpy(), one["grad"])


def test_host_and_device_pointers(gp_ctx):
    kname, theta = KERNELS[2]
    th = np.array(theta)
    x, y = series(1000)
    host = gp_ctx.chol_large_grad(kname, th, x, y)
    dev = gp_ctx.chol_large_grad(kname, th, torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda())
    assert isinstance(dev["grad"], torch.Tensor) and dev["grad"].is_cuda
    assert host["lml"] == dev["lml"] and np.array_equal(host["grad"], dev["grad"].cpu().numpy())


def test_not_positive_definite(gp_ctx):
    from corenav_gp_b200.api import CngpError
    x, y = series(600)
    th = np.array([1.0, 50.0, -0.5])                    # negative noise: Ky indefinite
    with pytest.raises(CngpError, match="positive definite at pivot") as e:
        gp_ctx.chol_large("rbf", th, x, y)
    pivot = int(str(e.value).rsplit(" ", 1)[1])
    out = gp_ctx.chol_large_grad("rbf", th, x, y)
    assert out["pivot"] == pivot and np.all(np.isnan(out["grad"])) and np.isnan(out["lml"])
    fac = large.chol_large(gp_ctx, "rbf", th, x, y)
    g = large.lml_grad_large_distributed(fac["window"], 0, 1)
    assert fac["pivot"] == pivot and g["pivot"] == pivot
    assert torch.isnan(g["grad"]).all() and g["grad"].shape == (3,)


def test_full_size_central_difference(gp_ctx):
    """N = 32768 (configs[4]) with the deployed rbf*brownian: theta_p dLML/dtheta_p against the central difference
    (LML(theta_p e^h) - LML(theta_p e^-h)) / 2h of the factorisation's own LML, h = 1e-3.  The truncation error is
    O(h^2) relative; the tolerance is 1e-5 of max(1, |difference|)."""
    N, h = 32768, 1e-3
    kname, theta = KERNELS[0]
    th = np.array(theta)
    x, y = series(N)
    dx, dy = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    fac = large.chol_large(gp_ctx, kname, th, dx, dy)
    g = large.lml_grad_large_distributed(fac["window"], 0, 1)["grad"].cpu().numpy()
    del fac
    assert np.all(np.isfinite(g))
    for p in range(len(th)):
        lp, lm = th.copy(), th.copy()
        lp[p] *= np.exp(h)
        lm[p] *= np.exp(-h)
        fd = (gp_ctx.chol_large(kname, lp, dx, dy)["lml"] - gp_ctx.chol_large(kname, lm, dx, dy)["lml"]) / (2 * h)
        assert abs(th[p] * g[p] - fd) < 1e-5 * max(1.0, abs(fd)), (p, th[p] * g[p], fd)
