"""The Toeplitz path of phase A (csrc/gp_fit_toeplitz.cuh, DESIGN.md section 4.1).

Windows with uniform integer stamps and a stationary expression have a Toeplitz Ky; gp_fit_toeplitz_kernel factors them
with the Schur algorithm and gp_fit_kernel takes every other window.  These tests hold the Toeplitz path to the oracle and
to the lazy evaluators (CNGP_NO_LAG_TABLES=1 sends every window to the tile Cholesky), check that the split of a batch
between the two kernels does not change any window's bits, and that the windows the Schur recursion must not take
(ill-conditioned, not positive definite) come out as they do on the tile path.  The Schur path runs for batches of more
problems than SMs (below that the tile kernel is faster), so every batch here has more than 148 windows; the oracle is
run on a few of them."""
import numpy as np
import pytest

from corenav_gp_b200 import synthetic as syn
from corenav_gp_b200.api import GpContext
from oracle import gp_oracle as go

pytestmark = pytest.mark.gpu
TOL = 1e-9
B_MIN = 160          # > the B200's 148 SMs: the batch takes the Schur path
ORACLE_WINDOWS = (0, 1, B_MIN - 1)

FAMILIES = [
    ("rbf", [0.01, 10.0]),
    ("rbf+stdperiodic", [0.01, 10.0, 0.0025, 37.0, 1.0]),
    ("mat32+bias", [0.02, 7.0, 0.001]),
    ("mat52+white", [0.5, 15.0, 1e-4]),
    ("ratquad+stdperiodic*rbf", [0.01, 8.0, 1.5, 0.5, 37.0, 1.2, 0.01, 50.0]),
]


def relerr(a, ref):
    a, ref = np.asarray(a, dtype=float), np.asarray(ref, dtype=float)
    scale = max(float(np.max(np.abs(ref))), 1e-300)
    return float(np.max(np.abs(a - ref) / np.maximum(np.abs(ref), 1e-3 * scale)))


def predict_both(ctx, kname, th, x, y, xs, monkeypatch):
    monkeypatch.delenv("CNGP_NO_LAG_TABLES", raising=False)
    out = ctx.predict(kname, th, x, y, xs)
    monkeypatch.setenv("CNGP_NO_LAG_TABLES", "1")
    lazy = ctx.predict(kname, th, x, y, xs)
    monkeypatch.delenv("CNGP_NO_LAG_TABLES", raising=False)
    return out, lazy


def uniform_windows(first, B, N, M):
    """B windows on uniform integer stamps (each window shifted by a few counts) and their test grids"""
    x, y = syn.slip_windows(first, B, N)
    x = x + 2.0 * (np.arange(B) % 7)[:, None]
    xs = np.stack([syn.test_grid(x[b], M) for b in range(B)])
    return x, y, xs


def check_oracle(kname, th, x, y, xs, mean, var, lml, tol=TOL, windows=ORACLE_WINDOWS):
    e = go.KernelExpr(kname)
    for b in windows:
        xsb = xs if xs.ndim == 1 else xs[b]
        inf = go.inference(e, th[:-1], th[-1], x[b], y[b])
        mu, v = go.predict(e, th[:-1], th[-1], x[b], y[b], xsb, inf)
        assert relerr(mean[b], mu) < tol and relerr(var[b], v) < tol and relerr(lml[b], inf.lml) < tol, (kname, b)


@pytest.mark.parametrize("kname,theta", FAMILIES)
@pytest.mark.parametrize("N,M", [(256, 600), (255, 601), (100, 600), (37, 13), (8, 20)])
def test_uniform_windows_match_oracle_and_tile_path(gp_ctx, monkeypatch, kname, theta, N, M):
    x, y, xs = uniform_windows(31, B_MIN, N, M)
    th = np.array(theta + [1e-3])
    (mean, var, lml, status), (mean0, var0, lml0, status0) = predict_both(gp_ctx, kname, th, x, y, xs, monkeypatch)
    assert np.all(status == 0) and np.all(status0 == 0)
    check_oracle(kname, th, x, y, xs, mean, var, lml)
    assert relerr(mean, mean0) < 1e-10 and relerr(var, var0) < 1e-10 and relerr(lml, lml0) < 1e-10


def test_stride_two_stamps(gp_ctx, monkeypatch):
    """Uniform stamps with step d = 2: Ky is Toeplitz in the lags 0, 2, 4, ..."""
    N, M = 128, 300
    x, y = syn.slip_windows(3, B_MIN, N)
    x = x[:, :1] + 2.0 * np.arange(N)[None, :]
    xs = np.stack([x[b, -1] + 1.0 + np.arange(M) for b in range(B_MIN)])
    th = syn.theta_for("rbf+stdperiodic")
    (mean, var, lml, status), (mean0, var0, lml0, _) = predict_both(gp_ctx, "rbf+stdperiodic", th, x, y, xs, monkeypatch)
    assert np.all(status == 0)
    check_oracle("rbf+stdperiodic", th, x, y, xs, mean, var, lml)
    assert relerr(mean, mean0) < 1e-10 and relerr(var, var0) < 1e-10 and relerr(lml, lml0) < 1e-10


def test_mixed_batch_gives_each_window_its_own_bits(gp_ctx):
    """Uniform (Toeplitz kernel), gapped and fractional (tile kernel) windows in one batch: every window's phase A
    results (LML, status, LML gradient) have the bits they have in a batch of its own kind.  Mean and variance agree to
    rounding: a batch with any window off the lag table runs phase B on the lazy evaluators for all of its windows."""
    rng = np.random.default_rng(11)
    B, N, M = 3 * B_MIN, 200, 300
    x, y = syn.slip_windows(40, B, N)
    for b in range(1, B, 3):   # gaps of 1..3 counts
        x[b] = x[b, 0] + np.concatenate([[0.0], np.cumsum(rng.integers(1, 4, N - 1))]).astype(float)
    for b in range(2, B, 3):   # fractional stamps
        x[b] = x[b] + 0.25
    xs = np.stack([np.floor(x[b, -1]) + 1.0 + np.arange(M) for b in range(B)])
    kname = "rbf+stdperiodic"
    th = syn.theta_for(kname)
    full = gp_ctx.predict(kname, th, x, y, xs)
    full_g = gp_ctx.lml_grad(kname, th[None, :], x, y)
    assert np.all(full[3] == 0) and np.all(full_g[2] == 0)
    for group in (np.arange(0, B, 3), np.arange(1, B, 3), np.arange(2, B, 3)):
        part = gp_ctx.predict(kname, th, x[group], y[group], xs[group])
        assert np.array_equal(full[2][group], part[2]) and np.array_equal(full[3][group], part[3]), group
        assert relerr(full[0][group], part[0]) < 1e-10 and relerr(full[1][group], part[1]) < 1e-10, group
        part_g = gp_ctx.lml_grad(kname, th[None, :], x[group], y[group])
        assert np.array_equal(full_g[0][:, group], part_g[0]) and np.array_equal(full_g[2][:, group], part_g[2]), group
        assert relerr(full_g[1][:, group], part_g[1]) < 1e-12, group
    check_oracle(kname, th, x, y, xs, *full[:3], windows=range(6))


def test_ill_conditioned_uniform_window(gp_ctx):
    """stdperiodic at noise 1e-6 (cond(Ky) ~ 2e8) is below the conditioning guard and stays on the tile path: it has the
    bits of its mirror image (stamps and grid reflected about the first stamp: the same Ky and K*, but stamps that
    decrease, which the Schur path never takes).  Against the oracle it is as close as the tile Cholesky gets at this
    condition number (5.6e-6 measured on a B200)."""
    N, M = 256, 600
    x, y, xs = uniform_windows(0, B_MIN, N, M)
    th = np.array([1.0, 37.0, 1.0, 1e-6])
    mean, var, lml, status = gp_ctx.predict("stdperiodic", th, x, y, xs)
    x0 = x[:, :1]
    mirror = gp_ctx.predict("stdperiodic", th, 2.0 * x0 - x, y, 2.0 * x0 - xs)
    assert np.all(status == 0)
    for a, b in zip((mean, var, lml, status), mirror):
        assert np.array_equal(a, b)
    check_oracle("stdperiodic", th, x, y, xs, mean, var, lml, tol=1e-4)


@pytest.mark.parametrize("jitter", [False, True], ids=["plain", "jitter_retry"])
def test_non_pd_uniform_window_keeps_tile_path_status(monkeypatch, jitter):
    """A negative noise variance makes Ky indefinite: the Schur recursion meets |rho| >= 1, leaves the window to the tile
    Cholesky, and status and outputs are what the tile path gives without lag tables."""
    ctx = GpContext(device=0, jitter_retry=jitter)
    try:
        N, M = 64, 40
        x, y, xs = uniform_windows(5, B_MIN, N, M)
        th = np.array([0.01, 10.0, -0.005])
        (mean, var, lml, status), (mean0, var0, lml0, status0) = predict_both(ctx, "rbf", th, x, y, xs, monkeypatch)
        assert np.all(status != 0)
        assert np.array_equal(status, status0)
        assert np.array_equal(np.isnan(lml), np.isnan(lml0)) and np.all(np.isnan(lml))
        assert np.array_equal(np.isnan(mean), np.isnan(mean0)) and np.array_equal(np.isnan(var), np.isnan(var0))
    finally:
        ctx.close()


def test_fp32_mode_on_uniform_windows(gp_ctx32):
    N, M = 256, 600
    x, y, xs = uniform_windows(12, B_MIN, N, M)
    kname = "rbf+stdperiodic"
    th = syn.theta_for(kname)
    mean, var, lml, status = gp_ctx32.predict(kname, th, x, y, xs)
    assert np.all(status == 0)
    e = go.KernelExpr(kname)
    for b in ORACLE_WINDOWS:
        inf = go.inference(e, th[:-1], th[-1], x[b], y[b])
        mu, v = go.predict(e, th[:-1], th[-1], x[b], y[b], xs[b], inf)
        assert np.max(np.abs(mean[b] - mu)) < 1e-4 * np.max(np.abs(mu))
        assert np.max(np.abs(var[b] - v)) < 1e-4 * np.max(np.abs(v))
        assert abs(lml[b] - inf.lml) < 1e-4 * abs(inf.lml)


@pytest.mark.parametrize("kname,theta", [FAMILIES[1], FAMILIES[3]])
def test_lml_grad_on_uniform_windows(gp_ctx, kname, theta):
    B, N = B_MIN // 2, 256
    x, y = syn.slip_windows(17, B, N)
    x = x + 2.0 * (np.arange(B) % 7)[:, None]
    th = np.array(theta + [1e-3])[None, :] * np.array([[1.0], [1.15]])
    lml, grad, status = gp_ctx.lml_grad(kname, th, x, y)
    assert np.all(status == 0)
    e = go.KernelExpr(kname)
    for c in range(th.shape[0]):
        for b in (0, 1, B - 1):
            inf = go.inference(e, th[c, :-1], th[c, -1], x[b], y[b], want_grad=True)
            assert relerr(lml[c, b], inf.lml) < TOL
            assert relerr(grad[c, b], inf.grad) < 1e-8, (kname, c, b)
