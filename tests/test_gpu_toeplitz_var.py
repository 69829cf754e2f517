"""The Toeplitz path of phase B (csrc/gp_var_toeplitz.cuh, DESIGN.md section 4.2c).

Windows on uniform integer stamps whose test points are consecutive points of the same lattice get their mean and
variance from the displacement recurrence; every other window goes to gp_var_kernel.  These tests hold the recurrence to
the oracle and to the lazy evaluators (CNGP_NO_LAG_TABLES=1 sends every window to gp_var_kernel), check that the grids the
recurrence does not take still come out right, that the split of a batch does not change any window's bits, and that a
window just below the conditioning guard stays on gp_var_kernel.  The path runs for batches of more windows than SMs, so
every batch here has more than 148 windows; the oracle is run on a few of them."""
import numpy as np
import pytest
import torch

from corenav_gp_b200 import synthetic as syn
from oracle import gp_oracle as go

pytestmark = pytest.mark.gpu
TOL = 1e-9
B_MIN = 160          # > the B200's 148 SMs
ORACLE_WINDOWS = (0, 1, B_MIN - 1)


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


def check_oracle(kname, th, x, y, xs, mean, var, tol=TOL, windows=ORACLE_WINDOWS):
    e = go.KernelExpr(kname)
    for b in windows:
        mu, v = go.predict(e, th[:-1], th[-1], x[b], y[b], xs[b])
        assert relerr(mean[b], mu) < tol and relerr(var[b], v) < tol, (kname, b, relerr(mean[b], mu), relerr(var[b], v))


def lattice_windows(B, N, d=1):
    x, y = syn.slip_windows(21, B, N)
    x = x[:, :1] + 3.0 * (np.arange(B) % 5)[:, None] + d * np.arange(N)[None, :]
    return x, y


def check_both(gp_ctx, monkeypatch, kname, th, x, y, xs):
    (mean, var, lml, status), (mean0, var0, lml0, status0) = predict_both(gp_ctx, kname, th, x, y, xs, monkeypatch)
    assert np.all(status == 0) and np.array_equal(status, status0)
    check_oracle(kname, th, x, y, xs, mean, var)
    assert relerr(mean, mean0) < 1e-10 and relerr(var, var0) < 1e-10
    return mean, var


@pytest.mark.parametrize("kname,theta", [
    ("rbf+stdperiodic", None),
    ("rbf", [0.01, 10.0, 1e-3]),
    ("mat32+bias", [0.02, 7.0, 0.001, 1e-3]),
    ("mat52+white", [0.5, 15.0, 1e-4, 1e-3]),   # below the guard: gp_var_kernel
    ("ratquad+stdperiodic*rbf", [0.01, 8.0, 1.5, 0.5, 37.0, 1.2, 0.01, 50.0, 1e-3]),
])
def test_benchmark_shape(gp_ctx, monkeypatch, kname, theta):
    """N = 256, M = 600, grid x_{N-1} + 1 + j: the chain starts at m0 = n-1"""
    th = syn.theta_for(kname) if theta is None else np.array(theta)
    x, y = lattice_windows(B_MIN, 256)
    xs = np.stack([syn.test_grid(x[b], 600) for b in range(B_MIN)])
    check_both(gp_ctx, monkeypatch, kname, th, x, y, xs)


@pytest.mark.parametrize("N", [256, 100, 9])
def test_reference_grid_from_first_stamp(gp_ctx, monkeypatch, N):
    """arange(min, max + 600): the grid starts at x_0, inside the training span (m0 = 0)"""
    kname = "rbf+stdperiodic"
    th = syn.theta_for(kname)
    x, y = lattice_windows(B_MIN, N)
    xs = np.stack([x[b, 0] + np.arange(N - 1 + 600, dtype=float) for b in range(B_MIN)])
    check_both(gp_ctx, monkeypatch, kname, th, x, y, xs)


@pytest.mark.parametrize("grid", ["lattice", "step1", "before_x0", "shuffled"])
def test_stride_two_and_off_lattice_grids(gp_ctx, monkeypatch, grid):
    """d = 2: a grid on the lattice is taken; a step-1 grid, a grid starting before x_0 and a permuted lattice grid fall
    back to gp_var_kernel.  All must match the oracle and the lazy path."""
    kname = "rbf+stdperiodic"
    th = syn.theta_for(kname)
    N, M = 128, 300
    x, y = lattice_windows(B_MIN, N, d=2)
    rng = np.random.default_rng(4)
    if grid == "lattice":
        xs = x[:, -1:] + 2.0 + 2.0 * np.arange(M)[None, :]
    elif grid == "step1":
        xs = x[:, -1:] + 1.0 + np.arange(M)[None, :]
    elif grid == "before_x0":
        xs = x[:, :1] - 20.0 + 2.0 * np.arange(M)[None, :]
    else:
        xs = x[:, -1:] + 2.0 + 2.0 * rng.permutation(M)[None, :]
    check_both(gp_ctx, monkeypatch, kname, th, x, y, np.ascontiguousarray(xs))


def test_ragged_counts(gp_ctx, monkeypatch):
    """per-window n and m: the recurrence honours both, and entries beyond m are not written"""
    kname = "rbf+stdperiodic"
    th = syn.theta_for(kname)
    B, ld, ldm = 2 * B_MIN, 256, 600
    rng = np.random.default_rng(8)
    x, y = lattice_windows(B, ld)
    n = rng.integers(200, ld + 1, B).astype(np.int32)
    m = rng.integers(1, ldm + 1, B).astype(np.int32)
    xs = np.stack([x[b, n[b] - 1] + 1.0 + np.arange(ldm, dtype=float) for b in range(B)])
    mean, var, lml, status = gp_ctx.predict_ragged(kname, th, x, y, n, xs, m)
    assert np.all(status == 0)
    e = go.KernelExpr(kname)
    for b in (0, 1, 2, B - 1):
        mu, v = go.predict(e, th[:-1], th[-1], x[b, :n[b]], y[b, :n[b]], xs[b, :m[b]])
        assert relerr(mean[b, :m[b]], mu) < TOL and relerr(var[b, :m[b]], v) < TOL, b
    monkeypatch.setenv("CNGP_NO_LAG_TABLES", "1")
    mean0, var0, _, _ = gp_ctx.predict_ragged(kname, th, x, y, n, xs, m)
    monkeypatch.delenv("CNGP_NO_LAG_TABLES", raising=False)
    valid = np.arange(ldm)[None, :] < m[:, None]
    assert relerr(mean[valid], mean0[valid]) < 1e-10 and relerr(var[valid], var0[valid]) < 1e-10


def test_sigma_mode_through_the_callback(gp_ctx, monkeypatch):
    """gp_slip: grid arange(min, max + 600) and sigma = 2 sqrt(var) written by the recurrence"""
    kname = "rbf+stdperiodic"
    th = syn.theta_for(kname)
    x, y = lattice_windows(B_MIN, 149)
    mean, sigma, status = gp_ctx.gp_slip(kname, x, y, theta=th)
    monkeypatch.setenv("CNGP_NO_LAG_TABLES", "1")
    mean0, sigma0, status0 = gp_ctx.gp_slip(kname, x, y, theta=th)
    monkeypatch.delenv("CNGP_NO_LAG_TABLES", raising=False)
    assert np.all(status == 0) and np.array_equal(status, status0)
    assert relerr(mean, mean0) < 1e-10 and relerr(sigma, sigma0) < 1e-10
    e = go.KernelExpr(kname)
    for b in (0, B_MIN - 1):
        mu, sg = go.gp_slip_callback(x[b], y[b], e, th[:-1], th[-1])
        assert relerr(mean[b], mu) < TOL and relerr(sigma[b], sg) < TOL


def test_mixed_batch_gives_each_window_its_own_bits(gp_ctx):
    """lattice grids (recurrence), step-1 grids on d = 2 stamps and gapped stamps (gp_var_kernel) in one batch: every
    window's mean and variance have the bits they have in a batch of its own kind"""
    kname = "rbf+stdperiodic"
    th = syn.theta_for(kname)
    B, N, M = 3 * B_MIN, 128, 300
    rng = np.random.default_rng(2)
    x, y = lattice_windows(B, N, d=2)
    xs = x[:, -1:] + 2.0 + 2.0 * np.arange(M)[None, :]
    xs[1::3] = x[1::3, -1:] + 1.0 + np.arange(M)[None, :]
    for b in range(2, B, 3):
        x[b] = x[b, 0] + np.concatenate([[0.0], np.cumsum(rng.integers(1, 4, N - 1))]).astype(float)
        xs[b] = x[b, -1] + 1.0 + np.arange(M)
    xs = np.ascontiguousarray(xs)
    full = gp_ctx.predict(kname, th, x, y, xs)
    assert np.all(full[3] == 0)
    for group in (np.arange(0, B, 3), np.arange(1, B, 3), np.arange(2, B, 3)):
        part = gp_ctx.predict(kname, th, x[group], y[group], xs[group])
        for a, b in zip(full, part):
            assert np.array_equal(a[group], b), group
    check_oracle(kname, th, x, y, xs, full[0], full[1], windows=range(6))


def test_device_tensors(gp_ctx):
    """device-memory call on the benchmark shape gives the bits of the host-memory call"""
    kname = "rbf+stdperiodic"
    th = syn.theta_for(kname)
    x, y = lattice_windows(B_MIN, 256)
    xs = np.stack([syn.test_grid(x[b], 600) for b in range(B_MIN)])
    host = gp_ctx.predict(kname, th, x, y, xs)
    dev = gp_ctx.predict(kname, *(torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (th, x, y, xs)))
    for a, b in zip(host, dev):
        assert np.array_equal(a, b.cpu().numpy())


def min_pivot_ratio(kname, th, x):
    e = go.KernelExpr(kname)
    Ky = go.kernel_K(e, th[:-1], x) + (th[-1] + 1e-8) * np.eye(x.size)
    return float(np.min(np.diag(np.linalg.cholesky(Ky)) ** 2) / Ky[0, 0])


def test_window_just_below_the_guard_stays_on_gp_var_kernel(gp_ctx):
    """rbf at noise 4.5e-5 has min L_kk^2 / t0 just below 1e-2: both Toeplitz kernels leave it alone, so it has the bits
    of its mirror image (stamps and grid reflected about x_0: the same Ky and K*, decreasing stamps, never taken)"""
    kname = "rbf"
    th = np.array([0.01, 10.0, 4.5e-5])
    x, y = lattice_windows(B_MIN, 256)
    assert 0.8e-2 < min_pivot_ratio(kname, th, x[0]) < 1e-2
    xs = np.stack([syn.test_grid(x[b], 600) for b in range(B_MIN)])
    out = gp_ctx.predict(kname, th, x, y, xs)
    x0 = x[:, :1]
    mirror = gp_ctx.predict(kname, th, 2.0 * x0 - x, y, 2.0 * x0 - xs)
    assert np.all(out[3] == 0)
    for a, b in zip(out, mirror):
        assert np.array_equal(a, b)
    check_oracle(kname, th, x, y, xs, out[0], out[1], tol=1e-7)
