"""Windows that share one covariance (csrc/gp_toep_group.cuh, DESIGN.md section 4.2d).

With one theta for the call, the Toeplitz windows with the same key (n, m, d, m_s) are factored once and every member gets
its z, mean and LML from that factor.  Passing the same theta once per window turns the grouping off, so the per-window
Toeplitz path is the reference: every case here must agree with it bit for bit in mean, variance, LML and status, and
with the oracle.  The path runs for batches of more windows than SMs."""
import numpy as np
import pytest
import torch

from corenav_gp_b200 import synthetic as syn
from oracle import gp_oracle as go

pytestmark = pytest.mark.gpu
TOL = 1e-9
B_MIN = 160          # > the B200's 148 SMs
KNAME = "rbf+stdperiodic"


def relerr(a, ref):
    a, ref = np.asarray(a, dtype=float), np.asarray(ref, dtype=float)
    scale = max(float(np.max(np.abs(ref))), 1e-300)
    return float(np.max(np.abs(a - ref) / np.maximum(np.abs(ref), 1e-3 * scale)))


def lattice_windows(B, N, d=1, seed=21):
    x, y = syn.slip_windows(seed, B, N)
    x = x[:, :1] + 3.0 * (np.arange(B) % 5)[:, None] + d * np.arange(N)[None, :]
    return x, y


def per_window(th, B):
    return np.ascontiguousarray(np.tile(th, (B, 1)))


def same_bits(shared, ref, valid=None):
    for a, b in zip(shared, ref):
        a, b = np.asarray(a), np.asarray(b)
        if valid is not None and a.ndim == 2:
            a, b = a[valid], b[valid]
        assert a.tobytes() == b.tobytes()


def check_oracle(th, x, y, xs, mean, var, windows, kname=KNAME, tol=TOL):
    e = go.KernelExpr(kname)
    for b in windows:
        mu, v = go.predict(e, th[:-1], th[-1], x[b], y[b], xs[b])
        assert relerr(mean[b], mu) < tol and relerr(var[b], v) < tol, (b, relerr(mean[b], mu), relerr(var[b], v))


def check(ctx, th, x, y, xs, kname=KNAME, oracle=(0, 1, -1), tol=TOL):
    out = ctx.predict(kname, th, x, y, xs)
    ref = ctx.predict(kname, per_window(th, x.shape[0]), x, y, xs)
    same_bits(out, ref)
    ok = np.flatnonzero(out[3] == 0)
    check_oracle(th, x, y, xs, out[0], out[1], [ok[i] for i in oracle], kname, tol)
    return out


@pytest.mark.parametrize("B", [B_MIN, 4096])
def test_benchmark_shape(gp_ctx, B):
    """N = 256, M = 600 on the grid x_{N-1} + 1 + j; start stamps and y differ from window to window"""
    th = syn.theta_for(KNAME)
    x, y = lattice_windows(B, 256)
    xs = np.stack([syn.test_grid(x[b], 600) for b in range(B)])
    out = check(gp_ctx, th, x, y, xs)
    assert np.all(out[3] == 0)


def test_without_lml(gp_ctx):
    """a call that does not ask for the LML (the Monte-Carlo shard, the node callback)"""
    th = syn.theta_for(KNAME)
    x, y = lattice_windows(B_MIN, 256)
    xs = np.stack([syn.test_grid(x[b], 600) for b in range(B_MIN)])
    out = gp_ctx.predict(KNAME, th, x, y, xs, want_lml=False)
    ref = gp_ctx.predict(KNAME, per_window(th, B_MIN), x, y, xs, want_lml=False)
    assert out[2] is None and ref[2] is None
    same_bits([out[0], out[1], out[3]], [ref[0], ref[1], ref[3]])
    full = gp_ctx.predict(KNAME, th, x, y, xs)
    same_bits([out[0], out[1], out[3]], [full[0], full[1], full[3]])


def test_two_keys_and_a_shifted_grid(gp_ctx):
    """d = 1 and d = 2 windows and a shifted grid in one batch: the first key forms the group, the others stay per
    window, and a batch of each kind alone gives the same bits"""
    th = syn.theta_for(KNAME)
    B, N, M = 3 * B_MIN, 128, 300
    x1, y = lattice_windows(B, N)
    x2, _ = lattice_windows(B, N, d=2)
    x = np.where((np.arange(B) % 3 == 1)[:, None], x2, x1)
    d = np.where(np.arange(B) % 3 == 1, 2.0, 1.0)[:, None]
    xs = x[:, -1:] + d + d * np.arange(M)[None, :]
    xs[2::3] += 5.0                                      # m_s = n + 5 instead of n
    xs = np.ascontiguousarray(xs)
    out = check(gp_ctx, th, x, y, xs, oracle=(0, 1, 2, -1))
    assert np.all(out[3] == 0)
    for sel in (np.arange(0, B, 3), np.arange(1, B, 3), np.arange(2, B, 3)):
        part = gp_ctx.predict(KNAME, th, x[sel], y[sel], xs[sel])
        for a, b in zip(out, part):
            assert np.asarray(a)[sel].tobytes() == np.asarray(b).tobytes()


def test_stamps_beyond_two_to_the_26(gp_ctx):
    """members whose stamps pass 2^26 leave the lag tables, and so the group"""
    th = syn.theta_for(KNAME)
    x, y = lattice_windows(B_MIN, 256)
    x[5::7] += 2.0 ** 26
    xs = np.stack([syn.test_grid(x[b], 600) for b in range(B_MIN)])
    check(gp_ctx, th, x, y, xs, oracle=(0, 5, -1), tol=1e-7)


def test_members_with_non_finite_or_huge_y(gp_ctx):
    """a NaN in y and y ~ 1e200 (quad overflows): each such member ends as the per-window path leaves it"""
    th = syn.theta_for(KNAME)
    x, y = lattice_windows(B_MIN, 256)
    y[3, 17] = np.nan
    y[0] *= 1e200
    y[9] *= 1e200
    y[11, :] = 1e300
    xs = np.stack([syn.test_grid(x[b], 600) for b in range(B_MIN)])
    out = gp_ctx.predict(KNAME, th, x, y, xs)
    ref = gp_ctx.predict(KNAME, per_window(th, B_MIN), x, y, xs)
    same_bits(out, ref)
    check_oracle(th, x, y, xs, out[0], out[1], [1, 2, B_MIN - 1])


def test_group_below_the_guard(gp_ctx):
    """rbf at noise 4.5e-5 is just below the Schur fit's conditioning guard: the whole group goes back to the tile
    Cholesky and gp_var_kernel"""
    th = np.array([0.01, 10.0, 4.5e-5])
    x, y = lattice_windows(B_MIN, 256)
    xs = np.stack([syn.test_grid(x[b], 600) for b in range(B_MIN)])
    out = check(gp_ctx, th, x, y, xs, kname="rbf", tol=1e-7)
    assert np.all(out[3] == 0)


def test_ragged_counts(gp_ctx):
    """per-window n and m: windows group by (n, m); entries beyond m are not written"""
    th = syn.theta_for(KNAME)
    B, ld, ldm = 4 * B_MIN, 256, 600
    rng = np.random.default_rng(8)
    x, y = lattice_windows(B, ld)
    n = np.where(rng.random(B) < 0.5, ld, rng.integers(200, ld + 1, B)).astype(np.int32)
    m = np.where(rng.random(B) < 0.5, ldm, rng.integers(1, ldm + 1, B)).astype(np.int32)
    xs = np.stack([x[b, n[b] - 1] + 1.0 + np.arange(ldm, dtype=float) for b in range(B)])
    out = gp_ctx.predict_ragged(KNAME, th, x, y, n, xs, m)
    ref = gp_ctx.predict_ragged(KNAME, per_window(th, B), x, y, n, xs, m)
    valid = np.arange(ldm)[None, :] < m[:, None]
    same_bits(out, ref, valid)
    assert np.all(out[3] == 0)
    e = go.KernelExpr(KNAME)
    for b in (0, 1, 2, B - 1):
        mu, v = go.predict(e, th[:-1], th[-1], x[b, :n[b]], y[b, :n[b]], xs[b, :m[b]])
        assert relerr(out[0][b, :m[b]], mu) < TOL and relerr(out[1][b, :m[b]], v) < TOL, b


def test_sigma_mode_through_the_callback(gp_ctx):
    """gp_slip: grid arange(min, max + 600) (m_s = 0) and sigma = 2 sqrt(var)"""
    th = syn.theta_for(KNAME)
    x, y = lattice_windows(B_MIN, 149)
    n = np.full(B_MIN, 149, np.int32)
    out = gp_ctx.gp_slip_ragged(KNAME, x, y, n, theta=th)
    ref = gp_ctx.gp_slip_ragged(KNAME, x, y, n, theta=per_window(th, B_MIN))
    valid = np.arange(out[0].shape[1])[None, :] < out[2][:, None]
    same_bits(out, ref, valid)
    assert np.all(out[3] == 0)
    e = go.KernelExpr(KNAME)
    for b in (0, B_MIN - 1):
        mu, sg = go.gp_slip_callback(x[b], y[b], e, th[:-1], th[-1])
        assert relerr(out[0][b, :out[2][b]], mu) < TOL and relerr(out[1][b, :out[2][b]], sg) < TOL


def test_device_tensors(gp_ctx):
    """device-memory calls give the bits of host-memory calls, grouped or not"""
    th = syn.theta_for(KNAME)
    x, y = lattice_windows(B_MIN, 256)
    xs = np.stack([syn.test_grid(x[b], 600) for b in range(B_MIN)])
    host = gp_ctx.predict(KNAME, th, x, y, xs)
    ref = gp_ctx.predict(KNAME, per_window(th, B_MIN), x, y, xs)
    dev = gp_ctx.predict(KNAME, *(torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (th, x, y, xs)))
    same_bits(host, ref)
    same_bits(host, [t.cpu().numpy() for t in dev])


def test_no_more_windows_than_sms(gp_ctx):
    """B <= SMs stays on the tile Cholesky and gp_var_kernel, shared theta or not"""
    th = syn.theta_for(KNAME)
    x, y = lattice_windows(100, 256)
    xs = np.stack([syn.test_grid(x[b], 600) for b in range(100)])
    check(gp_ctx, th, x, y, xs)
