"""Members of a shared covariance in CTAs that share the factor's tile columns (csrc/gp_toep_group.cuh,
DESIGN.md section 4.2d).

gp_toep_member_kernel runs TG_WARPS members per CTA, which walk the factor's tile columns together, so a member's
results must not depend on how many members share its CTA, on where the group ends inside a CTA, or on a neighbour
that fails.  The same theta passed once per window turns the grouping off: every case must agree with that per-window
Toeplitz path bit for bit in mean, variance, LML and status, and with the oracle on a sample."""
import numpy as np
import pytest

from corenav_gp_b200 import synthetic as syn
from oracle import gp_oracle as go

pytestmark = pytest.mark.gpu
TOL = 1e-9
KNAME = "rbf+stdperiodic"
TG_WARPS = 8         # members per CTA of gp_toep_member_kernel


def relerr(a, ref):
    a, ref = np.asarray(a, dtype=float), np.asarray(ref, dtype=float)
    scale = max(float(np.max(np.abs(ref))), 1e-300)
    return float(np.max(np.abs(a - ref) / np.maximum(np.abs(ref), 1e-3 * scale)))


def lattice_windows(B, N, d=1, seed=33):
    x, y = syn.slip_windows(seed, B, N)
    x = x[:, :1] + 3.0 * (np.arange(B) % 5)[:, None] + d * np.arange(N)[None, :]
    return x, y


def per_window(th, B):
    return np.ascontiguousarray(np.tile(th, (B, 1)))


def same_bits(out, ref, valid=None):
    for a, b in zip(out, ref):
        a, b = np.asarray(a), np.asarray(b)
        if valid is not None and a.ndim == 2:
            a, b = a[valid], b[valid]
        assert a.tobytes() == b.tobytes()


def check(ctx, th, x, y, xs, sample, tol=TOL):
    out = ctx.predict(KNAME, th, x, y, xs)
    ref = ctx.predict(KNAME, per_window(th, x.shape[0]), x, y, xs)
    same_bits(out, ref)
    e = go.KernelExpr(KNAME)
    for b in sample:
        mu, v = go.predict(e, th[:-1], th[-1], x[b], y[b], xs[b])
        assert relerr(out[0][b], mu) < tol and relerr(out[1][b], v) < tol, (b, relerr(out[0][b], mu))
    return out


@pytest.mark.parametrize("B", [149, 150, 4097])
def test_group_sizes(gp_ctx, B):
    """every window one group; the last CTA of members is partly empty"""
    th = syn.theta_for(KNAME)
    x, y = lattice_windows(B, 256)
    xs = np.stack([syn.test_grid(x[b], 600) for b in range(B)])
    out = check(gp_ctx, th, x, y, xs, (0, B // 2, B - 1))
    assert np.all(out[3] == 0)


@pytest.mark.parametrize("members", [TG_WARPS - 1, TG_WARPS + 1, 2 * TG_WARPS + 1])
def test_group_of_block_size_plus_minus_one(gp_ctx, members):
    """a group of TG_WARPS +- 1 members (the windows with the first window's stamp step) among windows of another stamp
    step, which stay per window"""
    th = syn.theta_for(KNAME)
    B, N, M = 200, 128, 300
    x1, y = lattice_windows(B, N)
    x2, _ = lattice_windows(B, N, d=2)
    pick = np.zeros(B, bool)
    pick[np.linspace(0, B - 1, members).astype(int)] = True
    x = np.where(pick[:, None], x1, x2)
    d = np.where(pick, 1.0, 2.0)[:, None]
    xs = np.ascontiguousarray(x[:, -1:] + d + d * np.arange(M)[None, :])
    out = check(gp_ctx, th, x, y, xs, (0, 1, B - 1))
    assert np.all(out[3] == 0)


def test_failing_members_leave_their_neighbours(gp_ctx):
    """a NaN y and y = 1e300 in the middle of a CTA of members; the other members of that CTA keep their bits"""
    th = syn.theta_for(KNAME)
    B = 4 * TG_WARPS * 8
    x, y = lattice_windows(B, 256)
    y[TG_WARPS + 3, 40] = np.nan
    y[TG_WARPS + 5, :] = 1e300
    xs = np.stack([syn.test_grid(x[b], 600) for b in range(B)])
    out = check(gp_ctx, th, x, y, xs, (TG_WARPS + 2, TG_WARPS + 4, TG_WARPS + 6))
    assert np.all(np.delete(out[3], [TG_WARPS + 3, TG_WARPS + 5]) == 0)


def test_tiny_y(gp_ctx):
    """y scaled to 1e-300: z, alpha and the mean run through subnormal values"""
    th = syn.theta_for(KNAME)
    x, y = lattice_windows(160, 256)
    y = y * 1e-300
    xs = np.stack([syn.test_grid(x[b], 600) for b in range(160)])
    out = gp_ctx.predict(KNAME, th, x, y, xs)
    ref = gp_ctx.predict(KNAME, per_window(th, 160), x, y, xs)
    same_bits(out, ref)


@pytest.mark.parametrize("N", [97, 250])
def test_counts_off_the_tile(gp_ctx, N):
    """n not a multiple of 8, and ragged n and m inside one call: the windows group by (n, m)"""
    th = syn.theta_for(KNAME)
    B, ldm = 320, 600
    rng = np.random.default_rng(N)
    x, y = lattice_windows(B, N)
    n = np.where(rng.random(B) < 0.7, N, rng.integers(N - 20, N + 1, B)).astype(np.int32)
    m = np.where(rng.random(B) < 0.7, ldm, rng.integers(1, ldm + 1, B)).astype(np.int32)
    xs = np.stack([x[b, n[b] - 1] + 1.0 + np.arange(ldm, dtype=float) for b in range(B)])
    out = gp_ctx.predict_ragged(KNAME, th, x, y, n, xs, m)
    ref = gp_ctx.predict_ragged(KNAME, per_window(th, B), x, y, n, xs, m)
    same_bits(out, ref, np.arange(ldm)[None, :] < m[:, None])
    assert np.all(out[3] == 0)
    e = go.KernelExpr(KNAME)
    for b in (0, 1, B - 1):
        mu, v = go.predict(e, th[:-1], th[-1], x[b, :n[b]], y[b, :n[b]], xs[b, :m[b]])
        assert relerr(out[0][b, :m[b]], mu) < TOL and relerr(out[1][b, :m[b]], v) < TOL, b


@pytest.mark.parametrize("mc", [1, 7, 600])
@pytest.mark.parametrize("start", [0, 1])
def test_grid_sizes_on_and_after_the_last_stamp(gp_ctx, mc, start):
    """d = 2 stamps, mc test points from x_{n-1} (start 0) or x_{n-1} + d (start 1)"""
    th = syn.theta_for(KNAME)
    B, N, d = 160, 200, 2.0
    x, y = lattice_windows(B, N, d=2)
    xs = np.ascontiguousarray(x[:, -1:] + d * (start + np.arange(mc))[None, :])
    out = check(gp_ctx, th, x, y, xs, (0, B - 1))
    assert np.all(out[3] == 0)


def test_n128(gp_ctx):
    """N = 128, M = 600 (the configs[3] window)"""
    th = syn.theta_for(KNAME)
    x, y = lattice_windows(1024, 128)
    xs = np.stack([syn.test_grid(x[b], 600) for b in range(1024)])
    out = check(gp_ctx, th, x, y, xs, (0, 511, 1023))
    assert np.all(out[3] == 0)
