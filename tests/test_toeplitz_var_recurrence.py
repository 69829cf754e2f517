"""The displacement recurrence of csrc/gp_var_toeplitz.cuh (DESIGN.md section 4.2c), restated in float64 numpy and held
to the oracle's predict.  Runs without a GPU.

For stamps x_0 + i d, Ky = K + s I is symmetric Toeplitz (s = Ky(0,0) - k*(0)), and for the lattice points
p_m = x_0 + m d the quadratic form q_m = k_m^T Ky^-1 k_m obeys
    q_{m+1} = q_m + ((a^T k_{m+1})^2 - (t^T k_m)^2) / gamma,   a = Ky^-1 e_0, t = reversed a, gamma = a_0,
anchored at m = 0 and m = n-1 by q = t0 - 2 s + s^2 gamma."""
import numpy as np
import pytest
from scipy import linalg

from corenav_gp_b200 import synthetic as syn
from oracle import gp_oracle as go

JITTER = 1e-8


def relerr(a, ref):
    scale = max(float(np.max(np.abs(ref))), 1e-300)
    return float(np.max(np.abs(a - ref) / np.maximum(np.abs(ref), 1e-3 * scale)))


def recurrence_predict(kname, th, x, y, d, m_first, count):
    """mean and variance at the lattice points x_0 + (m_first + j) d, j < count, the way the kernel computes them"""
    e = go.KernelExpr(kname)
    theta, noise = th[:-1], th[-1]
    n = x.size
    kstar = lambda lag: go.kernel_K(e, theta, np.zeros(1), np.atleast_1d(np.asarray(lag, float) * d))[0]
    K = go.kernel_K(e, theta, x)
    Ky = K + (noise + JITTER) * np.eye(n)
    t0 = Ky[0, 0]
    s = t0 - kstar(0.0)[0]
    kss = go.kernel_Kdiag(e, theta, x[:1])[0]
    cf = linalg.cho_factor(Ky, lower=True)
    alpha = linalg.cho_solve(cf, y)
    w = linalg.cho_solve(cf, np.eye(n)[:, n - 1])   # A e_{n-1} = t
    t, a = w, w[::-1]
    gam = w[n - 1]
    m0 = n - 1 if m_first >= n - 1 else 0
    m_end = m_first + count - 1
    i = np.arange(n)
    q = t0 - 2.0 * s + s * s * gam
    mean, var = [], []
    v_prev = None
    for m in range(m0, m_end + 1):
        k = kstar(np.abs(i - m))
        u = a @ k
        if v_prev is not None:
            q = q + (u * u - v_prev * v_prev) / gam
        v_prev = t @ k
        if m >= m_first:
            mean.append(alpha @ k)
            var.append(max(kss - q, 1e-15) + noise)
    return np.array(mean), np.array(var)


def window(N, d=1):
    x, y = syn.slip_windows(7, 1, N)
    return x[0, 0] + d * np.arange(N, dtype=float), y[0]


CASES = [
    # kernel, theta (noise last), N, d, first lattice index of the grid (None: x_{N-1} + 1), M, tolerance
    ("rbf+stdperiodic", None, 256, 1, None, 600, 1e-11),          # the benchmark window
    ("rbf+stdperiodic", None, 256, 1, 0, 855, 1e-11),             # the reference's grid from x_0
    ("rbf+stdperiodic", None, 128, 2, None, 300, 1e-10),          # d = 2 on the lattice
    ("rbf", [0.01, 10.0, 1e-3], 100, 3, 40, 200, 1e-10),          # d = 3, grid starting inside the span
    ("mat32+bias", [0.02, 7.0, 0.001, 1e-3], 256, 1, None, 600, 1e-10),
    ("mat52+white", [0.5, 15.0, 1e-4, 1e-3], 256, 1, None, 600, 1e-9),
    ("stdperiodic", [1.0, 37.0, 1.0, 1e-4], 256, 1, None, 600, 1e-8),
    ("rbf", [0.01, 10.0, 1e-5], 256, 1, None, 600, 1e-8),
]


@pytest.mark.parametrize("kname,theta,N,d,m_first,M,tol", CASES)
def test_recurrence_matches_oracle(kname, theta, N, d, m_first, M, tol):
    th = syn.theta_for(kname) if theta is None else np.array(theta)
    x, y = window(N, d)
    mf = N if m_first is None else m_first
    mean, var = recurrence_predict(kname, th, x, y, d, mf, M)
    xs = x[0] + d * (mf + np.arange(M, dtype=float))
    e = go.KernelExpr(kname)
    mu, v = go.predict(e, th[:-1], th[-1], x, y, xs)
    assert relerr(mean, mu) < tol and relerr(var, v) < tol, (relerr(mean, mu), relerr(var, v))


def test_anchor_is_the_quadratic_form_at_both_ends():
    kname = "rbf+stdperiodic"
    th = syn.theta_for(kname)
    x, y = window(64)
    e = go.KernelExpr(kname)
    Ky = go.kernel_K(e, th[:-1], x) + (th[-1] + JITTER) * np.eye(x.size)
    A = np.linalg.inv(Ky)
    kx = go.kernel_K(e, th[:-1], x, x)   # no White in this expression: K* = K
    s = Ky[0, 0] - kx[0, 0]
    closed = Ky[0, 0] - 2.0 * s + s * s * A[0, 0]
    for m in (0, x.size - 1):
        assert abs(kx[:, m] @ A @ kx[:, m] - closed) < 1e-12 * closed
    assert abs(A[0, 0] - A[-1, -1]) < 1e-12 * A[0, 0]
