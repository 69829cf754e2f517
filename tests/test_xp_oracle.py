"""oracle/xp_oracle.py, the float80 exact GP that the Toeplitz conditioning tests hold the kernels to.  Runs without a GPU.

Its own error must stay well below anything those tests resolve: it agrees with the float64 oracle where both are
accurate, with a 40-digit mpmath restatement at the largest conditioning the GPU cases reach (cond(Ky) ~ 3e4) to
1e-14 and at cond ~ 1e8 to 1e-10 (an error that grows as cond eps_80, not faster), its gradient with central
differences of its own LML, and its pivot ratio with the float64 LAPACK factor."""
import mpmath
import numpy as np
import pytest
from scipy.linalg import lapack

from corenav_gp_b200 import synthetic as syn
from oracle import gp_oracle as go
from oracle import xp_oracle as xp

# the seven expression families of tests/test_gpu_predict.py, noise 1e-3
KERNELS = [
    ("rbf", [0.01, 10.0]),
    ("rbf+stdperiodic", [0.01, 10.0, 0.0025, 37.0, 1.0]),
    ("rbf*brownian", [0.01, 10.0, 0.05]),
    ("mat32+bias", [0.02, 7.0, 0.001]),
    ("mat52*linear+white", [0.5, 15.0, 1e-5, 1e-4]),
    ("ratquad+stdperiodic*rbf", [0.01, 8.0, 1.5, 0.5, 37.0, 1.2, 0.01, 50.0]),
    ("(rbf+linear)*brownian+white", [0.02, 12.0, 1e-6, 0.03, 2e-4]),
]


def err(a, ref):
    """max |a - ref| / max(1, |ref|), elementwise (the parity metric)"""
    a, ref = np.asarray(a, dtype=np.longdouble), np.asarray(ref, dtype=np.longdouble)
    return float(np.max(np.abs(a - ref) / np.maximum(1, np.abs(ref))))


def nrel(a, ref):
    """normwise relative error max |a - ref| / max |ref|"""
    a, ref = np.asarray(a, dtype=np.longdouble), np.asarray(ref, dtype=np.longdouble)
    return float(np.max(np.abs(a - ref)) / np.max(np.abs(ref)))


@pytest.mark.parametrize("kname,theta", KERNELS)
def test_matches_float64_oracle_at_benchmark_theta(kname, theta):
    N, M = 100, 600
    x, y = syn.slip_windows(3, 1, N)
    x, y = x[0], y[0]
    xs = syn.test_grid(x, M)
    th = np.array(theta + [1e-3])
    e = go.KernelExpr(kname)
    i64 = go.inference(e, th[:-1], th[-1], x, y, want_grad=True)
    m64, v64 = go.predict(e, th[:-1], th[-1], x, y, xs, i64)
    ixp = xp.inference(e, th[:-1], th[-1], x, y, want_grad=True)
    mxp, vxp = xp.predict(e, th[:-1], th[-1], x, y, xs, ixp)
    for name, a, b in (("lml", i64.lml, ixp.lml), ("alpha", i64.alpha, ixp.alpha), ("mean", m64, mxp),
                       ("var", v64, vxp), ("grad", i64.grad, ixp.grad)):
        assert err(a, b) < 1e-12, (kname, name, err(a, b))


# ---------------------------------------------------------------------------------------------------------------------
# 40-digit reference
# ---------------------------------------------------------------------------------------------------------------------
def _mp_leaf(nm, th, r2, dx, cross):
    """one stationary leaf at squared distance r2 / signed difference dx (both exact floats), mpmath; cross: an entry
    of K(X, X*), where White is zero"""
    if nm in ("rbf", "mat32", "mat52", "ratquad"):
        r = mpmath.sqrt(r2) / th[1]
        if nm == "rbf":
            k = mpmath.exp(-r * r / 2)
        elif nm == "mat32":
            k = (1 + mpmath.sqrt(3) * r) * mpmath.exp(-mpmath.sqrt(3) * r)
        elif nm == "mat52":
            k = (1 + mpmath.sqrt(5) * r + mpmath.mpf(5) / 3 * r * r) * mpmath.exp(-mpmath.sqrt(5) * r)
        else:
            k = mpmath.exp(-th[2] * mpmath.log1p(r * r / 2))
        return th[0] * k
    if nm == "stdperiodic":
        s = mpmath.sin(mpmath.pi * dx / th[1])
        return th[0] * mpmath.exp(-(s / th[2]) ** 2 / 2)
    if nm == "bias":
        return th[0]
    if nm == "white":
        return th[0] if dx == 0 and not cross else mpmath.mpf(0)
    raise AssertionError(nm)


def _mp_k(expr, th, a, b, cross=False):
    dx = mpmath.mpf(float(a) - float(b))              # exact for the integer stamps used here
    r2 = mpmath.mpf(float(go._r2_expanded(np.array([a]), np.array([b]))[0, 0]) if a != b else 0.0)
    stack, p = [], 0
    for op in expr.program:
        if op < go.OP_ADD:
            nm = go.OPNAME[op]
            n = go.LEAVES[nm][1]
            stack.append(_mp_leaf(nm, th[p:p + n], r2, dx, cross))
            p += n
        else:
            v = stack.pop()
            u = stack.pop()
            stack.append(u + v if op == go.OP_ADD else u * v)
    return stack.pop()


def _mp_ky(expr, th, x):
    n = len(x)
    Ky = mpmath.matrix(n, n)
    for i in range(n):
        for j in range(i + 1):
            Ky[i, j] = Ky[j, i] = _mp_k(expr, th, x[i], x[j])
        Ky[i, i] += th[-1] + mpmath.mpf(go.JITTER)
    return Ky


def _mp_lml(expr, th, x, y):
    Ky = _mp_ky(expr, th, x)
    L = mpmath.cholesky(Ky)
    alpha = mpmath.cholesky_solve(Ky, y)
    logdet = 2 * mpmath.fsum(mpmath.log(L[i, i]) for i in range(len(x)))
    return (-len(x) * mpmath.log(2 * mpmath.pi) - logdet - mpmath.fdot(y, alpha)) / 2, Ky, L, alpha


def mp_reference(kname, theta, x, y, xs):
    """(lml, alpha, mean, var, grad) at 40 digits; the gradient by central differences with step 1e-12 theta_j
    (truncation ~1e-24, cancellation ~1e-28 relative)"""
    expr = go.KernelExpr(kname)
    with mpmath.workdps(40):
        th = [mpmath.mpf(float(t)) for t in theta]
        ym = mpmath.matrix([mpmath.mpf(float(v)) for v in y])
        lml, Ky, L, alpha = _mp_lml(expr, th, x, ym)
        mean, var = [], []
        for p in xs:
            k = mpmath.matrix([_mp_k(expr, th, xi, p, cross=True) for xi in x])
            mean.append(mpmath.fdot(k, alpha))
            t = mpmath.lu_solve(L, k)   # L is lower triangular: L^-1 k
            kss = _mp_k(expr, th, p, p)
            var.append(max(kss - mpmath.fdot(t, t), mpmath.mpf(go.VAR_FLOOR)) + th[-1])
        grad = []
        for j in range(len(th)):
            h = th[j] * mpmath.mpf("1e-12")
            up = list(th)
            dn = list(th)
            up[j] += h
            dn[j] -= h
            grad.append((_mp_lml(expr, up, x, ym)[0] - _mp_lml(expr, dn, x, ym)[0]) / (2 * h))
        to = lambda v: np.array([mpmath.nstr(u, 30) for u in v], dtype=np.longdouble)
        return np.longdouble(mpmath.nstr(lml, 30)), to(alpha), to(mean), to(var), to(grad)


# cond(Ky) of each case is asserted below; N = 24 - 40
MP_CASES = [
    # kernel, theta (noise last), N, cond range, tolerance
    ("rbf", [1.0, 6.0, 4.5e-4], 32, (1e4, 1e5), 1e-14),
    ("mat52+white", [0.5, 15.0, 4e-4, 2e-4], 40, (1e4, 1e5), 1e-14),
    ("rbf+stdperiodic", [0.01, 10.0, 0.0025, 7.0, 1.0, 7e-6], 24, (1e4, 1e5), 1e-14),
    ("rbf", [1.0, 6.0, 6e-8], 32, (5e7, 5e8), 1e-10),
    ("mat52+white", [0.5, 20.0, 1e-9, 1e-8], 40, (5e7, 5e8), 1e-10),
]


@pytest.mark.parametrize("kname,theta,N,cond,tol", MP_CASES)
def test_matches_mpmath(kname, theta, N, cond, tol):
    x, y = syn.slip_windows(5, 1, N)
    x, y = x[0], y[0]
    xs = x[0] + np.arange(N + 8, dtype=float)[::3]   # inside the span and beyond it
    th = np.array(theta)
    e = go.KernelExpr(kname)
    Ky = go.kernel_K(e, th[:-1], x) + (th[-1] + go.JITTER) * np.eye(N)
    c = np.linalg.cond(Ky)
    assert cond[0] < c < cond[1], c
    ixp = xp.inference(e, th[:-1], th[-1], x, y, want_grad=True)
    mxp, vxp = xp.predict(e, th[:-1], th[-1], x, y, xs, ixp)
    lml, alpha, mean, var, grad = mp_reference(kname, th, x, y, xs)
    errs = dict(lml=nrel([ixp.lml], [lml]), alpha=nrel(ixp.alpha, alpha), mean=nrel(mxp, mean), var=nrel(vxp, var),
                grad=nrel(ixp.grad, grad))
    assert max(errs.values()) < tol, (kname, c, errs)


@pytest.mark.parametrize("kname,theta", [KERNELS[1], KERNELS[4], ("mat52+white", [0.5, 15.0, 1e-4])])
def test_gradient_matches_central_differences(kname, theta):
    N = 40
    x, y = syn.slip_windows(9, 1, N)
    x, y = x[0], y[0]
    th = np.array(theta + [1e-3])
    e = go.KernelExpr(kname)
    g = xp.inference(e, th[:-1], th[-1], x, y, want_grad=True).grad
    for j in range(th.size):
        h = 1e-6 * th[j]
        up, dn = th.copy(), th.copy()
        up[j] += h
        dn[j] -= h
        h = up[j] - dn[j]   # the step the float64 parameters actually take
        fd = (xp.inference(e, up[:-1], up[-1], x, y).lml - xp.inference(e, dn[:-1], dn[-1], x, y).lml) / h
        assert abs(g[j] - fd) < 1e-8 * max(1.0, abs(float(g[j]))), (kname, j, float(g[j]), float(fd))


@pytest.mark.parametrize("kname,theta,d", [("rbf+stdperiodic", syn.theta_for("rbf+stdperiodic"), 1),
                                           ("mat52+white", [0.5, 15.0, 1e-4, 1e-3], 1),
                                           ("mat32+bias", [0.02, 7.0, 0.001, 1e-3], 2),
                                           ("stdperiodic", [1.0, 37.0, 1.0, 1e-2], 1)])
def test_pivot_ratio_matches_lapack(kname, theta, d):
    N = 256
    th = np.asarray(theta, dtype=float)
    e = go.KernelExpr(kname)
    x = d * np.arange(N, dtype=float)
    Ky = go.kernel_K(e, th[:-1], x) + (th[-1] + go.JITTER) * np.eye(N)
    L, info = lapack.dpotrf(Ky, lower=1)
    assert info == 0
    t0 = go.kernel_Kdiag(e, th[:-1], x[:1])[0] + th[-1] + go.JITTER
    ref = np.min(np.diag(L)) ** 2 / t0
    assert abs(xp.pivot_ratio(kname, th, N, d) - ref) < 1e-10 * ref


@pytest.mark.parametrize("target", [1.5e-2, 0.7e-2])
def test_theta_at_ratio_hits_target(target):
    th0 = np.array([0.01, 10.0, 1e-3])
    th = xp.theta_at_ratio("rbf", th0, 100, 1, target)
    assert np.array_equal(th[:-1], th0[:-1])
    assert abs(xp.pivot_ratio("rbf", th, 100, 1) - target) < 1e-4 * target
