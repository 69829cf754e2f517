"""Extended-precision exact GP: oracle/gp_oracle.py's inference, predict and LML gradient in float80.

THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE (see oracle/gp_oracle.py).

gp_oracle is float64 LAPACK: near the conditioning guard of the Toeplitz paths (cond(Ky) ~ 1e3 - 3e4) its own error is
of the order cond(Ky) eps_64, the same as the kernels it checks, so agreement with it cannot show that either is right.
This restatement carries everything after the squared distance in numpy long double (x86 extended precision,
eps = 1.1e-19), so its error at those conditionings stays about four orders of magnitude below the 1e-9 parity target.

What the device sees is reproduced exactly: theta, x, y and x* are the float64 values passed to it, and r^2 is GPy's
float64 expanded form (gp_oracle._r2_expanded), promoted afterwards - exact for the integer stamps below 2^26 that the
Toeplitz paths take.  Everything after r^2 is long double: the constants pi, sqrt 3, sqrt 5, exp / log1p / sin, a dense
Cholesky, the triangular solves, log det, alpha, Ky^-1 for dL_dK, the 1e-15 variance clip and + noise.

pivot_ratio / theta_at_ratio place a theta against TOEP_MIN_PIVOT2 (csrc/gp_fit_toeplitz.cuh) without a GPU:
min_k L_kk^2 / t0 of Ky on the stamps 0, d, 2d, ..., t0 = k(0) + noise + 1e-8."""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np
from scipy.linalg import lapack

from oracle import gp_oracle as go

LD = np.longdouble
PI = LD("3.14159265358979323846264338327950288")
SQRT3 = np.sqrt(LD(3))
SQRT5 = np.sqrt(LD(5))
LOG_2_PI = np.log(2 * PI)
JITTER = LD(go.JITTER)
VAR_FLOOR = LD(go.VAR_FLOOR)

KernelExpr = go.KernelExpr


def _ld(a):
    return np.asarray(a, dtype=np.float64).astype(LD)


def _leaf_K(op: int, th, x: np.ndarray, x2: Optional[np.ndarray]):
    """(K, [dK/dtheta_j]) of one leaf in long double; th long double, x / x2 float64 stamps"""
    nm = go.OPNAME[op]
    xx2 = x if x2 is None else x2
    if nm in ("rbf", "mat32", "mat52", "ratquad"):
        var, ls = th[0], th[1]
        r = np.sqrt(go._r2_expanded(x, x2).astype(LD)) / ls
        if nm == "rbf":
            kr = np.exp(-r * r / 2)
            dk_dr = -r * kr
        elif nm == "mat32":
            e = np.exp(-SQRT3 * r)
            kr = (1 + SQRT3 * r) * e
            dk_dr = -3 * r * e
        elif nm == "mat52":
            e = np.exp(-SQRT5 * r)
            kr = (1 + SQRT5 * r + LD(5) / 3 * r * r) * e
            dk_dr = (LD(10) / 3 * r - 5 * r - 5 * SQRT5 / 3 * r * r) * e
        else:
            a = th[2]
            l1p = np.log1p(r * r / 2)
            kr = np.exp(-a * l1p)
            dk_dr = -a * r * np.exp(-(a + 1) * l1p)
        K = var * kr
        grads = [kr, -(var * dk_dr) * r / ls]
        if nm == "ratquad":
            grads.append(-K * l1p)
        return K, grads
    if nm == "stdperiodic":
        var, per, ls = th
        base = PI * (x[:, None] - xx2[None, :]).astype(LD) / per   # the difference of float64 stamps, as GPy forms it
        sb = np.sin(base)
        ed = np.exp(-(sb / ls) ** 2 / 2)
        K = var * ed
        dwl = var / (ls * ls) * sb * np.cos(base) * (base / per)
        dl = var * sb * sb / ls ** 3
        return K, [ed, dwl * ed, dl * ed]
    if nm == "brownian":
        a, b = x[:, None], xx2[None, :]
        base = np.where(np.sign(a) == np.sign(b), np.fmin(np.abs(a), np.abs(b)), 0.0).astype(LD)
        return th[0] * base, [base]
    if nm == "linear":
        base = np.multiply.outer(x.astype(LD), xx2.astype(LD))
        return th[0] * base, [base]
    if nm == "bias":
        base = np.ones((x.size, xx2.size), dtype=LD)
        return th[0] * base, [base]
    if nm == "white":
        base = np.eye(x.size, dtype=LD) if x2 is None else np.zeros((x.size, xx2.size), dtype=LD)
        return th[0] * base, [base]
    raise AssertionError(nm)


def kernel_K(expr: KernelExpr, theta, x, x2=None, want_grads=False):
    """K(X, X2) of the composite in long double; with want_grads also dK/dtheta_j (Add / Prod rules)"""
    th = _ld(theta)
    x = np.asarray(x, dtype=np.float64).ravel()
    x2 = None if x2 is None else np.asarray(x2, dtype=np.float64).ravel()
    stack = []
    p = 0
    for op in expr.program:
        if op < go.OP_ADD:
            n = go.LEAVES[go.OPNAME[op]][1]
            K, g = _leaf_K(op, th[p:p + n], x, x2)
            stack.append((K, {p + j: g[j] for j in range(n)}))
            p += n
        else:
            Kb, gb = stack.pop()
            Ka, ga = stack.pop()
            if op == go.OP_ADD:
                stack.append((Ka + Kb, {**ga, **gb}))
            else:
                stack.append((Ka * Kb, {**{k: v * Kb for k, v in ga.items()}, **{k: v * Ka for k, v in gb.items()}}))
    K, g = stack.pop()
    if want_grads:
        return K, [g[j] for j in range(expr.n_params)]
    return K


def kernel_Kdiag(expr: KernelExpr, theta, x) -> np.ndarray:
    th = _ld(theta)
    x = np.asarray(x, dtype=np.float64).ravel()
    stack = []
    p = 0
    for op in expr.program:
        if op < go.OP_ADD:
            nm = go.OPNAME[op]
            n = go.LEAVES[nm][1]
            if nm == "brownian":
                stack.append(th[p] * np.abs(x).astype(LD))
            elif nm == "linear":
                stack.append(th[p] * np.square(x.astype(LD)))
            else:
                stack.append(th[p] * np.ones(x.size, dtype=LD))
            p += n
        else:
            b = stack.pop()
            a = stack.pop()
            stack.append(a + b if op == go.OP_ADD else a * b)
    return stack.pop()


# ----------------------------------------------------------------------------------------------------------------------
# dense linear algebra in long double
# ----------------------------------------------------------------------------------------------------------------------
def cholesky(A: np.ndarray) -> np.ndarray:
    """Lower Cholesky factor (right-looking, one rank-1 update per column); raises go.NotPositiveDefinite"""
    A = np.array(A, dtype=LD)
    n = A.shape[0]
    L = np.zeros_like(A)
    for j in range(n):
        d = A[j, j]
        if not d > 0:
            raise go.NotPositiveDefinite(f"pivot {j} = {float(d)}")
        ljj = np.sqrt(d)
        col = A[j + 1:, j] / ljj
        L[j, j] = ljj
        L[j + 1:, j] = col
        A[j + 1:, j + 1:] -= np.multiply.outer(col, col)
    return L


def solve_lower(L: np.ndarray, B: np.ndarray) -> np.ndarray:
    """L^-1 B by forward substitution (B a vector or a matrix of columns)"""
    X = np.array(B, dtype=LD)
    for j in range(L.shape[0]):
        X[j] /= L[j, j]
        if X.ndim == 1:
            X[j + 1:] -= L[j + 1:, j] * X[j]
        else:
            X[j + 1:] -= np.multiply.outer(L[j + 1:, j], X[j])
    return X


def solve_upper_t(L: np.ndarray, b: np.ndarray) -> np.ndarray:
    """L^-T b by back substitution"""
    x = np.array(b, dtype=LD)
    for j in range(L.shape[0] - 1, -1, -1):
        x[j] = (x[j] - L[j + 1:, j] @ x[j + 1:]) / L[j, j]
    return x


@dataclass
class Inference:
    L: np.ndarray
    alpha: np.ndarray
    lml: LD
    logdet: LD
    Kinv: Optional[np.ndarray]
    grad: Optional[np.ndarray]      # d LML / d [theta..., noise], long double


def _ky(expr, theta, noise, x, want_grads):
    if want_grads:
        K, dKs = kernel_K(expr, theta, x, None, want_grads=True)
    else:
        K, dKs = kernel_K(expr, theta, x), None
    K[np.diag_indices(K.shape[0])] += LD(float(noise)) + JITTER
    return K, dKs


def inference(expr: KernelExpr, theta, noise: float, x, y, want_grad: bool = False, L: Optional[np.ndarray] = None,
              Kinv: Optional[np.ndarray] = None) -> Inference:
    """ExactGaussianInference.inference (gp_oracle.inference) in long double.  No jitter ladder: a Ky that is not
    positive definite in long double raises go.NotPositiveDefinite.  L (and Kinv) may be passed from the inference of
    another window with the same Ky - windows on stamps x_0 + i d with the same n and d share it, whatever x_0."""
    x = np.asarray(x, dtype=np.float64).ravel()
    y = _ld(y).ravel()
    n = x.size
    Ky, dKs = _ky(expr, theta, noise, x, want_grad)
    if L is None:
        L = cholesky(Ky)
    z = solve_lower(L, y)
    alpha = solve_upper_t(L, z)
    logdet = 2 * np.sum(np.log(np.diag(L)))
    lml = (-n * LOG_2_PI - logdet - y @ alpha) / 2
    grad = None
    if want_grad:
        if Kinv is None:
            Li = solve_lower(L, np.eye(n, dtype=LD))
            Kinv = Li.T @ Li
        dL_dK = (np.multiply.outer(alpha, alpha) - Kinv) / 2
        grad = np.array([np.sum(dL_dK * dK) for dK in dKs] + [np.trace(dL_dK)], dtype=LD)
    return Inference(L, alpha, lml, logdet, Kinv, grad)


def predict(expr: KernelExpr, theta, noise: float, x, y, xnew, inf: Optional[Inference] = None,
            include_likelihood: bool = True):
    """(mean [M], var [M]) in long double, as gp_oracle.predict"""
    x = np.asarray(x, dtype=np.float64).ravel()
    xnew = np.asarray(xnew, dtype=np.float64).ravel()
    if inf is None:
        inf = inference(expr, theta, noise, x, y)
    Kx = kernel_K(expr, theta, x, xnew)
    mu = Kx.T @ inf.alpha
    tmp = solve_lower(inf.L, Kx)
    var = np.maximum(kernel_Kdiag(expr, theta, xnew) - np.sum(tmp * tmp, axis=0), VAR_FLOOR)
    if include_likelihood:
        var = var + LD(float(noise))
    return mu, var


# ----------------------------------------------------------------------------------------------------------------------
# where a theta sits against the conditioning guard of the Toeplitz paths
# ----------------------------------------------------------------------------------------------------------------------
def _ky_lattice(kname, theta, N, d, dtype):
    expr = KernelExpr(kname)
    th = np.asarray(theta, dtype=np.float64)
    x = d * np.arange(N, dtype=np.float64)
    if dtype == LD:
        Ky, _ = _ky(expr, th[:-1], th[-1], x, False)
        t0 = kernel_Kdiag(expr, th[:-1], x[:1])[0] + LD(float(th[-1])) + JITTER
    else:
        Ky = go.kernel_K(expr, th[:-1], x)
        Ky[np.diag_indices(N)] += th[-1] + go.JITTER
        t0 = go.kernel_Kdiag(expr, th[:-1], x[:1])[0] + (th[-1] + go.JITTER)
    return Ky, t0


def pivot_ratio(kname: str, theta, N: int, d: int = 1) -> float:
    """min_k L_kk^2 / t0 of Ky on the stamps 0, d, ..., (N-1) d (theta with the noise last), in long double: the
    quantity gp_fit_toeplitz_kernel holds against TOEP_MIN_PIVOT2"""
    Ky, t0 = _ky_lattice(kname, theta, N, d, LD)
    return float(np.min(np.diag(cholesky(Ky))) ** 2 / t0)


def _pivot_ratio64(kname, theta, N, d):
    Ky, t0 = _ky_lattice(kname, theta, N, d, np.float64)
    L, info = lapack.dpotrf(Ky, lower=1)
    if info != 0:
        return 0.0
    return float(np.min(np.diag(L)) ** 2 / t0)


def theta_at_ratio(kname: str, theta, N: int, d: int, target: float, rtol: float = 1e-6) -> np.ndarray:
    """theta with its noise (last entry) set so that pivot_ratio(kname, theta, N, d) = target.  The ratio grows with
    the noise; the bisection runs on log(noise) with the float64 factor (at ratios near the guard its pivots carry about
    14 correct digits), and the result is checked in long double."""
    th = np.array(theta, dtype=np.float64)
    lo, hi = np.log(1e-14), np.log(1e3)
    for _ in range(200):
        mid = 0.5 * (lo + hi)
        th[-1] = np.exp(mid)
        if _pivot_ratio64(kname, th, N, d) < target:
            lo = mid
        else:
            hi = mid
        if hi - lo < rtol:
            break
    th[-1] = np.exp(0.5 * (lo + hi))
    r = pivot_ratio(kname, th, N, d)
    if not abs(r - target) <= 1e-4 * target:
        raise ValueError(f"{kname}: no noise gives a pivot ratio of {target} (reached {r})")
    return th
