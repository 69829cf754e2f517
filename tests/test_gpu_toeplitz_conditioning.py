"""The Toeplitz paths at their conditioning guard, against the float80 exact GP (oracle/xp_oracle.py).

The Schur fit (csrc/gp_fit_toeplitz.cuh), the variance recurrence (csrc/gp_var_toeplitz.cuh) and the shared-covariance
group (csrc/gp_toep_group.cuh) take a uniform-stamp window only while min_k L_kk^2 >= TOEP_MIN_PIVOT2 t0 (1e-2).  Near
that guard cond(Ky) is 1e3 - 3e4, where the float64 oracle carries the same cond eps error as the kernels; the float80
restatement does not.  Every case places its theta with xp.theta_at_ratio at a pivot ratio of 1.5e-2 (just admitted)
or 0.7e-2 (just refused), at x1, x10 and x100 the lengthscales of the families' test theta, or at that theta itself
(noise 1e-3, the control).  Each case runs B = 160 windows (more than the 148 SMs, so the Toeplitz kernels are on) four
ways:
  (a) theta per window ([B, P]: no grouping): the Schur fit and the recurrence;
  (b) one theta ([P]): the shared-covariance group;
  (c) the mirror image, stamps and grid reflected about x_0: the same Ky and K*, but decreasing stamps, which the
      Toeplitz paths never take - the tile Cholesky with lag tables;
  (d) CNGP_NO_LAG_TABLES=1: the lazy tile path,
on two grids: x_{n-1} + d (1 + j), M = 600 (the benchmark) and x_0 + d j, M = n + 600 (the reference's grid, whose
chain is anchored at x_0 and crosses the training span).

What must hold: the paths land on the side of the guard the case is on (an admitted case's Schur LML differs in bits
from the mirror on most windows, a refused case's (a) and (b) have the mirror's bits, (b) always has (a)'s); every path
is within 1e-9 max(1, |ref|) of xp in mean, variance and LML; the Toeplitz paths are no worse than 10x the tile path
(+1e-13), also in the posterior variance var - noise relative to k(0), which the parity floor of 1 would hide.  The LML
gradient of C = 2 candidates x 80 windows (the Schur factor feeds it) is held to xp and to the same windows in calls of
80 problems (the tile path).  `pytest -s` prints the worst error per path and case."""
import numpy as np
import pytest

from corenav_gp_b200 import synthetic as syn
from oracle import gp_oracle as go
from oracle import xp_oracle as xp

pytestmark = pytest.mark.gpu
B = 160                     # > the B200's 148 SMs: the Toeplitz kernels run
GUARD = 1e-2                # TOEP_MIN_PIVOT2
ADMIT, REFUSE = 1.5e-2, 0.7e-2
XP_WINDOWS = (0, 1, B - 1)
TOL = 1e-9
HORIZON = 600

# the Toeplitz-eligible families and their test theta (tests/test_gpu_toeplitz_fit.py), noise not included
FAMILIES = {
    "rbf": [0.01, 10.0],
    "rbf+stdperiodic": [0.01, 10.0, 0.0025, 37.0, 1.0],
    "mat32+bias": [0.02, 7.0, 0.001],
    "mat52+white": [0.5, 15.0, 1e-4],
    "ratquad+stdperiodic*rbf": [0.01, 8.0, 1.5, 0.5, 37.0, 1.2, 0.01, 50.0],
    "stdperiodic": [1.0, 37.0, 1.0],
}


def case_theta(kname, scale, ratio, N, d):
    """the family's theta with every lengthscale times scale and the noise at the pivot ratio (None: noise 1e-3)"""
    th = np.array(FAMILIES[kname] + [1e-3])
    names = go.KernelExpr(kname).param_names()
    for j, nm in enumerate(names):
        if nm.endswith(".lengthscale"):
            th[j] *= scale
    return th if ratio is None else xp.theta_at_ratio(kname, th, N, d, ratio)


# mat32+bias at its test lengthscale stays above the guard at any noise (pivot ratio 2.2e-2 at noise 0): the Matern 3/2
# spectrum decays too slowly for Ky to get ill-conditioned on unit steps
CASES = [(k, N, 1, s, r) for N in (256, 100) for k in FAMILIES for s in (1, 10, 100) for r in (ADMIT, REFUSE)
         if (k, s) != ("mat32+bias", 1)]
CASES += [(k, N, 1, 1, None) for N in (256, 100) for k in FAMILIES]
CASES += [("rbf+stdperiodic", 128, 2, 10, r) for r in (ADMIT, REFUSE)]


def case_id(c):
    k, N, d, s, r = c
    return f"{k}-N{N}-d{d}-ls{s}-" + ("bench" if r is None else f"r{r:g}")


def lattice_windows(N, d, first=31):
    """B windows on stamps x_0 + i d, x_0 = 20 + 2 (b mod 7), different y; the two grids"""
    _, y = syn.slip_windows(first, B, N)
    x0 = syn.T0 + 2.0 * (np.arange(B) % 7)[:, None]
    x = x0 + d * np.arange(N, dtype=float)[None, :]
    bench = x[:, -1:] + d * (1.0 + np.arange(HORIZON, dtype=float))[None, :]
    ref = x0 + d * np.arange(N + HORIZON, dtype=float)[None, :]
    return x, y, {"bench": bench, "ref": ref}


# ---------------------------------------------------------------------------------------------------------------------
# float80 references, one per case (windows with the same n and d share Ky and K*: one factor for all of them)
# ---------------------------------------------------------------------------------------------------------------------
_XP = {}


def xp_predict(c, th, x, y, xs_ref):
    if c in _XP:
        return _XP[c]
    kname, N = c[0], c[1]
    e = xp.KernelExpr(kname)
    w0 = XP_WINDOWS[0]
    out = {}
    inf0 = xp.inference(e, th[:-1], th[-1], x[w0], y[w0])
    _, var = xp.predict(e, th[:-1], th[-1], x[w0], y[w0], xs_ref[w0], inf0)
    for b in XP_WINDOWS:
        assert np.array_equal(x[b] - x[b, 0], x[w0] - x[w0, 0]) and np.array_equal(xs_ref[b] - x[b, 0], xs_ref[w0] - x[w0, 0])
        inf = xp.inference(e, th[:-1], th[-1], x[b], y[b], L=inf0.L)
        mean = xp.kernel_K(e, th[:-1], x[b], xs_ref[b]).T @ inf.alpha
        out[b] = (mean, var, inf.lml)
    kss = xp.kernel_Kdiag(e, th[:-1], x[w0, :1])[0]
    _XP[c] = out, kss
    return _XP[c]


def nerr(a, ref):
    """the parity metric: max |a - ref| / max(1, |ref|)"""
    a, ref = np.asarray(a, dtype=np.longdouble), np.asarray(ref, dtype=np.longdouble)
    return float(np.max(np.abs(a - ref) / np.maximum(1, np.abs(ref))))


def path_errors(out, refs, kss, sl):
    """worst (mean, var, lml, posterior var / k(0)) error over the xp windows; sl: the grid's slice of the xp grid"""
    e = np.zeros(4)
    for b, (mu, v, lml) in refs.items():
        e = np.maximum(e, [nerr(out[0][b], mu[sl]), nerr(out[1][b], v[sl]), nerr(out[2][b], lml),
                           float(np.max(np.abs(out[1][b] - v[sl])) / kss)])
    return e


def same_bits(p, q):
    return all(np.asarray(a).tobytes() == np.asarray(b).tobytes() for a, b in zip(p, q))


@pytest.mark.parametrize("c", CASES, ids=case_id)
def test_predict_at_the_guard(gp_ctx, monkeypatch, c):
    kname, N, d, scale, ratio = c
    th = case_theta(kname, scale, ratio, N, d)
    r = xp.pivot_ratio(kname, th, N, d)
    assert abs(r - GUARD) > 0.2 * GUARD, r            # every case is clearly on one side
    admitted = r >= GUARD
    x, y, grids = lattice_windows(N, d)
    refs, kss = xp_predict(c, th, x, y, grids["ref"])
    x0 = x[:, :1]
    thB = np.ascontiguousarray(np.tile(th, (B, 1)))
    report = []
    for gname, xs in grids.items():
        monkeypatch.delenv("CNGP_NO_LAG_TABLES", raising=False)
        out = {"a": gp_ctx.predict(kname, thB, x, y, xs), "b": gp_ctx.predict(kname, th, x, y, xs),
               "c": gp_ctx.predict(kname, th, 2.0 * x0 - x, y, 2.0 * x0 - xs)}
        monkeypatch.setenv("CNGP_NO_LAG_TABLES", "1")
        out["d"] = gp_ctx.predict(kname, th, x, y, xs)
        monkeypatch.delenv("CNGP_NO_LAG_TABLES", raising=False)
        for p in out.values():
            assert np.all(p[3] == 0)

        # which side of the guard each path took
        assert same_bits(out["b"], out["a"]), (gname, "the group path differs from the per-window path")
        if admitted:
            differ = np.mean(out["a"][2] != out["c"][2])
            assert differ > 0.5, (gname, r, differ, "an admitted case did not take the Schur fit")
        else:
            assert same_bits(out["a"], out["c"]), (gname, r, "a refused case did not stay on the tile path")

        sl = slice(0, N + HORIZON) if gname == "ref" else slice(N, N + HORIZON)
        errs = {p: path_errors(o, refs, kss, sl) for p, o in out.items()}
        for p, e in errs.items():
            assert np.all(e[:3] < TOL), (gname, p, r, e)
            report.append(f"{gname:5s} {p} mean {e[0]:.1e} var {e[1]:.1e} lml {e[2]:.1e} post {e[3]:.1e}")
        for p in ("a", "b"):
            assert np.all(errs[p] <= 10.0 * errs["c"] + 1e-13), (gname, p, r, errs[p], errs["c"])
    print(f"\n[{case_id(c)}] pivot ratio {r:.3e} ({'admitted' if admitted else 'refused'}) noise {th[-1]:.3e}\n  "
          + "\n  ".join(report))


# ---------------------------------------------------------------------------------------------------------------------
# LML gradient from the Schur factor
# ---------------------------------------------------------------------------------------------------------------------
GRAD_B = 80
GRAD_CASES = [(k, 256, 1, s) for k in FAMILIES for s in (1, 10, 100) if (k, s) != ("mat32+bias", 1)]
GRAD_CASES += [("rbf+stdperiodic", 128, 2, 10)]


@pytest.mark.parametrize("c", GRAD_CASES, ids=lambda c: f"{c[0]}-N{c[1]}-d{c[2]}-ls{c[3]}")
def test_lml_grad_at_the_guard(gp_ctx, c):
    """C = 2 candidates (pivot ratios 1.5e-2 and 2e-2) x 80 windows = 160 problems: the Schur fit feeds the gradient
    (the uniform diagonal-sum contraction for d = 1, the general one for d = 2); the same windows one candidate per
    call (80 problems) take the tile Cholesky"""
    kname, N, d, scale = c
    x, y, _ = lattice_windows(N, d, first=17)
    x, y = x[:GRAD_B], y[:GRAD_B]
    th = np.stack([case_theta(kname, scale, ADMIT, N, d), case_theta(kname, scale, 2e-2, N, d)])
    lml, grad, status = gp_ctx.lml_grad(kname, th, x, y)
    assert np.all(status == 0)
    tile = [gp_ctx.lml_grad(kname, th[i:i + 1], x, y) for i in range(2)]
    assert all(np.all(t[2] == 0) for t in tile)
    # the Schur fit ran: its LML bits differ from the tile path's on most windows
    assert np.mean(lml != np.concatenate([t[0] for t in tile])) > 0.5
    e = xp.KernelExpr(kname)
    worst = np.zeros((2, 3))
    for ci in range(2):
        inf0 = None
        for b in (0, 1, GRAD_B - 1):
            inf = xp.inference(e, th[ci, :-1], th[ci, -1], x[b], y[b], want_grad=True,
                               L=None if inf0 is None else inf0.L, Kinv=None if inf0 is None else inf0.Kinv)
            if inf0 is None:
                inf0 = inf
            es = nerr(grad[ci, b], inf.grad)
            et = nerr(tile[ci][1][0, b], inf.grad)
            worst[ci] = np.maximum(worst[ci], [es, et, nerr(lml[ci, b], inf.lml)])
            assert es < 1e-8 and et < 1e-8, (ci, b, es, et)
            assert nerr(lml[ci, b], inf.lml) < TOL
        assert worst[ci, 0] <= 10.0 * worst[ci, 1] + 1e-12, (ci, worst[ci])
    print(f"\n[grad {kname} N{N} d{d} ls{scale}] " + " | ".join(
        f"ratio {xp.pivot_ratio(kname, th[ci], N, d):.2e}: schur {worst[ci, 0]:.1e} tile {worst[ci, 1]:.1e} "
        f"lml {worst[ci, 2]:.1e}" for ci in range(2)))
