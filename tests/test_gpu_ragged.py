"""GPU parity of the ragged entry points (cngp_*_ragged): every window of a call has its own number of training points
n[b] and test points m[b], as the recorder's windows do.  Each window is compared with the oracle on its own valid
entries (true-relative 1e-9 in FP64, as tests/test_gpu_predict.py), with the fixed-size entry points where the shapes
agree (bit for bit), and padding beyond n[b] / m[b] is shown to be neither read nor written."""
import ctypes as C

import numpy as np
import pytest
import torch

from corenav_gp_b200 import synthetic as syn
from corenav_gp_b200 import _lib as L
from corenav_gp_b200.api import CngpError, GpContext, parse_kernel
from oracle import gp_oracle as go
from oracle import stop_oracle as so

pytestmark = pytest.mark.gpu
TOL = 1e-9

KERNELS = [
    ("rbf", [0.01, 10.0]),
    ("rbf+stdperiodic", [0.01, 10.0, 0.0025, 37.0, 1.0]),
    ("rbf*brownian", [0.01, 10.0, 0.05]),
    ("mat32+bias", [0.02, 7.0, 0.001]),
    ("mat52*linear+white", [0.5, 15.0, 1e-5, 1e-4]),
    ("ratquad+stdperiodic*rbf", [0.01, 8.0, 1.5, 0.5, 37.0, 1.2, 0.01, 50.0]),
    ("(rbf+linear)*brownian+white", [0.02, 12.0, 1e-6, 0.03, 2e-4]),
]


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.max(np.abs(a - b) / np.maximum(1.0, np.abs(b)))) if a.size else 0.0


@pytest.fixture(scope="module")
def small_ctx():
    """A context whose scratch holds only a few hundred windows: chunks split the buckets."""
    ctx = GpContext(device=0, scratch_bytes=48 << 20)
    yield ctx
    ctx.close()


def ragged_set(seed=0, integer=True, fill=0.0, mmax=40):
    """~300 windows: n covers every tile bucket 1..32 and every residue n % 8; m varies per window (0 included)."""
    rng = np.random.default_rng(seed)
    n = np.concatenate([np.arange(1, 257), rng.integers(1, 257, 44)]).astype(np.int32)
    rng.shuffle(n)
    B, ld = n.size, 256
    m = rng.integers(0, mmax + 1, B).astype(np.int32)
    ldm = mmax + 3
    x = np.full((B, ld), fill)
    y = np.full((B, ld), fill)
    xs = np.full((B, ldm), fill)
    xw, yw = syn.slip_windows(0, B, ld)
    for b in range(B):
        k = n[b]
        t = xw[b, :k] + 7.0 * b
        if not integer:
            t = t + np.linspace(0.0, 0.37, k) + 0.013 * b
        x[b, :k], y[b, :k] = t, yw[b, :k]
        xs[b, :m[b]] = t[0] + (np.arange(m[b]) * 1.5 - 3.0 if integer else np.linspace(-2.3, k + 5.1, m[b]))
    return x, y, n, xs, m


def check_predict(kname, th, x, y, n, xs, m, mean, var, lml, status, tol=TOL):
    e = go.KernelExpr(kname)
    assert np.all(status == 0)
    for b in range(x.shape[0]):
        k, mb = n[b], m[b]
        tb = th[b] if th.ndim == 2 else th
        inf = go.inference(e, tb[:-1], tb[-1], x[b, :k], y[b, :k])
        assert rel(lml[b], inf.lml) < tol, (b, k)
        if mb:
            mu, v = go.predict(e, tb[:-1], tb[-1], x[b, :k], y[b, :k], xs[b, :mb], inf)
            assert rel(mean[b, :mb], mu) < tol and rel(var[b, :mb], v) < tol, (b, k, mb)


@pytest.mark.parametrize("integer", [True, False], ids=["table", "lazy"])
@pytest.mark.parametrize("kname,theta", KERNELS)
def test_predict_ragged_matches_oracle(gp_ctx, kname, theta, integer):
    x, y, n, xs, m = ragged_set(1, integer)
    rng = np.random.default_rng(2)
    th = np.array(theta + [2e-3])[None, :] * rng.uniform(0.8, 1.25, (x.shape[0], len(theta) + 1))
    mean, var, lml, status = gp_ctx.predict_ragged(kname, th, x, y, n, xs, m)
    check_predict(kname, th, x, y, n, xs, m, mean, var, lml, status)


def test_predict_ragged_fp32_mode(gp_ctx32):
    kname, theta = KERNELS[2]
    x, y, n, xs, m = ragged_set(3)
    th = np.array(theta + [2e-3])
    mean, var, lml, status = gp_ctx32.predict_ragged(kname, th, x, y, n, xs, m)
    assert np.all(status == 0)
    e = go.KernelExpr(kname)
    for b in range(x.shape[0]):
        k, mb = n[b], m[b]
        if not mb:
            continue
        mu, v = go.predict(e, th[:-1], th[-1], x[b, :k], y[b, :k], xs[b, :mb])
        assert np.linalg.norm(mean[b, :mb] - mu) <= 1e-4 * max(1.0, np.linalg.norm(mu))
        assert np.linalg.norm(var[b, :mb] - v) <= 1e-4 * max(1.0, np.linalg.norm(v))


@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
def test_padding_is_invisible(gp_ctx, device):
    kname, theta = KERNELS[1]
    th = np.array(theta + [2e-3])
    x0, y0, n, xs0, m = ragged_set(4, fill=0.0)
    xn, yn, _, xsn, _ = ragged_set(4, fill=np.nan)
    n = n.copy()
    n[::17] = 0                                           # skipped windows
    runs = []
    for x, y, xs in ((x0, y0, xs0), (xn, yn, xsn)):
        args = [th, x, y, n, xs, m]
        if device:
            args = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in args]
        runs.append(gp_ctx.predict_ragged(kname, *args))
    out = [[np.asarray(a.cpu() if device else a) for a in r] for r in runs]
    valid = np.arange(xs0.shape[1])[None, :] < m[:, None]
    live = n > 0
    for a, b in zip(out[0][:2], out[1][:2]):
        assert np.array_equal(a[valid & live[:, None]], b[valid & live[:, None]])
    assert np.array_equal(out[0][2][live], out[1][2][live])
    assert np.array_equal(out[0][3], out[1][3]) and np.all(out[0][3][~live] == 0)
    # outputs beyond m[b] (and of skipped windows) are not written: sentinel buffers come back untouched
    B, ldm = xs0.shape
    sent = -12345.0
    mean = np.full((B, ldm), sent); var = np.full((B, ldm), sent); lml = np.full(B, sent); st = np.full(B, 7, np.int32)
    kp = parse_kernel(kname)
    xn_, yn_, xsn_ = (np.ascontiguousarray(a) for a in (xn, yn, xsn))
    rc = gp_ctx.lib.cngp_predict_ragged(gp_ctx.h, C.byref(kp), th.ctypes.data, 0, xn_.ctypes.data, yn_.ctypes.data,
                                        n.ctypes.data, xn_.shape[1], xsn_.ctypes.data, m.ctypes.data, ldm, B,
                                        mean.ctypes.data, var.ctypes.data, lml.ctypes.data, st.ctypes.data, L.MEM_HOST)
    assert rc == 0
    assert np.all(mean[~(valid & live[:, None])] == sent) and np.all(var[~(valid & live[:, None])] == sent)
    assert np.all(lml[~live] == sent) and np.all(st[~live] == 0)
    assert np.array_equal(mean[valid & live[:, None]], out[1][0][valid & live[:, None]])


@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("N", [149, 64, 5])
def test_all_equal_batch_equals_predict_batch(gp_ctx, device, N):
    kname, theta = KERNELS[2]
    B, M = 40, 57
    x, y = syn.slip_windows(9, B, N)
    x = x + 3.0 * np.arange(B)[:, None]
    xs = np.stack([syn.test_grid(x[b], M) for b in range(B)])
    th = np.array(theta + [1e-3])
    n = np.full(B, N, np.int32)
    m = np.full(B, M, np.int32)
    conv = (lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()) if device else (lambda a: a)
    ref = gp_ctx.predict(kname, conv(th), conv(x), conv(y), conv(xs))
    out = gp_ctx.predict_ragged(kname, conv(th), conv(x), conv(y), conv(n), conv(xs), conv(m))
    g = (lambda a: a.cpu().numpy()) if device else (lambda a: a)
    for a, b in zip(ref, out):
        assert np.array_equal(g(a), g(b))


def test_gp_slip_ragged_equals_batch_on_equal_windows(gp_ctx):
    B, n = 6, 149
    x, y = syn.slip_windows(50, B, n)
    x = x + 10.0 * np.arange(B)[:, None]
    th = syn.theta_for("rbf*brownian")
    mean, sigma, status = gp_ctx.gp_slip("rbf*brownian", x, y, theta=th)
    mr, sr, mo, st = gp_ctx.gp_slip_ragged("rbf*brownian", x, y, np.full(B, n, np.int32), theta=th)
    M = mean.shape[1]
    assert np.all(mo == M)
    assert np.array_equal(mr[:, :M], mean) and np.array_equal(sr[:, :M], sigma) and np.array_equal(st, status)


@pytest.mark.parametrize("integer", [True, False], ids=["uniform", "irregular"])
@pytest.mark.parametrize("kname,theta", KERNELS)
def test_lml_grad_ragged_matches_oracle(gp_ctx, kname, theta, integer):
    rng = np.random.default_rng(8)
    n = np.array([1, 7, 8, 9, 30, 64, 100, 134, 149, 152, 153, 200, 255, 256, 0, 17], np.int32)
    B, ld = n.size, 260
    x = np.full((B, ld), np.nan)
    y = np.full((B, ld), np.nan)
    xw, yw = syn.slip_windows(20, B, 256)
    for b in range(B):
        t = xw[b, :n[b]] + 5.0 * b
        if not integer:
            t = t + np.cumsum(rng.uniform(0.0, 0.4, n[b]))
        x[b, :n[b]], y[b, :n[b]] = t, yw[b, :n[b]]
    th = np.array(theta + [2e-3])[None, :] * np.array([[1.0], [1.2]])
    lml, grad, status = gp_ctx.lml_grad_ragged(kname, th, x, y, n)
    e = go.KernelExpr(kname)
    for c in range(th.shape[0]):
        for b in range(B):
            if n[b] == 0:
                assert status[c, b] == 0
                continue
            assert status[c, b] == 0
            inf = go.inference(e, th[c, :-1], th[c, -1], x[b, :n[b]], y[b, :n[b]], want_grad=True)
            assert rel(lml[c, b], inf.lml) < 1e-8
            assert rel(grad[c, b], inf.grad) < 1e-8, (kname, c, b, n[b])


def test_optimize_ragged_equals_per_window_fits(gp_ctx):
    """Windows of 20..150 points in one call: every window ends where a fit of that window alone ends (same kernels,
    same state machine), its LML is the oracle's at the returned theta, and host and device calls agree bit for bit."""
    kname = "rbf*brownian"
    n = np.array([20, 45, 64, 97, 134, 150], np.int32)
    B, ld = n.size, 150
    x = np.full((B, ld), np.nan)
    y = np.full((B, ld), np.nan)
    xw, yw = syn.slip_windows(70, B, ld)
    for b in range(B):
        x[b, :n[b]], y[b, :n[b]] = xw[b, :n[b]] + 9.0 * b, yw[b, :n[b]]
    th, lml, it = gp_ctx.optimize_ragged(kname, x, y, n)
    dev = gp_ctx.optimize_ragged(kname, *(torch.from_numpy(a).cuda() for a in (x, y, n)))
    assert np.array_equal(th, dev[0].cpu().numpy()) and np.array_equal(lml, dev[1].cpu().numpy())
    e = go.KernelExpr(kname)
    for b in range(B):
        k = n[b]
        t1, l1, i1 = gp_ctx.optimize(kname, x[b:b + 1, :k], y[b:b + 1, :k])
        assert np.array_equal(th[b], t1[0]) and lml[b] == l1[0] and it[b] == i1[0]
        inf = go.inference(e, th[b, :-1], th[b, -1], x[b, :k], y[b, :k])
        assert rel(lml[b], inf.lml) < TOL


def recorder_windows(count, T=420, max_windows=3, seed_first=0):
    d = syn.drives(seed_first, count, T=T, pauses=True)
    dev = {k: torch.from_numpy(v).cuda() for k, v in d.items()}
    return d, dev


def test_gp_slip_ragged_on_recorder_output(gp_ctx):
    cap = 150
    d, dev = recorder_windows(48)
    rec = gp_ctx.slip_record(dev["joint"], dev["att"], dev["vel"], dev["cmd"], dev["stop_cmd"], max_windows=3, cap=cap)
    ns, pub = rec["n_samples"], rec["published"]
    assert int(ns.max()) <= cap
    n = torch.where(pub != 0, ns, torch.zeros_like(ns)).reshape(-1).to(torch.int32)
    t = rec["time_array"].reshape(-1, cap)
    s = rec["slip_array"].reshape(-1, cap)
    kname = "rbf*brownian"
    th = syn.theta_for(kname)
    mean, sigma, m_out, status = gp_ctx.gp_slip_ragged(kname, t, s, n, theta=torch.from_numpy(th).cuda())
    torch.cuda.synchronize()
    nh, th_, sh = n.cpu().numpy(), t.cpu().numpy(), s.cpu().numpy()
    mh, sgh, moh, sth = (a.cpu().numpy() for a in (mean, sigma, m_out, status))
    assert (nh > 0).sum() >= 40 and len(set(nh[nh > 0].tolist())) > 5      # the fixture is ragged
    e = go.KernelExpr(kname)
    for b in np.nonzero(nh)[0]:
        k = nh[b]
        mu, sg = go.gp_slip_callback(th_[b, :k], sh[b, :k], e, theta=th[:-1], noise=th[-1])
        assert moh[b] == mu.size and sth[b] == 0
        assert rel(mh[b, :mu.size], mu) < TOL and rel(sgh[b, :mu.size], sg) < TOL
    assert np.all(moh[nh == 0] == 0) and np.all(sth[nh == 0] == 0)
    # with the fit, on a few windows (the bars of test_gp_slip_callback_with_fit)
    pick = np.nonzero(nh)[0][[0, 3, 7]]
    sel = torch.from_numpy(pick).cuda()
    mf, sf, mof, stf = gp_ctx.gp_slip_ragged(kname, t[sel], s[sel], n[sel])
    for i, b in enumerate(pick):
        k = nh[b]
        mu, sg = go.gp_slip_callback(th_[b, :k], sh[b, :k], e)
        mfi, sfi = mf[i].cpu().numpy()[:mu.size], sf[i].cpu().numpy()[:mu.size]
        assert int(stf[i]) == 0 and np.max(np.abs(mfi - mu)) < 1e-5 and np.max(np.abs(sfi - sg) / sg) < 1e-4
    # n < 2 publishes nothing; n > ld is refused
    n2 = n.clone()
    n2[0] = 1
    _, _, mo2, st2 = gp_ctx.gp_slip_ragged(kname, t, s, n2, theta=torch.from_numpy(th).cuda())
    assert int(mo2[0]) == 0 and int(st2[0]) == 0
    n2[1] = cap + 1
    with pytest.raises(CngpError):
        gp_ctx.gp_slip_ragged(kname, t, s, n2, theta=torch.from_numpy(th).cuda())


def ocfg():
    return so.default_cfg(trig_mode=1)


def lookahead_ref(mean, sigma, m, ctx, b):
    pw = lambda a: a[b] if a.ndim == 2 else a
    if m == 0:
        return dict(triggered=0, i_stop=0, step_stop=0, xy_err=0.0)
    return so.lookahead(mean[:m], sigma[:m], pw(ctx["P"]), pw(ctx["Q"]), pw(ctx["STM"]), pw(ctx["Hvec"]), pw(ctx["pos"]),
                        ocfg())


@pytest.mark.parametrize("kern", ["tc", "warp", "cta"])
def test_lookahead_ragged_matches_oracle(gp_ctx, monkeypatch, kern):
    monkeypatch.setenv("CNGP_LOOKAHEAD_KERNEL", kern)
    B, ldm = 96, 620
    rng = np.random.default_rng(11)
    m = rng.integers(0, ldm + 1, B).astype(np.int32)
    m[:3] = [0, 1, ldm]
    k = np.arange(ldm)
    mean = 0.05 * np.exp(-k / 80.0)[None, :] * rng.uniform(-1, 1, (B, 1)) + 0.01 * rng.standard_normal((B, ldm))
    sigma = 2.0 * np.sqrt(1e-3 + 0.01 * (1 - np.exp(-k / 150.0)))[None, :] * rng.uniform(0.7, 1.3, (B, 1))
    mask = k[None, :] >= m[:, None]
    mean[mask] = np.nan
    sigma[mask] = np.nan
    ctx = syn.monte_carlo_contexts(0, B)
    out = gp_ctx.zupt_lookahead(mean, sigma, ctx["P"], ctx["Q"], ctx["STM"], ctx["Hvec"], ctx["pos"], m=m)
    for b in range(B):
        ref = lookahead_ref(mean[b], sigma[b], m[b], ctx, b)
        for key in ("triggered", "i_stop", "step_stop", "xy_err"):
            assert out[key][b] == ref[key], (kern, b, m[b], key)
    # equal m: the fixed-size call, bit for bit
    mean2, sigma2 = np.nan_to_num(mean[:, :300]), np.nan_to_num(sigma[:, :300])
    full = gp_ctx.zupt_lookahead(mean2, sigma2, ctx["P"], ctx["Q"], ctx["STM"], ctx["Hvec"], ctx["pos"], want_state=True)
    rag = gp_ctx.zupt_lookahead(mean2, sigma2, ctx["P"], ctx["Q"], ctx["STM"], ctx["Hvec"], ctx["pos"], want_state=True,
                                m=np.full(B, 300, np.int32))
    for key in full:
        assert np.array_equal(full[key], rag[key]), key


@pytest.mark.parametrize("which", ["default", "small_scratch"])
def test_end_to_end_at_size(gp_ctx, small_ctx, which):
    """~4096 recorder windows: recorder -> callback -> look-ahead on the device with no host copy in between; 64 windows
    (first and last of every bucket, the last window overall) checked against the oracles."""
    ctx_ = gp_ctx if which == "default" else small_ctx
    cap, W = 150, 2
    d, dev = recorder_windows(2048, T=420, seed_first=100)
    rec = ctx_.slip_record(dev["joint"], dev["att"], dev["vel"], dev["cmd"], dev["stop_cmd"], max_windows=W, cap=cap)
    assert int(rec["n_samples"].max()) <= cap
    n = torch.where(rec["published"] != 0, rec["n_samples"], torch.zeros_like(rec["n_samples"])).reshape(-1).to(torch.int32)
    t, s = rec["time_array"].reshape(-1, cap), rec["slip_array"].reshape(-1, cap)
    kname = "rbf*brownian"
    th = syn.theta_for(kname)
    mean, sigma, m_out, status = ctx_.gp_slip_ragged(kname, t, s, n, theta=torch.from_numpy(th).cuda())
    B = n.numel()
    mc = syn.monte_carlo_contexts(0, B)
    cdev = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in mc.items()}
    la = ctx_.zupt_lookahead(mean, sigma, cdev["P"], cdev["Q"], cdev["STM"], cdev["Hvec"], cdev["pos"], m=m_out)
    torch.cuda.synchronize()
    nh = n.cpu().numpy()
    live = np.nonzero(nh)[0]
    ntr = (0.9 * nh).astype(np.int64)
    bucket = (ntr + 7) // 8
    pick = set()
    for k in np.unique(bucket[live]):
        idx = live[bucket[live] == k]
        pick.update([idx[0], idx[-1]])
    pick.add(live[-1])
    rng = np.random.default_rng(0)
    rest = np.setdiff1d(live, list(pick))
    pick.update(rng.choice(rest, 64 - len(pick), replace=False).tolist())
    th_, sh = t.cpu().numpy(), s.cpu().numpy()
    mh, sgh, moh, sth = (a.cpu().numpy() for a in (mean, sigma, m_out, status))
    lah = {k: v.cpu().numpy() for k, v in la.items()}
    e = go.KernelExpr(kname)
    for b in sorted(pick):
        k = nh[b]
        mu, sg = go.gp_slip_callback(th_[b, :k], sh[b, :k], e, theta=th[:-1], noise=th[-1])
        assert moh[b] == mu.size and sth[b] == 0
        assert rel(mh[b, :mu.size], mu) < TOL and rel(sgh[b, :mu.size], sg) < TOL
        ref = lookahead_ref(mh[b], sgh[b], moh[b], mc, b)
        for key in ("triggered", "i_stop", "step_stop", "xy_err"):
            assert lah[key][b] == ref[key], (b, key)
    assert np.all(moh[nh == 0] == 0) and np.all(lah["triggered"][nh == 0] == 0)
