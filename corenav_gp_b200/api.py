"""Python host API over the C ABI (include/cngp.h).

`GpContext` is one GPU context.  Every method takes either host arrays (numpy / CPU torch tensors, pinned or not:
the library copies in and out inside the call) or CUDA torch tensors (device pointers are passed straight through
and the kernels are enqueued on torch's current stream).  Nothing here computes: it only marshals pointers.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Union

import numpy as np

from . import _lib as L

try:  # torch is plumbing (device memory, streams, torch.distributed); the library itself does not need it
    import torch
except Exception:  # pragma: no cover
    torch = None


class CngpError(RuntimeError):
    pass


def parse_kernel(text: Union[str, L.Kernel]) -> L.Kernel:
    """'rbf*brownian', 'se+periodic', '(rbf+linear)*brownian+white' ... -> postfix program (cngp_kernel)."""
    if isinstance(text, L.Kernel):
        return text
    k = L.Kernel()
    rc = L.load().cngp_kernel_parse(text.encode(), C.byref(k))
    if rc != 0:
        raise CngpError(f"cannot parse kernel expression {text!r} (rc={rc})")
    return k


def _is_cuda(a) -> bool:
    return torch is not None and isinstance(a, torch.Tensor) and a.is_cuda


class _Arg:
    """Pointer + keep-alive for one array argument."""

    def __init__(self, a, dtype, device_mode: bool, allow_none=False, output=False):
        """Inputs are coerced (dtype, contiguity).  OUTPUTS are never coerced: the library writes through the pointer,
        so a converted copy would leave the caller's buffer untouched - a wrong dtype or a non-contiguous output raises."""
        self.keep = None
        self.ptr = None
        if a is None:
            assert allow_none
            return
        is_tensor = torch is not None and isinstance(a, torch.Tensor)
        if device_mode and not _is_cuda(a):
            raise CngpError("mixing host and device arrays in one call")
        if is_tensor:
            tdt = torch.float64 if dtype == np.float64 else torch.int32
            if a.dtype != tdt or not a.is_contiguous():
                if output:
                    raise CngpError(f"output buffer must be a contiguous {tdt} tensor (got {a.dtype}, "
                                    f"contiguous={a.is_contiguous()})")
                a = a.to(tdt).contiguous()
            self.keep = a
            self.ptr = a.data_ptr()
        else:
            if output:
                if not (isinstance(a, np.ndarray) and a.dtype == dtype and a.flags.c_contiguous and a.flags.writeable):
                    raise CngpError(f"output buffer must be a writeable C-contiguous numpy array of {np.dtype(dtype)}")
            else:
                a = np.ascontiguousarray(a, dtype=dtype)
            self.keep = a
            self.ptr = a.ctypes.data


class GpContext:
    PRECISIONS = {"f64": 0, "f32": 1}

    def __init__(self, device: int = 0, jitter_retry: bool = False, scratch_bytes: int = 0, precision: str = "f64"):
        """precision: "f64" (1e-9 parity, default) or "f32" (north_star's 1e-4 mode: the predictive mean / variance
        phase runs as 3xTF32 on the tensor cores; arrays stay float64 at the interface)."""
        self.lib = L.load()
        cfg = L.Config()
        self.lib.cngp_default_config(C.byref(cfg))
        cfg.device = device
        cfg.jitter_retry = int(jitter_retry)
        cfg.scratch_bytes = scratch_bytes
        cfg.precision = self.PRECISIONS[precision]
        h = C.c_void_p()
        rc = self.lib.cngp_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise CngpError(f"cngp_create failed (rc={rc}): {self.lib.cngp_last_error(None).decode()}")
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.cngp_destroy(self.h)
            self.h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise CngpError(f"{what} failed (rc={rc}): {self.lib.cngp_last_error(self.h).decode()}")

    def sync(self):
        self._check(self.lib.cngp_sync(self.h), "cngp_sync")

    def set_precision(self, precision: str):
        self._check(self.lib.cngp_set_precision(self.h, self.PRECISIONS[precision]), "cngp_set_precision")

    def launch_count(self) -> int:
        return int(self.lib.cngp_launch_count(self.h))

    def set_profiling(self, on: bool):
        self._check(self.lib.cngp_set_profiling(self.h, int(on)), "cngp_set_profiling")

    def profile_read(self, kernel_id: int, reset: bool = True):
        """(total milliseconds, launches) of one kernel class since the last reset (CUDA events, launching stream)."""
        ms, n = C.c_double(0.0), C.c_int64(0)
        self._check(self.lib.cngp_profile_read(self.h, kernel_id, C.byref(ms), C.byref(n), int(reset)),
                    "cngp_profile_read")
        return ms.value, n.value

    def _bind_stream(self, device_mode: bool):
        if device_mode:
            self.lib.cngp_set_stream(self.h, C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream), 0)
        else:
            self.lib.cngp_set_stream(self.h, None, 1)

    def _empty(self, shape, dtype, device_mode, like=None):
        if device_mode:
            return torch.empty(shape, dtype=torch.float64 if dtype == np.float64 else torch.int32,
                               device=f"cuda:{self.device}")
        return np.empty(shape, dtype=dtype)

    # ------------------------------------------------------------------------------------------------------
    def predict(self, kernel, theta, x, y, xstar, want_lml: bool = True, out=None):
        """Exact-GP predictive mean / variance for B windows.  theta [P] or [B,P]; x, y [B,N]; xstar [M] or [B,M].

        Returns (mean [B,M], var [B,M], lml [B] or None, status [B]).  `out` = (mean, var, lml, status) buffers to
        reuse (host: numpy or pinned torch tensors; device: CUDA tensors)."""
        k = parse_kernel(kernel)
        dev = _is_cuda(x)
        B, N = x.shape
        P = k.n_params + 1
        th_shape = tuple(theta.shape)
        theta_stride = 0 if len(th_shape) == 1 else th_shape[1]
        if th_shape[-1] != P:
            raise CngpError(f"theta has {th_shape[-1]} entries, kernel needs {P} (noise last)")
        xs_shape = tuple(xstar.shape)
        M = xs_shape[-1]
        xstar_stride = 0 if len(xs_shape) == 1 else M
        if out is None:
            mean = self._empty((B, M), np.float64, dev)
            var = self._empty((B, M), np.float64, dev)
            lml = self._empty((B,), np.float64, dev) if want_lml else None
            status = self._empty((B,), np.int32, dev)
        else:
            mean, var, lml, status = out
        a = [_Arg(theta, np.float64, dev), _Arg(x, np.float64, dev), _Arg(y, np.float64, dev),
             _Arg(xstar, np.float64, dev), _Arg(mean, np.float64, dev, output=True),
             _Arg(var, np.float64, dev, output=True), _Arg(lml, np.float64, dev, True, output=True),
             _Arg(status, np.int32, dev, output=True)]
        self._bind_stream(dev)
        rc = self.lib.cngp_predict_batch(self.h, C.byref(k), a[0].ptr, theta_stride, a[1].ptr, a[2].ptr, a[3].ptr,
                                         xstar_stride, B, N, M, a[4].ptr, a[5].ptr, a[6].ptr, a[7].ptr,
                                         L.MEM_DEVICE if dev else L.MEM_HOST)
        self._check(rc, "cngp_predict_batch")
        return mean, var, lml, status

    def lml_grad(self, kernel, theta, x, y, want_grad: bool = True):
        """LML (and d LML / d theta) for C candidates x B windows.  theta [C,P]; returns lml [C,B], grad [C,B,P], status."""
        k = parse_kernel(kernel)
        dev = _is_cuda(x)
        B, N = x.shape
        Cn, P = theta.shape
        if P != k.n_params + 1:
            raise CngpError(f"theta has {P} entries, kernel needs {k.n_params + 1} (noise last)")
        lml = self._empty((Cn, B), np.float64, dev)
        grad = self._empty((Cn, B, P), np.float64, dev) if want_grad else None
        status = self._empty((Cn, B), np.int32, dev)
        a = [_Arg(theta, np.float64, dev), _Arg(x, np.float64, dev), _Arg(y, np.float64, dev),
             _Arg(lml, np.float64, dev, output=True), _Arg(grad, np.float64, dev, True, output=True),
             _Arg(status, np.int32, dev, output=True)]
        self._bind_stream(dev)
        rc = self.lib.cngp_lml_grad_batch(self.h, C.byref(k), a[0].ptr, Cn, a[1].ptr, a[2].ptr, B, N, a[3].ptr,
                                          a[4].ptr, a[5].ptr, L.MEM_DEVICE if dev else L.MEM_HOST)
        self._check(rc, "cngp_lml_grad_batch")
        return lml, grad, status

    def optimize(self, kernel, x, y, theta0=None, max_iters: int = 1000):
        """Batched m.optimize(): returns (theta [B,P], lml [B], iters [B]).  Host arrays, or CUDA tensors (then the
        results are CUDA tensors too and the whole fit stays on the device)."""
        k = parse_kernel(kernel)
        if _is_cuda(x):
            B, N = x.shape
            P = k.n_params + 1
            th0 = torch.ones(P, dtype=torch.float64, device=x.device) if theta0 is None else theta0
            stride = 0 if th0.dim() == 1 else P
            theta = torch.empty((B, P), dtype=torch.float64, device=x.device)
            lml = torch.empty(B, dtype=torch.float64, device=x.device)
            iters = torch.empty(B, dtype=torch.int32, device=x.device)
            a = [_Arg(th0, np.float64, True), _Arg(x, np.float64, True), _Arg(y, np.float64, True),
                 _Arg(theta, np.float64, True, output=True), _Arg(lml, np.float64, True, output=True),
                 _Arg(iters, np.int32, True, output=True)]
            self._bind_stream(True)
            rc = self.lib.cngp_optimize_batch_mem(self.h, C.byref(k), a[0].ptr, stride, a[1].ptr, a[2].ptr, B, N, max_iters,
                                                  a[3].ptr, a[4].ptr, a[5].ptr, L.MEM_DEVICE)
            self._check(rc, "cngp_optimize_batch_mem")
            return theta, lml, iters
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.ascontiguousarray(y, dtype=np.float64)
        B, N = x.shape
        P = k.n_params + 1
        if theta0 is None:
            theta0 = np.ones(P)
        theta0 = np.ascontiguousarray(theta0, dtype=np.float64)
        stride = 0 if theta0.ndim == 1 else P
        theta = np.empty((B, P))
        lml = np.empty(B)
        iters = np.empty(B, dtype=np.int32)
        self._bind_stream(False)
        rc = self.lib.cngp_optimize_batch(self.h, C.byref(k), theta0.ctypes.data, stride, x.ctypes.data, y.ctypes.data,
                                          B, N, max_iters, theta.ctypes.data, lml.ctypes.data, iters.ctypes.data)
        self._check(rc, "cngp_optimize_batch")
        return theta, lml, iters

    def gp_slip(self, kernel, time_array, slip_array, theta=None, horizon: int = 600):
        """The node callback for B windows [B,n]: returns (mean [B,m], sigma [B,m], status [B]); sigma = 2 sqrt(var)."""
        k = parse_kernel(kernel)
        t = np.ascontiguousarray(time_array, dtype=np.float64)
        s = np.ascontiguousarray(slip_array, dtype=np.float64)
        B, n = t.shape
        # gp_slip_node.py:45,59-61: len(arange(min, max + horizon, 1)) - n published points; the same for every window
        # of a batch (the library checks), so the outputs can be allocated at their exact size
        lens = np.ceil((t.max(axis=1) + float(horizon)) - t.min(axis=1))
        m_cap = max(1, int(lens.max()) - n)
        mean = np.empty((B, m_cap))
        sigma = np.empty((B, m_cap))
        m_out = C.c_int32(0)
        status = np.zeros(B, dtype=np.int32)
        if theta is not None:
            theta = np.ascontiguousarray(theta, dtype=np.float64)
            stride = 0 if theta.ndim == 1 else theta.shape[1]
            tptr = theta.ctypes.data
        else:
            stride, tptr = 0, None
        self._bind_stream(False)
        rc = self.lib.cngp_gp_slip_batch(self.h, C.byref(k), tptr, stride, t.ctypes.data, s.ctypes.data, B, n, horizon,
                                         m_cap, mean.ctypes.data, sigma.ctypes.data, C.addressof(m_out),
                                         status.ctypes.data)
        self._check(rc, "cngp_gp_slip_batch")
        m = m_out.value
        if m == m_cap:
            return mean, sigma, status
        return mean[:, :m].copy(), sigma[:, :m].copy(), status

    # ---- ragged windows: window b has n[b] valid entries in its row of x / y, m[b] in its row of xstar / outputs ----
    def _ragged_common(self, kernel, x, n):
        k = parse_kernel(kernel)
        dev = _is_cuda(x)
        B, ld = (int(v) for v in tuple(x.shape))
        if int(np.prod(tuple(n.shape))) != B:
            raise CngpError(f"n has {int(np.prod(tuple(n.shape)))} entries for {B} windows")
        return k, dev, B, ld, k.n_params + 1

    @staticmethod
    def _theta_stride(theta, P):
        shape = tuple(theta.shape)
        if shape[-1] != P:
            raise CngpError(f"theta has {shape[-1]} entries, kernel needs {P} (noise last)")
        return 0 if len(shape) == 1 else P

    def predict_ragged(self, kernel, theta, x, y, n, xstar, m):
        """predict() for windows of different sizes: x, y [B,ld] with n[b] valid entries in row b; xstar [B,ldm] with
        m[b] valid test points.  theta [P] or [B,P].  Returns (mean [B,ldm], var [B,ldm], lml [B], status [B]) on the
        device of the inputs; entries of mean / var beyond m[b] (and lml of windows with n[b] = 0) are left as allocated."""
        k, dev, B, ld, P = self._ragged_common(kernel, x, n)
        stride = self._theta_stride(theta, P)
        ldm = int(tuple(xstar.shape)[-1])
        mean = self._empty((B, ldm), np.float64, dev)
        var = self._empty((B, ldm), np.float64, dev)
        lml = self._empty((B,), np.float64, dev)
        status = self._empty((B,), np.int32, dev)
        a = [_Arg(theta, np.float64, dev), _Arg(x, np.float64, dev), _Arg(y, np.float64, dev), _Arg(n, np.int32, dev),
             _Arg(xstar, np.float64, dev), _Arg(m, np.int32, dev), _Arg(mean, np.float64, dev, output=True),
             _Arg(var, np.float64, dev, output=True), _Arg(lml, np.float64, dev, output=True),
             _Arg(status, np.int32, dev, output=True)]
        self._bind_stream(dev)
        rc = self.lib.cngp_predict_ragged(self.h, C.byref(k), a[0].ptr, stride, a[1].ptr, a[2].ptr, a[3].ptr, ld,
                                          a[4].ptr, a[5].ptr, ldm, B, a[6].ptr, a[7].ptr, a[8].ptr, a[9].ptr,
                                          L.MEM_DEVICE if dev else L.MEM_HOST)
        self._check(rc, "cngp_predict_ragged")
        return mean, var, lml, status

    def lml_grad_ragged(self, kernel, theta, x, y, n, want_grad: bool = True):
        """lml_grad() for windows of different sizes: theta [C,P]; x, y [B,ld] with n[b] valid entries.
        Returns lml [C,B], grad [C,B,P] (or None), status [C,B]."""
        k, dev, B, ld, P = self._ragged_common(kernel, x, n)
        Cn = int(tuple(theta.shape)[0])
        if tuple(theta.shape)[-1] != P:
            raise CngpError(f"theta has {tuple(theta.shape)[-1]} entries, kernel needs {P} (noise last)")
        lml = self._empty((Cn, B), np.float64, dev)
        grad = self._empty((Cn, B, P), np.float64, dev) if want_grad else None
        status = self._empty((Cn, B), np.int32, dev)
        a = [_Arg(theta, np.float64, dev), _Arg(x, np.float64, dev), _Arg(y, np.float64, dev), _Arg(n, np.int32, dev),
             _Arg(lml, np.float64, dev, output=True), _Arg(grad, np.float64, dev, True, output=True),
             _Arg(status, np.int32, dev, output=True)]
        self._bind_stream(dev)
        rc = self.lib.cngp_lml_grad_ragged(self.h, C.byref(k), a[0].ptr, Cn, a[1].ptr, a[2].ptr, a[3].ptr, ld, B,
                                           a[4].ptr, a[5].ptr, a[6].ptr, L.MEM_DEVICE if dev else L.MEM_HOST)
        self._check(rc, "cngp_lml_grad_ragged")
        return lml, grad, status

    def optimize_ragged(self, kernel, x, y, n, theta0=None, max_iters: int = 1000):
        """optimize() for windows of different sizes: x, y [B,ld] with n[b] valid entries.  theta0 None (all ones),
        [P] or [B,P].  Returns (theta [B,P], lml [B], iters [B]) on the device of the inputs."""
        k, dev, B, ld, P = self._ragged_common(kernel, x, n)
        stride = 0 if theta0 is None else self._theta_stride(theta0, P)
        theta = self._empty((B, P), np.float64, dev)
        lml = self._empty((B,), np.float64, dev)
        iters = self._empty((B,), np.int32, dev)
        a = [_Arg(theta0, np.float64, dev, True), _Arg(x, np.float64, dev), _Arg(y, np.float64, dev),
             _Arg(n, np.int32, dev), _Arg(theta, np.float64, dev, output=True), _Arg(lml, np.float64, dev, output=True),
             _Arg(iters, np.int32, dev, output=True)]
        self._bind_stream(dev)
        rc = self.lib.cngp_optimize_ragged(self.h, C.byref(k), a[0].ptr, stride, a[1].ptr, a[2].ptr, a[3].ptr, ld, B,
                                           max_iters, a[4].ptr, a[5].ptr, a[6].ptr, L.MEM_DEVICE if dev else L.MEM_HOST)
        self._check(rc, "cngp_optimize_ragged")
        return theta, lml, iters

    def gp_slip_ragged(self, kernel, time_array, slip_array, n, theta=None, horizon: int = 600, ldm: Optional[int] = None):
        """The node callback for windows of different sizes: time_array, slip_array [B,ld] with n[b] samples in row b
        (e.g. slip_record's [B*max_windows, cap] rows with n = where(published, n_samples, 0)).  Returns (mean [B,ldm],
        sigma [B,ldm], m_out [B], status [B]) on the device of the inputs; row b holds m_out[b] published points.
        ldm defaults to the largest ld + horizon (every window of ld stamps fits)."""
        k, dev, B, ld, P = self._ragged_common(kernel, time_array, n)
        if ldm is None:
            ldm = ld + int(horizon)
        stride, targ = 0, _Arg(None, np.float64, dev, True)
        if theta is not None:
            stride = self._theta_stride(theta, P)
            targ = _Arg(theta, np.float64, dev)
        mean = self._empty((B, ldm), np.float64, dev)
        sigma = self._empty((B, ldm), np.float64, dev)
        m_out = self._empty((B,), np.int32, dev)
        status = self._empty((B,), np.int32, dev)
        a = [_Arg(time_array, np.float64, dev), _Arg(slip_array, np.float64, dev), _Arg(n, np.int32, dev),
             _Arg(mean, np.float64, dev, output=True), _Arg(sigma, np.float64, dev, output=True),
             _Arg(m_out, np.int32, dev, output=True), _Arg(status, np.int32, dev, output=True)]
        self._bind_stream(dev)
        rc = self.lib.cngp_gp_slip_ragged(self.h, C.byref(k), targ.ptr, stride, a[0].ptr, a[1].ptr, a[2].ptr, ld, B,
                                          int(horizon), ldm, a[3].ptr, a[4].ptr, a[5].ptr, a[6].ptr,
                                          L.MEM_DEVICE if dev else L.MEM_HOST)
        self._check(rc, "cngp_gp_slip_ragged")
        return mean, sigma, m_out, status

    # ------------------------------------------------------------------------------------------------------
    @staticmethod
    def stop_config(**over) -> L.StopConfig:
        c = L.StopConfig()
        L.load().cngp_default_stop_config(C.byref(c))
        for key, v in over.items():
            if key in ("init_llh", "init_ecef"):
                for j in range(3):
                    getattr(c, key)[j] = float(v[j])
            else:
                setattr(c, key, v)
        return c

    def zupt_lookahead(self, mean, sigma, P, Q, STM, Hvec, pos, cfg: Optional[L.StopConfig] = None,
                       want_state: bool = False, m=None):
        """Batched GpPredictor look-ahead.  mean, sigma [B,M]; each of P,Q,STM ([225] or [B,225]), Hvec ([60] or
        [B,60]), pos ([3] or [B,3]) is shared or per window.  Returns dict(triggered, i_stop, step_stop, xy_err);
        want_state adds P_final [B,225], K_final [B,60], R_final [B,16] - what the reference leaves in the public
        members P_pred, K_pred, R_IP after the callback (gp_predictor.h:36-43).  m [B] (optional): row b of mean / sigma
        holds m[b] points (cngp_zupt_lookahead_ragged), e.g. the m_out of gp_slip_ragged."""
        dev = _is_cuda(mean)
        B, M = mean.shape
        cfg = cfg or self.stop_config()
        mask = 0
        ctx_args = []
        for bit, (arr, sz) in enumerate(zip((P, Q, STM, Hvec, pos), (225, 225, 225, 60, 3))):
            shape = tuple(arr.shape)
            n_el = int(np.prod(shape))
            if len(shape) >= 2 and shape[0] == B and n_el == sz * B:
                mask |= 1 << bit          # one entry per window
            elif n_el != sz:
                raise CngpError(f"context array {bit} has {n_el} elements, expected {sz} or [{B},{sz}]")
            ctx_args.append(_Arg(arr, np.float64, dev))
        trig = self._empty((B,), np.int32, dev)
        i_stop = self._empty((B,), np.int32, dev)
        step = self._empty((B,), np.int32, dev)
        xy = self._empty((B,), np.float64, dev)
        a = [_Arg(mean, np.float64, dev), _Arg(sigma, np.float64, dev), _Arg(trig, np.int32, dev),
             _Arg(i_stop, np.int32, dev), _Arg(step, np.int32, dev), _Arg(xy, np.float64, dev)]
        self._bind_stream(dev)
        if m is not None:
            if int(np.prod(tuple(m.shape))) != B:
                raise CngpError(f"m has {int(np.prod(tuple(m.shape)))} entries for {B} windows")
            ma = _Arg(m, np.int32, dev)
            st = [None, None, None]
            if want_state:
                st = [self._empty((B, n), np.float64, dev) for n in (225, 60, 16)]
            s3 = [_Arg(v, np.float64, dev, True, output=True) for v in st]
            rc = self.lib.cngp_zupt_lookahead_ragged(self.h, a[0].ptr, a[1].ptr, B, ma.ptr, M, *[c.ptr for c in ctx_args],
                                                     mask, C.byref(cfg), a[2].ptr, a[3].ptr, a[4].ptr, a[5].ptr,
                                                     s3[0].ptr, s3[1].ptr, s3[2].ptr, L.MEM_DEVICE if dev else L.MEM_HOST)
            self._check(rc, "cngp_zupt_lookahead_ragged")
            res = dict(triggered=trig, i_stop=i_stop, step_stop=step, xy_err=xy)
            if want_state:
                res.update(P_final=st[0], K_final=st[1], R_final=st[2])
            return res
        if want_state:
            Pf, Kf, Rf = (self._empty((B, n), np.float64, dev) for n in (225, 60, 16))
            s3 = [_Arg(Pf, np.float64, dev, output=True), _Arg(Kf, np.float64, dev, output=True),
                  _Arg(Rf, np.float64, dev, output=True)]
            rc = self.lib.cngp_zupt_lookahead_batch_ex(self.h, a[0].ptr, a[1].ptr, B, M, *[c.ptr for c in ctx_args], mask,
                                                       C.byref(cfg), a[2].ptr, a[3].ptr, a[4].ptr, a[5].ptr,
                                                       s3[0].ptr, s3[1].ptr, s3[2].ptr,
                                                       L.MEM_DEVICE if dev else L.MEM_HOST)
            self._check(rc, "cngp_zupt_lookahead_batch_ex")
            return dict(triggered=trig, i_stop=i_stop, step_stop=step, xy_err=xy, P_final=Pf, K_final=Kf, R_final=Rf)
        rc = self.lib.cngp_zupt_lookahead_batch(self.h, a[0].ptr, a[1].ptr, B, M, *[c.ptr for c in ctx_args], mask,
                                                C.byref(cfg), a[2].ptr, a[3].ptr, a[4].ptr, a[5].ptr,
                                                L.MEM_DEVICE if dev else L.MEM_HOST)
        self._check(rc, "cngp_zupt_lookahead_batch")
        return dict(triggered=trig, i_stop=i_stop, step_stop=step, xy_err=xy)

    def ekf_covariance(self, P0, Q, STM, H, R, n_steps: int, ratio: int = 5):
        """The EKF's covariance recursion (CoreNav.cpp:101, 226-230) for B operating points: n_steps IMU steps with an
        odometry update every `ratio`-th.  P0 [B,225]; Q, STM ([225] or [B,225]); H ([60] true row-major 4x15 or [B,60]);
        R ([16] or [B,16]).  Returns P [B,225] - the P_pred of the SetStopping service (CoreNav.cpp:291-292)."""
        dev = _is_cuda(P0)
        B = P0.shape[0]
        mask = 1                                   # P0 is per window
        args = [_Arg(P0, np.float64, dev)]
        for bit, (arr, sz) in ((1, (Q, 225)), (2, (STM, 225)), (3, (H, 60)), (4, (R, 16))):
            n_el = int(np.prod(tuple(arr.shape)))
            if n_el == sz * B and (B > 1 or len(arr.shape) >= 2):
                mask |= 1 << bit
            elif n_el != sz:
                raise CngpError(f"ekf_covariance: array {bit} has {n_el} elements, expected {sz} or [{B},{sz}]")
            args.append(_Arg(arr, np.float64, dev))
        out = self._empty((B, 225), np.float64, dev)
        o = _Arg(out, np.float64, dev, output=True)
        self._bind_stream(dev)
        rc = self.lib.cngp_ekf_covariance_batch(self.h, *[a.ptr for a in args], B, n_steps, ratio, mask, o.ptr,
                                                L.MEM_DEVICE if dev else L.MEM_HOST)
        self._check(rc, "cngp_ekf_covariance_batch")
        return out

    def ekf_context(self, llh, vel, att, f_ib_b, dt: float = 0.02, dt_odo: float = 0.1, want_h: bool = True):
        """STM, Q (and the packed odometry H) of the SetStopping service for B operating points
        (CoreNav::insErrorStateModel_LNF / calc_Q, CoreNav.cpp:411-527).  Inputs [B,3]; returns (STM [B,225], Q [B,225],
        Hvec [B,60] or None)."""
        dev = _is_cuda(llh)
        B = int(tuple(llh.shape)[0])
        S = self._empty((B, 225), np.float64, dev)
        Q = self._empty((B, 225), np.float64, dev)
        H = self._empty((B, 60), np.float64, dev) if want_h else None
        a = [_Arg(llh, np.float64, dev), _Arg(vel, np.float64, dev), _Arg(att, np.float64, dev),
             _Arg(f_ib_b, np.float64, dev), _Arg(S, np.float64, dev), _Arg(Q, np.float64, dev),
             _Arg(H, np.float64, dev, True)]
        self._bind_stream(dev)
        rc = self.lib.cngp_ekf_context_batch(self.h, a[0].ptr, a[1].ptr, a[2].ptr, a[3].ptr, B, float(dt), float(dt_odo),
                                             a[4].ptr, a[5].ptr, a[6].ptr, L.MEM_DEVICE if dev else L.MEM_HOST)
        self._check(rc, "cngp_ekf_context_batch")
        return S, Q, H

    @staticmethod
    def slip_config(**over) -> L.SlipConfig:
        c = L.SlipConfig()
        L.load().cngp_default_slip_config(C.byref(c))
        for key, v in over.items():
            setattr(c, key, v)
        return c

    def slip_record(self, joint, att, vel, cmd, stop_cmd=None, max_windows: int = 2, cap: int = 149,
                    cfg: Optional[L.SlipConfig] = None, want_slip: bool = True):
        """Slip extraction + GP_Input recorder of CoreNav::Update for B drives (CoreNav.cpp:244-329).

        joint [B,T,4], att [B,T,3], vel [B,T,3], cmd [B,T], stop_cmd [B,T] (NaN = no command) or None.  Returns
        dict(slip [B,T], time_array / slip_array [B,W,cap], n_samples / published / stop_update [B,W], n_windows [B])."""
        dev = _is_cuda(joint)
        B, T = tuple(cmd.shape)
        cfg = cfg or self.slip_config()
        slip = self._empty((B, T), np.float64, dev) if want_slip else None
        ta = self._empty((B, max_windows, cap), np.float64, dev)
        sa = self._empty((B, max_windows, cap), np.float64, dev)
        ns = self._empty((B, max_windows), np.int32, dev)
        pu = self._empty((B, max_windows), np.int32, dev)
        su = self._empty((B, max_windows), np.int32, dev)
        nw = self._empty((B,), np.int32, dev)
        a = [_Arg(joint, np.float64, dev), _Arg(att, np.float64, dev), _Arg(vel, np.float64, dev),
             _Arg(cmd, np.float64, dev), _Arg(stop_cmd, np.float64, dev, True), _Arg(slip, np.float64, dev, True),
             _Arg(ta, np.float64, dev), _Arg(sa, np.float64, dev), _Arg(ns, np.int32, dev), _Arg(pu, np.int32, dev),
             _Arg(su, np.int32, dev), _Arg(nw, np.int32, dev)]
        self._bind_stream(dev)
        rc = self.lib.cngp_slip_record_batch(self.h, a[0].ptr, a[1].ptr, a[2].ptr, a[3].ptr, a[4].ptr, B, T,
                                             C.byref(cfg), max_windows, cap, a[5].ptr, a[6].ptr, a[7].ptr, a[8].ptr,
                                             a[9].ptr, a[10].ptr, a[11].ptr, L.MEM_DEVICE if dev else L.MEM_HOST)
        self._check(rc, "cngp_slip_record_batch")
        return dict(slip=slip, time_array=ta, slip_array=sa, n_samples=ns, published=pu, stop_update=su, n_windows=nw)

    def llh_to_enu(self, llh, cfg: Optional[L.StopConfig] = None):
        dev = _is_cuda(llh)
        n = int(np.prod(tuple(llh.shape))) // 3
        cfg = cfg or self.stop_config()
        enu = self._empty((n, 3), np.float64, dev)
        a = [_Arg(llh, np.float64, dev), _Arg(enu, np.float64, dev)]
        self._bind_stream(dev)
        rc = self.lib.cngp_llh_to_enu(self.h, a[0].ptr, n, C.byref(cfg), a[1].ptr, L.MEM_DEVICE if dev else L.MEM_HOST)
        self._check(rc, "cngp_llh_to_enu")
        return enu

    def chol_large(self, kernel, theta, x, y, want_alpha: bool = False):
        """Single large window (BASELINE.json configs[4], N = 32768) on this GPU: blocked FP64 Cholesky in HBM.
        theta: host [P]; x, y: host arrays or CUDA tensors [N].  Returns dict(logdet, quad, lml[, alpha]).
        Raises CngpError when the matrix is not positive definite (rc = failing pivot)."""
        k = parse_kernel(kernel)
        dev = _is_cuda(x)
        N = int(np.prod(tuple(x.shape)))
        th = np.ascontiguousarray(np.asarray(theta, dtype=np.float64))
        if th.size != k.n_params + 1:
            raise CngpError(f"theta has {th.size} entries, kernel needs {k.n_params + 1} (noise last)")
        outs = np.empty(3)
        alpha = self._empty((N,), np.float64, dev) if want_alpha else None
        a = [_Arg(x, np.float64, dev), _Arg(y, np.float64, dev), _Arg(alpha, np.float64, dev, True)]
        self._bind_stream(dev)
        rc = self.lib.cngp_chol_large(self.h, C.byref(k), th.ctypes.data, a[0].ptr, a[1].ptr, N, outs.ctypes.data,
                                      outs.ctypes.data + 8, outs.ctypes.data + 16, a[2].ptr,
                                      L.MEM_DEVICE if dev else L.MEM_HOST)
        if rc > 0:
            raise CngpError(f"cngp_chol_large: matrix not positive definite at pivot {rc}")
        self._check(rc, "cngp_chol_large")
        res = dict(logdet=float(outs[0]), quad=float(outs[1]), lml=float(outs[2]))
        if want_alpha:
            res["alpha"] = alpha
        return res

    def chol_large_predict(self, kernel, theta, x, y, xstar):
        """chol_large, then the predictive mean and variance at xstar [M] from the factor (GPy m.predict with
        include_likelihood=True).  x, y, xstar: host arrays or CUDA tensors, all alike.  Returns dict(mean, var, logdet,
        quad, lml, pivot): pivot = 0, or the (1-based) pivot at which Ky was found not positive definite - then every
        other value is NaN."""
        k = parse_kernel(kernel)
        dev = _is_cuda(x)
        N = int(np.prod(tuple(x.shape)))
        M = int(np.prod(tuple(xstar.shape)))
        th = np.ascontiguousarray(np.asarray(theta, dtype=np.float64))
        if th.size != k.n_params + 1:
            raise CngpError(f"theta has {th.size} entries, kernel needs {k.n_params + 1} (noise last)")
        outs = np.empty(3)
        mean = self._empty((M,), np.float64, dev)
        var = self._empty((M,), np.float64, dev)
        a = [_Arg(x, np.float64, dev), _Arg(y, np.float64, dev), _Arg(xstar, np.float64, dev),
             _Arg(mean, np.float64, dev, output=True), _Arg(var, np.float64, dev, output=True)]
        self._bind_stream(dev)
        rc = self.lib.cngp_chol_large_predict(self.h, C.byref(k), th.ctypes.data, a[0].ptr, a[1].ptr, N, a[2].ptr, M,
                                              a[3].ptr, a[4].ptr, outs.ctypes.data, outs.ctypes.data + 8,
                                              outs.ctypes.data + 16, L.MEM_DEVICE if dev else L.MEM_HOST)
        if rc < 0:
            self._check(rc, "cngp_chol_large_predict")
        return dict(mean=mean, var=var, logdet=float(outs[0]), quad=float(outs[1]), lml=float(outs[2]), pivot=int(rc))

    def chol_large_grad(self, kernel, theta, x, y):
        """chol_large, then the gradient of the LML with respect to theta [P] (natural parameters, noise last) from the
        factor: GPy's ExactGaussianInference dL_dK with kern.update_gradients_full, as lml_grad.  x, y: host arrays or
        CUDA tensors, alike; grad follows them.  Returns dict(lml, grad, logdet, quad, pivot): pivot = 0, or the (1-based)
        pivot at which Ky was found not positive definite - then every other value is NaN."""
        k = parse_kernel(kernel)
        dev = _is_cuda(x)
        N = int(np.prod(tuple(x.shape)))
        th = np.ascontiguousarray(np.asarray(theta, dtype=np.float64))
        if th.size != k.n_params + 1:
            raise CngpError(f"theta has {th.size} entries, kernel needs {k.n_params + 1} (noise last)")
        outs = np.empty(3)
        grad = self._empty((th.size,), np.float64, dev)
        a = [_Arg(x, np.float64, dev), _Arg(y, np.float64, dev), _Arg(grad, np.float64, dev, output=True)]
        self._bind_stream(dev)
        rc = self.lib.cngp_chol_large_grad(self.h, C.byref(k), th.ctypes.data, a[0].ptr, a[1].ptr, N, outs.ctypes.data,
                                           outs.ctypes.data + 8, outs.ctypes.data + 16, a[2].ptr,
                                           L.MEM_DEVICE if dev else L.MEM_HOST)
        if rc < 0:
            self._check(rc, "cngp_chol_large_grad")
        return dict(lml=float(outs[2]), grad=grad, logdet=float(outs[0]), quad=float(outs[1]), pivot=int(rc))

    def large_matvec(self, kernel, theta, x, v):
        """r = (K(x,x) + (noise + 1e-8) I) v evaluated on the fly on the device; x, v CUDA tensors [N]."""
        k = parse_kernel(kernel)
        th = np.ascontiguousarray(np.asarray(theta, dtype=np.float64))
        N = int(x.numel())
        r = torch.empty(N, dtype=torch.float64, device=x.device)
        self._bind_stream(True)
        rc = self.lib.cngp_large_matvec(self.h, C.byref(k), th.ctypes.data, x.data_ptr(), v.data_ptr(), N, r.data_ptr())
        self._check(rc, "cngp_large_matvec")
        return r
