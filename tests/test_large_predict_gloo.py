"""The multi-rank driver of the large-window predict pass (corenav_gp_b200/large.py, predict_large_distributed) under
world_size-2 gloo on CPU.  The engine is a TEST DOUBLE: the dense block-cyclic engine of test_large_driver_gloo.py with
the predict interface added (dense torch-CPU R = K(x*, x) block columns).  What is exercised is the driver's schedule:
owners, look-ahead order, double-buffered payload broadcasts and the reduction of the block sums.  Mean and variance
must equal a direct scipy Cholesky solve."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from test_large_driver_gloo import NB, DenseEngine, _free_port, _problem

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NOISE = 1e-2


def _kern(a, b):
    """The covariance of _problem without its noise: rbf (0.01, l = 10) + periodic (0.0025, p = 37, l = 1)."""
    d = a[:, None] - b[None, :]
    return 0.01 * np.exp(-0.5 * d * d / 100.0) + 0.0025 * np.exp(-0.5 * np.sin(np.pi * d / 37.0) ** 2)


def _xstar(n):
    """Before, between, on and after the training stamps (x = 20 .. 20 + n - 1)."""
    return np.concatenate([[3.0, 19.5], 20.0 + np.arange(0, n, 37) + 0.25, 20.0 + np.arange(0, n, 50),
                           20.0 + n + np.arange(0.0, 40.0)])


class PredictEngine(DenseEngine):
    """DenseEngine + the predict interface of large.LargeWindow.  Payload k = [W_k (M x NB) ; L(rows > k, k)]."""

    def __init__(self, K, y, rank, world, Ks, kss):
        super().__init__(K, y, rank, world)
        self.Ks, self.kss = Ks, kss          # K(x*, x) [M, n], k(x*, x*) [M]

    def predict_begin(self, xstar):
        self.M = len(xstar)
        self.R = {c: self.Ks[:, c * NB:(c + 1) * NB].clone() for c in self.cols}
        self.s = torch.zeros(self.n_blockcols * self.M, dtype=torch.float64)
        self.pay = [torch.zeros(self.M * NB + (self.n_pad - NB) * NB, dtype=torch.float64) for _ in range(2)]

    def predict_payload(self, k):
        return self.pay[k % 2][: self.M * NB + (self.n_pad - (k + 1) * NB) * NB]

    def predict_panel(self, k):
        assert k % self.world == self.rank
        self.calls.append(("predict_panel", k))
        W = self.R[k] @ self.diag_inv[k].T
        buf = self.predict_payload(k)
        buf[: self.M * NB] = W.reshape(-1)
        buf[self.M * NB:] = self.cols[k][(k + 1) * NB:self.n_pad].reshape(-1)
        self.s[k * self.M:(k + 1) * self.M] = (W * W).sum(1)

    def predict_update(self, k, c_lo, c_hi):
        self.calls.append(("predict_update", k, c_lo, c_hi))
        buf = self.predict_payload(k)
        W, Lk = buf[: self.M * NB].reshape(self.M, NB), buf[self.M * NB:].reshape(-1, NB)   # Lk rows (k+1) NB ...
        for c in range(max(c_lo, k + 1), min(c_hi, self.n_blockcols)):
            if c % self.world == self.rank:
                r = (c - k - 1) * NB
                self.R[c] -= W @ Lk[r:r + NB].T

    def predict_sums(self):
        return self.s

    def predict_finish(self):
        mean = self.Ks @ self.alpha
        var = torch.clamp(self.kss - self.s.reshape(self.n_blockcols, self.M).sum(0), min=1e-15) + NOISE
        return mean, var


def _engine(n, rank, world):
    K, y = _problem(n)
    x, xs = np.arange(n, dtype=np.float64) + 20.0, _xstar(n)
    Ks = torch.from_numpy(_kern(xs, x))
    kss = torch.full((len(xs),), 0.01 + 0.0025, dtype=torch.float64)
    return PredictEngine(K, y, rank, world, Ks, kss), xs


def _reference(n):
    from scipy.linalg import cho_factor, cho_solve, solve_triangular
    K, y = _problem(n)
    x, xs = np.arange(n, dtype=np.float64) + 20.0, _xstar(n)
    Ks = _kern(xs, x)
    c = cho_factor(K.numpy(), lower=True)
    mean = Ks @ cho_solve(c, y.numpy())
    W = solve_triangular(np.tril(c[0]), Ks.T, lower=True)
    var = np.clip(0.0125 - np.sum(W * W, 0), 1e-15, None) + NOISE
    return mean, var


def _worker(rank, world, port, n, lookahead, outdir):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from corenav_gp_b200 import large
    eng, xs = _engine(n, rank, world)
    coll = large.TorchCollectives()
    large.chol_large_distributed(eng, rank, world, coll=coll, lookahead=lookahead)
    out = large.predict_large_distributed(eng, xs, rank, world, coll=coll, lookahead=lookahead)
    np.savez(os.path.join(outdir, f"rank{rank}.npz"), mean=out["mean"].numpy(), var=out["var"].numpy(),
             n_panel=len([c for c in eng.calls if c[0] == "predict_panel"]))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("lookahead", [True, False])
def test_two_rank_gloo_predict_matches_scipy(tmp_path, lookahead):
    world, n = 2, 5 * NB
    mp.spawn(_worker, args=(world, _free_port(), n, lookahead, str(tmp_path)), nprocs=world, join=True)
    mean, var = _reference(n)
    n_panel = 0
    for r in range(world):
        got = np.load(tmp_path / f"rank{r}.npz")
        assert np.max(np.abs(got["mean"] - mean)) < 1e-10 * np.max(np.abs(mean))
        assert np.max(np.abs(got["var"] - var) / var) < 1e-10
        n_panel += int(got["n_panel"])
    assert n_panel == n // NB             # every block column's payload formed exactly once, by its owner


def test_single_rank_predict_order_and_reuse():
    """Look-ahead order of the sweep, and two predict passes from one factorisation."""
    from corenav_gp_b200 import large
    n = 3 * NB
    eng, xs = _engine(n, 0, 1)
    with pytest.raises(large.CngpError, match="factored"):
        large.predict_large_distributed(eng, xs, 0, 1)
    large.chol_large_distributed(eng, 0, 1)
    first = large.predict_large_distributed(eng, xs, 0, 1)
    i_p1 = eng.calls.index(("predict_panel", 1))
    assert eng.calls[i_p1 - 1] == ("predict_update", 0, 1, 2) and eng.calls[i_p1 + 1] == ("predict_update", 0, 2, 3)
    second = large.predict_large_distributed(eng, xs, 0, 1)
    assert torch.equal(first["mean"], second["mean"]) and torch.equal(first["var"], second["var"])
    mean, var = _reference(n)
    assert np.max(np.abs(first["mean"].numpy() - mean)) < 1e-10 * np.max(np.abs(mean))
    assert np.max(np.abs(first["var"].numpy() - var) / var) < 1e-10


def test_predict_sizes_helper():
    """Buffer sizes from the plan and M: R of this rank, payload k = [W_k ; L rows below block k], s."""
    import ctypes as C
    from corenav_gp_b200 import _lib as L
    from corenav_gp_b200 import large
    lib = L.load()
    for N, world, M in ((32768, 8, 600), (1300, 8, 1), (2049, 3, 129), (200, 1, 8)):
        for r in range(world):
            p = large.make_plan(N, world, r)
            m_tiles = -(-M // 128) * 16
            for k in (0, int(p.n_blockcols) - 1):
                rd, pay, sd = C.c_int64(), C.c_int64(), C.c_int64()
                assert lib.cngp_large_predict_sizes(C.byref(p), M, k, C.byref(rd), C.byref(pay), C.byref(sd)) == 0
                assert rd.value == p.n_local_blockcols * 32 * m_tiles * 64
                assert pay.value == 32 * 64 * (m_tiles + p.n_pad // 8 - (k + 1) * 32)
                assert sd.value == p.n_blockcols * M
            assert lib.cngp_large_predict_sizes(C.byref(p), 0, 0, None, None, None) != 0
            assert lib.cngp_large_predict_sizes(C.byref(p), M, p.n_blockcols, None, None, None) != 0
