"""The multi-rank driver of the large-window LML gradient pass (corenav_gp_b200/large.py, lml_grad_large_distributed)
under world_size-2 gloo on CPU.  The engine is a TEST DOUBLE: the dense block-cyclic engine of test_large_driver_gloo.py
with the gradient interface added (dense torch-CPU block columns of R, then G).  What is exercised is the driver's
schedule: owners, look-ahead order, double-buffered payload broadcasts, the accumulation of Ky^-1 into the block columns
already swept and the reduction of the parts.  The gradient must equal a numpy / LAPACK dpotri gradient."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from test_large_driver_gloo import NB, DenseEngine, _free_port, _problem

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
THETA = np.array([0.01, 10.0, 0.0025, 37.0, 1.0, 1e-2])     # _problem: rbf + periodic, noise last


def _dK(n):
    """dK/dtheta of _problem's covariance (stamps 20 .. 20 + n - 1), one dense matrix per parameter."""
    v1, l1, v2, p, l2, _ = THETA
    x = np.arange(n, dtype=np.float64) + 20.0
    d = x[:, None] - x[None, :]
    e1 = np.exp(-0.5 * d * d / l1 ** 2)
    s, c = np.sin(np.pi * d / p), np.cos(np.pi * d / p)
    e2 = np.exp(-0.5 * s * s / l2 ** 2)
    return [e1, v1 * e1 * d * d / l1 ** 3, e2, v2 * e2 * s * c * np.pi * d / (p * p * l2 ** 2), v2 * e2 * s * s / l2 ** 3,
            np.eye(n)]


class GradEngine(DenseEngine):
    """DenseEngine + the gradient interface of large.LargeWindow.  Payload k = [W_k (rows < NB (k+1)) ; L(rows > k, k)];
    block column c of RG holds R(:, c) until W_c is formed, then G(:, c) = -(Ky^-1)(:, c)."""

    def __init__(self, K, y, rank, world):
        super().__init__(K, y, rank, world)
        self.theta = THETA
        self.dK = [torch.from_numpy(m) for m in _dK(K.shape[0])]

    def grad_begin(self):
        eye = torch.eye(self.n_pad, dtype=torch.float64)
        self.RG = {c: eye[:, c * NB:(c + 1) * NB].clone() for c in self.cols}
        self.gpay = [torch.zeros(self.n_pad * NB, dtype=torch.float64) for _ in range(2)]

    def grad_payload(self, k):
        return self.gpay[k % 2]

    def _split(self, k):
        r0 = (k + 1) * NB
        buf = self.gpay[k % 2]
        return buf[: r0 * NB].reshape(r0, NB), buf[r0 * NB:].reshape(-1, NB)

    def grad_panel(self, k):
        assert k % self.world == self.rank
        self.calls.append(("grad_panel", k))
        r0 = (k + 1) * NB
        W, Lk = self._split(k)
        W[:] = self.RG[k][:r0] @ self.diag_inv[k].T
        Lk[:] = self.cols[k][r0:self.n_pad]
        self.RG[k][k * NB:r0] = 0.0

    def grad_update(self, k, c_lo, c_hi):
        self.calls.append(("grad_update", k, c_lo, c_hi))
        r0 = (k + 1) * NB
        W, Lk = self._split(k)
        for c in range(max(c_lo, 0), min(c_hi, self.n_blockcols)):
            if c % self.world != self.rank:
                continue
            if c > k:
                r = (c - k - 1) * NB
                self.RG[c][:r0] -= W @ Lk[r:r + NB].T
            else:
                self.RG[c][c * NB:r0] -= W[c * NB:] @ W[c * NB:(c + 1) * NB].T

    def grad_contract(self):
        P = len(self.theta)
        self.part = torch.zeros(self.n_blockcols * P, dtype=torch.float64)
        n = self.N
        for c, G in self.RG.items():
            w = torch.outer(self.alpha, self.alpha[c * NB:(c + 1) * NB]) + G
            i = torch.arange(n)[:, None]
            j = torch.arange(c * NB, (c + 1) * NB)[None, :]
            w = torch.where(i > j, 2.0 * w, torch.where(i == j, w, torch.zeros_like(w)))
            for p in range(P):
                self.part[c * P + p] = (w * self.dK[p][:, c * NB:(c + 1) * NB]).sum()
        return self.part

    def grad_finish(self):
        return 0.5 * self.part.reshape(self.n_blockcols, -1).sum(0)


def _reference(n):
    from scipy.linalg import cho_solve, lapack
    K, y = _problem(n)
    Kn = K.numpy()
    c, info = lapack.dpotrf(Kn, lower=1)
    assert info == 0
    inv, info = lapack.dpotri(c, lower=1)
    assert info == 0
    Kinv = np.tril(inv) + np.tril(inv, -1).T
    alpha = cho_solve((c, True), y.numpy())
    dL = np.outer(alpha, alpha) - Kinv
    return np.array([0.5 * np.sum(dL * m) for m in _dK(n)])


def _worker(rank, world, port, n, lookahead, outdir):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from corenav_gp_b200 import large
    K, y = _problem(n)
    eng = GradEngine(K, y, rank, world)
    coll = large.TorchCollectives()
    large.chol_large_distributed(eng, rank, world, coll=coll, lookahead=lookahead)
    out = large.lml_grad_large_distributed(eng, rank, world, coll=coll, lookahead=lookahead)
    np.savez(os.path.join(outdir, f"rank{rank}.npz"), grad=out["grad"].numpy(),
             n_panel=len([c for c in eng.calls if c[0] == "grad_panel"]))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("lookahead", [True, False])
def test_two_rank_gloo_grad_matches_dpotri(tmp_path, lookahead):
    world, n = 2, 5 * NB
    mp.spawn(_worker, args=(world, _free_port(), n, lookahead, str(tmp_path)), nprocs=world, join=True)
    ref = _reference(n)
    got = [np.load(tmp_path / f"rank{r}.npz") for r in range(world)]
    for g in got:
        assert np.max(np.abs(g["grad"] - ref) / np.maximum(1.0, np.abs(ref))) < 1e-10
    assert np.array_equal(got[0]["grad"], got[1]["grad"])
    assert sum(int(g["n_panel"]) for g in got) == n // NB     # every payload formed exactly once, by its owner


def test_single_rank_grad_order_and_reuse():
    """Look-ahead order of the sweep, the accumulation after it, and two gradient passes from one factorisation."""
    from corenav_gp_b200 import large
    n = 3 * NB
    K, y = _problem(n)
    eng = GradEngine(K, y, 0, 1)
    with pytest.raises(large.CngpError, match="factored"):
        large.lml_grad_large_distributed(eng, 0, 1)
    large.chol_large_distributed(eng, 0, 1)
    first = large.lml_grad_large_distributed(eng, 0, 1)
    i_p1 = eng.calls.index(("grad_panel", 1))
    assert eng.calls[i_p1 - 1] == ("grad_update", 0, 1, 2)
    assert eng.calls[i_p1 + 1: i_p1 + 3] == [("grad_update", 0, 2, 3), ("grad_update", 0, 0, 1)]
    second = large.lml_grad_large_distributed(eng, 0, 1)
    assert first["pivot"] == 0 and torch.equal(first["grad"], second["grad"])
    ref = _reference(n)
    assert np.max(np.abs(first["grad"].numpy() - ref) / np.maximum(1.0, np.abs(ref))) < 1e-10


def test_grad_sizes_helper():
    """Buffer sizes from the plan: RG of this rank (n_pad/8 row tiles per column tile), one payload = n_pad x NB,
    the parts [n_blockcols][MAX_PARAMS + 1]."""
    import ctypes as C
    from corenav_gp_b200 import _lib as L
    from corenav_gp_b200 import large
    lib = L.load()
    for N, world in ((32768, 8), (1300, 8), (2049, 3), (200, 1)):
        for r in range(world):
            p = large.make_plan(N, world, r)
            rg, pay, part = C.c_int64(), C.c_int64(), C.c_int64()
            assert lib.cngp_large_grad_sizes(C.byref(p), C.byref(rg), C.byref(pay), C.byref(part)) == 0
            assert rg.value == p.n_local_blockcols * 32 * (p.n_pad // 8) * 64
            assert pay.value == p.n_pad * NB
            assert part.value == p.n_blockcols * L.LARGE_GRAD_STRIDE
