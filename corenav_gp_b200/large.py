"""One large slip window (BASELINE.json configs[4]: N = 32768) factored across the GPUs of one box.

Same inference as the batched windows (row a3 of SURVEY.md section 8: GPy ExactGaussianInference as reached from
core_navigation/script/gp_slip_node.py:35) - Ky = K + (noise + 1e-8) I, Cholesky, log det, y' Ky^-1 y, LML, alpha - for
a window far beyond what the reference ever runs.  1-D block-cyclic column distribution: block column c (256 columns)
lives on rank c % world.  Per block column k

    owner(k):   factor the diagonal block, form the panel                    cngp_large_factor_panel   (CUDA)
    all ranks:  broadcast of the panel (C2 - the only data-path collective)   torch.distributed / NCCL over NVLink
    all ranks:  A(:, own columns > k) -= panel panel^T                        cngp_large_update         (CUDA, FP64 DMMA)

with a look-ahead of one block column: the owner of k+1 updates that block column first, factors it and starts its
broadcast while every rank is still busy with the rest of update k, so the broadcast and the (latency-bound) diagonal
factorisation hide behind the trailing update.  y rides along as an extra matrix row, so after the last panel each rank
holds its slice of z = L^-1 y; one all-reduce gives log det, z'z and z, and alpha = L^-T z is a backward sweep with
one 2 KB broadcast per block column.

`engine` is anything with the LargeWindow methods below - the CUDA one here, or a test double (tests/ uses a numpy
engine to exercise this driver under world_size-2 gloo on CPU).  Nothing in this module computes.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import Dict, Optional

import numpy as np

from . import _lib as L
from .api import CngpError, GpContext, parse_kernel

try:
    import torch
    import torch.distributed as dist
except Exception:  # pragma: no cover
    torch = None
    dist = None

LOG_2PI = math.log(2.0 * math.pi)


def make_plan(N: int, world: int = 1, rank: int = 0) -> L.LargePlan:
    p = L.LargePlan()
    rc = L.load().cngp_large_make_plan(N, world, rank, C.byref(p))
    if rc != 0:
        raise CngpError(f"cngp_large_make_plan(N={N}, world={world}, rank={rank}) failed (rc={rc})")
    return p


class LargeWindow:
    """This rank's share of one large window on its GPU: block columns, three panel buffers (panel k+1 is produced /
    received while the trailing updates of panels k-1 and k still read theirs), inverted diagonal blocks, and a
    high-priority stream for the panel chain."""
    N_PANELS = 3

    def __init__(self, ctx: GpContext, kernel, theta, x, y, rank: int = 0, world: int = 1,
                 chunk_rows: Optional[int] = None):
        self.ctx, self.lib = ctx, ctx.lib
        self.kernel = parse_kernel(kernel)
        self.theta = np.ascontiguousarray(np.asarray(theta, dtype=np.float64))
        if self.theta.size != self.kernel.n_params + 1:
            raise CngpError(f"theta has {self.theta.size} entries, kernel needs {self.kernel.n_params + 1} (noise last)")
        dev = torch.device(f"cuda:{ctx.device}")
        self.x = torch.as_tensor(x, dtype=torch.float64).to(dev).contiguous()
        self.y = torch.as_tensor(y, dtype=torch.float64).to(dev).contiguous()
        self.N = int(self.x.numel())
        self.rank, self.world = rank, world
        self.plan = make_plan(self.N, world, rank)
        p = self.plan
        # panel chunks (cngp.h, chunk_blocks): the unit of the pipelined panel chain.  OFF by default: with NCCL broadcasts
        # (~50 us each whatever the size) the pipelining loses more than it gains - 8 GPUs, N = 32768: 80-90 ms in one
        # piece, 95 ms in chunks of 4096 rows, 107 ms in chunks of 2048 (profiles/bench_large_8gpu_c*_r02o.json)
        if chunk_rows is None:
            chunk_rows = int(os.environ.get("CNGP_LARGE_CHUNK_ROWS", "0"))
        if chunk_rows > 0:
            rb = int(p.row_tiles) // 16
            cs = max(chunk_rows // 128, -(-rb // L.LARGE_MAX_CHUNKS))
            p.chunk_blocks = cs + (cs & 1)
        self.n_blockcols, self.nb, self.n_pad = int(p.n_blockcols), L.LARGE_NB, int(p.n_pad)
        f64 = dict(dtype=torch.float64, device=dev)
        self.A = torch.empty(max(1, p.local_doubles), **f64)
        self.panels = [torch.zeros(p.panel_doubles, **f64) for _ in range(self.N_PANELS)]
        self.chain_stream = torch.cuda.Stream(device=dev, priority=-1)   # the serial panel chain runs here
        self.side_stream = torch.cuda.Stream(device=dev, priority=-1)    # ... and the rows below the block being factored
        self.winv = torch.zeros(max(1, p.winv_doubles), **f64)
        self.logdet = torch.zeros(p.n_blockcols, **f64)
        self.status = torch.zeros(p.n_blockcols, dtype=torch.int32, device=dev)
        self.z = torch.zeros(p.n_pad, **f64)
        self.alpha = torch.zeros(p.n_pad, **f64)
        self.s_acc = torch.zeros(p.n_pad, **f64)
        self.sums = torch.zeros(4, **f64)
        self._chunk_cache: Dict[int, tuple] = {}

    def _bind(self):
        self.ctx._bind_stream(True)

    def _chk(self, rc, what):
        self.ctx._check(rc, what)

    # ---- the engine interface used by chol_large_distributed ----
    def panel_buffer(self, k: int):
        return self.panels[k % self.N_PANELS]

    def panel_payload(self, k: int):
        """The contiguous part of panel k's buffer the other ranks need (rows below the diagonal block)."""
        rows = int(self.plan.row_tiles) - (k + 1) * (self.nb // 8)
        return self.panels[k % self.N_PANELS][: (self.nb // 8) * rows * 64]

    def panel_chunks(self, k: int):
        """-> (absolute id of the first chunk of panel k that holds rows, [contiguous views of the panel buffer, one per
        chunk]): the broadcast payloads of panel k, in row order."""
        if k not in self._chunk_cache:
            first, count = C.c_int32(), C.c_int32()
            offs = (C.c_int64 * (L.LARGE_MAX_CHUNKS + 1))()
            rc = self.lib.cngp_large_panel_chunks(C.byref(self.plan), k, C.byref(first), C.byref(count), offs)
            if rc != 0:
                raise CngpError(f"cngp_large_panel_chunks(k={k}) failed (rc={rc})")
            self._chunk_cache[k] = (int(first.value), [int(offs[i]) for i in range(count.value + 1)])
        first, offs = self._chunk_cache[k]
        buf = self.panels[k % self.N_PANELS]
        return first, [buf[offs[i]:offs[i + 1]] for i in range(len(offs) - 1)]

    def assemble(self):
        self._bind()
        self._chk(self.lib.cngp_large_assemble(self.ctx.h, C.byref(self.plan), C.byref(self.kernel), self.theta.ctypes.data,
                                               self.x.data_ptr(), self.y.data_ptr(), self.A.data_ptr()),
                  "cngp_large_assemble")

    DEFER_COPY, DIAG_ONLY, PANEL_ONLY = 1, 2, 4          # cngp.h CNGP_LARGE_*
    ROWS_ALL, ROWS_DIAG, ROWS_BELOW = 0, 1, 2

    def factor_panel(self, k: int, flags: int = 0, chunk: int = -1):
        self._bind()
        self._chk(self.lib.cngp_large_factor_panel_ex(self.ctx.h, C.byref(self.plan), self.A.data_ptr(), k,
                                                      self.panels[k % self.N_PANELS].data_ptr(), self.winv.data_ptr(),
                                                      self.logdet.data_ptr(), self.status.data_ptr(), int(flags), int(chunk)),
                  "cngp_large_factor_panel")

    def update_part(self, k: int, c: int, rows: int, chunk: int = -1):
        """Update block column c with panel k: its diagonal block only / only the rows below it / (chunk >= 0) only the
        rows of one chunk of the panel."""
        self._bind()
        self._chk(self.lib.cngp_large_update_part(self.ctx.h, C.byref(self.plan), self.A.data_ptr(), k,
                                                  self.panels[k % self.N_PANELS].data_ptr(), c, c + 1, rows, int(chunk)),
                  "cngp_large_update_part")

    def copy_back(self, k: int):
        """Store panel k as block column k of L (deferred step of factor_panel; needed by the backward sweep only)."""
        self._bind()
        self._chk(self.lib.cngp_large_copy_back(self.ctx.h, C.byref(self.plan), self.A.data_ptr(), k,
                                                self.panels[k % self.N_PANELS].data_ptr()), "cngp_large_copy_back")

    def update(self, k: int, c_lo: int, c_hi: int):
        self._bind()
        self._chk(self.lib.cngp_large_update(self.ctx.h, C.byref(self.plan), self.A.data_ptr(), k,
                                             self.panels[k % self.N_PANELS].data_ptr(), c_lo, c_hi), "cngp_large_update")

    def reduce(self):
        """-> (z [n_pad] with this rank's columns, sums [3] = logdet part, z'z part, first failing pivot or 0)."""
        self._bind()
        self._chk(self.lib.cngp_large_reduce(self.ctx.h, C.byref(self.plan), self.A.data_ptr(), self.logdet.data_ptr(),
                                             self.status.data_ptr(), self.z.data_ptr(), self.sums.data_ptr()),
                  "cngp_large_reduce")
        return self.z, self.sums[:3]

    def backsolve_step(self, j: int):
        self._bind()
        self._chk(self.lib.cngp_large_backsolve_step(self.ctx.h, C.byref(self.plan), self.A.data_ptr(),
                                                     self.winv.data_ptr(), j, self.z.data_ptr(), self.alpha.data_ptr()),
                  "cngp_large_backsolve_step")

    def backsolve_begin(self):
        self.s_acc.zero_()

    def backsolve_finish(self, j: int):
        self._bind()
        self._chk(self.lib.cngp_large_backsolve_finish(self.ctx.h, C.byref(self.plan), self.winv.data_ptr(), j,
                                                       self.z.data_ptr(), self.s_acc.data_ptr(), self.alpha.data_ptr()),
                  "cngp_large_backsolve_finish")

    def backsolve_apply(self, j: int):
        """s_c += L(block row j, c)^T alpha_j for this rank's block columns c < j."""
        self._bind()
        self._chk(self.lib.cngp_large_backsolve_apply(self.ctx.h, C.byref(self.plan), self.A.data_ptr(), j,
                                                      self.alpha.data_ptr(), self.s_acc.data_ptr()),
                  "cngp_large_backsolve_apply")

    def alpha_block(self, j: int):
        return self.alpha[j * self.nb:(j + 1) * self.nb]

    # ---- the engine interface used by predict_large_distributed ----
    def _pred_sizes(self, M: int, k: int):
        r, pay, s = C.c_int64(), C.c_int64(), C.c_int64()
        rc = self.lib.cngp_large_predict_sizes(C.byref(self.plan), M, k, C.byref(r), C.byref(pay), C.byref(s))
        if rc != 0:
            raise CngpError(f"cngp_large_predict_sizes(M={M}, k={k}) failed (rc={rc})")
        return int(r.value), int(pay.value), int(s.value)

    def predict_begin(self, xstar):
        """R = K(x*, x) for this rank's block columns, s = 0.  R, the two payload buffers (payload k+1 is formed while
        the update with payload k still reads it) and s are allocated on first use and kept while M does not grow."""
        self._bind()
        dev = self.x.device
        self.xstar = torch.as_tensor(xstar, dtype=torch.float64).to(dev).contiguous().reshape(-1)
        self.M = M = int(self.xstar.numel())
        r, pay, s = self._pred_sizes(M, 0)
        f64 = dict(dtype=torch.float64, device=dev)
        if getattr(self, "R", None) is None or self.R.numel() < max(1, r) or self.payloads[0].numel() < pay:
            self.R = torch.empty(max(1, r), **f64)
            self.payloads = [torch.empty(pay, **f64) for _ in range(2)]
        self.s = torch.zeros(s, **f64)
        self._chk(self.lib.cngp_large_predict_assemble(self.ctx.h, C.byref(self.plan), C.byref(self.kernel),
                                                       self.theta.ctypes.data, self.x.data_ptr(), self.xstar.data_ptr(),
                                                       M, self.R.data_ptr()), "cngp_large_predict_assemble")

    def predict_payload(self, k: int):
        """[W_k ; L(rows below the diagonal block, k)]: what the owner of k broadcasts."""
        return self.payloads[k % 2][: self._pred_sizes(self.M, k)[1]]

    def predict_panel(self, k: int):
        self._bind()
        self._chk(self.lib.cngp_large_predict_panel(self.ctx.h, C.byref(self.plan), self.A.data_ptr(), self.winv.data_ptr(),
                                                    self.R.data_ptr(), self.M, k, self.payloads[k % 2].data_ptr(),
                                                    self.s.data_ptr()), "cngp_large_predict_panel")

    def predict_update(self, k: int, c_lo: int, c_hi: int):
        self._bind()
        self._chk(self.lib.cngp_large_predict_update(self.ctx.h, C.byref(self.plan), self.R.data_ptr(), self.M, k,
                                                     self.payloads[k % 2].data_ptr(), c_lo, c_hi),
                  "cngp_large_predict_update")

    def predict_sums(self):
        """s [n_blockcols * M]: this rank's rows of the per-block-column sums of W^2, zero elsewhere."""
        return self.s

    def predict_finish(self):
        """-> (mean [M], var [M]) from alpha and the rank-summed s."""
        self._bind()
        mean = torch.empty(self.M, dtype=torch.float64, device=self.x.device)
        var = torch.empty_like(mean)
        self._chk(self.lib.cngp_large_predict_finish(self.ctx.h, C.byref(self.plan), C.byref(self.kernel),
                                                     self.theta.ctypes.data, self.x.data_ptr(), self.alpha.data_ptr(),
                                                     self.xstar.data_ptr(), self.M, self.s.data_ptr(), mean.data_ptr(),
                                                     var.data_ptr()), "cngp_large_predict_finish")
        return mean, var

    # ---- the engine interface used by lml_grad_large_distributed ----
    def grad_begin(self):
        """RG = I for this rank's block columns.  RG (R, then G, like A), the two payload buffers and the parts are
        allocated on first use and kept."""
        self._bind()
        if getattr(self, "RG", None) is None:
            rg, pay, part = C.c_int64(), C.c_int64(), C.c_int64()
            rc = self.lib.cngp_large_grad_sizes(C.byref(self.plan), C.byref(rg), C.byref(pay), C.byref(part))
            if rc != 0:
                raise CngpError(f"cngp_large_grad_sizes failed (rc={rc})")
            f64 = dict(dtype=torch.float64, device=self.x.device)
            self.RG = torch.empty(max(1, rg.value), **f64)
            self.grad_payloads = [torch.empty(pay.value, **f64) for _ in range(2)]
            self.part = torch.zeros(part.value, **f64)
        self._chk(self.lib.cngp_large_grad_begin(self.ctx.h, C.byref(self.plan), self.RG.data_ptr()), "cngp_large_grad_begin")

    def grad_payload(self, k: int):
        """[W_k ; L(rows below the diagonal block, k)]: what the owner of k broadcasts (n_pad x NB doubles for every k)."""
        return self.grad_payloads[k % 2]

    def grad_panel(self, k: int):
        self._bind()
        self._chk(self.lib.cngp_large_grad_panel(self.ctx.h, C.byref(self.plan), self.A.data_ptr(), self.winv.data_ptr(),
                                                 self.RG.data_ptr(), k, self.grad_payloads[k % 2].data_ptr()),
                  "cngp_large_grad_panel")

    def grad_update(self, k: int, c_lo: int, c_hi: int):
        """This rank's block columns c in [c_lo, c_hi) with payload k: c > k swept, c <= k accumulated into G."""
        self._bind()
        self._chk(self.lib.cngp_large_grad_update(self.ctx.h, C.byref(self.plan), self.RG.data_ptr(), k,
                                                  self.grad_payloads[k % 2].data_ptr(), c_lo, c_hi),
                  "cngp_large_grad_update")

    def grad_contract(self):
        """-> part [n_blockcols * stride]: this rank's rows of the contraction, zero elsewhere."""
        self._bind()
        self._chk(self.lib.cngp_large_grad_contract(self.ctx.h, C.byref(self.plan), C.byref(self.kernel),
                                                    self.theta.ctypes.data, self.x.data_ptr(), self.alpha.data_ptr(),
                                                    self.RG.data_ptr(), self.part.data_ptr()), "cngp_large_grad_contract")
        return self.part

    def grad_finish(self):
        """-> grad [P] from the rank-summed parts."""
        self._bind()
        grad = torch.empty(self.theta.size, dtype=torch.float64, device=self.x.device)
        self._chk(self.lib.cngp_large_grad_finish(self.ctx.h, C.byref(self.plan), C.byref(self.kernel),
                                                  self.part.data_ptr(), grad.data_ptr()), "cngp_large_grad_finish")
        return grad


class TorchCollectives:
    """broadcast / all-reduce through torch.distributed (NCCL for CUDA tensors, gloo for CPU tensors)."""

    def __init__(self, group=None):
        self.group = group

    def broadcast_async(self, t, src: int):
        return dist.broadcast(t, src=src, group=self.group, async_op=True)

    def all_reduce_sum(self, t):
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)

    def all_reduce_max(self, t):
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)


class NoCollectives:
    """world == 1.  A broadcast moves nothing, but its wait() still orders the stream that waits after the stream that
    produced the payload, as NCCL's does: the two-stream schedule forms panel k+1 on the chain stream, and the trailing
    update on the main stream must not read it earlier."""

    class _Done:
        def wait(self):
            return True

    class _Ready:
        def __init__(self, ev):
            self.ev = ev

        def wait(self):
            torch.cuda.current_stream().wait_event(self.ev)
            return True

    def broadcast_async(self, t, src: int):
        if torch is not None and isinstance(t, torch.Tensor) and t.is_cuda:
            ev = torch.cuda.Event()
            ev.record()                                          # the payload is complete here on the current stream
            return self._Ready(ev)
        return self._Done()

    def all_reduce_sum(self, t):
        pass

    def all_reduce_max(self, t):
        pass


class _PhaseTimer:
    """Optional per-phase device timing of the distributed driver (CUDA events on the current stream)."""

    def __init__(self, on: bool):
        self.on = on
        self.spans = []

    def mark(self, name):
        if not self.on:
            return None
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.spans.append((name, e))
        return e

    def summary(self):
        if not self.on:
            return None
        torch.cuda.synchronize()
        out: Dict[str, float] = {}
        for (n0, e0), (n1, e1) in zip(self.spans[:-1], self.spans[1:]):
            out[n0] = out.get(n0, 0.0) + e0.elapsed_time(e1)
        return out


def _factor_one_stream(engine, rank, world, coll, nblk, lookahead, pt):
    """Everything in program order on one stream (CPU engines of the gloo tests; lookahead = False on the GPU)."""
    pt.mark("assemble")
    engine.assemble()
    if rank == 0 % world:
        engine.factor_panel(0)
    pending = coll.broadcast_async(engine.panel_payload(0), src=0)
    for k in range(nblk):
        pt.mark("wait_panel")
        pending.wait()                                           # panel k is here
        nxt = k + 1
        if nxt < nblk:
            if lookahead:
                if nxt % world == rank:                          # bring block column k+1 up to date first and factor it
                    pt.mark("update_next_column")
                    engine.update(k, nxt, nxt + 1)
                    pt.mark("factor_panel")
                    engine.factor_panel(nxt)
                pt.mark("bcast_enqueue")
                pending = coll.broadcast_async(engine.panel_payload(nxt), src=nxt % world)   # overlaps the update below
                pt.mark("trailing_update")
                engine.update(k, nxt + 1, nblk)
            else:
                engine.update(k, nxt, nblk)
                if nxt % world == rank:
                    engine.factor_panel(nxt)
                pending = coll.broadcast_async(engine.panel_payload(nxt), src=nxt % world)


def _factor_two_streams(engine, rank, world, coll, nblk, chain, pt):
    """The GPU schedule.  The panel chain - update block column k+1 with panel k, factor it, broadcast it - is the serial
    part of a right-looking factorisation; on ONE stream it queues behind the owner's trailing update of the previous
    panel, so every column costs trailing + chain (measured on 8 GPUs: 49 ms of 114 waiting for panels).  Here the chain
    runs on a high-priority stream of its own, next to the trailing updates on the main stream:
      main,  step k: wait panel k; update column k+2 with it FIRST (event: that column is current through panel k),
                     then columns k+3...; event: panel k's buffer is no longer read
      chain, step k: wait "column k+1 current through panel k-1", wait "the buffer of panel k-2 is free";
                     owner: update column k+1 with panel k, factor; everybody: broadcast panel k+1 into the third buffer.
    and the chain itself is pipelined over CHUNKS of panel rows (engine.panel_chunks; fixed absolute row ranges, each a
    contiguous payload): the owner of k+1 updates its diagonal block as soon as the FIRST chunk of panel k is there and
    factors it while the later chunks are still arriving; on a side stream it updates the rows of chunk c of its column
    when chunk c of panel k has arrived; the panel GEMM of chunk c follows and its broadcast starts while the GEMM of
    chunk c+1 runs.  Per column the chain then costs about  first chunk + diagonal block + one chunk GEMM  instead of
    whole broadcast + update + whole panel GEMM.
    Each block column still receives its updates in increasing panel order, so the results are the same bits."""
    main = torch.cuda.current_stream()
    side = engine.side_stream
    pt.mark("assemble")
    engine.assemble()
    if rank == 0 % world:
        engine.factor_panel(0)
    first, views = engine.panel_chunks(0)
    pending = {first + i: coll.broadcast_async(v, src=0) for i, v in enumerate(views)}
    col_current = torch.cuda.Event()          # block column k+1 is current through panel k-1 (recorded on main)
    col_current.record(main)
    buffer_free = {}                          # k -> event: trailing update k done, panel k's buffer may be overwritten
    for k in range(nblk):
        pt.mark("wait_panel")
        for w in pending.values():
            w.wait()                                             # main: panel k is here, all of it
        nxt = k + 1
        if nxt < nblk:
            with torch.cuda.stream(chain):
                chain.wait_event(col_current)
                if k - 2 in buffer_free:
                    chain.wait_event(buffer_free.pop(k - 2))     # panel k+1 goes where panel k-2 was
                nxt_first, nxt_views = engine.panel_chunks(nxt)
                nxt_pending = {}
                if nxt % world == rank:
                    # diagonal block first (its panel rows are the head of the first chunk), then its factorisation +
                    # inversion WHILE the rows below are brought up to date, chunk by chunk, on the side stream
                    pending[min(pending)].wait()
                    engine.update_part(k, nxt, engine.ROWS_DIAG)
                    fork = torch.cuda.Event()
                    fork.record(chain)
                    rows_current = {}
                    with torch.cuda.stream(side):
                        side.wait_event(fork)
                        for c in sorted(pending):
                            pending[c].wait()
                            engine.update_part(k, nxt, engine.ROWS_BELOW, c)
                            rows_current[c] = torch.cuda.Event()
                            rows_current[c].record(side)
                    engine.factor_panel(nxt, engine.DIAG_ONLY)
                    for i, v in enumerate(nxt_views):
                        c = nxt_first + i
                        chain.wait_event(rows_current[c])
                        engine.factor_panel(nxt, engine.PANEL_ONLY | engine.DEFER_COPY, c)
                        nxt_pending[c] = coll.broadcast_async(v, src=nxt % world)
                else:
                    for i, v in enumerate(nxt_views):
                        nxt_pending[nxt_first + i] = coll.broadcast_async(v, src=nxt % world)
            pt.mark("trailing_update")
            if k > 0 and k % world == rank:
                engine.copy_back(k)                              # off the chain: main has waited for panel k above
            engine.update(k, nxt + 1, nxt + 2)                   # the column the chain needs next goes first
            col_current = torch.cuda.Event()
            col_current.record(main)
            engine.update(k, nxt + 2, nblk)
            ev = torch.cuda.Event()
            ev.record(main)
            buffer_free[k] = ev
            pending = nxt_pending
    done = torch.cuda.Event()
    done.record(chain)
    main.wait_event(done)
    done_side = torch.cuda.Event()
    done_side.record(side)
    main.wait_event(done_side)
    if nblk > 1 and (nblk - 1) % world == rank:
        engine.copy_back(nblk - 1)                               # the last panel has no rows below its diagonal block


def chol_large_distributed(engine, rank: int, world: int, coll=None, want_alpha: bool = True,
                           lookahead: bool = True, profile: bool = False) -> Dict[str, object]:
    """Run the blocked factorisation of `engine`'s window over `world` ranks (SPMD: every rank calls this).

    Returns dict(logdet, quad, lml, pivot[, alpha]) - identical on every rank; pivot = 0, or the first (1-based) pivot
    at which the matrix was found not positive definite (then the other values are NaN)."""
    if coll is None:
        coll = TorchCollectives() if world > 1 else NoCollectives()
    nblk = engine.n_blockcols
    pt = _PhaseTimer(profile and torch.cuda.is_available())
    chain = getattr(engine, "chain_stream", None) if lookahead else None
    import time as _time
    _t0 = _time.perf_counter()
    if chain is not None:
        _factor_two_streams(engine, rank, world, coll, nblk, chain, pt)
    else:
        _factor_one_stream(engine, rank, world, coll, nblk, lookahead, pt)
    host_enqueue_ms = (_time.perf_counter() - _t0) * 1e3     # host time to ENQUEUE the factorisation (no sync inside)
    pt.mark("reduce")
    z, sums = engine.reduce()
    # pivot: smallest non-zero over ranks  ->  max of (BIG - pivot)
    BIG = 1.0e15
    enc = sums.clone()
    enc[2] = torch.where(sums[2] > 0, BIG - sums[2], torch.zeros_like(sums[2]))
    both = enc[:2].clone()
    coll.all_reduce_sum(both)
    piv = enc[2:3].clone()
    coll.all_reduce_max(piv)
    coll.all_reduce_sum(z)
    logdet, quad = float(both[0]), float(both[1])
    pivot = int(round(BIG - float(piv[0]))) if float(piv[0]) > 0 else 0
    res: Dict[str, object] = dict(pivot=pivot)
    engine.pivot, engine.have_alpha = pivot, False       # what predict_large_distributed may read
    if pivot:
        nan = float("nan")
        res.update(logdet=nan, quad=nan, lml=nan)
        return res
    res.update(logdet=logdet, quad=quad, lml=0.5 * (-engine.N * LOG_2PI - logdet - quad))
    if want_alpha:
        pt.mark("backsolve")
        if hasattr(engine, "backsolve_apply"):
            # lazy sweep: the owner only finishes its block (256 x 256), every rank then folds alpha_j into the sums of
            # all its block columns to the left - the pass over the column is off the serial path.  What is left per
            # block column is the broadcast itself (~50 us for 2 KB on 8 GPUs).  Measured and not kept: replicating the
            # blocks that couple `world` consecutive block columns so that a group costs one all-reduce and every rank
            # runs its serial part alone - 8 GPUs: 90.7 ms against 89.2 ms (the group's 18 MB of blocks read by
            # one CTA, or its 16 dependent small kernels, cost what the seven broadcasts did)
            engine.backsolve_begin()
            for j in range(nblk - 1, -1, -1):
                if j % world == rank:
                    engine.backsolve_finish(j)
                coll.broadcast_async(engine.alpha_block(j), src=j % world).wait()
                if j > 0:
                    engine.backsolve_apply(j)
        else:
            for j in range(nblk - 1, -1, -1):
                if j % world == rank:
                    engine.backsolve_step(j)
                coll.broadcast_async(engine.alpha_block(j), src=j % world).wait()
        res["alpha"] = engine.alpha[: engine.N]
        engine.have_alpha = True
    pt.mark("end")
    if pt.on:
        res["phase_ms"] = pt.summary()
    res["host_enqueue_ms"] = host_enqueue_ms
    return res


def predict_large_distributed(engine, xstar, rank: int, world: int, coll=None,
                              lookahead: bool = True) -> Dict[str, object]:
    """Predictive mean and variance at xstar [M] from `engine`'s stored factor (SPMD: every rank calls this after
    chol_large_distributed(engine, ..., want_alpha=True); any number of calls may follow one factorisation).

    A forward sweep W = L^-1 K(x, x*) over the block columns, in the shape of the factorisation: the owner of k forms
    W_k and broadcasts it with L(:, k), every rank updates its own block columns of R = K(x*, x).  With the look-ahead
    the owner of k+1 brings its block column up to date first and starts the next broadcast before the rest of update k.
    Returns dict(mean, var, pivot) - identical on every rank and on every world size; if the factorisation found Ky not
    positive definite (pivot > 0), mean and var are NaN and the factor is not read."""
    if coll is None:
        coll = TorchCollectives() if world > 1 else NoCollectives()
    pivot = getattr(engine, "pivot", None)
    if pivot is None or not (pivot or getattr(engine, "have_alpha", False)):
        raise CngpError("predict_large_distributed: the window has not been factored with want_alpha=True")
    if pivot:
        nan = torch.full((int(np.prod(np.shape(xstar))),), float("nan"), dtype=torch.float64, device=engine.alpha.device)
        return dict(mean=nan, var=nan.clone(), pivot=pivot)
    nblk = engine.n_blockcols
    engine.predict_begin(xstar)
    if rank == 0 % world:
        engine.predict_panel(0)
    pending = coll.broadcast_async(engine.predict_payload(0), src=0)
    for k in range(nblk):
        pending.wait()                                           # payload k is here
        nxt = k + 1
        if nxt >= nblk:
            break
        if lookahead:
            if nxt % world == rank:
                engine.predict_update(k, nxt, nxt + 1)
                engine.predict_panel(nxt)
            pending = coll.broadcast_async(engine.predict_payload(nxt), src=nxt % world)   # overlaps the update below
            engine.predict_update(k, nxt + 1, nblk)
        else:
            engine.predict_update(k, nxt, nblk)
            if nxt % world == rank:
                engine.predict_panel(nxt)
            pending = coll.broadcast_async(engine.predict_payload(nxt), src=nxt % world)
    s = engine.predict_sums()
    coll.all_reduce_sum(s)                                       # each row comes from one rank: x + 0, exact
    mean, var = engine.predict_finish()
    return dict(mean=mean, var=var, pivot=0)


def lml_grad_large_distributed(engine, rank: int, world: int, coll=None, lookahead: bool = True) -> Dict[str, object]:
    """Gradient of the LML with respect to theta (natural parameters, noise last) from `engine`'s stored factor (SPMD:
    every rank calls this after chol_large_distributed(engine, ..., want_alpha=True); any number of gradient and predict
    passes may follow one factorisation).

    The predict sweep with R = I: the owner of k forms W_k = (L^-T)(:, k) and broadcasts it with L(:, k); every rank
    sweeps its block columns c > k and accumulates Ky^-1 = sum_k W_k W_k^T into its block columns c <= k; at the end each
    rank contracts its block columns against dK/dtheta.  Returns dict(grad, pivot) - identical on every rank and on every
    world size; if the factorisation found Ky not positive definite (pivot > 0), grad is NaN and the factor is not read."""
    if coll is None:
        coll = TorchCollectives() if world > 1 else NoCollectives()
    pivot = getattr(engine, "pivot", None)
    if pivot is None or not (pivot or getattr(engine, "have_alpha", False)):
        raise CngpError("lml_grad_large_distributed: the window has not been factored with want_alpha=True")
    if pivot:
        nan = torch.full((int(np.size(engine.theta)),), float("nan"), dtype=torch.float64, device=engine.alpha.device)
        return dict(grad=nan, pivot=pivot)
    nblk = engine.n_blockcols
    engine.grad_begin()
    if rank == 0 % world:
        engine.grad_panel(0)
    pending = coll.broadcast_async(engine.grad_payload(0), src=0)
    for k in range(nblk):
        pending.wait()                                           # payload k is here
        nxt = k + 1
        if nxt < nblk:
            if lookahead:
                if nxt % world == rank:
                    engine.grad_update(k, nxt, nxt + 1)
                    engine.grad_panel(nxt)
                pending = coll.broadcast_async(engine.grad_payload(nxt), src=nxt % world)   # overlaps the updates below
                engine.grad_update(k, nxt + 1, nblk)
            else:
                engine.grad_update(k, nxt, nblk)
                if nxt % world == rank:
                    engine.grad_panel(nxt)
                pending = coll.broadcast_async(engine.grad_payload(nxt), src=nxt % world)
        engine.grad_update(k, 0, nxt)                            # G(:, c <= k) -= W_k W_k(c)^T
    part = engine.grad_contract()
    coll.all_reduce_sum(part)                                    # each row comes from one rank: x + 0, exact
    return dict(grad=engine.grad_finish(), pivot=0)


def chol_large(ctx: GpContext, kernel, theta, x, y, rank: int = 0, world: int = 1, coll=None, want_alpha: bool = True,
               lookahead: bool = True, chunk_rows: Optional[int] = None) -> Dict[str, object]:
    """Convenience: build this rank's LargeWindow and run the distributed factorisation.  The window is returned as
    out["window"]: predict_large_distributed(out["window"], xstar, rank, world, coll) predicts from its factor, and
    lml_grad_large_distributed(out["window"], rank, world, coll) gives the LML gradient from it."""
    win = LargeWindow(ctx, kernel, theta, x, y, rank=rank, world=world, chunk_rows=chunk_rows)
    out = chol_large_distributed(win, rank, world, coll=coll, want_alpha=want_alpha, lookahead=lookahead)
    out["window"] = win
    return out
