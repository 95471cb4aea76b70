"""Row-sharded solves: ONE graph spread over the GPUs of a node (SURVEY 8(e), BASELINE.json configs[4] "row-sharded A at largest n").

Rank r holds rows ``[r n/P, (r+1) n/P)`` of the adjacency path AND of its transpose (twice the memory, no reduce-scatter), and the
same rows of the state.  RMSNorm -> Linear, the Runge-Kutta updates and the weight gradients are row-local; per layer the only
exchange is the operand ``V^T`` of the n x n x d contraction plus two d-vectors of column sums, done by the library's own kernels over
peer memory (``k_shard_push`` / ``k_shard_wait``, see ``PegShard`` in include/pegncde.h): no NCCL on the data path.  The peer-visible
buffers come from ``torch.distributed._symmetric_memory`` (CUDA IPC / fabric handles over NVLink); the only NCCL collectives are the
one-off reductions of the plane totals / maxima at pack time and the all-reduce of the small parameter-gradient buffer per solve.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Tuple

import numpy as np
import torch
import torch.distributed as dist

from ._lib import PEG_WS_SOLVE_BWD, PEG_WS_SOLVE_FWD, PegControl, PegDims, PegShard, check, lib
from .control import PackedControl, _stream_ptr
from .solve import constant_step_table
from .vector_field import PermEquivGraphVectorField, workspace


def row_range(n: int, rank: int, world: int) -> Tuple[int, int]:
    """Rows of rank ``rank``: equal strips, each a multiple of 128 (the row block of the contraction kernel)."""
    if n % (128 * world) != 0:
        raise ValueError(f"row sharding needs n ({n}) to be a multiple of 128 * world ({128 * world})")
    per = n // world
    return rank * per, (rank + 1) * per


def _symmetric(nbytes: int, device, group):
    """A zeroed peer-visible byte buffer and the base pointers of every rank's copy."""
    import torch.distributed._symmetric_memory as symm_mem

    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:
        t = torch.zeros(max(nbytes, 16), dtype=torch.uint8, device=device)
        return t, [t.data_ptr()], None
    t = symm_mem.empty(max(nbytes, 16), dtype=torch.uint8, device=device)
    hdl = symm_mem.rendezvous(t, group=group if group is not None else dist.group.WORLD)
    t.zero_()
    return t, [int(p) for p in hdl.buffer_ptrs], hdl


class RowShardedControl:
    """This rank's strip of a control path (planes of the strip and of the transposed strip) plus the peer-visible exchange buffers.

    ``snapshots_rows``: ``A_k[:, rows, :]`` -> ``[T, n_loc, n]`` (or batched ``[B, T, n_loc, n]``);
    ``snapshots_cols_t``: ``A_k[:, :, rows]`` transposed to ``[T, n_loc, n]`` -- the same strip of the transposed path."""

    def __init__(self, ts: torch.Tensor, snapshots_rows: torch.Tensor, snapshots_cols_t: torch.Tensor, hidden_dim: int, num_layers: int,
                 group=None, flags: int = 1):
        if isinstance(snapshots_rows, PackedControl) or isinstance(snapshots_cols_t, PackedControl):
            raise TypeError("RowShardedControl takes dense snapshot strips; sparse (CSR) controls cannot be row-sharded")
        dev = snapshots_rows.device
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        A = (snapshots_rows if snapshots_rows.dim() == 4 else snapshots_rows.unsqueeze(0)).to(torch.float32).contiguous()
        At = (snapshots_cols_t if snapshots_cols_t.dim() == 4 else snapshots_cols_t.unsqueeze(0)).to(torch.float32).contiguous()
        B, T, nloc, n = A.shape
        if At.shape != A.shape:
            raise ValueError("the transposed strip must have the shape of the row strip")
        r0, r1 = row_range(n, self.rank, self.world)
        if r1 - r0 != nloc:
            raise ValueError(f"rank {self.rank} of {self.world} owns {r1 - r0} rows of n = {n}, got a strip of {nloc}")
        self.n_glob, self.row0 = n, r0
        pc = PackedControl.__new__(PackedControl)
        pc.B, pc.n, pc.T, pc.e, pc.ldn = B, nloc, T, 0, nloc
        f = dict(dtype=torch.float32, device=dev)
        pc.ts = torch.empty((B, T), **f)
        pc.ts.copy_(ts.to(dev, torch.float32).reshape(-1, T).expand(B, T))
        pc.adj_coef = torch.empty((B, T - 1, 4 * nloc * n), **f)
        pc.adj_rowsum = torch.empty((B, T - 1, 4, nloc), **f)
        pc.adj_diag = torch.zeros((B, T - 1, 4, nloc), **f)
        pc.adj_total = torch.empty((B, T - 1, 4), **f)
        pc.tch_coef = torch.empty((B, T - 1, 3, nloc), **f)
        pc.adj_absmax = torch.empty((B, T - 1, 4), **f)
        pc.x_coef, pc.x_packed = None, None
        pc._adj = {"colsum": None, "pending": None, "host_ts": None}
        self.pc = pc
        self.adj_coef_t = torch.empty((B, T - 1, 4 * nloc * n), **f)
        absmax_t = torch.empty((B, T - 1, 4), **f)
        l, st, dims = lib(), _stream_ptr(dev), pc.dims(h=4, L=1)
        check(l.pegncde_build_adj_rect(st, dims, n, r0, pc.ts.data_ptr(), A.data_ptr(), pc.adj_coef.data_ptr(), pc.adj_rowsum.data_ptr(),
                                       pc.adj_diag.data_ptr(), pc.adj_total.data_ptr(), pc.tch_coef.data_ptr(), pc.adj_absmax.data_ptr()),
              "pegncde_build_adj_rect")
        check(l.pegncde_build_adj_rect(st, dims, n, -1, pc.ts.data_ptr(), At.data_ptr(), self.adj_coef_t.data_ptr(), None, None, None, None,
                                       absmax_t.data_ptr()), "pegncde_build_adj_rect (transposed strip)")
        # totals and maxima refer to the WHOLE path: reduce the per-strip values once
        torch.maximum(pc.adj_absmax, absmax_t, out=pc.adj_absmax)
        if self.world > 1:
            dist.all_reduce(pc.adj_total, op=dist.ReduceOp.SUM, group=group)
            dist.all_reduce(pc.adj_absmax, op=dist.ReduceOp.MAX, group=group)
        # ---- peer-visible exchange buffers ----
        d = PegDims(B, nloc, nloc, hidden_dim, 0, num_layers, T, flags)
        sizes = (ctypes.c_size_t * 4)()
        check(l.pegncde_shard_buffer_bytes(d, self.world, sizes), "pegncde_shard_buffer_bytes")
        self._bufs, self._ptr_tables, self._handles = [], [], []
        for nbytes in (sizes[0], sizes[0], sizes[1], sizes[2], sizes[3]):
            t, ptrs, hdl = _symmetric(int(nbytes), dev, group)
            self._bufs.append(t)
            self._handles.append(hdl)
            self._ptr_tables.append((ctypes.c_void_p * self.world)(*ptrs))
        self._epoch = ctypes.c_uint32(0)
        # device-side epoch base: every call advances it past its own exchanges, so a captured solve can be replayed as a CUDA graph
        self._epoch_dev = torch.zeros(1, dtype=torch.int32, device=dev)
        self.shard = PegShard(self.rank, self.world, n, r0, self.adj_coef_t.data_ptr(), self._ptr_tables[0], self._ptr_tables[1],
                              self._ptr_tables[2], self._ptr_tables[3], self._ptr_tables[4], ctypes.pointer(self._epoch),
                              self._epoch_dev.data_ptr())
        self._keep = (A, At)
        if self.world > 1:
            dist.barrier(group=group)     # every rank's buffers exist (and are zeroed) before the first push

    def struct(self) -> PegControl:
        c = self.pc.struct()
        c.shard = ctypes.pointer(self.shard)
        return c

    def dims(self, h: int, L: int, flags: int) -> PegDims:
        return PegDims(self.pc.B, self.pc.n, self.pc.ldn, h, 0, L, self.pc.T, flags)


class _RowShardedSolve(torch.autograd.Function):
    @staticmethod
    def forward(ctx, y0, flat, ctl: RowShardedControl, dims, step_ts, reduce_grads=True):
        y0, flat = y0.contiguous(), flat.contiguous()
        l, dev = lib(), y0.device
        S = len(step_ts) - 1
        ws = workspace(dev, max(l.pegncde_workspace_bytes(dims, PEG_WS_SOLVE_FWD, S), l.pegncde_workspace_bytes(dims, PEG_WS_SOLVE_BWD, S)))
        y_ckpt = torch.empty((S + 1,) + tuple(y0.shape), dtype=torch.float32, device=dev)
        host_ts = np.ascontiguousarray(step_ts, dtype=np.float32)
        need_grad = any(ctx.needs_input_grad[:2])
        store = torch.empty(l.pegncde_stage_store_bytes(dims, S) // 4, dtype=torch.float32, device=dev) if need_grad else None
        check(l.pegncde_solve_fwd(_stream_ptr(dev), dims, ctl.struct(), flat.data_ptr(), host_ts.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), S,
                                  y0.data_ptr(), None, y_ckpt.data_ptr(), store.data_ptr() if store is not None else None, ws.data_ptr(), ws.numel()),
              "pegncde_solve_fwd (row-sharded)")
        ctx.save_for_backward(flat, y_ckpt)
        ctx.store, ctx.ctl, ctx.dims, ctx.host_ts, ctx.S, ctx.reduce_grads = store, ctl, dims, host_ts, S, reduce_grads
        return y_ckpt[S]

    @staticmethod
    def backward(ctx, g_yT):
        flat, y_ckpt = ctx.saved_tensors
        l, dev, dims, S, ctl = lib(), flat.device, ctx.dims, ctx.S, ctx.ctl
        ws = workspace(dev, l.pegncde_workspace_bytes(dims, PEG_WS_SOLVE_BWD, S))
        g_yT = g_yT.contiguous().to(torch.float32)
        g_y0 = torch.empty_like(y_ckpt[0])
        g_flat = torch.zeros_like(flat)
        store = ctx.store
        check(l.pegncde_solve_bwd(_stream_ptr(dev), dims, ctl.struct(), flat.data_ptr(), ctx.host_ts.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), S,
                                  y_ckpt.data_ptr(), store.data_ptr() if store is not None else None, g_yT.data_ptr(), None, None, g_y0.data_ptr(),
                                  g_flat.data_ptr(), None, ws.data_ptr(), ws.numel()), "pegncde_solve_bwd (row-sharded)")
        ctx.store = None
        if ctl.world > 1 and ctx.reduce_grads:      # every rank holds the partial sums over its rows: the parameter gradient is their sum
            dist.all_reduce(g_flat, op=dist.ReduceOp.SUM, group=ctl.group)
        return g_y0, g_flat, None, None, None, None


def diffeqsolve_rowsharded(vf: PermEquivGraphVectorField, ctl: RowShardedControl, y0_rows: torch.Tensor, t0: float, t1: float, dt0: float,
                           max_steps: int = 4096, reduce_grads: bool = True) -> torch.Tensor:
    """Fixed-step Tsit5 solve of the row-sharded graph: ``y0_rows`` = this rank's rows ``[n_loc, h]`` (or ``[B, n_loc, h]``) of the initial
    state; returns the same rows of ``y(t1)``.  Differentiable: the cotangent w.r.t. ``y0_rows`` is row-local, the parameter gradients
    are all-reduced over the group (every rank ends up with the full gradient) unless ``reduce_grads=False`` (the caller then reduces
    the per-rank partial sums itself, e.g. outside a captured CUDA graph; the solve itself -- exchanges included -- is capturable)."""
    if vf.uses_control() or vf.directed:
        raise NotImplementedError("row-sharded mode: ODETerm(PermEquivGraphVectorField) without the CDE wrapper, undirected layer")
    unb = y0_rows.dim() == 2
    yb = (y0_rows.unsqueeze(0) if unb else y0_rows).to(torch.float32)
    dims = ctl.dims(vf.hidden_dim, vf.num_layers, vf.flags)
    step_ts = constant_step_table(float(t0), float(t1), float(dt0), "state", max_steps)
    out = _RowShardedSolve.apply(yb, vf.checked_flat_params(dims), ctl, dims, step_ts, reduce_grads)
    return out.squeeze(0) if unb else out


def vector_field_rowsharded(vf: PermEquivGraphVectorField, ctl: RowShardedControl, t: float, y_rows: torch.Tensor) -> torch.Tensor:
    """One evaluation ``f(t, y)`` on the row-sharded graph (this rank's rows in, this rank's rows out; forward only)."""
    from ._lib import PEG_WS_VF_VJP

    unb = y_rows.dim() == 2
    yb = (y_rows.unsqueeze(0) if unb else y_rows).to(torch.float32).contiguous()
    dims = ctl.dims(vf.hidden_dim, vf.num_layers, vf.flags)
    l, dev = lib(), yb.device
    ws = workspace(dev, l.pegncde_workspace_bytes(dims, PEG_WS_VF_VJP, 0))
    dy = torch.empty_like(yb)
    flat = vf.checked_flat_params(dims).detach().contiguous()
    check(l.pegncde_vf_fwd(_stream_ptr(dev), dims, ctl.struct(), flat.data_ptr(), float(t), yb.data_ptr(), dy.data_ptr(), ws.data_ptr(), ws.numel()),
          "pegncde_vf_fwd (row-sharded)")
    return dy.squeeze(0) if unb else dy
