"""diffrax-compatible term / solve API for the fused path.

Mirrors the call the reference makes
(src/models/pgt_graph_neural_cde.py:119-129, graph_neural_cde.py:94-104, tgb_graph_neural_cde.py:152-162)::

    diffeqsolve(terms=ODETerm(vf), solver=Tsit5(), t0=ts[0], t1=ts[-1], dt0=0.1, y0=y0,
                args=[control_adj, control_data], stepsize_controller=ConstantStepSize(),
                saveat=SaveAt(t1=True))  ->  Solution(.ys, .ts, .stats)

The whole integration (all steps x 7 stages x L layers) is enqueued by ONE C-ABI call
(``pegncde_solve_fwd``); reverse mode (``torch.autograd`` standing in for ``jax.custom_vjp``)
is ONE call of ``pegncde_solve_bwd`` -- the exact discrete adjoint of Tsit5, i.e. the
gradients diffrax's default ``RecursiveCheckpointAdjoint`` produces.

The adaptive call of the dynamical-systems models (src/models/graph_neural_cde.py:86-104)::

    diffeqsolve(ODETerm(vf), Tsit5(), t0=ts[0], t1=ts[-1], dt0=None, y0=y0, args=control,
                stepsize_controller=PIDController(rtol=1e-3, atol=1e-6), saveat=SaveAt(ts=ts))

runs with the step-size controller ON THE DEVICE: one ``pegncde_step_fwd_batched`` launch attempts a step of every
trajectory of the batch (each with its own start time and step size, ``jax.vmap`` of the reference's while-loop),
``pegncde_adaptive_control`` accepts / rejects per trajectory, emits the dense-output samples and advances the state;
the host only polls the `done` flags every few attempts.  The adjoint runs over every trajectory's accepted steps.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass, field
from typing import Optional

import numpy as np
import torch

from ._lib import PEG_WS_SOLVE_BWD, PEG_WS_SOLVE_FWD, PEG_WS_STEP, PEG_WS_VF_FWD, check, lib
from .control import _stream_ptr
from .vector_field import CDEWrapperVectorField, PermEquivGraphVectorField, adj_grad_buffer, resolve_control, workspace


STREAM_MIN_PIECE_BYTES = 128 << 20   # host coefficient arrays are streamed piece by piece above this size per cubic piece


class Tsit5:
    """Marker for ``diffrax.Tsit5()`` -- the only solver the fused kernels implement."""


class ODETerm:
    def __init__(self, vector_field):
        self.vector_field = vector_field


class ConstantStepSize:
    """``diffrax.ConstantStepSize()``.  ``rule`` selects how the next step start is accumulated in fp32:
    "state" (t + dt0, diffrax >= 0.7) or "prev_diff" (t + (t - tprev), diffrax <= 0.6)."""

    def __init__(self, rule: str = "state"):
        self.rule = rule


class PIDController:
    """``diffrax.PIDController(rtol, atol)`` -- with the defaults the reference uses (pcoeff=0, icoeff=1, dcoeff=0,
    i.e. the classical I-controller) plus diffrax's safety / factormin / factormax defaults.

    Restated from diffrax (unpinned, see DESIGN.md): ``keep = err < 1``; ``factor = clip(safety * err**(-1/5),
    factormin if rejected else 1, factormax)``; the next step is ``dt * factor`` and is clipped to ``t1``."""

    def __init__(self, rtol: float, atol: float, pcoeff: float = 0.0, icoeff: float = 1.0, dcoeff: float = 0.0,
                 safety: float = 0.9, factormin: float = 0.2, factormax: float = 10.0, error_order: int = 5):
        if pcoeff != 0.0 or dcoeff != 0.0 or icoeff != 1.0:
            raise NotImplementedError("only the I-controller the reference configures (pcoeff=0, icoeff=1, dcoeff=0)")
        self.rtol, self.atol = float(rtol), float(atol)
        self.safety, self.factormin, self.factormax, self.error_order = safety, factormin, factormax, error_order

    def adapt(self, scaled_error: float, dt):
        """-> (keep_step, next dt) for a step of size ``dt`` (np.float32) whose scaled error norm is ``scaled_error``."""
        f = np.float32
        err = f(scaled_error)
        keep = bool(err < f(1.0))
        with np.errstate(divide="ignore", over="ignore"):
            inv = f(1.0) / err
        if not np.isfinite(inv):
            inv = f(1.0) if np.isnan(inv) else f(np.finfo(np.float32).max)
        factor = f(self.safety) * f(inv ** f(1.0 / self.error_order))
        lo = f(1.0) if keep else f(self.factormin)
        factor = min(max(factor, lo), f(self.factormax))
        return keep, f(f(dt) * f(factor))


def clip_to_end(tprev, tnext, t1, keep_step: bool):
    """diffrax ``_clip_to_end`` for fp32 times: a step that would end within 1e-6 of (or beyond) ``t1`` ends at ``t1``
    (after a rejection: half way), so dense output never sees a vanishing last interval."""
    f = np.float32
    if f(tnext) > f(f(t1) - f(1e-6)):
        return f(t1) if keep_step else f(f(tprev) + f(0.5) * f(f(t1) - f(tprev)))
    return f(tnext)


@dataclass
class SaveAt:
    t1: bool = False
    steps: bool = False
    ts: Optional[torch.Tensor] = None


@dataclass
class Solution:
    ts: torch.Tensor
    ys: torch.Tensor
    stats: dict = field(default_factory=dict)


def constant_step_table(t0: float, t1: float, dt0: float, rule: str = "state", max_steps: int = 4096) -> np.ndarray:
    """fp32 step boundaries [S+1] under diffrax's ConstantStepSize + ``_clip_to_end``
    (``tnext > t1 - 1e-6 -> t1`` for fp32 times); raises like ``throw=True`` past ``max_steps``."""
    f = np.float32
    t0, t1, dt0 = f(t0), f(t1), f(dt0)
    if not dt0 > 0 or not t1 > t0:
        raise ValueError("need dt0 > 0 and t1 > t0")
    out = [t0]
    tprev, tnext = t0, f(t0 + dt0)
    while True:
        if tnext > f(t1 - f(1e-6)):
            tnext = t1
        out.append(tnext)
        if tnext >= t1:
            break
        if len(out) > max_steps:
            raise RuntimeError(f"max_steps={max_steps} reached")
        step = f(tnext - tprev) if rule == "prev_diff" else dt0
        tprev, tnext = tnext, f(tnext + step)
    return np.asarray(out, dtype=np.float32)


def _solve_bwd(l, g_adj, *args) -> None:
    """pegncde_solve_bwd, or pegncde_solve_bwd_adj when the cotangent of the sparse coefficients is asked for (``args`` = the
    arguments up to g_xcoef, then the workspace pointer and size)."""
    if g_adj is None:
        check(l.pegncde_solve_bwd(*args), "pegncde_solve_bwd")
    else:
        check(l.pegncde_solve_bwd_adj(*args[:-2], g_adj.data_ptr(), *args[-2:]), "pegncde_solve_bwd_adj")


class _SolveFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, y0, flat, x_packed, adj_packed, pc, dims, step_ts, save_steps, store_stages):
        y0 = y0.contiguous()
        flat = flat.contiguous()
        S = len(step_ts) - 1
        l = lib()
        dev = y0.device
        nbytes = max(l.pegncde_workspace_bytes(dims, PEG_WS_SOLVE_FWD, S), l.pegncde_workspace_bytes(dims, PEG_WS_SOLVE_BWD, S))
        ws = workspace(dev, nbytes)
        y_ckpt = torch.empty((S + 1,) + tuple(y0.shape), dtype=torch.float32, device=dev)
        host_ts = np.ascontiguousarray(step_ts, dtype=np.float32)
        ctl = pc.struct()
        need_grad = any(ctx.needs_input_grad[:4])
        store = None
        if store_stages and need_grad:
            nbytes_store = l.pegncde_stage_store_bytes(dims, S)
            capturing = torch.cuda.is_current_stream_capturing()
            free = torch.cuda.mem_get_info(dev)[0] if not capturing else float("inf")
            if nbytes_store < 0.5 * free:   # otherwise fall back to checkpoint-per-step + recompute
                store = torch.empty(nbytes_store // 4, dtype=torch.float32, device=dev)
        def run_steps(s0, s1):   # solver steps [s0, s1) -- the whole table in one call unless the control is streamed
            start = y0 if s0 == 0 else y_ckpt[s0].clone()
            seg_ts = np.ascontiguousarray(host_ts[s0:s1 + 1])
            store_ptr = None if store is None else store.data_ptr() + s0 * l.pegncde_stage_store_bytes(dims, 1)
            check(l.pegncde_solve_fwd(_stream_ptr(dev), dims, ctl, flat.data_ptr(),
                                      seg_ts.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), s1 - s0, start.data_ptr(), None,
                                      y_ckpt[s0].data_ptr(), store_ptr, ws.data_ptr(), ws.numel()), "pegncde_solve_fwd")

        if pc.pending is not None:
            # streaming pays when a cubic piece is big (its copy hides behind the steps inside the previous piece); many small
            # pieces (SIR: 119 pieces of 16 MB) are cheaper to copy in one go
            piece_bytes = 4 * pc.B * pc.n * pc.n * 2 * 4
            if pc.host_ts is None or piece_bytes < STREAM_MIN_PIECE_BYTES:
                pc.materialize()
        if pc.pending is None:
            run_steps(0, S)
        else:
            _stream_pieces(pc, host_ts, run_steps)
        ctx.save_for_backward(flat, y_ckpt)
        ctx.store = store
        ctx.pc, ctx.dims, ctx.host_ts, ctx.S, ctx.save_steps = pc, dims, host_ts, S, save_steps
        return y_ckpt if save_steps else y_ckpt[S]

    @staticmethod
    def backward(ctx, g_out):
        flat, y_ckpt = ctx.saved_tensors
        l = lib()
        dims, pc, S = ctx.dims, ctx.pc, ctx.S
        dev = flat.device
        nbytes = l.pegncde_workspace_bytes(dims, PEG_WS_SOLVE_BWD, S)
        ws = workspace(dev, nbytes)
        g_out = g_out.contiguous().to(torch.float32)
        if ctx.save_steps:
            g_ckpt = g_out
            g_yT = torch.zeros_like(y_ckpt[0])
        else:
            g_ckpt = None
            g_yT = g_out
        g_y0 = torch.empty_like(y_ckpt[0])
        g_flat = torch.zeros_like(flat)
        g_x = torch.zeros_like(pc.x_coef) if ctx.needs_input_grad[2] else None
        g_adj = adj_grad_buffer(pc, ctx.needs_input_grad[3])
        ctl = pc.struct()
        store = ctx.store
        _solve_bwd(l, g_adj, _stream_ptr(dev), dims, ctl, flat.data_ptr(),
                   ctx.host_ts.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), S, y_ckpt.data_ptr(),
                   store.data_ptr() if store is not None else None, g_yT.data_ptr(), g_ckpt.data_ptr() if g_ckpt is not None else None, None, g_y0.data_ptr(),
                   g_flat.data_ptr(), g_x.data_ptr() if g_x is not None else None, ws.data_ptr(), ws.numel())
        ctx.store = None
        return g_y0, g_flat, g_x, g_adj, None, None, None, None, None


def dense_samples_of_table(step_ts: np.ndarray, save_ts: np.ndarray):
    """For every save time the step that produces it and the position inside the step, as diffrax's SaveAt(ts=...) does
    it: a save time t is emitted by the step with ``tprev < t <= tnext`` (``t == t0`` by the first step, theta = 0).
    -> list of (save index, step index, theta)."""
    f = np.float32
    out = []
    S = len(step_ts) - 1
    for m, t in enumerate(save_ts):
        t = f(t)
        if t < step_ts[0] or t > step_ts[-1]:
            raise ValueError("SaveAt(ts=...) holds times outside [t0, t1]")
        s = int(np.searchsorted(step_ts, t, side="left")) - 1
        s = min(max(s, 0), S - 1)
        h = f(step_ts[s + 1] - step_ts[s])
        theta = f(min(max(f(t - step_ts[s]) / h, f(0.0)), f(1.0)))
        out.append((m, s, float(theta)))
    return out


class _FixedDenseFunction(torch.autograd.Function):
    """Fixed-step solve with ``SaveAt(ts=...)`` (src/models/pgt_graph_neural_cde.py:114-117, tgb_graph_neural_cde.py:147-150):
    the forward solve keeps y at every step boundary; every step that holds a save time is re-evaluated once with
    ``pegncde_step_fwd`` (all seven slopes) and sampled with Tsit5's interpolant (``pegncde_tsit5_dense``).  Backward = the exact
    discrete adjoint over the step table, the samples entering as cotangents of their step's start state and stage slopes."""

    @staticmethod
    def forward(ctx, y0, flat, x_packed, adj_packed, pc, dims, step_ts, save_ts):
        y0 = y0.contiguous()
        flat = flat.contiguous()
        l = lib()
        dev = y0.device
        S = len(step_ts) - 1
        pc.materialize()
        ws = workspace(dev, max(l.pegncde_workspace_bytes(dims, PEG_WS_SOLVE_FWD, S), l.pegncde_workspace_bytes(dims, PEG_WS_SOLVE_BWD, S),
                                l.pegncde_workspace_bytes(dims, PEG_WS_STEP, 1)))
        host_ts = np.ascontiguousarray(step_ts, dtype=np.float32)
        y_ckpt = torch.empty((S + 1,) + tuple(y0.shape), dtype=torch.float32, device=dev)
        ctl = pc.struct()
        st = _stream_ptr(dev)
        check(l.pegncde_solve_fwd(st, dims, ctl, flat.data_ptr(), host_ts.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), S,
                                  y0.data_ptr(), None, y_ckpt.data_ptr(), None, ws.data_ptr(), ws.numel()), "pegncde_solve_fwd")
        samples = dense_samples_of_table(host_ts, save_ts)
        ys = torch.empty((len(save_ts),) + tuple(y0.shape), dtype=torch.float32, device=dev)
        k1, k7, y1 = torch.empty_like(y0), torch.empty_like(y0), torch.empty_like(y0)
        kst = torch.empty((5,) + tuple(y0.shape), dtype=torch.float32, device=dev)
        done_step = -1
        for (m, s, theta) in sorted(samples, key=lambda r: r[1]):
            h = float(np.float32(host_ts[s + 1] - host_ts[s]))
            if s != done_step:
                check(l.pegncde_step_fwd(st, dims, ctl, flat.data_ptr(), float(host_ts[s]), h, y_ckpt[s].data_ptr(), k1.data_ptr(), 0,
                                         y1.data_ptr(), None, k7.data_ptr(), kst.data_ptr(), ws.data_ptr(), ws.numel()), "pegncde_step_fwd")
                done_step = s
            check(l.pegncde_tsit5_dense(st, dims, h, theta, y_ckpt[s].data_ptr(), k1.data_ptr(), kst.data_ptr(), k7.data_ptr(),
                                        ys[m].data_ptr()), "pegncde_tsit5_dense")
        ctx.save_for_backward(flat, y_ckpt)
        ctx.pc, ctx.dims, ctx.host_ts, ctx.S, ctx.samples = pc, dims, host_ts, S, samples
        return ys

    @staticmethod
    def backward(ctx, g_out):
        flat, y_ckpt = ctx.saved_tensors
        l = lib()
        dims, pc, S, host_ts = ctx.dims, ctx.pc, ctx.S, ctx.host_ts
        dev = flat.device
        ws = workspace(dev, l.pegncde_workspace_bytes(dims, PEG_WS_SOLVE_BWD, S))
        g_out = g_out.contiguous().to(torch.float32)
        g_ckpt = torch.zeros_like(y_ckpt)
        g_stage = torch.zeros((S, 7) + tuple(y_ckpt.shape[1:]), dtype=torch.float32, device=dev)
        for (m, s, theta) in ctx.samples:
            g_ckpt[s] += g_out[m]
            w = dense_weights(theta) * np.float32(host_ts[s + 1] - host_ts[s])
            for i in range(7):
                if w[i] != 0.0:
                    g_stage[s, i].add_(g_out[m], alpha=float(w[i]))
        g_y0 = torch.empty_like(y_ckpt[0])
        g_flat = torch.zeros_like(flat)
        g_x = torch.zeros_like(pc.x_coef) if ctx.needs_input_grad[2] else None
        g_adj = adj_grad_buffer(pc, ctx.needs_input_grad[3])
        _solve_bwd(l, g_adj, _stream_ptr(dev), dims, pc.struct(), flat.data_ptr(), host_ts.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), S,
                   y_ckpt.data_ptr(), None, None, g_ckpt.data_ptr(), g_stage.data_ptr(), g_y0.data_ptr(), g_flat.data_ptr(),
                   g_x.data_ptr() if g_x is not None else None, ws.data_ptr(), ws.numel())
        return g_y0, g_flat, g_x, g_adj, None, None, None, None


def _stream_pieces(pc, step_ts, run_steps) -> None:
    """Streamed control (host coefficient arrays): copy + pack cubic piece i+1 on a side stream while the solver steps that
    end inside piece i run on the main stream.  A step may start once the piece holding its end time is packed (the lookup
    is left-continuous like diffrax's: index = searchsorted(ts, t, 'left') - 1)."""
    dev = pc.device
    main = torch.cuda.current_stream(dev)
    side = torch.cuda.Stream(dev)
    side.wait_stream(main)
    B, Tm1, n = pc.B, pc.T - 1, pc.n
    S = len(step_ts) - 1
    piece_of_step = np.clip(np.searchsorted(pc.host_ts, step_ts[1:], side="left") - 1, 0, Tm1 - 1)
    staging = [[torch.empty((B, 1, n, n, 2), dtype=torch.float32, device=dev) for _ in range(4)] for _ in range(2)]
    packed_ev = [None, None]
    done = 0
    for iv in range(Tm1):
        buf = staging[iv & 1]
        with torch.cuda.stream(side):
            if packed_ev[iv & 1] is not None:
                side.wait_event(packed_ev[iv & 1])          # the pack that last read this staging buffer has finished
            for q in range(4):
                for b in range(B):
                    buf[q][b, 0].copy_(pc.pending[q][b, iv], non_blocking=True)
            copied = torch.cuda.Event()
            copied.record(side)
        main.wait_event(copied)
        pc.pack_pieces(iv, 1, buf, main.cuda_stream)
        packed_ev[iv & 1] = torch.cuda.Event()
        packed_ev[iv & 1].record(main)
        end = done
        while end < S and piece_of_step[end] <= iv:
            end += 1
        if end > done:
            run_steps(done, end)
            done = end
    if done < S:
        run_steps(done, S)
    for buf in staging:
        for t in buf:
            t.record_stream(side)
    pc.pending = None


def _unwrap(term):
    vf = term.vector_field if isinstance(term, ODETerm) else term
    if isinstance(vf, CDEWrapperVectorField):
        return vf.vector_field, True
    if isinstance(vf, PermEquivGraphVectorField):
        return vf, False
    raise TypeError("the fused solve supports ODETerm(PermEquivGraphVectorField) and ODETerm(CDEWrapperVectorField(...))")


def diffeqsolve(terms, solver, t0, t1, dt0, y0, args=None, *, saveat: Optional[SaveAt] = None,
                stepsize_controller=None, max_steps: int = 4096, **unused) -> Solution:
    """Fused drop-in for ``diffrax.diffeqsolve`` on the hot path: Tsit5 with ``ConstantStepSize()`` (one C-ABI call
    per solve) or ``PIDController(rtol, atol)`` (+ ``SaveAt(ts=...)`` dense output; host-driven step loop).

    ``y0``: ``[n,h]`` or batched ``[B,n,h]`` (the reference's ``jax.vmap(model)`` batch)."""
    if not isinstance(solver, Tsit5):
        raise NotImplementedError("only Tsit5 is implemented by the fused kernels")
    controller = stepsize_controller or ConstantStepSize()
    if not isinstance(controller, (ConstantStepSize, PIDController)):
        raise NotImplementedError("stepsize_controller must be ConstantStepSize() or PIDController(rtol, atol)")
    adaptive = isinstance(controller, PIDController)
    if dt0 is None and not adaptive:
        raise ValueError("ConstantStepSize needs dt0")
    saveat = saveat or SaveAt(t1=True)
    vf, wrapped = _unwrap(terms)
    if y0.device.type != "cuda":
        raise RuntimeError("the fused solve runs on CUDA only (no CPU fallback)")
    if wrapped:
        control_adj, control_data = args
    else:
        control_adj, control_data = (args[0] if isinstance(args, (list, tuple)) else args), None
    pc = resolve_control(control_adj, control_data, y0.device)
    dims = vf.dims_for(pc, with_wrapper=wrapped)
    unb = y0.dim() == 2
    yb = (y0.unsqueeze(0) if unb else y0).to(torch.float32)
    if yb.shape[0] != pc.B:
        raise ValueError(f"state batch {yb.shape[0]} != control batch {pc.B}")
    if adaptive:
        pc.materialize()
        return _diffeqsolve_adaptive(vf, wrapped, pc, t0, t1, dt0, yb, unb, controller, saveat, max_steps)
    step_ts = constant_step_table(float(t0), float(t1), float(dt0), controller.rule, max_steps)
    if saveat.ts is not None:   # SaveAt(ts=...) with ConstantStepSize: evolving_out=True of the PGT / TGB models
        save_ts = np.asarray(torch.as_tensor(saveat.ts).detach().cpu().numpy(), dtype=np.float32).reshape(-1)
        out = _FixedDenseFunction.apply(yb, vf.checked_flat_params(dims), pc.x_packed, pc.adj_packed, pc, dims, step_ts, save_ts)
        S = len(step_ts) - 1
        return Solution(ts=torch.from_numpy(save_ts.copy()), ys=out.squeeze(1) if unb else out,
                        stats={"num_steps": S, "num_accepted_steps": S, "num_rejected_steps": 0})
    out = _SolveFunction.apply(yb, vf.checked_flat_params(dims), pc.x_packed, pc.adj_packed, pc, dims, step_ts, bool(saveat.steps),
                               bool(getattr(vf, "store_stages", True)))
    S = len(step_ts) - 1
    if saveat.steps:
        ys = out.squeeze(1) if unb else out
        ts_out = torch.from_numpy(step_ts.copy())
    else:
        ys = (out.squeeze(0) if unb else out).unsqueeze(0)  # diffrax: ys has a leading save axis of length 1
        ts_out = torch.tensor([float(step_ts[-1])])
    return Solution(ts=ts_out, ys=ys, stats={"num_steps": S, "num_accepted_steps": S, "num_rejected_steps": 0})


# ----------------------------------------------------------------------------------------------
# adaptive path: Tsit5 + PIDController + SaveAt(ts=...)   (graph_neural_cde.py:53-54, 86-104)
# ----------------------------------------------------------------------------------------------
def dense_weights(theta: float) -> np.ndarray:
    """b_i(theta), i = 1..7, of Tsit5's 4th-order interpolant (``pegncde_tsit5_dense_weights``)."""
    w = (ctypes.c_float * 7)()
    lib().pegncde_tsit5_dense_weights(float(theta), w)
    return np.asarray(list(w), dtype=np.float32)


def _initial_step(dims, pc1, flat, y, k1, t0, ctrl: PIDController):
    """diffrax ``_select_initial_step`` (Hairer, Norsett & Wanner II.4, error order 5) for ONE trajectory (B = 1): a few scaled
    norms and one extra evaluation, done once per solve (the only host round trips of the adaptive path besides the polling)."""
    l = lib()
    dev = y.device
    f = np.float32
    st = _stream_ptr(dev)
    ctl = pc1.struct()
    ws = workspace(dev, max(l.pegncde_workspace_bytes(dims, PEG_WS_STEP, 1), l.pegncde_workspace_bytes(dims, PEG_WS_VF_FWD, 1)))
    nh = y[0].numel()
    norm_out = torch.empty(1, dtype=torch.float32, device=dev)

    def norm(x, x2, s0, s1):
        check(l.pegncde_scaled_sumsq(st, dims, x.data_ptr(), x2.data_ptr() if x2 is not None else None, s0.data_ptr(),
                                     s1.data_ptr() if s1 is not None else None, ctrl.rtol, ctrl.atol, norm_out.data_ptr()), "pegncde_scaled_sumsq")
        return f(np.sqrt(f(norm_out.item()) / f(nh)))

    d0, d1 = norm(y, None, y, None), norm(k1, None, y, None)
    small = d0 < f(1e-5) or d1 < f(1e-5)
    h0 = f(1e-6) if small else f(f(0.01) * f(d0 / d1))
    f1 = torch.empty_like(y)
    y_probe = torch.add(y, k1, alpha=float(h0))
    check(l.pegncde_vf_fwd(st, dims, ctl, flat.data_ptr(), float(f(t0 + h0)), y_probe.data_ptr(), f1.data_ptr(), ws.data_ptr(), ws.numel()), "pegncde_vf_fwd")
    d2 = f(norm(f1, k1, y, None) / h0)
    dmax = max(d1, d2)
    h1 = max(f(1e-6), f(h0 * f(1e-3))) if dmax <= f(1e-15) else f((f(0.01) / dmax) ** f(1.0 / ctrl.error_order))
    return min(f(100.0) * h0, h1)


def _adaptive_batch(vf, wrapped, pc, flat, y0, t0, t1, dt0, ctrl: PIDController, save_ts, max_steps):
    """Forward solve of ALL trajectories of the batch under the PID controller, the controller running on the device
    (``pegncde_step_fwd_batched`` + ``pegncde_adaptive_control``): one step launch per attempt for the whole batch, every trajectory with
    its own accepted-step sequence, the host polling the `done` flags every few attempts.  Returns per-trajectory records for the
    adjoint (accepted step table, checkpoints, which step emitted which dense-output sample) and the saved states."""
    from ._lib import PegAdaptState

    l = lib()
    dev = y0.device
    f = np.float32
    st = _stream_ptr(dev)
    B = pc.B
    dims = vf.dims_for(pc, with_wrapper=wrapped)
    ctl = pc.struct()
    ws = workspace(dev, max(l.pegncde_workspace_bytes(dims, PEG_WS_STEP, 1), l.pegncde_workspace_bytes(dims, PEG_WS_VF_FWD, 1)))
    t0, t1 = f(t0), f(t1)
    y = y0.clone()
    k1 = torch.empty_like(y)
    check(l.pegncde_vf_fwd(st, dims, ctl, flat.data_ptr(), float(t0), y.data_ptr(), k1.data_ptr(), ws.data_ptr(), ws.numel()), "pegncde_vf_fwd")   # FSAL: f(t0, y0)
    state = np.zeros(B, dtype=np.dtype([("tprev", "<f4"), ("tnext", "<f4"), ("done", "<i4"), ("nacc", "<i4"), ("attempts", "<i4"), ("rejected", "<i4"),
                                        ("mi", "<i4"), ("mi0", "<i4"), ("mi1", "<i4"), ("keep", "<i4"), ("h", "<f4"), ("overflow", "<i4")]))
    assert state.dtype.itemsize == ctypes.sizeof(PegAdaptState)
    for b in range(B):
        if dt0 is None:
            pc1 = pc.select(b)
            dt = _initial_step(vf.dims_for(pc1, with_wrapper=wrapped), pc1, flat, y[b:b + 1], k1[b:b + 1], t0, ctrl)
        else:
            dt = f(dt0)
        state["tprev"][b] = t0
        state["tnext"][b] = clip_to_end(t0, f(t0 + dt), t1, True)
    M = 0 if save_ts is None else len(save_ts)
    save_dev = torch.from_numpy(np.ascontiguousarray(save_ts, dtype=np.float32)).to(dev) if M else None
    shape = tuple(y.shape[1:])
    cap = 64

    def alloc(cap_):
        return (torch.empty((B, cap_ + 1) + shape, dtype=torch.float32, device=dev), torch.zeros((B, cap_ + 1), dtype=torch.float32, device=dev))

    y_ckpt, step_tab = alloc(cap)
    y_ckpt[:, 0] = y
    step_tab[:, 0] = float(t0)
    ys_save = torch.empty((M, B) + shape, dtype=torch.float32, device=dev) if M else None
    sample_step = torch.zeros((max(M, 1), B), dtype=torch.int32, device=dev)
    sample_theta = torch.zeros((max(M, 1), B), dtype=torch.float32, device=dev)
    state_dev = torch.from_numpy(state.view(np.uint8).copy()).to(dev)
    t_dev = torch.from_numpy(state["tprev"].copy()).to(dev)
    dt_dev = torch.from_numpy((state["tnext"] - state["tprev"]).astype(np.float32)).to(dev)
    y1, yerr, k7 = torch.empty_like(y), torch.empty_like(y), torch.empty_like(y)
    kst = torch.empty((5,) + tuple(y.shape), dtype=torch.float32, device=dev)
    sumsq = torch.empty(B, dtype=torch.float32, device=dev)
    poll = 8
    host = None
    for it in range(max_steps + poll):
        check(l.pegncde_step_fwd_batched(st, dims, ctl, flat.data_ptr(), t_dev.data_ptr(), dt_dev.data_ptr(), y.data_ptr(), k1.data_ptr(), 1,
                                         y1.data_ptr(), yerr.data_ptr(), k7.data_ptr(), kst.data_ptr(), ws.data_ptr(), ws.numel()), "pegncde_step_fwd_batched")
        check(l.pegncde_adaptive_control(st, dims, state_dev.data_ptr(), ctrl.rtol, ctrl.atol, float(t1), ctrl.safety, ctrl.factormin, ctrl.factormax,
                                         int(ctrl.error_order), save_dev.data_ptr() if M else None, M, cap, y.data_ptr(), y1.data_ptr(), yerr.data_ptr(),
                                         k1.data_ptr(), k7.data_ptr(), kst.data_ptr(), y_ckpt.data_ptr(), ys_save.data_ptr() if M else None,
                                         step_tab.data_ptr(), sample_step.data_ptr(), sample_theta.data_ptr(), t_dev.data_ptr(), dt_dev.data_ptr(),
                                         sumsq.data_ptr()), "pegncde_adaptive_control")
        if it % poll != poll - 1:
            continue
        host = state_dev.cpu().numpy().view(state.dtype)        # the one synchronisation per `poll` attempts
        if int(host["attempts"].max()) > max_steps:
            raise RuntimeError(f"max_steps={max_steps} reached")   # diffrax throw=True
        if host["overflow"].any():                                # grow the accepted-step tables, re-arm the stalled trajectories
            new_cap = 2 * cap
            y_new, tab_new = alloc(new_cap)
            y_new[:, : cap + 1] = y_ckpt
            tab_new[:, : cap + 1] = step_tab
            y_ckpt, step_tab, cap = y_new, tab_new, new_cap
            host = host.copy()
            host["overflow"][:] = 0
            state_dev.copy_(torch.from_numpy(host.view(np.uint8).copy()))
            dt_dev.copy_(torch.from_numpy(np.where(host["done"] != 0, 0.0, host["tnext"] - host["tprev"]).astype(np.float32)))
            continue
        if host["done"].all():
            break
    else:
        raise RuntimeError(f"max_steps={max_steps} reached")
    if M and int(host["mi"].min()) < M:
        raise ValueError("SaveAt(ts=...) holds times outside [t0, t1]")
    tab = step_tab.cpu().numpy()
    s_step, s_theta = sample_step.cpu().numpy(), sample_theta.cpu().numpy()
    recs = []
    for b in range(B):
        S = int(host["nacc"][b])
        table = np.ascontiguousarray(tab[b, : S + 1], dtype=np.float32)
        recs.append(dict(step_ts=table, y_ckpt=y_ckpt[b, : S + 1].unsqueeze(1), samples=[(m, int(s_step[m, b]), float(s_theta[m, b])) for m in range(M)],
                         stats={"num_steps": int(host["attempts"][b]), "num_accepted_steps": S, "num_rejected_steps": int(host["rejected"][b]),
                                "step_ts": table}))
    out = ys_save if M else y.unsqueeze(0)
    return recs, out


class _AdaptiveSolveFunction(torch.autograd.Function):
    """Adaptive solve of a batch of trajectories (each with its own accepted-step sequence).  Backward = the exact
    discrete adjoint over the accepted steps with the step sizes held fixed (``pegncde_solve_bwd``), the dense-output
    samples entering as cotangents of the step's start state and of its seven stage slopes."""

    @staticmethod
    def forward(ctx, y0, flat, adj_packed, vf, wrapped, pc, t0, t1, dt0, ctrl, save_ts, max_steps, stats_out):
        y0 = y0.contiguous()
        flat = flat.contiguous()
        recs, out = _adaptive_batch(vf, wrapped, pc, flat, y0, t0, t1, dt0, ctrl, save_ts, max_steps)
        for b, rec in enumerate(recs):
            pc1 = pc.select(b)
            rec["dims"], rec["pc1"] = vf.dims_for(pc1, with_wrapper=wrapped), pc1
            stats_out.append(rec["stats"])
        ctx.recs, ctx.has_ts = recs, save_ts is not None
        ctx.save_for_backward(flat)
        return out   # [M or 1, B, n, h]

    @staticmethod
    def backward(ctx, g_out):
        (flat,) = ctx.saved_tensors
        l = lib()
        dev = flat.device
        g_out = g_out.contiguous().to(torch.float32)
        g_flat = torch.zeros_like(flat)
        g_adj = adj_grad_buffer(ctx.recs[0]["pc1"], ctx.needs_input_grad[2])   # shared by the per-graph views: entries are absolute
        g_y0s = []
        for b, rec in enumerate(ctx.recs):
            dims, pc1, y_ckpt, step_ts = rec["dims"], rec["pc1"], rec["y_ckpt"], rec["step_ts"]
            S = len(step_ts) - 1
            ws = workspace(dev, l.pegncde_workspace_bytes(dims, PEG_WS_SOLVE_BWD, S))
            g_y0 = torch.empty_like(y_ckpt[0])
            g_ckpt = torch.zeros_like(y_ckpt)
            g_stage = None
            if ctx.has_ts:
                g_stage = torch.zeros((S, 7) + tuple(y_ckpt.shape[1:]), dtype=torch.float32, device=dev)
                for (m, s, theta) in rec["samples"]:
                    gm = g_out[m, b:b + 1]
                    g_ckpt[s] += gm
                    w = dense_weights(theta) * np.float32(step_ts[s + 1] - step_ts[s])
                    for i in range(7):
                        if w[i] != 0.0:
                            g_stage[s, i].add_(gm, alpha=float(w[i]))
            else:
                g_ckpt[S] = g_out[0, b:b + 1]
            _solve_bwd(l, g_adj, _stream_ptr(dev), dims, pc1.struct(), flat.data_ptr(),
                       step_ts.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), S, y_ckpt.data_ptr(), None, None,
                       g_ckpt.data_ptr(), g_stage.data_ptr() if g_stage is not None else None, g_y0.data_ptr(),
                       g_flat.data_ptr(), None, ws.data_ptr(), ws.numel())
            g_y0s.append(g_y0)
        return (torch.cat(g_y0s, dim=0), g_flat, g_adj) + (None,) * 10


def _diffeqsolve_adaptive(vf, wrapped, pc, t0, t1, dt0, yb, unb, ctrl, saveat, max_steps) -> Solution:
    if saveat.steps:
        raise NotImplementedError("SaveAt(steps=True) with an adaptive controller (ragged per trajectory) is not implemented")
    save_ts = None
    if saveat.ts is not None:
        save_ts = np.asarray(torch.as_tensor(saveat.ts).detach().cpu().numpy(), dtype=np.float32)
    stats_list = []
    out = _AdaptiveSolveFunction.apply(yb, vf.flat_params(), pc.adj_packed, vf, wrapped, pc, float(t0), float(t1), dt0, ctrl, save_ts, max_steps,
                                       stats_list)
    ys = out.squeeze(1) if unb else out
    ts_out = torch.from_numpy(save_ts.copy()) if save_ts is not None else torch.tensor([float(t1)])
    stats = stats_list[0] if unb else {k: [s[k] for s in stats_list] for k in stats_list[0]}
    return Solution(ts=ts_out, ys=ys, stats=stats)


def tsit5_step(vf_term, t: float, dt: float, y: torch.Tensor, args, k1: Optional[torch.Tensor] = None):
    """One Tsit5 step through ``pegncde_step_fwd`` -> ``(y1, y_err, k7)`` (forward only; the adaptive
    ``diffeqsolve`` path below is built on the same entry point)."""
    vf, wrapped = _unwrap(vf_term)
    if wrapped:
        control_adj, control_data = args
    else:
        control_adj, control_data = (args[0] if isinstance(args, (list, tuple)) else args), None
    pc = resolve_control(control_adj, control_data, y.device).materialize()
    dims = vf.dims_for(pc, with_wrapper=wrapped)
    unb = y.dim() == 2
    yb = (y.unsqueeze(0) if unb else y).to(torch.float32).contiguous()
    l = lib()
    ws = workspace(y.device, l.pegncde_workspace_bytes(dims, PEG_WS_STEP, 1))
    k1_valid = k1 is not None
    k1b = (k1.unsqueeze(0) if (unb and k1_valid) else k1)
    k1b = k1b.contiguous().clone() if k1_valid else torch.empty_like(yb)
    y1, yerr, k7 = torch.empty_like(yb), torch.empty_like(yb), torch.empty_like(yb)
    flat = vf.flat_params().detach().contiguous()
    ctl = pc.struct()
    check(l.pegncde_step_fwd(_stream_ptr(y.device), dims, ctl, flat.data_ptr(), float(t), float(dt), yb.data_ptr(),
                             k1b.data_ptr(), 1 if k1_valid else 0, y1.data_ptr(), yerr.data_ptr(), k7.data_ptr(), None,
                             ws.data_ptr(), ws.numel()), "pegncde_step_fwd")
    if unb:
        return y1.squeeze(0), yerr.squeeze(0), k7.squeeze(0)
    return y1, yerr, k7
