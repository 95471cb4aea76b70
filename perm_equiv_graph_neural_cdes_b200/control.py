"""Control paths: the host-side mirror of ``diffrax.backward_hermite_coefficients`` /
``diffrax.CubicInterpolation`` as the reference uses them
(src/configs/dataset_configs.py:147-173, 1073-1100; src/models/pgt_graph_neural_cde.py:101-107),
plus the packed planar device layout the kernels consume.

Coefficient tuples keep diffrax's order ``(d, c, b, a)`` and the reference's layout
``[..., T-1, n, n, 2]`` with the last axis interleaved (time, adjacency).
"""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import torch

from ._lib import PegControl, PegDims, check, lib


def backward_hermite_coefficients(ts: torch.Tensor, ys: torch.Tensor) -> Tuple[torch.Tensor, ...]:
    """``diffrax.backward_hermite_coefficients(ts, ys)`` -> ``(d, c, b, a)``, each ``[T-1, ...]``.

    Elementwise torch ops (runs on whatever device ``ys`` lives on).  Per interval i with
    dt = t[i+1]-t[i] and secant m_i: a = y_i, b = m_{i-1} (m_0 first), c = 2(m_i-b)/dt, d = -(m_i-b)/dt^2."""
    ts = ts.to(ys.dtype)
    dt = (ts[1:] - ts[:-1]).reshape((-1,) + (1,) * (ys.dim() - 1))
    m = (ys[1:] - ys[:-1]) / dt
    b = torch.cat([m[:1], m[:-1]], dim=0)
    a = ys[:-1]
    c = 2.0 * (m - b) / dt
    d = -(m - b) / (dt * dt)
    return d, c, b, a


def _pad32(n: int) -> int:
    return (n + 31) // 32 * 32


def tiled_offsets(npad: int) -> torch.Tensor:
    """Float offset, inside one slab, of element (plane q, row i, col k) of the 32x32-tiled plane layout
    (``peg_tile_off`` in csrc/peg_common.cuh) as an int64 tensor [4, npad, npad] -- for inspection / tests."""
    nt = npad // 32
    i = torch.arange(npad).view(1, npad, 1)
    k = torch.arange(npad).view(1, 1, npad)
    q = torch.arange(4).view(4, 1, 1)
    rt, ct, r, c = i // 32, k // 32, i % 32, k % 32
    rq, m, cq, e = r // 4, r % 4, c // 4, c % 4
    s = (rq - cq) % 8
    g, lane = s // 4, (s % 4) * 8 + cq
    return (rt * nt + ct) * 4096 + ((g * 4 + q) * 4 + m) * 128 + lane * 4 + e


class CubicInterpolation:
    """Drop-in for ``diffrax.CubicInterpolation(ts, coeffs)`` on the fused path.

    ``coeffs = (d, c, b, a)``; for the adjacency control each is ``[T-1, n, n, 2]`` (or batched
    ``[B, T-1, n, n, 2]``), for the node-signal control ``[T-1, n, e, 2]``.  ``evaluate`` /
    ``derivative`` exist for API parity (torch ops on the device); the solver never calls them --
    it consumes the packed planes built lazily by :meth:`packed_adj` / :meth:`packed_x`.
    """

    def __init__(self, ts: torch.Tensor, coeffs: Sequence[torch.Tensor]):
        if isinstance(coeffs, torch.Tensor):  # the PGT trainer passes the 4 arrays stacked (trainer_pgt.py:203)
            coeffs = tuple(coeffs[i] for i in range(4))
        self.ts = ts
        self.d, self.c, self.b, self.a = coeffs
        self._packed = None

    # -- diffrax API -------------------------------------------------------------------
    def _interpret_t(self, t):
        ts = self.ts.to(torch.float32)
        t = torch.as_tensor(t, dtype=torch.float32, device=ts.device)
        idx = torch.searchsorted(ts.contiguous(), t, right=False) - 1
        idx = int(idx.clamp(0, ts.numel() - 2))
        return idx, t - ts[idx]

    def evaluate(self, t):
        i, s = self._interpret_t(t)
        return self.a[i] + s * (self.b[i] + s * (self.c[i] + s * self.d[i]))

    def derivative(self, t):
        i, s = self._interpret_t(t)
        return self.b[i] + s * (2.0 * self.c[i] + 3.0 * s * self.d[i])


class LinearInterpolation(CubicInterpolation):
    """Drop-in for ``diffrax.LinearInterpolation(ts, ys)`` (``interpolation="linear"`` of the PGT / TGB models,
    src/models/pgt_graph_neural_cde.py:101-103): ``ys`` are the knot values ``[T, n, n, 2]`` (what ``diffrax.linear_interpolation``
    returns for data without NaNs).  A piecewise-linear path is the cubic path with ``a = y_i``, ``b = (y_{i+1} - y_i) / dt``,
    ``c = d = 0``, so the fused kernels run it unchanged (same left-continuous piece lookup)."""

    def __init__(self, ts: torch.Tensor, ys: torch.Tensor):
        tsv = ts.to(ys.dtype)
        batched = ys.dim() == 5 or (ys.dim() == 4 and ts.dim() == 2)
        t_axis = 1 if batched else 0
        dt = (tsv[..., 1:] - tsv[..., :-1])
        shape = [1] * ys.dim()
        shape[t_axis] = -1
        if tsv.dim() == 2:
            shape[0] = tsv.shape[0]
        a = ys.narrow(t_axis, 0, ys.shape[t_axis] - 1)
        b = (ys.narrow(t_axis, 1, ys.shape[t_axis] - 1) - a) / dt.reshape(shape)
        z = torch.zeros_like(a)
        super().__init__(ts, (z, z, b, a))


class PackedControl:
    """Planar device layout of one batch of control paths (``PegControl`` in pegncde.h).

    Built once per batch; owns the device tensors and hands raw pointers to the C-ABI."""

    adj_packed = None   # differentiable source of the adjacency coefficients: sparse controls only (SparseControl)

    def __init__(self, B: int, n: int, T: int, e: int, device):
        self.B, self.n, self.T, self.e = B, n, T, e
        self.ldn = _pad32(n)  # planes are stored as 32x32 tiles, zero padded
        f = dict(dtype=torch.float32, device=device)
        self.ts = torch.empty((B, T), **f)
        self.adj_coef = torch.empty((B, T - 1, 4 * self.ldn * self.ldn), **f)
        self.adj_rowsum = torch.empty((B, T - 1, 4, n), **f)
        self.adj_diag = torch.empty((B, T - 1, 4, n), **f)
        self.adj_total = torch.empty((B, T - 1, 4), **f)
        self.tch_coef = torch.empty((B, T - 1, 3, n), **f)
        self.adj_absmax = torch.empty((B, T - 1, 4), **f)   # max |entry| of each plane: range bound of the fp16x2 operand format
        self.x_coef = torch.empty((B, T - 1, 3, n, 2 * e), **f) if e > 0 else None
        self.x_packed = None   # differentiable source of x_coef when the node-signal coefficients require grad
        # state of the adjacency part, SHARED by every view made with with_x(): column sums of the planes ([B,T-1,4,n], built on
        # demand for the directed fusion layer), the host (d,c,b,a) arrays whose planes have not been copied / packed yet
        # (streamed controls) and the knot times shared by the batch (streaming needs one time grid; numpy fp32)
        self._adj = {"colsum": None, "pending": None, "host_ts": None}

    adj_colsum = property(lambda self: self._adj["colsum"], lambda self, v: self._adj.__setitem__("colsum", v))
    pending = property(lambda self: self._adj["pending"], lambda self, v: self._adj.__setitem__("pending", v))
    host_ts = property(lambda self: self._adj["host_ts"], lambda self, v: self._adj.__setitem__("host_ts", v))

    def with_x(self, x_coeffs) -> "PackedControl":
        """The same adjacency planes (shared tensors, shared streaming state -- no copy, no re-pack) paired with the
        node-signal coefficients ``x_coeffs = (d,c,b,a)``, each ``[T-1,n,e,2]`` or ``[B,T-1,n,e,2]``."""
        v = PackedControl.__new__(PackedControl)
        v.B, v.n, v.T, v.ldn = self.B, self.n, self.T, self.ldn
        for name in ("ts", "adj_coef", "adj_rowsum", "adj_diag", "adj_total", "tch_coef", "adj_absmax"):
            setattr(v, name, getattr(self, name))
        v._adj = self._adj
        v._keepalive = self
        _attach_x(v, x_coeffs, self.device)
        return v

    def pack_pieces(self, begin: int, count: int, staging, stream_ptr: int) -> None:
        """Packs cubic pieces [begin, begin+count) from device staging arrays (d,c,b,a each [B,count,n,n,2])."""
        check(lib().pegncde_pack_adj_range(stream_ptr, self.dims(h=4, L=1), begin, count, staging[0].data_ptr(), staging[1].data_ptr(),
                                           staging[2].data_ptr(), staging[3].data_ptr(), self.adj_coef.data_ptr(),
                                           self.adj_rowsum.data_ptr(), self.adj_diag.data_ptr(), self.adj_total.data_ptr(),
                                           self.tch_coef.data_ptr()), "pegncde_pack_adj_range")
        self.plane_maxima(begin, count, stream_ptr)

    def plane_maxima(self, begin: int = 0, count: int = -1, stream_ptr: Optional[int] = None) -> None:
        """``adj_absmax`` of the cubic pieces [begin, begin+count) from the tiled planes (``pegncde_adj_absmax``)."""
        count = self.T - 1 - begin if count < 0 else count
        st = _stream_ptr(self.device) if stream_ptr is None else stream_ptr
        check(lib().pegncde_adj_absmax(st, self.dims(h=4, L=1), begin, count, self.adj_coef.data_ptr(), self.adj_absmax.data_ptr()),
              "pegncde_adj_absmax")

    def materialize(self) -> "PackedControl":
        """Copies and packs every pending piece now (adaptive solves, single evaluations, ragged time grids)."""
        if self.pending is not None:
            dev = self.device
            total = 4 * self.pending[0].numel() * 4
            chunk = self.T - 1 if total <= (8 << 30) else max(1, (self.T - 1) * (8 << 30) // total)   # <= 8 GB of staging at a time
            for iv in range(0, self.T - 1, chunk):
                cnt = min(chunk, self.T - 1 - iv)
                staging = [c[:, iv:iv + cnt].to(dev, non_blocking=True).contiguous() for c in self.pending]
                self.pack_pieces(iv, cnt, staging, _stream_ptr(dev))
            self.pending = None
        return self

    def select(self, b: int) -> "PackedControl":
        """View of graph ``b`` as a batch of one (no copy): adaptive solves step every trajectory on its own."""
        v = PackedControl.__new__(PackedControl)
        v.B, v.n, v.T, v.e, v.ldn = 1, self.n, self.T, self.e, self.ldn
        for name in ("ts", "adj_coef", "adj_rowsum", "adj_diag", "adj_total", "tch_coef", "adj_absmax"):
            setattr(v, name, getattr(self, name)[b:b + 1])
        v.x_coef = self.x_coef[b:b + 1] if self.x_coef is not None else None
        v.x_packed = None
        cs = self.adj_colsum
        v._adj = {"colsum": cs[b:b + 1] if cs is not None else None, "pending": None, "host_ts": None}
        v._keepalive = self
        return v

    def dims(self, h: int, L: int, flags: int = 0) -> PegDims:
        return PegDims(self.B, self.n, self.ldn, h, self.e, L, self.T, flags)

    def dense_planes(self) -> torch.Tensor:
        """Un-tiles ``adj_coef`` to [B, T-1, 4(a,b,c,d), n, n] (inspection / tests)."""
        off = tiled_offsets(self.ldn).to(self.adj_coef.device)
        dense = self.adj_coef[:, :, off.reshape(-1)].reshape(self.B, self.T - 1, 4, self.ldn, self.ldn)
        return dense[..., : self.n, : self.n]

    def struct(self) -> PegControl:
        return PegControl(
            self.ts.data_ptr(), self.adj_coef.data_ptr(), self.adj_rowsum.data_ptr(), self.adj_diag.data_ptr(),
            self.adj_total.data_ptr(), self.tch_coef.data_ptr(), self.x_coef.data_ptr() if self.x_coef is not None else None,
            self.adj_colsum.data_ptr() if self.adj_colsum is not None else None,
            self.adj_absmax.data_ptr() if getattr(self, "adj_absmax", None) is not None else None,
        )

    def ensure_colsums(self) -> "PackedControl":
        """Column sums of the planes (``pegncde_adj_colsums``), needed by ``PEG_FLAG_DIRECTED`` only; computed once."""
        if self.adj_colsum is None:
            self.materialize()
            self.adj_colsum = torch.empty((self.B, self.T - 1, 4, self.n), dtype=torch.float32, device=self.device)
            check(lib().pegncde_adj_colsums(_stream_ptr(self.device), self.dims(h=4, L=1), self.adj_coef.data_ptr(),
                                            self.adj_colsum.data_ptr()), "pegncde_adj_colsums")
        return self

    @property
    def device(self):
        return self.ts.device


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _as_batched(x: torch.Tensor, nd_unbatched: int) -> torch.Tensor:
    return x.unsqueeze(0) if x.dim() == nd_unbatched else x


def _attach_x(pc: "PackedControl", x_coeffs, device) -> None:
    """Sets the node-signal part (e, x_coef, x_packed) of ``pc`` from reference-layout coefficients (or clears it)."""
    pc.x_packed = None
    if x_coeffs is None:
        pc.e, pc.x_coef = 0, None
        return
    if isinstance(x_coeffs, torch.Tensor):
        x_coeffs = tuple(x_coeffs[i] for i in range(4))
    cx = [_as_batched(c, 4).to(device=device, dtype=torch.float32, non_blocking=True).contiguous() for c in x_coeffs]
    B, Tm1, n, e = cx[0].shape[0], cx[0].shape[1], cx[0].shape[2], cx[0].shape[3]
    if (B, Tm1, n) != (pc.B, pc.T - 1, pc.n):
        raise ValueError(f"node-signal coefficients [B={B},T-1={Tm1},n={n}] do not match the adjacency control [B={pc.B},T-1={pc.T - 1},n={pc.n}]")
    pc.e = e
    if any(c.requires_grad for c in cx):
        # learnable node-signal path (TGB models, tgb_graph_neural_cde.py:118-137): the re-layout stays on the autograd
        # tape so that pegncde_solve_bwd's g_xcoef flows back into backward_hermite_coefficients / the data encoder
        pc.x_packed = torch.stack([cx[2], cx[1], cx[0]], dim=2).reshape(B, Tm1, 3, n, 2 * e)
        pc.x_coef = pc.x_packed.detach().contiguous()
    else:
        pc.x_coef = torch.empty((B, Tm1, 3, n, 2 * e), dtype=torch.float32, device=device)
        check(lib().pegncde_pack_x(_stream_ptr(device), pc.dims(h=4, L=1), cx[0].data_ptr(), cx[1].data_ptr(), cx[2].data_ptr(),
                                   cx[3].data_ptr(), pc.x_coef.data_ptr()), "pegncde_pack_x")
        pc._x_keepalive = cx   # sources stay alive until the pack kernel has run (stream-ordered)


def pack_control(
    ts: torch.Tensor,
    coeffs_adj: Sequence[torch.Tensor],
    x_coeffs: Optional[Sequence[torch.Tensor]] = None,
    device=None,
) -> PackedControl:
    """Reference-layout coefficients -> :class:`PackedControl` (runs ``pegncde_pack_adj`` / ``pegncde_pack_x``).

    ``coeffs_adj``: ``(d,c,b,a)`` each ``[T-1,n,n,2]`` or ``[B,T-1,n,n,2]`` (or the 4 stacked on axis 0);
    ``x_coeffs``: ``(d,c,b,a)`` each ``[T-1,n,e,2]`` or ``[B,T-1,n,e,2]``; ``ts``: ``[T]`` or ``[B,T]``."""
    if isinstance(coeffs_adj, torch.Tensor):
        coeffs_adj = tuple(coeffs_adj[i] for i in range(4))
    if isinstance(x_coeffs, torch.Tensor):
        x_coeffs = tuple(x_coeffs[i] for i in range(4))
    device = torch.device(device if device is not None else coeffs_adj[0].device)
    if device.type != "cuda":
        raise RuntimeError("pack_control needs a CUDA device: the fused path has no CPU fallback")
    if all(c.device.type == "cpu" for c in coeffs_adj):
        return _pack_control_streamed(ts, coeffs_adj, x_coeffs, device)
    cad = [_as_batched(c, 4).to(device=device, dtype=torch.float32).contiguous() for c in coeffs_adj]
    B, Tm1, n = cad[0].shape[0], cad[0].shape[1], cad[0].shape[2]
    pc = PackedControl(B, n, Tm1 + 1, 0, device)
    tsb = _as_batched(ts, 1).to(device=device, dtype=torch.float32)
    pc.ts.copy_(tsb.expand(B, Tm1 + 1))
    check(
        lib().pegncde_pack_adj(_stream_ptr(device), pc.dims(h=4, L=1), cad[0].data_ptr(), cad[1].data_ptr(), cad[2].data_ptr(),
                               cad[3].data_ptr(), pc.adj_coef.data_ptr(), pc.adj_rowsum.data_ptr(), pc.adj_diag.data_ptr(),
                               pc.adj_total.data_ptr(), pc.tch_coef.data_ptr()),
        "pegncde_pack_adj",
    )
    pc.plane_maxima()
    _attach_x(pc, x_coeffs, device)
    pc._keepalive = cad   # keep the sources alive until the pack kernels have run (stream-ordered)
    return pc


def _pack_control_streamed(ts, coeffs_adj, x_coeffs, device) -> PackedControl:
    """HOST coefficient arrays (what the reference's trainers hold: numpy / torch-CPU batches, trainer_pgt.py:201-207): the
    adjacency planes are NOT copied here.  The returned control is *pending*: a fixed-step solve copies and packs cubic piece
    i+1 (``pegncde_pack_adj_range``, side stream) while the steps inside piece i run; anything else calls
    :meth:`PackedControl.materialize` first.  The node-signal coefficients (small) are packed right away."""
    cad = []
    for c in coeffs_adj:
        c = _as_batched(c, 4).to(torch.float32).contiguous()
        cad.append(c if c.is_pinned() else c.pin_memory())
    B, Tm1, n = cad[0].shape[0], cad[0].shape[1], cad[0].shape[2]
    pc = PackedControl(B, n, Tm1 + 1, 0, device)
    tsb = _as_batched(ts, 1).to(torch.float32)
    pc.ts.copy_(tsb.expand(B, Tm1 + 1), non_blocking=True)
    _attach_x(pc, x_coeffs, device)
    pc.pending = cad
    grid = tsb.reshape(-1, Tm1 + 1)
    pc.host_ts = grid[0].cpu().numpy().copy() if bool((grid == grid[0]).all()) else None
    pc._keepalive = cad
    return pc


def build_control(ts: torch.Tensor, snapshots: torch.Tensor, x_t: Optional[torch.Tensor] = None, device=None) -> PackedControl:
    """Graph snapshots -> :class:`PackedControl` in one device pass (``pegncde_build_adj``): the fused replacement of
    ``get_graph_interpolation_coeffs`` (src/configs/dataset_configs.py:147-173, 1073-1100), which stacks a time channel
    onto ``A_k``, calls ``diffrax.backward_hermite_coefficients`` on the host and ships four ``[T-1,n,n,2]`` arrays.

    ``snapshots``: ``[T,n,n]`` or ``[B,T,n,n]``; ``ts``: ``[T]`` or ``[B,T]``; ``x_t`` (optional node signals
    ``[T,n,e]`` / ``[B,T,n,e]``): their coefficients are small and are built with :func:`backward_hermite_coefficients`."""
    device = torch.device(device if device is not None else snapshots.device)
    if device.type != "cuda":
        raise RuntimeError("build_control needs a CUDA device: the fused path has no CPU fallback")
    A = _as_batched(snapshots, 3).to(device=device, dtype=torch.float32).contiguous()
    B, T, n = A.shape[0], A.shape[1], A.shape[2]
    e = 0
    cx = None
    if x_t is not None:
        xb = _as_batched(x_t, 3).to(device=device, dtype=torch.float32)
        e = xb.shape[-1]
        tsx = _as_batched(ts, 1).to(device=device, dtype=torch.float32).expand(B, T)
        per = []
        for b in range(B):
            X = torch.stack([tsx[b][:, None, None].expand(T, n, e), xb[b]], dim=-1)
            per.append(backward_hermite_coefficients(tsx[b], X))
        cx = [torch.stack([per[b][i] for b in range(B)]).contiguous() for i in range(4)]
    pc = PackedControl(B, n, T, 0, device)
    pc.ts.copy_(_as_batched(ts, 1).to(device=device, dtype=torch.float32).expand(B, T))
    check(lib().pegncde_build_adj(_stream_ptr(device), pc.dims(h=4, L=1), pc.ts.data_ptr(), A.data_ptr(), pc.adj_coef.data_ptr(),
                                  pc.adj_rowsum.data_ptr(), pc.adj_diag.data_ptr(), pc.adj_total.data_ptr(), pc.tch_coef.data_ptr()),
          "pegncde_build_adj")
    pc.plane_maxima()
    _attach_x(pc, cx, device)
    pc._keepalive = A
    return pc


# ------------------------------------------------------------------------------------------------------------------------
# sparse (CSR) controls: PegSparse in pegncde.h
# ------------------------------------------------------------------------------------------------------------------------
class SparsePattern:
    """Coalesced CSR pattern of a batch of B graphs (:func:`sparse_pattern`).  Every index array is absolute: graph b's rows point
    into one shared entry axis of ``nnz`` entries.

    ``row_ptr``/``row_ptr_t`` ``[B, n+1]``, ``col``/``col_t`` ``[nnz]`` (int32): the pattern and its transpose, columns ascending
    inside a row.  ``perm_t`` ``[nnz]`` (int32): entry e sits at position ``perm_t[e]`` of the transposed pattern.  ``edge_map[b]``
    ``[E_b]`` (int64): the entry every input edge of graph b was coalesced into."""

    def __init__(self, n, row_ptr, col, row_ptr_t, col_t, perm_t, edge_map):
        self.n, self.B, self.nnz = n, row_ptr.shape[0], int(col.numel())
        self.row_ptr, self.col, self.row_ptr_t, self.col_t, self.perm_t, self.edge_map = row_ptr, col, row_ptr_t, col_t, perm_t, edge_map


def _edge_list(edge_index) -> list:
    if isinstance(edge_index, torch.Tensor):
        return [edge_index]
    if isinstance(edge_index, (list, tuple)) and len(edge_index) > 0 and all(isinstance(e, torch.Tensor) for e in edge_index):
        return list(edge_index)
    raise ValueError("edge_index must be a [2, E] integer tensor or a non-empty list of them (one per graph)")


def sparse_pattern(edge_index, num_nodes: int) -> SparsePattern:
    """Edge list(s) -> the coalesced CSR pattern and its transpose (torch ops on the device of ``edge_index``).

    ``edge_index``: ``[2, E]`` (rows, columns) or a list of B of them with any E per graph.  Duplicate edges become one entry (their
    values are summed, as ``index_put_(accumulate=True)`` into a dense matrix would).  Malformed input raises ``ValueError``."""
    n = int(num_nodes)
    if n < 1:
        raise ValueError(f"num_nodes must be >= 1, got {num_nodes}")
    graphs = _edge_list(edge_index)
    rp, cols, rpt, colts, perms, maps = [], [], [], [], [], []
    base = 0
    for g, ei in enumerate(graphs):
        if ei.dim() != 2 or ei.shape[0] != 2:
            raise ValueError(f"edge_index of graph {g} must have shape [2, E], got {tuple(ei.shape)}")
        if ei.dtype.is_floating_point or ei.dtype.is_complex or ei.dtype == torch.bool:
            raise ValueError(f"edge_index of graph {g} must hold integers, got {ei.dtype}")
        ei = ei.to(torch.int64)
        if ei.numel() > 0 and (int(ei.min()) < 0 or int(ei.max()) >= n):
            raise ValueError(f"edge_index of graph {g} has a node index outside [0, {n})")
        key = ei[0] * n + ei[1]
        uniq, inv = torch.unique(key, sorted=True, return_inverse=True)
        rows, cs = uniq // n, uniq % n
        m = int(uniq.numel())
        if base + m > 2**31 - 1:
            raise ValueError("the batch has more than 2^31 - 1 entries")
        dev = ei.device
        counts = torch.bincount(rows, minlength=n)
        rp.append(torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), counts.cumsum(0)]) + base)
        cols.append(cs)
        order = torch.argsort(cs * n + rows)                     # transposed order: by column, then row
        pos = torch.empty_like(order)
        pos[order] = torch.arange(m, device=dev)
        counts_t = torch.bincount(cs, minlength=n)
        rpt.append(torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), counts_t.cumsum(0)]) + base)
        colts.append(rows[order])
        perms.append(pos + base)
        maps.append(inv.reshape(-1) + base)
        base += m
    i32 = lambda xs: torch.cat(xs).to(torch.int32).contiguous()
    return SparsePattern(n, torch.stack(rp).to(torch.int32).contiguous(), i32(cols), torch.stack(rpt).to(torch.int32).contiguous(),
                         i32(colts), i32(perms), maps)


class SparseControl(PackedControl):
    """A control path on a sparse (CSR) adjacency pattern: ``PegControl.sparse`` is set and ``adj_coef`` is NULL.  Used wherever a
    :class:`PackedControl` is (vector fields, ``diffeqsolve``, ``tsit5_step``, the models); built by :func:`build_sparse_control` or
    :func:`pack_sparse_control`.  ``coef``/``coef_t`` are ``[T-1, nnz, 4]`` (a,b,c,d per entry) in pattern and transposed order.

    When the builder's edge weights or coefficients require grad, ``adj_packed`` is ``coef`` on the autograd tape: the solves and
    vector fields then return the cotangent of the coefficients (``pegncde_solve_bwd_adj``) and it flows back to the caller's tensors."""

    def __init__(self, pattern: SparsePattern, T: int, device):
        B, n = pattern.B, pattern.n
        self.B, self.n, self.T, self.e, self.ldn = B, n, T, 0, _pad32(n)
        self.pattern = pattern
        f = dict(dtype=torch.float32, device=device)
        self.ts = torch.empty((B, T), **f)
        self.adj_coef = None
        self.adj_absmax = None
        self.adj_rowsum = torch.empty((B, T - 1, 4, n), **f)
        self.adj_diag = torch.empty((B, T - 1, 4, n), **f)
        self.adj_total = torch.empty((B, T - 1, 4), **f)
        self.tch_coef = torch.empty((B, T - 1, 3, n), **f)
        nnz = max(pattern.nnz, 1)
        self.coef = torch.empty((T - 1, nnz, 4), **f)
        self.coef_t = torch.empty((T - 1, nnz, 4), **f)
        self.row_ptr, self.row_ptr_t = pattern.row_ptr, pattern.row_ptr_t
        self.col, self.col_t = pattern.col, pattern.col_t
        self.x_coef, self.x_packed = None, None
        self.adj_packed = None
        self._adj = {"colsum": torch.empty((B, T - 1, 4, n), **f), "pending": None, "host_ts": None}

    @property
    def nnz(self) -> int:
        return self.pattern.nnz

    def sparse_struct(self):
        from ._lib import PegSparse
        return PegSparse(self.pattern.nnz, self.coef.shape[1], self.row_ptr.data_ptr(), self.col.data_ptr(), self.coef.data_ptr(),
                         self.row_ptr_t.data_ptr(), self.col_t.data_ptr(), self.coef_t.data_ptr())

    def struct(self) -> PegControl:
        import ctypes
        self._sp = self.sparse_struct()      # the PegControl below points at it: kept alive with the control
        return PegControl(self.ts.data_ptr(), None, self.adj_rowsum.data_ptr(), self.adj_diag.data_ptr(), self.adj_total.data_ptr(),
                          self.tch_coef.data_ptr(), self.x_coef.data_ptr() if self.x_coef is not None else None,
                          self.adj_colsum.data_ptr(), None, None, ctypes.pointer(self._sp))

    def _view(self) -> "SparseControl":
        v = SparseControl.__new__(SparseControl)
        v.B, v.n, v.T, v.e, v.ldn = self.B, self.n, self.T, self.e, self.ldn
        for name in ("pattern", "ts", "adj_coef", "adj_absmax", "adj_rowsum", "adj_diag", "adj_total", "tch_coef", "coef", "coef_t",
                     "row_ptr", "row_ptr_t", "col", "col_t", "x_coef", "x_packed", "adj_packed"):
            setattr(v, name, getattr(self, name))
        v._adj = self._adj
        v._keepalive = self
        return v

    def with_x(self, x_coeffs) -> "SparseControl":
        """The same pattern and coefficients (shared, no copy) paired with the node-signal coefficients ``x_coeffs``."""
        v = self._view()
        _attach_x(v, x_coeffs, self.device)
        return v

    def select(self, b: int) -> "SparseControl":
        """View of graph ``b`` as a batch of one (no copy: the row offsets are absolute into the shared entry axis, so ``coef`` and
        ``adj_packed`` stay the whole batch's)."""
        v = self._view()
        v.B = 1
        for name in ("ts", "adj_rowsum", "adj_diag", "adj_total", "tch_coef", "row_ptr", "row_ptr_t"):
            setattr(v, name, getattr(self, name)[b:b + 1])
        v.x_coef = self.x_coef[b:b + 1] if self.x_coef is not None else None
        v.x_packed = None
        v._adj = {"colsum": self.adj_colsum[b:b + 1], "pending": None, "host_ts": None}
        return v

    def materialize(self) -> "SparseControl":
        return self

    def ensure_colsums(self) -> "SparseControl":
        return self            # the sparse builders always write the column sums

    def pack_pieces(self, *args, **kwargs):
        raise TypeError("sparse controls are built in one go; they have no streamed pieces")

    def plane_maxima(self, *args, **kwargs):
        raise TypeError("sparse controls have no tiled planes (adj_absmax is unused)")

    def dense_planes(self) -> torch.Tensor:
        """The path densified to [B, T-1, 4(a,b,c,d), n, n] (inspection / tests: O(n^2) memory)."""
        out = torch.zeros((self.B, self.T - 1, 4, self.n, self.n), dtype=torch.float32, device=self.device)
        rp = self.row_ptr.to(torch.int64)
        for b in range(self.B):
            e0, e1 = int(rp[b, 0]), int(rp[b, -1])
            rows = torch.repeat_interleave(torch.arange(self.n, device=self.device), rp[b, 1:] - rp[b, :-1])
            cols = self.col[e0:e1].to(torch.int64)
            out[b][:, :, rows, cols] = self.coef[:, e0:e1].permute(0, 2, 1)
        return out


def _sparse_dims(pat: SparsePattern, T: int, e: int = 0) -> PegDims:
    return PegDims(pat.B, pat.n, _pad32(pat.n), 4, e, 1, T, 0)


def _per_graph(x, B: int, what: str) -> list:
    xs = list(x) if isinstance(x, (list, tuple)) else [x]
    if len(xs) != B:
        raise ValueError(f"{what}: expected {B} graphs, got {len(xs)}")
    return xs


def _node_signal_coeffs(ts_b: torch.Tensor, x_t: torch.Tensor, B: int, T: int, n: int, device):
    xb = _as_batched(x_t, 3).to(device=device, dtype=torch.float32)
    if tuple(xb.shape[:3]) != (B, T, n):
        raise ValueError(f"x_t must be [T={T}, n={n}, e] or [B={B}, T, n, e], got {tuple(x_t.shape)}")
    e = xb.shape[-1]
    per = []
    for b in range(B):
        X = torch.stack([ts_b[b][:, None, None].expand(T, n, e), xb[b]], dim=-1)
        per.append(backward_hermite_coefficients(ts_b[b], X))
    return [torch.stack([per[b][i] for b in range(B)]).contiguous() for i in range(4)]


def _new_sparse_control(ts, pattern: SparsePattern, T: int, device) -> SparseControl:
    if T < 2:
        raise ValueError("a control path needs at least two knots")
    sc = SparseControl(pattern, T, device)
    tsb = _as_batched(torch.as_tensor(ts), 1).to(device=device, dtype=torch.float32)
    if tsb.shape[-1] != T or tsb.shape[0] not in (1, pattern.B):
        raise ValueError(f"ts must be [T={T}] or [B={pattern.B}, T], got {tuple(tsb.shape)}")
    sc.ts.copy_(tsb.expand(pattern.B, T))
    return sc


class _HermiteOnPattern(torch.autograd.Function):
    """``values`` [T, nnz] (knot values of every entry) -> the coefficients ``[T-1, nnz, 4]`` (a,b,c,d) the CUDA builder wrote
    (``coef``, returned as is, so they stay bit-identical to the dense builder's).  Backward: the transpose of
    :func:`backward_hermite_coefficients` per graph (it is linear in the values), with that graph's knot times."""

    @staticmethod
    def forward(ctx, values, sc):
        ctx.ts = sc.ts
        ctx.bounds = sc.row_ptr[:, [0, -1]].cpu().tolist()    # each graph's entry range (on the host: no sync in backward)
        return sc.coef.detach()

    @staticmethod
    def backward(ctx, g):
        g = g.to(torch.float32)
        out = torch.zeros((ctx.ts.shape[1], g.shape[1]), dtype=torch.float32, device=g.device)
        for b, (e0, e1) in enumerate(ctx.bounds):
            if e1 == e0:
                continue
            with torch.enable_grad():
                v = torch.zeros((ctx.ts.shape[1], e1 - e0), dtype=torch.float32, device=g.device, requires_grad=True)
                d, c, bb, a = backward_hermite_coefficients(ctx.ts[b], v)
                out[:, e0:e1] = torch.autograd.grad((a, bb, c, d), v, tuple(g[:, e0:e1, q] for q in range(4)))[0]
        return out, None


def build_sparse_control(ts: torch.Tensor, edge_index, edge_weight, num_nodes: int, x_t: Optional[torch.Tensor] = None,
                         device=None) -> SparseControl:
    """Edge list(s) + per-knot edge weights -> :class:`SparseControl` (``pegncde_build_adj_sparse``: the sparse form of
    :func:`build_control`, with the same Hermite arithmetic, so the coefficients equal the dense builder's bit for bit).

    ``edge_index``: ``[2, E]`` or a list of B; ``edge_weight``: ``[T, E]`` (or a list of B, matching), the value of every edge at
    every knot (0 where it is absent); ``ts``: ``[T]`` or ``[B, T]``; ``x_t``: optional node signals ``[T, n, e]`` / ``[B, T, n, e]``.

    Edge weights that require grad receive their gradient through every solve and vector field run on this control (duplicate edges
    each get the gradient of the entry they were summed into); ``edge_index`` and ``ts`` get none."""
    graphs = _edge_list(edge_index)
    device = torch.device(device if device is not None else graphs[0].device)
    if device.type != "cuda":
        raise RuntimeError("build_sparse_control needs a CUDA device: the fused path has no CPU fallback")
    pat = sparse_pattern([g.to(device) for g in graphs], num_nodes)
    ws = [w.to(device=device, dtype=torch.float32) for w in _per_graph(edge_weight, pat.B, "edge_weight")]
    T = ws[0].shape[0]
    for b, (w, g) in enumerate(zip(ws, graphs)):
        if w.dim() != 2 or w.shape != (T, g.shape[1]):
            raise ValueError(f"edge_weight of graph {b} must be [T={T}, E={g.shape[1]}], got {tuple(w.shape)}")
    values = torch.zeros((T, max(pat.nnz, 1)), dtype=torch.float32, device=device)
    for w, m in zip(ws, pat.edge_map):
        values.index_add_(1, m, w)
    sc = _new_sparse_control(ts, pat, T, device)
    sp = sc.sparse_struct()
    check(lib().pegncde_build_adj_sparse(_stream_ptr(device), _sparse_dims(pat, T), sp, pat.perm_t.data_ptr(), sc.ts.data_ptr(),
                                         values.data_ptr(), sc.adj_rowsum.data_ptr(), sc.adj_diag.data_ptr(), sc.adj_total.data_ptr(),
                                         sc.adj_colsum.data_ptr(), sc.tch_coef.data_ptr()), "pegncde_build_adj_sparse")
    if values.requires_grad:
        sc.adj_packed = _HermiteOnPattern.apply(values, sc)
    if x_t is not None:
        _attach_x(sc, _node_signal_coeffs(sc.ts, x_t, pat.B, T, pat.n, device), device)
    sc._keepalive = values      # the source lives until the builder has run (stream-ordered)
    return sc


def pack_sparse_control(ts: torch.Tensor, edge_index, coeffs_adj, x_coeffs=None, num_nodes: Optional[int] = None,
                        device=None) -> SparseControl:
    """Coefficients on an edge list -> :class:`SparseControl` (``pegncde_pack_adj_sparse``): the sparse form of
    :func:`pack_control`'s ``coeffs_adj``.

    ``coeffs_adj``: ``(d, c, b, a)`` each ``[T-1, E]`` -- the adjacency channel only (the time channel is t itself) -- or a list of B
    such tuples, one per pattern of ``edge_index``.  Linear interpolation is ``c = d = 0``.  ``x_coeffs`` as in :func:`pack_control`.
    ``num_nodes`` defaults to the node count of ``x_coeffs`` (required without it).  Coefficients that require grad receive their
    gradient as in :func:`build_sparse_control`."""
    graphs = _edge_list(edge_index)
    device = torch.device(device if device is not None else graphs[0].device)
    if device.type != "cuda":
        raise RuntimeError("pack_sparse_control needs a CUDA device: the fused path has no CPU fallback")
    if num_nodes is None:
        if x_coeffs is None:
            raise ValueError("num_nodes is required without x_coeffs")
        num_nodes = int((x_coeffs[0] if not isinstance(x_coeffs, torch.Tensor) else x_coeffs[0]).shape[-3])
    pat = sparse_pattern([g.to(device) for g in graphs], num_nodes)
    one_graph = isinstance(coeffs_adj, torch.Tensor) or (len(coeffs_adj) == 4 and all(isinstance(c, torch.Tensor) for c in coeffs_adj))
    per = _per_graph([coeffs_adj] if one_graph else list(coeffs_adj), pat.B, "coeffs_adj")
    Tm1 = None
    for b, (co, g) in enumerate(zip(per, graphs)):
        if len(co) != 4:
            raise ValueError("coeffs_adj must be (d, c, b, a)")
        co = [c.to(device=device, dtype=torch.float32) for c in co]
        Tm1 = co[0].shape[0] if Tm1 is None else Tm1
        for c in co:
            if c.dim() != 2 or c.shape != (Tm1, g.shape[1]):
                raise ValueError(f"coefficients of graph {b} must be [T-1={Tm1}, E={g.shape[1]}], got {tuple(c.shape)}")
        per[b] = co
    cf = [torch.zeros((Tm1, max(pat.nnz, 1)), dtype=torch.float32, device=device) for _ in range(4)]
    for co, m in zip(per, pat.edge_map):
        for q in range(4):
            cf[q].index_add_(1, m, co[q])
    sc = _new_sparse_control(ts, pat, Tm1 + 1, device)
    sp = sc.sparse_struct()
    check(lib().pegncde_pack_adj_sparse(_stream_ptr(device), _sparse_dims(pat, Tm1 + 1), sp, pat.perm_t.data_ptr(), cf[0].data_ptr(),
                                        cf[1].data_ptr(), cf[2].data_ptr(), cf[3].data_ptr(), sc.adj_rowsum.data_ptr(),
                                        sc.adj_diag.data_ptr(), sc.adj_total.data_ptr(), sc.adj_colsum.data_ptr(),
                                        sc.tch_coef.data_ptr()), "pegncde_pack_adj_sparse")
    if any(c.requires_grad for c in cf):
        sc.adj_packed = torch.stack([cf[3], cf[2], cf[1], cf[0]], dim=-1)     # [T-1, nnz, 4] (a,b,c,d): coef, on the tape
    if x_coeffs is not None:
        _attach_x(sc, x_coeffs, device)
    sc._keepalive = cf
    return sc


# ------------------------------------------------------------------------------------------------------------------------
# static controls: PegControl.adj_static in pegncde.h
# ------------------------------------------------------------------------------------------------------------------------
class StaticControl(PackedControl):
    """A control whose graph does not change in time: A(t) = A on every piece, paired (optionally) with a time-varying node-signal
    path on the knots ``ts``.  ``adj_static`` holds ONE tiled fp32 plane per graph (``[B, ldn*ldn]``) instead of four per piece, so it
    costs ``4 ldn^2`` bytes per graph and every contraction reads a quarter of the bytes of the dense control of ``[A] * T`` -- whose
    results it reproduces bit for bit.  The O(n) tables keep the dense shapes (A's statistics in slot ``a``, zeros in b, c, d).

    Built by :func:`build_static_control`; used wherever a :class:`PackedControl` is.  Not differentiable in A."""

    def __init__(self, B: int, n: int, T: int, device):
        self.B, self.n, self.T, self.e, self.ldn = B, n, T, 0, _pad32(n)
        f = dict(dtype=torch.float32, device=device)
        self.ts = torch.empty((B, T), **f)
        self.adj_coef = None
        self.adj_static = torch.empty((B, self.ldn * self.ldn), **f)
        self.adj_rowsum = torch.empty((B, T - 1, 4, n), **f)
        self.adj_diag = torch.empty((B, T - 1, 4, n), **f)
        self.adj_total = torch.empty((B, T - 1, 4), **f)
        self.adj_absmax = torch.empty((B, T - 1, 4), **f)
        self.tch_coef = torch.empty((B, T - 1, 3, n), **f)
        self.x_coef, self.x_packed = None, None
        self._adj = {"colsum": torch.empty((B, T - 1, 4, n), **f), "pending": None, "host_ts": None}

    def struct(self) -> PegControl:
        return PegControl(self.ts.data_ptr(), None, self.adj_rowsum.data_ptr(), self.adj_diag.data_ptr(), self.adj_total.data_ptr(),
                          self.tch_coef.data_ptr(), self.x_coef.data_ptr() if self.x_coef is not None else None,
                          self.adj_colsum.data_ptr(), self.adj_absmax.data_ptr(), None, None, self.adj_static.data_ptr())

    def _view(self) -> "StaticControl":
        v = StaticControl.__new__(StaticControl)
        v.B, v.n, v.T, v.e, v.ldn = self.B, self.n, self.T, self.e, self.ldn
        for name in ("ts", "adj_coef", "adj_static", "adj_rowsum", "adj_diag", "adj_total", "adj_absmax", "tch_coef", "x_coef", "x_packed"):
            setattr(v, name, getattr(self, name))
        v._adj = self._adj
        v._keepalive = self
        return v

    def with_x(self, x_coeffs) -> "StaticControl":
        """The same plane and tables (shared, no copy) paired with the node-signal coefficients ``x_coeffs``."""
        v = self._view()
        _attach_x(v, x_coeffs, self.device)
        return v

    def select(self, b: int) -> "StaticControl":
        """View of graph ``b`` as a batch of one (no copy)."""
        v = self._view()
        v.B = 1
        for name in ("ts", "adj_static", "adj_rowsum", "adj_diag", "adj_total", "adj_absmax", "tch_coef"):
            setattr(v, name, getattr(self, name)[b:b + 1])
        v.x_coef = self.x_coef[b:b + 1] if self.x_coef is not None else None
        v.x_packed = None
        v._adj = {"colsum": self.adj_colsum[b:b + 1], "pending": None, "host_ts": None}
        return v

    def materialize(self) -> "StaticControl":
        return self

    def ensure_colsums(self) -> "StaticControl":
        return self            # the builder always writes the column sums

    def pack_pieces(self, *args, **kwargs):
        raise TypeError("static controls are built in one go; they have no streamed pieces")

    def plane_maxima(self, *args, **kwargs):
        raise TypeError("static controls get their plane maxima from build_static_control")

    def static_plane(self) -> torch.Tensor:
        """Un-tiles ``adj_static`` to the adjacency [B, n, n] (inspection / tests)."""
        off = tiled_offsets(self.ldn)[0]
        nt = self.ldn // 32
        tile = (torch.arange(self.ldn).view(-1, 1) // 32) * nt + torch.arange(self.ldn).view(1, -1) // 32
        off = off - tile * 4096                          # offset inside a 4-plane tile: [g][q][m][lane][e] with q = 0
        g = off // 2048
        off = tile * 1024 + g * 512 + (off - g * 2048)   # the single-plane tile: [g][m][lane][e]
        dense = self.adj_static[:, off.reshape(-1).to(self.adj_static.device)].reshape(self.B, self.ldn, self.ldn)
        return dense[:, : self.n, : self.n]

    def dense_planes(self) -> torch.Tensor:
        """The path as [B, T-1, 4(a,b,c,d), n, n]: A in plane a of every piece, zeros elsewhere (inspection / tests)."""
        out = torch.zeros((self.B, self.T - 1, 4, self.n, self.n), dtype=torch.float32, device=self.device)
        out[:, :, 0] = self.static_plane()[:, None]
        return out


def build_static_control(ts: torch.Tensor, adjacency: torch.Tensor, x_t: Optional[torch.Tensor] = None, device=None) -> StaticControl:
    """A graph that does not change in time -> :class:`StaticControl` (``pegncde_build_adj_static``).  The same results, bit for bit,
    as ``build_control(ts, adjacency.expand(T, n, n), x_t)`` at a quarter of the plane bytes per contraction and ``1 / (4 (T-1))`` of
    the control's memory.

    ``adjacency``: ``[n, n]`` or ``[B, n, n]`` (a host tensor is copied to the device once); ``ts``: ``[T]`` or ``[B, T]`` (T >= 2);
    ``x_t``: optional node signals ``[T, n, e]`` / ``[B, T, n, e]``.  The adjacency gets no gradient: one that requires grad raises."""
    if not isinstance(adjacency, torch.Tensor):
        raise TypeError("adjacency must be a torch tensor")
    if adjacency.requires_grad:
        raise ValueError("build_static_control: static controls are not differentiable in the adjacency; pass adjacency.detach()")
    if adjacency.dim() not in (2, 3) or adjacency.shape[-1] != adjacency.shape[-2] or adjacency.shape[-1] < 1:
        raise ValueError(f"adjacency must be [n, n] or [B, n, n], got {tuple(adjacency.shape)}")
    if adjacency.dtype.is_complex:
        raise ValueError(f"adjacency must hold real numbers, got {adjacency.dtype}")
    device = torch.device(device if device is not None else adjacency.device)
    if device.type != "cuda":
        raise RuntimeError("build_static_control needs a CUDA device: the fused path has no CPU fallback")
    A = _as_batched(adjacency, 2).to(device=device, dtype=torch.float32, non_blocking=True).contiguous()
    B, n = A.shape[0], A.shape[1]
    tsb = _as_batched(torch.as_tensor(ts), 1).to(device=device, dtype=torch.float32)
    T = tsb.shape[-1]
    if T < 2:
        raise ValueError("a control path needs at least two knots")
    if tsb.dim() != 2 or tsb.shape[0] not in (1, B):
        raise ValueError(f"ts must be [T] or [B={B}, T], got {tuple(ts.shape)}")
    sc = StaticControl(B, n, T, device)
    sc.ts.copy_(tsb.expand(B, T))
    check(lib().pegncde_build_adj_static(_stream_ptr(device), sc.dims(h=4, L=1), A.data_ptr(), sc.adj_static.data_ptr(),
                                         sc.adj_rowsum.data_ptr(), sc.adj_diag.data_ptr(), sc.adj_total.data_ptr(), sc.adj_colsum.data_ptr(),
                                         sc.adj_absmax.data_ptr(), sc.tch_coef.data_ptr()), "pegncde_build_adj_static")
    if x_t is not None:
        _attach_x(sc, _node_signal_coeffs(sc.ts, x_t, B, T, n, device), device)
    sc._keepalive = A          # the source lives until the builder has run (stream-ordered)
    return sc
