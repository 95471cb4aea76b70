"""Host-side mirror of the reference's vector-field modules for the fused sm_100a path.

Same class names, constructor arguments, leaf names and call protocol ``vf(t, y, args)`` as
``src/models/vector_fields/{layers,perm_equiv_graph_vector_field,cde_wrapper_vector_field}.py``,
so checkpoints / optimiser states keyed on leaf names line up.  ``torch.nn.Module`` stands in
for ``eqx.Module`` (JAX/Equinox are not installable in this image; the jax.ffi binding that
would sit here in a JAX environment is in ``jax_ffi/``).  All arithmetic runs in
``libpegncde.so``; there is no eager/CPU implementation behind these classes.
"""
from __future__ import annotations

import math

import torch
from torch import nn

from ._lib import PEG_FLAG_DIRECTED, PEG_FLAG_TENSOR_CORES, PEG_WS_VF_VJP, PegDims, check, lib
from .control import CubicInterpolation, PackedControl, StaticControl, _stream_ptr, pack_control

_WS_CACHE = {}


def workspace(device, nbytes: int) -> torch.Tensor:
    """Caller-owned scratch for the C-ABI (grown on demand, one per device and stream)."""
    key = (str(device), torch.cuda.current_stream(device).cuda_stream)
    buf = _WS_CACHE.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _WS_CACHE[key] = buf
    return buf


class RMSNorm(nn.Module):
    """Parameters of ``eqx.nn.RMSNorm(shape)`` (weight AND bias, eps 1e-5)."""

    def __init__(self, dim: int):
        super().__init__()
        self.weight = nn.Parameter(torch.ones(dim))
        self.bias = nn.Parameter(torch.zeros(dim))


class Linear(nn.Module):
    """Parameters of ``eqx.nn.Linear(in, out)``: weight [out, in], bias [out], U(+-1/sqrt(in))."""

    def __init__(self, input_dim: int, output_dim: int, generator=None):
        super().__init__()
        lim = 1.0 / math.sqrt(input_dim)
        self.weight = nn.Parameter((torch.rand((output_dim, input_dim), generator=generator) * 2 - 1) * lim)
        self.bias = nn.Parameter((torch.rand((output_dim,), generator=generator) * 2 - 1) * lim)


class ConvLayer(nn.Module):
    """src/models/vector_fields/layers.py:11-48 (parameters only; the arithmetic is fused)."""

    def __init__(self, input_dim: int, output_dim: int, generator=None):
        super().__init__()
        self.linear = Linear(input_dim, output_dim, generator)
        self.norm = RMSNorm(input_dim)


class ConvEquivFusionLayer(nn.Module):
    """src/models/vector_fields/layers.py:51-177: param1..param8 ~ U(-1,1)/15 plus a ConvLayer."""

    def __init__(self, input_dim: int, output_dim: int, generator=None):
        super().__init__()
        for i in range(1, 9):
            setattr(self, f"param{i}", nn.Parameter((torch.rand((2,), generator=generator) * 2 - 1) / 15.0))
        self.conv_layer = ConvLayer(input_dim, output_dim, generator)

    def fusion_params(self) -> torch.Tensor:
        return torch.cat([getattr(self, f"param{i}") for i in range(1, 9)])


class _FixedFusionConvLayer(ConvLayer):
    """A plain ``ConvLayer`` (layers.py:11-48) run through the equivariant kernel with CONSTANT fusion scalars:
    ``m + (c0 A + c1 A') m`` is the fused form with ``param1 = (c0 - 1, c1 - 1)`` and ``param2..8 = 0``.  Leaf names stay
    the reference's (``gnn_layers[i].linear`` / ``.norm``); the fusion vector is a buffer, so it gets no gradient."""

    def __init__(self, input_dim: int, output_dim: int, generator, c0: float, c1: float):
        super().__init__(input_dim, output_dim, generator)
        fus = torch.zeros(16)
        fus[0], fus[1] = c0 - 1.0, c1 - 1.0
        self.register_buffer("fusion_const", fus, persistent=False)   # not a checkpoint key: the reference has no such leaf

    @property
    def conv_layer(self):
        return self

    def fusion_params(self) -> torch.Tensor:
        return self.fusion_const


class ConvEquivFusionDirectedLayer(nn.Module):
    """src/models/vector_fields/layers.py:180-362: 11 parameter pairs ~ U(-1,1)/15 (row AND column sums of A, A') plus a
    ConvLayer.  Reference quirks kept: ``param6_prime`` is drawn with ``param5_prime``'s key (init only), term 4' mixes
    rowsum(A) with colsum(A'), term 7 uses sum(A) twice."""

    NAMES = ("param1", "param2", "param3", "param4", "param5", "param6", "param7", "param8", "param4_prime", "param5_prime", "param6_prime")

    def __init__(self, input_dim: int, output_dim: int, generator=None):
        super().__init__()
        for name in ("param1", "param2", "param3", "param4", "param4_prime", "param5", "param5_prime", "param6", "param6_prime", "param7", "param8"):
            setattr(self, name, nn.Parameter((torch.rand((2,), generator=generator) * 2 - 1) / 15.0))
        self.conv_layer = ConvLayer(input_dim, output_dim, generator)

    def fusion_params(self) -> torch.Tensor:
        """Kernel order (pegncde.h): param1..param8, then param4', param5', param6' and one pair of padding."""
        return torch.cat([getattr(self, name) for name in self.NAMES] + [torch.zeros(2, device=self.param1.device, dtype=self.param1.dtype)])


class PermEquivGraphVectorField(nn.Module):
    """src/models/vector_fields/perm_equiv_graph_vector_field.py:10-129 (enc_idx=False).

    ``vf(t, y, args)`` with ``args`` = the adjacency control (a :class:`CubicInterpolation`,
    or an already :class:`PackedControl`); ``y`` is ``[n, h]`` or batched ``[B, n, h]``."""

    def __init__(self, input_dim: int, hidden_dim: int, output_dim: int, num_layers: int, data_embed_dim: int,
                 num_nodes: int, enc_idx: bool = False, enc_type: str = "mlp", idx_dim: int = 512, *, key=None,
                 flags=None, **kwargs):
        super().__init__()
        if enc_idx:
            raise NotImplementedError("enc_idx=True is unreachable in the reference (fields commented out)")
        if input_dim != hidden_dim:
            # every reference config builds the field with input_dim == hidden_dim (vector_field_configs.py:62-75), and the
            # kernels' parameter packing (pegncde_param_count) assumes it
            raise NotImplementedError(f"the fused kernels need input_dim == hidden_dim (got {input_dim} and {hidden_dim})")
        gen = None
        if key is not None:
            gen = torch.Generator().manual_seed(int(key))
        layers = []
        for _ in range(num_layers - 1):
            layers.append(self._make_layer(input_dim, hidden_dim, gen))
            input_dim = hidden_dim
        layers.append(self._make_layer(input_dim, output_dim, gen))
        self.gnn_layers = nn.ModuleList(layers)
        self.data_embed_dim = data_embed_dim
        self.num_nodes = num_nodes
        self.enc_idx = enc_idx
        self.hidden_dim = hidden_dim
        self.output_dim = output_dim
        # tcgen05 contraction wherever the shape is a real dense contraction (n >= 128, widths multiples of 32): the library
        # falls back per layer to the CUDA-core kernels otherwise (tc_supported).  0 selects the CUDA-core path everywhere.
        self.flags = PEG_FLAG_TENSOR_CORES if flags is None else int(flags)
        # keep every stage's layer inputs in the forward solve so the adjoint needs no recompute (memory permitting)
        self.store_stages = True

    directed = False   # PEG_FLAG_DIRECTED: 22 fusion scalars per layer, column sums in the control

    def _make_layer(self, input_dim: int, output_dim: int, gen) -> nn.Module:
        return ConvEquivFusionLayer(input_dim, output_dim, gen)

    # ---- packing -------------------------------------------------------------------------
    @property
    def num_layers(self) -> int:
        return len(self.gnn_layers)

    def uses_control(self) -> bool:
        return self.output_dim != self.hidden_dim

    def flat_params(self) -> torch.Tensor:
        """The packed fp32 buffer of pegncde.h (differentiable torch.cat of the leaves)."""
        parts = []
        for layer in self.gnn_layers:
            cl = layer.conv_layer
            parts += [cl.linear.weight.reshape(-1), cl.linear.bias, cl.norm.weight, cl.norm.bias, layer.fusion_params()]
        return torch.cat(parts).to(torch.float32)

    def load_oracle_layers(self, layers) -> None:
        """Copies parameters given as (fusion[8,2], W, b, norm_w, norm_b) per layer (test helper)."""
        with torch.no_grad():
            for mine, lp in zip(self.gnn_layers, layers):
                fus, W, b, nw, nb = [torch.as_tensor(x, dtype=torch.float32) for x in lp]
                for i in range(8):
                    getattr(mine, f"param{i + 1}").copy_(fus[i])
                mine.conv_layer.linear.weight.copy_(W)
                mine.conv_layer.linear.bias.copy_(b)
                mine.conv_layer.norm.weight.copy_(nw)
                mine.conv_layer.norm.bias.copy_(nb)

    def dims_for(self, pc: PackedControl, with_wrapper: bool) -> PegDims:
        e = pc.e if with_wrapper else 0
        expect = 2 * self.hidden_dim * e if e > 0 else self.hidden_dim
        if expect != self.output_dim:
            raise ValueError(f"output_dim {self.output_dim} does not match hidden_dim*data_embed_dim*2 = {expect}")
        if pc.n != self.num_nodes:
            raise ValueError(f"control has {pc.n} nodes, vector field was built for {self.num_nodes}")
        flags = self.flags
        if self.directed:
            flags |= PEG_FLAG_DIRECTED
            pc.ensure_colsums()
        d = pc.dims(self.hidden_dim, self.num_layers, flags)
        d.e = e
        return d

    def checked_flat_params(self, dims: PegDims) -> torch.Tensor:
        """``flat_params()`` after checking its length against the library's packing for ``dims`` (a mismatch would make the
        kernels read weights at wrong offsets)."""
        flat = self.flat_params()
        want = lib().pegncde_param_count(dims)
        if flat.numel() != want:
            raise ValueError(f"packed parameter buffer has {flat.numel()} floats, pegncde_param_count says {want}")
        return flat

    # ---- the ODETerm callable ------------------------------------------------------------
    def forward(self, t, y: torch.Tensor, args) -> torch.Tensor:
        return fused_vector_field(self, t, y, args, None)


class PermEquivDirGraphVectorField(PermEquivGraphVectorField):
    """src/models/vector_fields/perm_equiv_dir_graph_vector_field.py:86-130 (enc_idx=False): the directed equivariant field --
    ``ConvEquivFusionDirectedLayer``s, ReLU between, time-gradient row scale; same kernels, different O(n) correction tables."""

    directed = True

    def _make_layer(self, input_dim: int, output_dim: int, gen) -> nn.Module:
        return ConvEquivFusionDirectedLayer(input_dim, output_dim, gen)


class GraphVectorField(PermEquivGraphVectorField):
    """src/models/vector_fields/graph_vector_field.py:80-115 (enc_idx=False): the plain GN-CDE field, message passing
    matrix ``A_s + A'_s`` -- the degenerate case of the same kernels (SURVEY N3)."""

    def _make_layer(self, input_dim: int, output_dim: int, gen) -> nn.Module:
        return _FixedFusionConvLayer(input_dim, output_dim, gen, 1.0, 1.0)


class GNODEVectorField(PermEquivGraphVectorField):
    """src/models/vector_fields/gnode_vector_field.py:57-81: message passing matrix ``A_s`` only."""

    def _make_layer(self, input_dim: int, output_dim: int, gen) -> nn.Module:
        return _FixedFusionConvLayer(input_dim, output_dim, gen, 1.0, 0.0)


class CDEWrapperVectorField(nn.Module):
    """src/models/vector_fields/cde_wrapper_vector_field.py:6-26."""

    def __init__(self, vector_field: nn.Module, hidden_dim: int):
        super().__init__()
        self.vector_field = vector_field
        self.hidden_dim = hidden_dim

    def forward(self, t, y: torch.Tensor, args) -> torch.Tensor:
        control_adj, control_data = args
        return fused_vector_field(self.vector_field, t, y, control_adj, control_data)


def resolve_control(control_adj, control_data, device) -> PackedControl:
    """Accepts the reference's ``args`` (CubicInterpolation objects) or a PackedControl.  The adjacency planes (the expensive
    pre-pass) are packed once and cached on the adjacency control object; the node-signal coefficients are taken from the
    ``control_data`` of THIS call every time (the TGB models rebuild them from their data encoder at every iteration, and a
    trainer may pair one adjacency window with different node signals)."""
    if isinstance(control_adj, PackedControl):
        base = control_adj
    elif isinstance(control_adj, CubicInterpolation):
        if control_adj._packed is None:
            control_adj._packed = pack_control(control_adj.ts, (control_adj.d, control_adj.c, control_adj.b, control_adj.a), None, device=device)
        base = control_adj._packed
    else:
        raise TypeError("args must be CubicInterpolation / PackedControl objects")
    if control_data is None:
        return base
    if isinstance(control_data, PackedControl):
        raise TypeError("control_data must be a CubicInterpolation (a PackedControl already carries its node-signal part)")
    return base.with_x((control_data.d, control_data.c, control_data.b, control_data.a))


def adj_grad_buffer(pc, needed: bool):
    """Zeroed cotangent of a sparse control's coefficients (``pegncde_*_adj``) or of a static control's adjacency, ``[B, ldn, ldn]``
    (``pegncde_*_adj_static``), or None when it is not asked for."""
    if not needed:
        return None
    if isinstance(pc, StaticControl):
        return torch.zeros((pc.B, pc.ldn, pc.ldn), dtype=torch.float32, device=pc.adj_static.device)
    return torch.zeros_like(pc.coef)


def adj_grad_out(pc, g):
    """The cotangent of ``pc.adj_packed`` from an :func:`adj_grad_buffer` buffer: a static control's ``[B, n, n]`` corner."""
    if g is None or not isinstance(pc, StaticControl):
        return g
    return g[:, :pc.n, :pc.n]


class _VFFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, y, flat, adj_packed, vf, pc, dims, t):
        y = y.contiguous()
        flat = flat.contiguous()
        l = lib()
        nbytes = l.pegncde_workspace_bytes(dims, PEG_WS_VF_VJP, 0)
        ws = workspace(y.device, nbytes)
        dy = torch.empty_like(y)
        ctl = pc.struct()
        check(l.pegncde_vf_fwd(_stream_ptr(y.device), dims, ctl, flat.data_ptr(), float(t), y.data_ptr(), dy.data_ptr(),
                               ws.data_ptr(), ws.numel()), "pegncde_vf_fwd")
        ctx.save_for_backward(y, flat)
        ctx.pc, ctx.dims, ctx.t = pc, dims, float(t)
        return dy

    @staticmethod
    def backward(ctx, g_dy):
        y, flat = ctx.saved_tensors
        l = lib()
        dims, pc = ctx.dims, ctx.pc
        nbytes = l.pegncde_workspace_bytes(dims, PEG_WS_VF_VJP, 0)
        ws = workspace(y.device, nbytes)
        g_y = torch.empty_like(y)
        g_flat = torch.zeros_like(flat)
        g_adj = adj_grad_buffer(pc, ctx.needs_input_grad[2])
        ctl = pc.struct()
        args = (_stream_ptr(y.device), dims, ctl, flat.data_ptr(), ctx.t, y.data_ptr(), g_dy.contiguous().data_ptr(), g_y.data_ptr(),
                g_flat.data_ptr(), None)
        if g_adj is None:
            check(l.pegncde_vf_vjp(*args, ws.data_ptr(), ws.numel()), "pegncde_vf_vjp")
        elif isinstance(pc, StaticControl):
            check(l.pegncde_vf_vjp_adj_static(*args, g_adj.data_ptr(), ws.data_ptr(), ws.numel()), "pegncde_vf_vjp_adj_static")
        else:
            check(l.pegncde_vf_vjp_adj(*args, g_adj.data_ptr(), ws.data_ptr(), ws.numel()), "pegncde_vf_vjp_adj")
        return g_y, g_flat, adj_grad_out(pc, g_adj), None, None, None, None


def fused_vector_field(vf: PermEquivGraphVectorField, t, y: torch.Tensor, control_adj, control_data) -> torch.Tensor:
    if y.device.type != "cuda":
        raise RuntimeError("the fused vector field runs on CUDA only (no CPU fallback)")
    pc = resolve_control(control_adj, control_data, y.device).materialize()
    dims = vf.dims_for(pc, with_wrapper=control_data is not None or (isinstance(control_adj, PackedControl) and vf.uses_control()))
    unb = y.dim() == 2
    yb = y.unsqueeze(0) if unb else y
    if yb.shape[0] != pc.B:
        raise ValueError(f"state batch {yb.shape[0]} != control batch {pc.B}")
    out = _VFFunction.apply(yb.to(torch.float32), vf.checked_flat_params(dims), pc.adj_packed, vf, pc, dims, t)
    return out.squeeze(0) if unb else out
