"""JAX host layer over the XLA FFI shim (``pegncde_ffi.cc``) -- the drop-in a maintainer adds to the reference:

* ``FusedPermEquivGraphVectorField`` -- an Equinox module with EXACTLY the pytree of the reference's
  ``PermEquivGraphVectorField`` (src/models/vector_fields/perm_equiv_graph_vector_field.py:10-83: ``gnn_layers[i].param1..8``,
  ``.conv_layer.linear.{weight,bias}``, ``.conv_layer.norm.{weight,bias}``), so ``VectorFieldCfg.build`` can select it by name
  (``getattr(vector_fields, self.name)``, src/configs/vector_field_configs.py:52) and checkpoints / optimiser states carry over.
  Its ``__call__(t, y, args)`` is one custom call (``peg_vf_fwd``, VJP ``peg_vf_vjp``), so it also runs under stock diffrax.
* ``fused_diffeqsolve`` -- the call-site signature of ``diffrax.diffeqsolve`` as the model wrappers use it
  (src/models/pgt_graph_neural_cde.py:119-129): the whole fixed-step solve is ONE custom call (``peg_solve_fwd``) with the exact
  discrete adjoint as its ``jax.custom_vjp`` (``peg_solve_bwd``), so ``eqx.filter_value_and_grad`` (src/engine/trainer_pgt.py:346)
  works unchanged.
* batching: every handler is registered with ``vmap_method="broadcast_all"`` -- under ``jax.vmap(model)``
  (src/configs/loss_configs.py:44) the call runs ONCE with a leading batch axis on every operand, which the shim maps onto
  ``PegDims.B`` (the kernels are batched over graphs).

STATUS: NOT IMPORTABLE IN THIS REPOSITORY'S IMAGE (no jax / equinox / diffrax wheels, no network).  The torch/ctypes host in the
parent package is the layer that is tested on B200, against the same C-ABI.  tests/test_host.py imports this file on recording
stand-ins for jax / equinox / diffrax and checks every ``ffi_call`` against the bindings of ``pegncde_ffi.cc``.
"""
import ctypes
import os

import diffrax
import equinox as eqx
import jax
import jax.numpy as jnp
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_shim = ctypes.CDLL(os.path.join(_HERE, "libpegncde_ffi.so"))
_core = ctypes.CDLL(os.path.join(os.path.dirname(_HERE), "libpegncde.so"))
for _name, _sym in (("peg_pack_adj", "PegPackAdj"), ("peg_pack_x", "PegPackX"), ("peg_vf_fwd", "PegVfFwd"), ("peg_vf_vjp", "PegVfVjp"),
                    ("peg_step_fwd", "PegStepFwd"), ("peg_solve_fwd", "PegSolveFwd"), ("peg_solve_bwd", "PegSolveBwd")):
    jax.ffi.register_ffi_target(_name, jax.ffi.pycapsule(getattr(_shim, _sym)), platform="CUDA")

PEG_FLAG_TENSOR_CORES = 1
PEG_WS_VF_VJP, PEG_WS_SOLVE_FWD, PEG_WS_SOLVE_BWD, PEG_WS_STEP = 1, 2, 3, 4


class _Dims(ctypes.Structure):
    _fields_ = [(k, ctypes.c_int32) for k in ("B", "n", "ldn", "h", "e", "L", "T", "flags")]


_core.pegncde_workspace_bytes.restype = ctypes.c_size_t
_core.pegncde_workspace_bytes.argtypes = [ctypes.POINTER(_Dims), ctypes.c_int32, ctypes.c_int32]
_core.pegncde_stage_store_bytes.restype = ctypes.c_size_t
_core.pegncde_stage_store_bytes.argtypes = [ctypes.POINTER(_Dims), ctypes.c_int32]


def _cdims(d):
    return _Dims(d["B"], d["n"], (d["n"] + 31) // 32 * 32, d["h"], d["e"], d["L"], d["T"], d["flags"])


def _call(name, out_types, *args, **attrs):
    return jax.ffi.ffi_call(name, out_types, vmap_method="broadcast_all")(*args, **attrs)


def _attrs(dims):
    return {k: np.int32(v) for k, v in dims.items()}


def _f32(*shape):
    return jax.ShapeDtypeStruct(shape, jnp.float32)


# ------------------------------------------------------------------------------------------------------------------
# parameters: Equinox pytree <-> the flat buffer of pegncde.h
# ------------------------------------------------------------------------------------------------------------------
def pack_params(vector_field):
    """Equinox PermEquivGraphVectorField pytree -> the flat buffer of pegncde.h (layer after layer:
    weight | bias | norm.weight | norm.bias | param1..param8).  Plain jnp ops: jax.grad flows back into the leaves."""
    parts = []
    for layer in vector_field.gnn_layers:
        cl = layer.conv_layer
        parts += [cl.linear.weight.reshape(-1), cl.linear.bias, cl.norm.weight, cl.norm.bias]
        parts += [getattr(layer, f"param{i}") for i in range(1, 9)]
    return jnp.concatenate(parts).astype(jnp.float32)


# ------------------------------------------------------------------------------------------------------------------
# control path
# ------------------------------------------------------------------------------------------------------------------
def pack_control(ts, coeffs_adj, x_coeffs, dims):
    """Once per batch: the reference-layout arrays the trainer passes to the model (``coeffs_adj`` = (d, c, b, a), each
    ``[B, T-1, n, n, 2]``; ``x_coeffs`` likewise ``[B, T-1, n, e, 2]`` or None) -> the control tuple
    (ts, adj_coef, adj_rowsum, adj_diag, adj_total, tch_coef, x_coef, adj_absmax) = the fields of ``PegControl`` in pegncde.h."""
    B, n, e, T = dims["B"], dims["n"], dims["e"], dims["T"]
    ldn = (n + 31) // 32 * 32
    outs = (_f32(B, T - 1, 4 * ldn * ldn), _f32(B, T - 1, 4, n), _f32(B, T - 1, 4, n), _f32(B, T - 1, 4), _f32(B, T - 1, 3, n), _f32(B, T - 1, 4))
    adj_coef, rowsum, diag, total, tch, absmax = _call("peg_pack_adj", outs, *[jnp.asarray(c, jnp.float32) for c in coeffs_adj], **_attrs(dims))
    if e > 0:
        (x_coef,) = _call("peg_pack_x", (_f32(B, T - 1, 3, n, 2 * e),), *[jnp.asarray(c, jnp.float32) for c in x_coeffs], **_attrs(dims))
    else:
        x_coef = jnp.zeros((1,), jnp.float32)      # placeholder operand: the shim passes NULL when e == 0
    ts_b = jnp.broadcast_to(jnp.asarray(ts, jnp.float32).reshape(-1, T)[:1] if jnp.ndim(ts) == 1 else jnp.asarray(ts, jnp.float32), (B, T))
    return (ts_b, adj_coef, rowsum, diag, total, tch, x_coef, absmax)


class PackedControl:
    """What ``diffrax.CubicInterpolation(ts, coeffs)`` is replaced by on the fused path: the control tuple + its dims.  Built by
    ``fused_control`` once per batch and handed to the vector field / ``fused_diffeqsolve`` as ``args``."""

    def __init__(self, control, dims):
        self.control, self.dims = tuple(control), dict(dims)


def fused_control(ts, coeffs_adj, x_coeffs, hidden_dim, num_layers, flags=PEG_FLAG_TENSOR_CORES):
    if hasattr(coeffs_adj, "row_ptr_t"):
        raise TypeError("the JAX handlers take dense coefficient arrays; sparse (CSR) controls run through the torch API only")
    d = jnp.ndim(coeffs_adj[0])
    cadj = [c if d == 5 else c[None] for c in coeffs_adj]
    cx = None if x_coeffs is None else [c if jnp.ndim(c) == 5 else c[None] for c in x_coeffs]
    B, Tm1, n = cadj[0].shape[0], cadj[0].shape[1], cadj[0].shape[2]
    dims = dict(B=B, n=n, h=hidden_dim, e=0 if cx is None else cx[0].shape[3], L=num_layers, T=Tm1 + 1, flags=flags)
    return PackedControl(pack_control(ts, cadj, cx, dims), dims)


# ------------------------------------------------------------------------------------------------------------------
# the ODETerm callable: one custom call per evaluation, VJP = one custom call
# ------------------------------------------------------------------------------------------------------------------
def make_fused_vf(dims):
    ws = int(_core.pegncde_workspace_bytes(ctypes.byref(_cdims(dims)), PEG_WS_VF_VJP, 0))
    B, n, h = dims["B"], dims["n"], dims["h"]

    def vf(t, params, control, y):
        @jax.custom_vjp
        def f(params, y):
            return _fwd(params, y)[0]

        def _fwd(params, y):
            dy, _ = _call("peg_vf_fwd", (_f32(B, n, h), jax.ShapeDtypeStruct((ws,), jnp.uint8)), params, *control, y, t=np.float32(t), **_attrs(dims))
            return dy, (params, y)

        def _bwd(res, g_dy):
            params, y = res
            g_y, g_params, _ = _call("peg_vf_vjp", (_f32(B, n, h), jax.ShapeDtypeStruct(params.shape, jnp.float32), jax.ShapeDtypeStruct((ws,), jnp.uint8)),
                                     params, *control, y, g_dy, t=np.float32(t), **_attrs(dims))
            return g_params, g_y

        f.defvjp(_fwd, _bwd)
        return f(params, y)

    return vf


class FusedPermEquivGraphVectorField(eqx.Module):
    """Same constructor, same leaves as the reference's PermEquivGraphVectorField (a checkpoint of one loads into the other);
    ``__call__(t, y, args)`` with ``args`` = a :class:`PackedControl` (or ``[PackedControl, ...]``) runs the fused kernels."""

    gnn_layers: list
    data_embed_dim: int = eqx.field(static=True)
    num_nodes: int = eqx.field(static=True)
    hidden_dim: int = eqx.field(static=True)

    def __init__(self, input_dim, hidden_dim, output_dim, num_layers, data_embed_dim, num_nodes, *, key, reference_cls=None, **kwargs):
        # the leaves are built by the reference's own module so that initialisation (layers.py:66-74) is the reference's
        if reference_cls is None:
            from src.models.vector_fields import PermEquivGraphVectorField as reference_cls
        ref = reference_cls(input_dim=input_dim, hidden_dim=hidden_dim, output_dim=output_dim, num_layers=num_layers,
                            data_embed_dim=data_embed_dim, num_nodes=num_nodes, key=key, **kwargs)
        self.gnn_layers = ref.gnn_layers
        self.data_embed_dim, self.num_nodes, self.hidden_dim = data_embed_dim, num_nodes, hidden_dim

    def __call__(self, t, y, args):
        pc = args[0] if isinstance(args, (list, tuple)) else args
        batched = jnp.ndim(y) == 3
        yb = y if batched else y[None]
        dy = make_fused_vf(pc.dims)(t, pack_params(self), pc.control, yb)
        return dy if batched else dy[0]


# ------------------------------------------------------------------------------------------------------------------
# the whole fixed-step solve
# ------------------------------------------------------------------------------------------------------------------
def constant_step_table(t0, t1, dt0):
    """fp32 step boundaries under diffrax's ConstantStepSize + _clip_to_end (tnext > t1 - 1e-6 -> t1)."""
    f = np.float32
    t0, t1, dt0 = f(t0), f(t1), f(dt0)
    out, tnext = [t0], f(t0 + dt0)
    while True:
        if tnext > f(t1 - f(1e-6)):
            tnext = t1
        out.append(tnext)
        if tnext >= t1:
            return np.asarray(out, dtype=np.float32)
        tnext = f(tnext + dt0)


def make_fused_solve(dims, step_ts, ws_bytes=None, store_elems=None):
    """dims = dict(B,n,h,e,L,T,flags); returns solve(params_flat, control_tuple, y0) -> y_ckpt [S+1,B,n,h] with a custom VJP."""
    S = len(step_ts) - 1
    B, n, h = dims["B"], dims["n"], dims["h"]
    cd = _cdims(dims)
    if ws_bytes is None:
        ws_bytes = int(max(_core.pegncde_workspace_bytes(ctypes.byref(cd), PEG_WS_SOLVE_FWD, S), _core.pegncde_workspace_bytes(ctypes.byref(cd), PEG_WS_SOLVE_BWD, S)))
    if store_elems is None:
        store_elems = int(_core.pegncde_stage_store_bytes(ctypes.byref(cd), S)) // 4
    attrs = dict(step_ts=np.asarray(step_ts, np.float32), **_attrs(dims))

    @jax.custom_vjp
    def solve(params, control, y0):
        return _fwd(params, control, y0)[0]

    def _fwd(params, control, y0):
        outs = (_f32(S + 1, B, n, h), _f32(store_elems), jax.ShapeDtypeStruct((ws_bytes,), jnp.uint8))
        y_ckpt, store, _ = _call("peg_solve_fwd", outs, params, *control, y0, **attrs)
        return y_ckpt, (params, control, y_ckpt, store)

    def _bwd(res, g_ckpt):
        params, control, y_ckpt, store = res
        outs = (_f32(B, n, h), jax.ShapeDtypeStruct(params.shape, jnp.float32), jax.ShapeDtypeStruct((ws_bytes,), jnp.uint8))
        g_y0, g_params, _ = _call("peg_solve_bwd", outs, params, *control, y_ckpt, store, g_ckpt, **attrs)
        return g_params, jax.tree_util.tree_map(jnp.zeros_like, control), g_y0

    solve.defvjp(_fwd, _bwd)
    return solve


class FusedSolution:
    def __init__(self, ts, ys, stats):
        self.ts, self.ys, self.stats = ts, ys, stats


def fused_diffeqsolve(terms, solver, t0, t1, dt0, y0, args=None, *, stepsize_controller=None, saveat=None, **unused):
    """``diffrax.diffeqsolve`` for the one combination the PGT / TGB models use (pgt_graph_neural_cde.py:119-129):
    ``ODETerm(FusedPermEquivGraphVectorField | CDEWrapperVectorField(...))``, ``Tsit5``, ``ConstantStepSize``, ``SaveAt(t1=True)``
    (or ``steps=True``).  ``args`` = ``[PackedControl]`` (``fused_control``).  Anything else is handed to diffrax unchanged --
    the vector field's own ``__call__`` is a custom call too, so the stock solver loop still runs on the fused kernels."""
    vf = getattr(terms.vector_field, "vector_field", terms.vector_field)      # unwrap CDEWrapperVectorField
    pc = args[0] if isinstance(args, (list, tuple)) else args
    fixed = isinstance(stepsize_controller, diffrax.ConstantStepSize) and isinstance(solver, diffrax.Tsit5) and isinstance(pc, PackedControl)
    if not (fixed and isinstance(vf, FusedPermEquivGraphVectorField) and getattr(saveat, "subs", saveat) is not None):
        return diffrax.diffeqsolve(terms, solver, t0, t1, dt0, y0, args=args, stepsize_controller=stepsize_controller, saveat=saveat, **unused)
    step_ts = constant_step_table(float(t0), float(t1), float(dt0))
    batched = jnp.ndim(y0) == 3
    y_ckpt = make_fused_solve(pc.dims, step_ts)(pack_params(vf), pc.control, y0 if batched else y0[None])
    if not batched:
        y_ckpt = y_ckpt[:, 0]
    steps = bool(getattr(saveat, "steps", False))
    ys = y_ckpt if steps else y_ckpt[-1:]
    return FusedSolution(jnp.asarray(step_ts if steps else step_ts[-1:]), ys, {"num_steps": len(step_ts) - 1})
