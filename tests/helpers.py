"""Glue between the oracle's Problem objects and the product's host API (tests only)."""
import torch

from oracle import reference_path as R

GOLDEN_CASES = {
    # name: make_problem kwargs.  Seeds are chosen well-conditioned (|fp32 oracle - fp64 oracle| << 1e-4).
    "tiny_nocontrol": dict(n=12, h=8, e=0, L=2, T=4, t1=3, dt0=0.1, seed=0),
    "tiny_control": dict(n=20, h=8, e=3, L=3, T=4, t1=3, dt0=0.1, seed=1),
    "ragged_n": dict(n=37, h=16, e=2, L=3, T=5, t1=2, dt0=0.1, seed=3),
    "sir_like": dict(n=100, h=32, e=3, L=3, T=12, t1=1, dt0=0.1, seed=4, float_ts=True),
    "england_like": dict(n=129, h=64, e=8, L=3, T=4, t1=3, dt0=0.1, seed=5),
}


FUSED = "fused"     # device_model(flags=FUSED): the product default, selected by name in parametrised tests


def per_operator(flags):
    """flags of a test that names a per-operator path: the small-graph cluster kernels are switched off"""
    from perm_equiv_graph_neural_cdes_b200 import _lib
    return int(flags) | _lib.PEG_FLAG_NO_FUSED_SMALL


def fused_flags():
    """the product default plus PEG_FLAG_FUSED_SMALL: the small-graph cluster kernels up to n = 256 (default: n < 128)"""
    from perm_equiv_graph_neural_cdes_b200 import _lib
    return _lib.PEG_FLAG_TENSOR_CORES | _lib.PEG_FLAG_FUSED_SMALL


def device_model(p, device, flags=None):
    """(vf, wrapped_vf_or_vf, control objects) of the product API for an oracle Problem."""
    import perm_equiv_graph_neural_cdes_b200 as P

    widths = R.layer_widths(p.h, p.L, p.e, p.e > 0)
    vf = P.PermEquivGraphVectorField(p.h, p.h, widths[-1], p.L, p.e, p.n, key=0)
    vf.load_oracle_layers([lp.tensors() for lp in p.layers])
    vf = vf.to(device)
    # None = the product default: the cluster-per-graph kernels for n < 128, tcgen05 wherever the shape allows it.
    # An explicit value names a per-operator path ("ffma" = 0, "tcgen05" = PEG_FLAG_TENSOR_CORES ...): the small-graph path is
    # switched off so that the test exercises the kernels it names at any n.  FUSED = the small-graph path up to n = 256.
    if isinstance(flags, str):
        assert flags == FUSED
        vf.flags = fused_flags()
    elif flags is not None:
        vf.flags = per_operator(flags)
    ts = p.ts.to(torch.float32)
    cadj = P.CubicInterpolation(ts.to(device), tuple(c.to(torch.float32).to(device) for c in p.coeffs_adj))
    cx = None
    if p.e > 0:
        cx = P.CubicInterpolation(ts.to(device), tuple(c.to(torch.float32).to(device) for c in p.x_coeffs))
    term_vf = P.CDEWrapperVectorField(vf, p.h) if p.e > 0 else vf
    args = [cadj, cx] if p.e > 0 else cadj
    return vf, term_vf, args


def product_grads_as_oracle(vf):
    """Gradients of the product module's leaves in the oracle's (fusion, W, b, nw, nb) per-layer order."""
    out = []
    for layer in vf.gnn_layers:
        fus = torch.stack([getattr(layer, f"param{i}").grad for i in range(1, 9)])
        cl = layer.conv_layer
        out.append([fus, cl.linear.weight.grad, cl.linear.bias.grad, cl.norm.weight.grad, cl.norm.bias.grad])
    return out


def rel_err(a, b):
    a = torch.as_tensor(a).detach().to(torch.float64).cpu()
    b = torch.as_tensor(b).detach().to(torch.float64).cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def union_pattern(planes):
    """planes [..., n, n] -> edge_index [2, E] of the union of nonzeros over the leading axes"""
    nz = (planes != 0).reshape(-1, planes.shape[-2], planes.shape[-1]).any(dim=0)
    return torch.nonzero(nz).t().contiguous()


def sparse_of_coeffs(ts, coeffs_adj, x_coeffs=None):
    """reference-layout coefficients (d,c,b,a) each [T-1, n, n, 2] -> SparseControl on the union of nonzeros of their adjacency channel"""
    import perm_equiv_graph_neural_cdes_b200 as P

    adj = torch.stack([c[..., 1] for c in coeffs_adj])             # [4, T-1, n, n]
    ei = union_pattern(adj)
    co = tuple(c[..., 1][:, ei[0], ei[1]].contiguous() for c in coeffs_adj)
    return P.pack_sparse_control(ts, ei, co, x_coeffs, num_nodes=adj.shape[-1])
