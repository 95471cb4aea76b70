"""Gradients with respect to a static control's adjacency (build_static_control(..., differentiable=True),
pegncde_vf_vjp_adj_static / pegncde_solve_bwd_adj_static).  Host: the C-ABI surface and argument checks.  GPU: against fp64 autograd
of the oracle on the constant path (a = A on every piece, b = c = d = 0, A a leaf), against the full-pattern sparse control's
edge-weight gradient, against a central difference at n = 16384, and the invariants (reproducible bit for bit, a batch equals its
graphs alone, the other outputs unchanged).  Each single-evaluation case names the gradient kernel it expects and checks it ran.
"""
import ctypes
import json
import os
import re

import pytest
import torch

import perm_equiv_graph_neural_cdes_b200 as P
from perm_equiv_graph_neural_cdes_b200 import _lib
from oracle import reference_path as R
from tests.helpers import per_operator, rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TC = _lib.PEG_FLAG_TENSOR_CORES
OFF_SMALL = _lib.PEG_FLAG_NO_FUSED_SMALL
FMTS = {"ffma": 0, "fp16x2": TC, "tf32x3": TC | _lib.PEG_FLAG_TF32X3, "bf16x2": TC | _lib.PEG_FLAG_BF16X2}
TOL_G = {"ffma": 3e-4, "fp16x2": 3e-4, "tf32x3": 3e-4, "bf16x2": 2e-3}   # bf16x2: the operand format's stated looser bound


def rel_l2(a, b):
    a = torch.as_tensor(a).detach().double().cpu()
    b = torch.as_tensor(b).detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


def grad_kernel(flags, n):
    """the rule of pegncde.cu (adj_grad_on_tc): tcgen05 with PEG_FLAG_TENSOR_CORES and n >= 128, the fp32 FFMA kernel otherwise"""
    return "k_tc_adj_grad" if (flags & TC) and n >= 128 else "k_adj_grad"


# ---------------------------------------------------------------------------------------------------
# host side
# ---------------------------------------------------------------------------------------------------
def test_static_adj_entries_match_the_header():
    hdr = open(os.path.join(ROOT, "include", "pegncde.h")).read()
    for name, base in (("pegncde_vf_vjp_adj_static", "pegncde_vf_vjp_adj"), ("pegncde_solve_bwd_adj_static", "pegncde_solve_bwd_adj")):
        decl = re.search(rf"\b{name}\s*\(([^;]*)\);", hdr).group(1)
        params = [p.strip() for p in decl.split(",")]
        bdecl = re.search(rf"\b{base}\s*\(([^;]*)\);", hdr).group(1)
        bparams = [p.strip() for p in bdecl.split(",")]
        assert len(params) == len(_lib.SIGNATURES[name][1]) == len(bparams), name
        # the sparse entry with g_adj_static in place of g_adj_coef
        assert params[-3] == "float* g_adj_static" and bparams[-3] == "float* g_adj_coef", name
        assert params[:-3] + params[-2:] == bparams[:-3] + bparams[-2:], name
        assert _lib.SIGNATURES[name] == _lib.SIGNATURES[base], name
        assert hasattr(_lib.lib(), name)
    assert "nor differentiable in A" not in hdr


def _control(static=True, sparse=None):
    fake = 4096
    return _lib.PegControl(fake, None if (static or sparse is not None) else fake, fake, fake, fake, fake, None, fake, fake, None,
                           ctypes.pointer(sparse) if sparse is not None else None, fake if static else None)


def _vjp(ctl, g, n=200, y=4096):
    """pegncde_vf_vjp_adj_static with fake (never dereferenced) device pointers: the argument checks return before anything runs"""
    fake = 4096
    dims = _lib.PegDims(1, n, (n + 31) // 32 * 32, 8, 0, 1, 3, 0)
    return _lib.lib().pegncde_vf_vjp_adj_static(None, dims, ctypes.byref(ctl), fake, 0.5, y, fake, fake, fake, None, g, fake, 1 << 30)


def _bwd(ctl, g, n=200, y=4096):
    fake = 4096
    dims = _lib.PegDims(1, n, (n + 31) // 32 * 32, 8, 0, 1, 3, 0)
    ts = (ctypes.c_float * 2)(0.0, 1.0)
    return _lib.lib().pegncde_solve_bwd_adj_static(None, dims, ctypes.byref(ctl), fake, ts, 1, y, None, fake, None, None, fake, fake,
                                                   None, g, fake, 1 << 30)


def test_c_abi_checks_the_static_gradient_without_a_device():
    sp = _lib.PegSparse(10, 10, 4096, 4096, 4096, 4096, 4096, 4096)
    for call in (_vjp, _bwd):
        assert call(_control(static=False), 8192) == 5, call                  # dense control: PEG_ERR_UNSUPPORTED
        assert call(_control(static=False, sparse=sp), 8192) == 5, call       # sparse control: PEG_ERR_UNSUPPORTED
        assert call(_control(), 8196) == 6, call                              # misaligned: PEG_ERR_ALIGNMENT
        assert call(_control(), 8192, y=None) == 2, call                      # past the gradient's checks: the plain entry's
        assert call(_control(), None, y=None) == 2, call                      # NULL gradient: the plain entry (NULL y)
    # the sparse entries keep refusing a static control
    dims = _lib.PegDims(1, 200, 224, 8, 0, 1, 3, 0)
    assert _lib.lib().pegncde_vf_vjp_adj(None, dims, ctypes.byref(_control()), 4096, 0.5, 4096, 4096, 4096, 4096, None, 8192, 4096,
                                         1 << 30) == 5


def test_differentiable_static_control_needs_a_cuda_device():
    A = torch.rand(6, 6, requires_grad=True)
    with pytest.raises(RuntimeError):
        P.build_static_control(torch.arange(3.0), A, device="cpu", differentiable=True)
    with pytest.raises(ValueError):
        P.build_static_control(torch.arange(3.0), A, device="cuda")          # without the flag: refused as before


# ---------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------
def _kernel_names(fn, tmp_path):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    path = tmp_path / "trace.json"
    prof.export_chrome_trace(str(path))
    names = {e.get("name", "") for e in json.loads(path.read_text())["traceEvents"] if e.get("cat") == "kernel"}
    return out, names


def _ran(names, kernel):
    return any(re.search(rf"(^|[\s:]){kernel}\b", s) for s in names)


def _graph(n, seed, B=None):
    g = torch.Generator().manual_seed(seed)
    shape = (n, n) if B is None else (B, n, n)
    mask = torch.rand(shape, generator=g) < min(1.0, 16.0 / n)
    A = torch.where(mask, torch.exp(torch.randn(shape, generator=g)), torch.zeros(()))
    A = A + torch.eye(n)
    return (A / A.sum(-1, keepdim=True)).to(torch.float64)


def _const_coeffs(p64, A64):
    """reference-layout (d, c, b, a) of the constant path A(t) = A (time channel: t itself) with A a leaf"""
    T1, n = p64.ts.numel() - 1, A64.shape[-1]
    z = torch.zeros((T1, n, n, 2), dtype=torch.float64)
    b = z.clone()
    b[..., 0] = 1.0
    a = torch.stack([p64.ts[:-1][:, None, None].expand(T1, n, n), A64.expand(T1, n, n)], dim=-1)
    return (z, z, b, a)


def _device_vf(p, cuda, flags, cls=P.PermEquivGraphVectorField):
    widths = R.layer_widths(p.h, p.L, p.e, p.e > 0)
    vf = cls(p.h, p.h, widths[-1], p.L, p.e, p.n, key=0)
    with torch.no_grad():
        for mine, lp in zip(vf.gnn_layers, p.layers):
            cl = mine.conv_layer
            cl.linear.weight.copy_(lp.weight); cl.linear.bias.copy_(lp.bias)
            cl.norm.weight.copy_(lp.norm_weight); cl.norm.bias.copy_(lp.norm_bias)
            if cls is P.PermEquivGraphVectorField:
                for i in range(8):
                    getattr(mine, f"param{i + 1}").copy_(lp.fusion[i])
    vf = vf.to(cuda)
    vf.flags = flags
    return vf


def _static_leaf(A64, ts, cuda, x_t=None):
    A = A64.to(torch.float32).to(cuda).requires_grad_(True)
    return P.build_static_control(ts.to(torch.float32).to(cuda), A, x_t, differentiable=True), A


# ---------------------------------------------------------------------------------------------------
# GPU 1: one evaluation + VJP against the fp64 oracle, every operand format, both gradient kernels
# ---------------------------------------------------------------------------------------------------
SHAPES = [(100, 32, 0, 2), (128, 64, 0, 2), (200, 128, 0, 2), (200, 128, 8, 2), (515, 32, 0, 3), (1000, 64, 8, 3), (300, 256, 0, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", list(FMTS))
@pytest.mark.parametrize("n,h,e,L", SHAPES)
def test_vector_field_adjacency_gradient_against_oracle(cuda, tmp_path, fmt, n, h, e, L):
    p = R.make_problem(n=n, h=h, e=e, L=L, T=3, t1=2, dt0=0.5, seed=21)
    flags = FMTS[fmt] if n < 128 else per_operator(FMTS[fmt])   # n < 128: the default plan would pick the small path; it falls back
    vf = _device_vf(p, cuda, flags)
    A64 = _graph(n, 3 + n)
    xc = None if e == 0 else tuple(c.to(torch.float32).to(cuda) for c in p.x_coeffs)
    sc, A = _static_leaf(A64, p.ts, cuda)
    t = 1.3
    y = p.y0.to(cuda).requires_grad_(True)
    term = P.CDEWrapperVectorField(vf, p.h) if e > 0 else vf
    args = [sc, P.CubicInterpolation(p.ts.to(torch.float32).to(cuda), xc)] if e > 0 else sc

    def run():
        dy = term(t, y, args)
        (dy * p.gyT.to(cuda)).sum().backward()
        return dy
    dy, names = _kernel_names(run, tmp_path)
    p64 = R.problem_to(p, torch.float64)
    Aref = A64.clone().requires_grad_(True)
    ca = R.CubicInterpolation(p64.ts, _const_coeffs(p64, Aref))
    if e > 0:
        ref = R.cde_wrapper_vector_field(t, p64.y0, ca, R.CubicInterpolation(p64.ts, p64.x_coeffs), p64.layers, p64.h, p64.e)
    else:
        ref = R.perm_equiv_vector_field(t, p64.y0, ca, p64.layers)
    (ref * p64.gyT).sum().backward()
    kernel = grad_kernel(flags, n)
    assert _ran(names, kernel), (kernel, sorted(names))
    assert not _ran(names, "k_tc_adj_grad" if kernel == "k_adj_grad" else "k_adj_grad")
    assert rel_err(dy, ref) < 2e-5
    assert rel_l2(A.grad, Aref.grad) <= TOL_G[fmt], rel_l2(A.grad, Aref.grad)


DIR_FIELDS = ("param1", "param2", "param3", "param4", "param4_prime", "param5", "param5_prime", "param6", "param6_prime", "param7", "param8")


@pytest.mark.gpu
@pytest.mark.parametrize("tc", [True, False], ids=["tcgen05", "ffma"])
@pytest.mark.parametrize("field", ["undirected", "directed", "GraphVectorField", "GNODEVectorField"])
def test_fields_adjacency_gradient_against_oracle(cuda, tmp_path, field, tc):
    p = R.make_problem(n=140, h=32, e=0, L=2, T=4, t1=3, dt0=0.75, seed=29)
    cls = {"undirected": P.PermEquivGraphVectorField, "directed": P.PermEquivDirGraphVectorField, "GraphVectorField": P.GraphVectorField,
           "GNODEVectorField": P.GNODEVectorField}[field]
    flags = per_operator(TC if tc else 0)
    vf = _device_vf(p, cuda, flags, cls)
    A64 = _graph(140, 8)
    sc, A = _static_leaf(A64, p.ts, cuda)
    y0 = p.y0.to(cuda).requires_grad_(True)

    def run():
        yT = P.diffeqsolve(P.ODETerm(vf), P.Tsit5(), 0.0, 3.0, 0.75, y0, sc).ys[-1]
        (yT * p.gyT.to(cuda)).sum().backward()
        return yT
    yT, names = _kernel_names(run, tmp_path)
    assert _ran(names, grad_kernel(flags, 140)), sorted(names)
    p64 = R.problem_to(p, torch.float64)
    Aref = A64.clone().requires_grad_(True)
    ca = R.CubicInterpolation(p64.ts, _const_coeffs(p64, Aref))
    if field == "directed":
        fus64 = [torch.stack([getattr(m, f).detach().double().cpu() for f in DIR_FIELDS]) for m in vf.gnn_layers]
        f = lambda t, y: R.perm_equiv_dir_vector_field(t, y, ca, p64.layers, fus64)
    elif field == "undirected":
        f = lambda t, y: R.perm_equiv_vector_field(t, y, ca, p64.layers)
    else:
        f = lambda t, y: R.plain_graph_vector_field(t, y, ca, p64.layers, field == "GraphVectorField")
    ref = R.tsit5_solve_fixed(f, p64.y0, R.constant_step_table(0.0, 3.0, 0.75))
    (ref * p64.gyT).sum().backward()
    assert rel_err(yT, ref) < 1e-4
    assert rel_l2(A.grad, Aref.grad) <= 1e-3


# ---------------------------------------------------------------------------------------------------
# GPU 2: solves
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("save", ["t1", "steps", "ts"])
@pytest.mark.parametrize("store", [True, False])
def test_fixed_step_solve_adjacency_gradient_against_oracle(cuda, save, store):
    p = R.make_problem(n=160, h=32, e=0, L=2, T=4, t1=3, dt0=0.5, seed=31)
    vf = _device_vf(p, cuda, TC)
    vf.store_stages = store
    A64 = _graph(160, 9)
    sc, A = _static_leaf(A64, p.ts, cuda)
    ts = p.ts.to(torch.float32)
    saveat = {"t1": P.SaveAt(t1=True), "steps": P.SaveAt(steps=True), "ts": P.SaveAt(ts=ts)}[save]
    y0 = p.y0.to(cuda).requires_grad_(True)
    ys = P.diffeqsolve(P.ODETerm(vf), P.Tsit5(), 0.0, 3.0, 0.5, y0, sc, saveat=saveat).ys
    g = torch.randn(ys.shape, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    (ys * g.to(torch.float32).to(cuda)).sum().backward()
    p64 = R.problem_to(p, torch.float64)
    Aref = A64.clone().requires_grad_(True)
    ca = R.CubicInterpolation(p64.ts, _const_coeffs(p64, Aref))
    f = lambda t, y: R.perm_equiv_vector_field(t, y, ca, p64.layers)
    step_ts = R.constant_step_table(0.0, 3.0, 0.5)
    if save == "ts":
        ref, _, _ = R.tsit5_solve_adaptive(f, p64.y0, 0.0, 3.0, save_ts=[float(t) for t in ts], forced_steps=step_ts)
    elif save == "steps":
        ref = torch.stack(R.tsit5_solve_fixed(f, p64.y0, step_ts, save_all=True))
    else:
        ref = R.tsit5_solve_fixed(f, p64.y0, step_ts)[None]
    (ref * g).sum().backward()
    assert rel_err(ys, ref) < 1e-4
    assert rel_l2(A.grad, Aref.grad) <= 1e-3


@pytest.mark.gpu
def test_small_graph_solve_falls_back_and_matches_the_oracle(cuda):
    """n < 128 on the product default: the forward runs the cluster kernels (no kept M_l in the stage store), the adjoint with the
    gradient the per-operator path"""
    p = R.make_problem(n=60, h=32, e=0, L=2, T=4, t1=3, dt0=0.5, seed=33)
    vf = _device_vf(p, cuda, TC)
    vf.store_stages = True
    A64 = _graph(60, 10)
    sc, A = _static_leaf(A64, p.ts, cuda)
    y0 = p.y0.to(cuda).requires_grad_(True)
    yT = P.diffeqsolve(P.ODETerm(vf), P.Tsit5(), 0.0, 3.0, 0.5, y0, sc).ys[-1]
    (yT * p.gyT.to(cuda)).sum().backward()
    p64 = R.problem_to(p, torch.float64)
    Aref, y64 = A64.clone().requires_grad_(True), p64.y0.clone().requires_grad_(True)
    ca = R.CubicInterpolation(p64.ts, _const_coeffs(p64, Aref))
    ref = R.tsit5_solve_fixed(lambda t, y: R.perm_equiv_vector_field(t, y, ca, p64.layers), y64, R.constant_step_table(0.0, 3.0, 0.5))
    (ref * p64.gyT).sum().backward()
    assert rel_err(yT, ref) < 1e-4
    assert rel_err(y0.grad, y64.grad) < 1e-3
    assert rel_l2(A.grad, Aref.grad) <= 1e-3


@pytest.mark.gpu
def test_batched_adaptive_solve_adjacency_gradient_against_oracle(cuda):
    B, n, h = 3, 150, 16
    p = R.make_problem(n=n, h=h, e=0, L=2, T=6, t1=5, dt0=0.1, seed=8)
    vf = _device_vf(p, cuda, TC)
    A64 = _graph(n, 12, B=B)
    sc, A = _static_leaf(A64, p.ts, cuda)
    ts = p.ts.to(torch.float32)
    gen = torch.Generator().manual_seed(4)
    y0 = (p.y0[None] + 0.1 * torch.randn((B, n, h), generator=gen)).to(cuda).requires_grad_(True)
    stats = []
    sol = P.diffeqsolve(P.ODETerm(vf), P.Tsit5(), 0.0, 5.0, None, y0, sc, stepsize_controller=P.PIDController(rtol=1e-3, atol=1e-6),
                        saveat=P.SaveAt(ts=ts))
    g = torch.randn(sol.ys.shape, generator=gen, dtype=torch.float64)
    (sol.ys * g.to(torch.float32).to(cuda)).sum().backward()
    p64 = R.problem_to(p, torch.float64)
    for b in range(B):
        Aref = A64[b].clone().requires_grad_(True)
        ca = R.CubicInterpolation(p64.ts, _const_coeffs(p64, Aref))
        step_ts = sol.stats["step_ts"][b] if isinstance(sol.stats["step_ts"], (list, tuple)) else sol.stats["step_ts"]
        ref, _, _ = R.tsit5_solve_adaptive(lambda t, y: R.perm_equiv_vector_field(t, y, ca, p64.layers), y0[b].detach().double().cpu(),
                                           0.0, 5.0, save_ts=[float(t) for t in ts], forced_steps=step_ts)
        (ref * g[:, b]).sum().backward()
        assert rel_err(sol.ys[:, b], ref) < 1e-4, b
        assert rel_l2(A.grad[b], Aref.grad) <= 1e-3, b


# ---------------------------------------------------------------------------------------------------
# GPU 3: the models with a learned adjacency softmax(relu(E E^T)), against the full-pattern sparse control's edge gradient
# ---------------------------------------------------------------------------------------------------
def _learned(E):
    return torch.softmax(torch.relu(E @ E.t()), dim=-1)


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["GraphNeuralCDE", "PGT", "TGB"])
def test_models_learn_the_adjacency(cuda, model):
    """E.grad through the static control against E.grad through build_sparse_control on all n^2 edges with A at every knot (the
    sparse edge-gradient path, itself checked against the oracle): different arithmetic, the same derivative"""
    n, h, e, T = 140, 16, 3, 5
    ts = torch.arange(T, dtype=torch.float32, device=cuda)
    g = torch.Generator().manual_seed(9)
    E0 = (0.3 * torch.randn((n, 8), generator=g)).to(cuda)
    x0 = torch.randn(n, 1, generator=g).to(cuda)
    xco = tuple(torch.randn((T - 1, n, e, 2), generator=g).to(cuda) for _ in range(4))
    x2 = torch.randn(n, 2, generator=g).to(cuda)
    x_data = torch.randn(T, n, n, generator=g).to(cuda)
    xt0 = torch.randn(n, n, generator=g).to(cuda)
    ii, jj = torch.meshgrid(torch.arange(n), torch.arange(n), indexing="ij")
    ei = torch.stack([ii.reshape(-1), jj.reshape(-1)]).to(cuda)

    def run(kind):
        E = E0.clone().requires_grad_(True)
        A = _learned(E)
        if kind == "static":
            ctl = P.build_static_control(ts, A, differentiable=True)
        else:
            ctl = P.build_sparse_control(ts, ei, A.reshape(1, -1).expand(T, n * n), n)
        if model == "GraphNeuralCDE":
            m = P.GraphNeuralCDE(16, P.PermEquivGraphVectorField(16, 16, 16, 2, 0, n, key=1), seed=3, dt0=0.25,
                                 controller=P.ConstantStepSize()).to(cuda)
            out = m(ts, ctl, x0)
        elif model == "PGT":
            m = P.PGTGraphNeuralCDE(h, 2, 3, P.PermEquivGraphVectorField(h, h, 2 * h * e, 2, e, n, key=2), seed=1, dt0=0.1).to(cuda)
            out = m(ts, ctl, P.CubicInterpolation(ts, xco), x2)
        else:
            m = P.TGBGraphNeuralCDE(h, P.PermEquivGraphVectorField(h, h, 2 * h * 4, 2, 4, n, key=3), use_mlps=True, seed=2,
                                    dt0=0.05).to(cuda)
            out = m(ts, ctl, x_data, xt0, None)
        out.square().mean().backward()
        return out.detach(), E.grad

    got, ref = run("static"), run("sparse")
    assert rel_err(got[0], ref[0]) < 1e-5
    assert float(ref[1].abs().max()) > 0
    assert rel_l2(got[1], ref[1]) <= 1e-4, rel_l2(got[1], ref[1])


# ---------------------------------------------------------------------------------------------------
# GPU 4: an independent cross-check and a large graph
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("tc", [True, False], ids=["tcgen05", "ffma"])
def test_gradient_equals_the_full_pattern_sparse_edge_gradient(cuda, tc):
    n, h, T = 512, 64, 4
    p = R.make_problem(n=n, h=h, e=0, L=3, T=T, t1=3, dt0=0.5, seed=14)
    vf = _device_vf(p, cuda, per_operator(TC if tc else 0))
    A32 = _graph(n, 15).to(torch.float32).to(cuda)
    ts = p.ts.to(torch.float32).to(cuda)
    y0 = p.y0.to(cuda)
    ii, jj = torch.meshgrid(torch.arange(n), torch.arange(n), indexing="ij")
    ei = torch.stack([ii.reshape(-1), jj.reshape(-1)]).to(cuda)

    A = A32.clone().requires_grad_(True)
    yT = P.diffeqsolve(P.ODETerm(vf), P.Tsit5(), 0.0, 3.0, 0.5, y0, P.build_static_control(ts, A, differentiable=True)).ys[-1]
    (yT * p.gyT.to(cuda)).sum().backward()
    w = A32.reshape(1, -1).expand(T, n * n).contiguous().requires_grad_(True)
    yS = P.diffeqsolve(P.ODETerm(vf), P.Tsit5(), 0.0, 3.0, 0.5, y0, P.build_sparse_control(ts, ei, w, n)).ys[-1]
    (yS * p.gyT.to(cuda)).sum().backward()
    ref = w.grad.sum(0).reshape(n, n)            # summed over the knots
    assert rel_err(yT, yS) < 1e-5
    assert rel_l2(A.grad, ref) <= 1e-4, rel_l2(A.grad, ref)


def _dense_vf64(t, y, A, layers, n):
    """PermEquivGraphVectorField on the constant path A(t) = A (A' = 0, time channel t), fp64 on the device"""
    rsA, dgA, totA = A.sum(1), torch.diagonal(A), A.sum()
    z = y
    for li, (p, W, bias, nw, nb) in enumerate(layers):
        m = R.rms_norm(z, nw, nb) @ W.t() + bias
        colm = m.sum(dim=0, keepdim=True)
        fused = ((1 + p[0, 0]) * (A @ m) + p[1, 0] * (A.t() @ m) + (p[2, 0] * dgA)[:, None] * m
                 + (p[3, 0] * rsA / n)[:, None] * colm + ((p[4, 0] * rsA / n)[:, None] * m).sum(dim=0, keepdim=True)
                 + (p[5, 0] * rsA / n)[:, None] * m + (p[6, 0] + p[6, 1]) / n ** 2 * totA * colm + p[7, 0] * totA / n ** 2 * m)
        z = m + fused
        if li < len(layers) - 1:
            z = torch.relu(z)
    return z


def test_fp64_dense_restatement_equals_the_oracle():
    """pins _dense_vf64 to the oracle's vector field on the constant path (CPU, fp64)"""
    p = R.problem_to(R.make_problem(n=37, h=16, e=0, L=3, T=4, t1=3, dt0=0.5, seed=5), torch.float64)
    A = _graph(37, 2)
    t = 1.3
    ref = R.perm_equiv_vector_field(t, p.y0, R.CubicInterpolation(p.ts, _const_coeffs(p, A)), p.layers)
    layers = [[lp.fusion.reshape(8, 2), lp.weight, lp.bias, lp.norm_weight, lp.norm_bias] for lp in p.layers]
    assert rel_err(_dense_vf64(t, p.y0, A, layers, 37), ref) < 1e-12


@pytest.mark.gpu
def test_large_graph_gradient_against_a_central_difference(cuda, tmp_path):
    n, h, L = 16384, 128, 2
    import bench
    A32 = bench.synth_adjacency(n, 1, 21, cuda)[0]
    ts = torch.tensor([0.0, 2.0], device=cuda)
    A = A32.clone().requires_grad_(True)
    vf = P.PermEquivGraphVectorField(h, h, h, L, 0, n, key=6, flags=TC).to(cuda)
    g = torch.Generator(device=cuda).manual_seed(2)
    y0, gy = torch.randn((n, h), generator=g, device=cuda), torch.randn((n, h), generator=g, device=cuda)
    t = 1.3

    def run():
        (vf(t, y0, P.build_static_control(ts, A, differentiable=True)) * gy).sum().backward()
    _, names = _kernel_names(run, tmp_path)
    assert _ran(names, "k_tc_adj_grad"), sorted(names)
    delta = torch.randn((n, n), generator=g, device=cuda, dtype=torch.float64)
    got = float((A.grad.double() * delta).sum())
    layers = []
    for layer in vf.gnn_layers:
        cl = layer.conv_layer
        layers.append([x.detach().double() for x in
                       (layer.fusion_params().reshape(8, 2), cl.linear.weight, cl.linear.bias, cl.norm.weight, cl.norm.bias)])
    A64, y64, g64 = A32.double(), y0.double(), gy.double()
    # a step small enough that the perturbed path crosses no ReLU kink: the field is only piecewise smooth in A
    eps = 1e-7 * float(A64.abs().max()) / float(delta.abs().max())
    loss = lambda a: float((_dense_vf64(t, y64, a, layers, n) * g64).sum())
    fd = (loss(A64 + eps * delta) - loss(A64 - eps * delta)) / (2 * eps)
    print(f"\n[n={n}] <G, delta> = {got:.6e}, central difference {fd:.6e}")
    assert abs(got - fd) <= 1e-3 * abs(fd)


# ---------------------------------------------------------------------------------------------------
# GPU 5: invariants
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("tc", [True, False], ids=["tcgen05", "ffma"])
def test_gradient_is_reproducible_and_leaves_the_other_outputs_alone(cuda, tc):
    n, h, T, B, e = 300, 32, 4, 2, 2
    ts = torch.arange(T, dtype=torch.float32, device=cuda)
    A0 = _graph(n, 5, B=B).to(torch.float32).to(cuda)
    gen = torch.Generator().manual_seed(3)
    x_t = torch.randn((B, T, n, e), generator=gen).to(cuda)
    y0, gy = torch.randn((B, n, h), generator=gen).to(cuda), torch.randn((B, n, h), generator=gen).to(cuda)
    vf = P.PermEquivGraphVectorField(h, h, 2 * h * e, 3, e, n, key=2, flags=per_operator(TC if tc else 0)).to(cuda)

    def run(grad_adj):
        vf.zero_grad(set_to_none=True)
        A = A0.clone().requires_grad_(grad_adj)
        sc = P.build_static_control(ts, A, x_t, differentiable=True)
        y = y0.clone().requires_grad_(True)
        yT = P.diffeqsolve(P.ODETerm(P.CDEWrapperVectorField(vf, h)), P.Tsit5(), 0.0, 3.0, 0.5, y, [sc, None]).ys[-1]
        (yT * gy).sum().backward()
        return yT.detach(), y.grad, [q.grad.clone() for q in vf.parameters()], A.grad

    a, b, off = run(True), run(True), run(False)
    assert torch.equal(a[3], b[3])                                     # bit for bit: one owner per element, no atomics
    assert torch.equal(a[0], off[0]) and torch.equal(a[1], off[1])
    for x, y in zip(a[2], off[2]):                                     # the parameter gradients' float-atomic reassociation
        assert float((x - y).abs().max()) <= 2e-5 * max(float(y.abs().max()), 1e-2 * max(float(q.abs().max()) for q in off[2]))
    assert torch.isfinite(a[3]).all() and float(a[3].abs().max()) > 0
    # g_xcoef of the exact adjoint, with and without the static gradient
    outs = []
    for want in (True, False):
        sc = P.build_static_control(ts, A0, x_t)
        dims = vf.dims_for(sc, with_wrapper=True)
        l = _lib.lib()
        flat = vf.checked_flat_params(dims).detach().contiguous()
        steps = [0.0, 0.5, 1.0]
        host_ts = (ctypes.c_float * 3)(*steps)
        S = 2
        ws = torch.zeros(max(l.pegncde_workspace_bytes(dims, _lib.PEG_WS_SOLVE_FWD, S), l.pegncde_workspace_bytes(dims, _lib.PEG_WS_SOLVE_BWD, S)),
                         dtype=torch.uint8, device=cuda)
        st = torch.cuda.current_stream().cuda_stream
        y_ckpt = torch.empty((S + 1, B, n, h), device=cuda)
        _lib.check(l.pegncde_solve_fwd(st, dims, sc.struct(), flat.data_ptr(), host_ts, S, y0.data_ptr(), None, y_ckpt.data_ptr(), None,
                                       ws.data_ptr(), ws.numel()), "fwd")
        g_y0, g_flat, g_x = torch.empty_like(y0), torch.zeros_like(flat), torch.zeros_like(sc.x_coef)
        g_adj = torch.zeros((B, sc.ldn, sc.ldn), device=cuda)
        args = (st, dims, sc.struct(), flat.data_ptr(), host_ts, S, y_ckpt.data_ptr(), None, gy.data_ptr(), None, None, g_y0.data_ptr(),
                g_flat.data_ptr(), g_x.data_ptr())
        if want:
            _lib.check(l.pegncde_solve_bwd_adj_static(*args, g_adj.data_ptr(), ws.data_ptr(), ws.numel()), "bwd_adj_static")
        else:
            _lib.check(l.pegncde_solve_bwd(*args, ws.data_ptr(), ws.numel()), "bwd")
        torch.cuda.synchronize()
        outs.append((g_y0, g_x, g_adj))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    pad = outs[0][2].clone()
    pad[:, :n, :n] = 0
    assert float(pad.abs().max()) == 0.0 and float(outs[0][2].abs().max()) > 0          # only i, j < n are touched


@pytest.mark.gpu
@pytest.mark.parametrize("tc", [True, False], ids=["tcgen05", "ffma"])
def test_batch_of_different_graphs_equals_each_graph_alone(cuda, tc):
    n, h, B = 256, 32, 3
    ts = torch.tensor([0.0, 1.0, 2.5], device=cuda)
    A0 = _graph(n, 17, B=B).to(torch.float32).to(cuda)
    y0 = torch.randn((B, n, h), generator=torch.Generator().manual_seed(7)).to(cuda)
    vf = P.PermEquivGraphVectorField(h, h, h, 2, 0, n, key=4, flags=per_operator(TC if tc else 0)).to(cuda)

    def run(Ab, y):
        A = Ab.clone().requires_grad_(True)
        yT = P.diffeqsolve(P.ODETerm(vf), P.Tsit5(), 0.0, 2.5, 0.25, y, P.build_static_control(ts, A, differentiable=True)).ys[-1]
        yT.square().sum().backward()
        return A.grad

    batch = run(A0, y0)
    for b in range(B):
        alone = run(A0[b:b + 1], y0[b:b + 1])
        assert torch.equal(batch[b], alone[0]), b
