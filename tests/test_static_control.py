"""Static controls (PegControl.adj_static, build_static_control): a graph that does not change in time, one tiled plane per graph.

The contract: states, state cotangents, g_xdot and the control's tables equal, bit for bit (torch.equal), the same call on the dense
control of the snapshots [A] * T (build_control(ts, A.expand(T, n, n), x_t)) -- on the tensor-core paths (fp16x2, 3xTF32, bf16x2),
FFMA and the small-graph cluster kernels.  Parameter gradients are float-atomic reductions whose order follows CTA timing; they are
checked to reassociation level (_assert_equal_to_reference).  Each case also proves from the profiler's kernel names that the static kernel of the path it names ran."""
import ctypes
import json

import pytest
import torch

import perm_equiv_graph_neural_cdes_b200 as P
from perm_equiv_graph_neural_cdes_b200 import _lib
from oracle import reference_path as R
from tests.helpers import device_model, rel_err

TC = _lib.PEG_FLAG_TENSOR_CORES
OFF_SMALL = _lib.PEG_FLAG_NO_FUSED_SMALL


# ---------------------------------------------------------------------------------------------------
# host: the C-ABI without a device
# ---------------------------------------------------------------------------------------------------
def _vf_fwd(ctl):
    dims = _lib.PegDims(1, 64, 64, 32, 0, 1, 3, 0)
    return _lib.lib().pegncde_vf_fwd(None, dims, ctypes.byref(ctl), 4096, 0.0, 4096, 4096, 4096, 1 << 30)


def _control(**kw):
    base = dict(ts=4096, adj_coef=None, adj_rowsum=4096, adj_diag=4096, adj_total=4096, tch_coef=4096, x_coef=None, adj_colsum=4096,
                adj_absmax=4096, adj_static=4096)
    return _lib.PegControl(**{**base, **kw})


def test_build_adj_static_signature_matches_the_header():
    import os
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, "include", "pegncde.h")).read()
    m = re.search(r"int pegncde_build_adj_static\(([^)]*)\);", hdr)
    assert m, "pegncde_build_adj_static is not declared"
    assert len(m.group(1).split(",")) == len(_lib.SIGNATURES["pegncde_build_adj_static"][1]) == 10
    assert _lib.PegControl._fields_[-1][0] == "adj_static"


def test_c_abi_checks_static_controls_without_a_device():
    sp = _lib.PegSparse(10, 10, 4096, 4096, 4096, 4096, 4096, 4096)
    assert _vf_fwd(_control(sparse=ctypes.pointer(sp))) == 5                   # static + sparse: PEG_ERR_UNSUPPORTED
    sh = _lib.PegShard(0, 1, 64, 0)
    assert _vf_fwd(_control(shard=ctypes.pointer(sh))) == 5                    # static + shard
    assert _vf_fwd(_control(adj_static=4100)) == 6                             # misaligned plane: PEG_ERR_ALIGNMENT
    assert _vf_fwd(_control(adj_rowsum=None)) == 2                             # NULL table: PEG_ERR_NULL_POINTER
    dims = _lib.PegDims(1, 64, 64, 32, 0, 1, 3, 0)
    ctl = _control()
    g = _lib.lib().pegncde_vf_vjp_adj(None, dims, ctypes.byref(ctl), 4096, 0.0, 4096, 4096, 4096, 4096, None, 4096, 4096, 1 << 30)
    assert g == 5                                                              # static + g_adj_coef: no gradient in A
    args = [None, dims] + [4096] * 8
    for i in range(2, 10):
        a = list(args)
        a[i] = None
        assert _lib.lib().pegncde_build_adj_static(*a) == 2, i
    a = list(args)
    a[3] = 4100
    assert _lib.lib().pegncde_build_adj_static(*a) == 6


@pytest.mark.parametrize("bad, err", [
    (torch.zeros(3), ValueError), (torch.zeros(2, 3), ValueError), (torch.zeros(2, 2, 3, 3), ValueError),
    (torch.zeros(3, 3, dtype=torch.complex64), ValueError), (torch.zeros(3, 3, requires_grad=True), ValueError), ([[0.0]], TypeError)])
def test_build_static_control_rejects_malformed_input(bad, err):
    with pytest.raises(err):
        P.build_static_control(torch.arange(3.0), bad, device="cuda")


def test_build_static_control_needs_a_cuda_device_and_two_knots():
    with pytest.raises(RuntimeError):
        P.build_static_control(torch.arange(3.0), torch.zeros(4, 4), device="cpu")


def test_jax_and_row_sharded_paths_reject_static_controls():
    from perm_equiv_graph_neural_cdes_b200.rowshard import RowShardedControl
    sc = P.StaticControl.__new__(P.StaticControl)
    with pytest.raises(TypeError, match="static"):
        RowShardedControl(torch.arange(3.0), sc, sc, 8, 1)
    src = open(P.__file__.replace("__init__.py", "jax_ffi/pegncde_jax.py")).read()
    assert 'hasattr(coeffs_adj, "adj_static")' in src


# ---------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------
def _graphs(B, n, seed, device):
    g = torch.Generator(device="cpu").manual_seed(seed)
    mask = torch.rand((B, n, n), generator=g) < min(1.0, 16.0 / n)
    A = torch.where(mask, torch.exp(torch.randn((B, n, n), generator=g)), torch.zeros(()))
    A = A + torch.eye(n)
    return (A / A.sum(-1, keepdim=True)).to(device)


def _pair(ts, A, x_t=None):
    """(static, replicated dense) controls of the same graph(s) A [B, n, n]"""
    T = ts.shape[-1]
    dense = P.build_control(ts, A[:, None].expand(A.shape[0], T, A.shape[1], A.shape[2]).contiguous(), x_t).ensure_colsums()
    return P.build_static_control(ts, A, x_t), dense


def _kernel_names(fn, tmp_path):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    path = tmp_path / "trace.json"
    prof.export_chrome_trace(str(path))
    names = {e.get("name", "") for e in json.loads(path.read_text())["traceEvents"] if e.get("cat") == "kernel"}
    return out, names


def _assert_equal(a, b, what):
    if isinstance(a, (list, tuple)):
        assert len(a) == len(b), what
        for i, (x, y) in enumerate(zip(a, b)):
            _assert_equal(x, y, f"{what}[{i}]")
        return
    if a is None:
        assert b is None, what
        return
    assert torch.equal(a, b), f"{what}: max |diff| {float((a - b).abs().max())}"


def _flat(x):
    if isinstance(x, (list, tuple)):
        return [t for v in x for t in _flat(v)]
    return [x]


def _assert_equal_to_reference(got, ref, what, nstate=2):
    """`got` against the replicated control's `ref`: the first `nstate` outputs (states, state cotangents, g_xdot) are computed in a
    fixed order and must be equal bit for bit.  The parameter gradients after them are reduced with float atomicAdd across CTAs
    (the fusion-scalar gradients of k_tc_contract / k_dual_contract / the cluster kernels, the Linear backward's weight, bias and
    norm gradients), so their last bits follow the order in which CTAs finish -- which depends on timing, and the static kernels
    time differently from the dense ones.  Those leaves are checked to fp32 reassociation level (2e-5 of the leaf's scale, or of 1e-2 of
    the largest parameter gradient for a leaf that is a sum with cancellation)."""
    g_all, r_all = _flat(got), _flat(ref)
    assert len(g_all) == len(r_all), what
    gmax = max([float(r.abs().max()) for r in r_all[nstate:] if r is not None] + [1e-30])
    for i, (g, r) in enumerate(zip(g_all, r_all)):
        if g is None:
            assert r is None, (what, i)
            continue
        diff = float((g - r).abs().max())
        if i < nstate:
            assert torch.equal(g, r), f"{what}[{i}]: max |diff| {diff}"
        else:
            # a leaf that is a sum with cancellation is compared relative to 1e-2 of the largest parameter gradient
            assert diff <= 2e-5 * max(float(r.abs().max()), 1e-2 * gmax), f"{what}[{i}] (parameter gradient): max |diff| {diff}"


def _vf(n, h, e, L, flags, directed=False, key=0):
    cls = P.PermEquivDirGraphVectorField if directed else P.PermEquivGraphVectorField
    return cls(h, h, 2 * h * e if e > 0 else h, L, e, n, key=key, flags=flags)


def _eval_vjp(vf, ctl, h, e, y0, gy, t=1.3):
    """one evaluation + its VJP through the public API: dy, g_y, every parameter leaf, and g_xcoef when e > 0"""
    vf.zero_grad(set_to_none=True)
    y = y0.clone().requires_grad_(True)
    dy = vf(t, y, ctl)          # e > 0: the control carries the node-signal path, the CDE wrapper is applied
    (dy * gy).sum().backward()
    return dy.detach(), y.grad, [q.grad.clone() for q in vf.parameters()]


# ---------------------------------------------------------------------------------------------------
# GPU 1: the builder's tables equal the replicated dense control's
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [37, 130, 300])
def test_static_builder_tables_equal_the_replicated_control(cuda, n):
    B, T = 2, 4
    ts = torch.tensor([0.0, 0.5, 1.25, 2.0], device=cuda)
    A = _graphs(B, n, n, cuda)
    sc, dense = _pair(ts, A)
    torch.cuda.synchronize()
    assert torch.equal(sc.static_plane(), A)
    assert torch.equal(sc.dense_planes(), dense.dense_planes())
    for name in ("ts", "adj_rowsum", "adj_diag", "adj_total", "adj_colsum", "adj_absmax", "tch_coef"):
        _assert_equal(getattr(sc, name), getattr(dense, name), name)
    # views share the plane
    assert sc.select(1).adj_static.data_ptr() == sc.adj_static[1:].data_ptr()
    assert sc.with_x(None).adj_static.data_ptr() == sc.adj_static.data_ptr()
    assert sc.materialize() is sc and sc.ensure_colsums() is sc
    # host adjacency, one graph
    one = P.build_static_control(ts, A[0].cpu(), device=cuda)
    assert torch.equal(one.adj_static, sc.adj_static[:1]) and torch.equal(one.adj_rowsum, sc.adj_rowsum[:1])
    # byte budget: one plane per graph
    assert sc.adj_static.numel() * 4 == B * 4 * sc.ldn * sc.ldn


# ---------------------------------------------------------------------------------------------------
# GPU 2: one evaluation + VJP, every contraction path
# ---------------------------------------------------------------------------------------------------
# (n, flags, expected static kernel name fragment)
PATHS = {
    "fp16x2": (256, TC | OFF_SMALL, "k_tc_contract<0, 2, true>"),
    "tf32x3": (256, TC | _lib.PEG_FLAG_TF32X3 | OFF_SMALL, "k_tc_contract<0, 0, true>"),
    "bf16x2": (256, TC | _lib.PEG_FLAG_BF16X2 | OFF_SMALL, "k_tc_contract<0, 1, true>"),
    "ffma": (100, OFF_SMALL, "k_dual_contract<1, true>"),
    "cluster_resident": (100, TC, "k_small_fwd<true>"),
    "cluster_streamed": (200, TC | _lib.PEG_FLAG_FUSED_SMALL, "k_small_fwd<true>"),
}
BWD_NAME = {"k_tc_contract<0, 2, true>": "k_tc_contract<1, 2, true>", "k_tc_contract<0, 0, true>": "k_tc_contract<1, 0, true>",
            "k_tc_contract<0, 1, true>": "k_tc_contract<1, 1, true>", "k_dual_contract<1, true>": "k_dual_contract<4, true>",
            "k_small_fwd<true>": "k_small_vjp<true>"}


@pytest.mark.gpu
@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("e", [0, 2])
@pytest.mark.parametrize("directed", [False, True])
def test_evaluation_and_vjp_equal_the_replicated_control(cuda, tmp_path, path, e, directed):
    n, flags, kname = PATHS[path]
    if directed and path.startswith("cluster"):
        pytest.skip("the small-graph kernels take the undirected layer only")
    B, T, h, L = 2, 4, 32, 2
    ts = torch.tensor([0.0, 0.7, 1.5, 2.5], device=cuda)
    A = _graphs(B, n, 7 + n, cuda)
    g = torch.Generator(device="cpu").manual_seed(3)
    x_t = torch.randn((B, T, n, e), generator=g).to(cuda) if e > 0 else None
    y0 = torch.randn((B, n, h), generator=g).to(cuda)
    gy = torch.randn((B, n, h), generator=g).to(cuda)
    sc, dense = _pair(ts, A, x_t)
    vf = _vf(n, h, e, L, flags, directed).to(cuda)
    (ref, names_d) = _kernel_names(lambda: _eval_vjp(vf, dense, h, e, y0, gy), tmp_path)
    (got, names_s) = _kernel_names(lambda: _eval_vjp(vf, sc, h, e, y0, gy), tmp_path)
    _assert_equal_to_reference(got, ref, f"{path} e={e} directed={directed}")
    assert any(kname in s for s in names_s), sorted(names_s)
    assert any(BWD_NAME[kname] in s for s in names_s), sorted(names_s)
    assert not any(", true>" in s or "<true>" in s for s in names_d)
    if e > 0:   # the cotangent of the node-signal derivative through the C-ABI
        outs = []
        for ctl in (sc, dense):
            dims = vf.dims_for(ctl, with_wrapper=True)
            l = _lib.lib()
            flat = vf.checked_flat_params(dims).detach().contiguous()
            ws = torch.zeros(l.pegncde_workspace_bytes(dims, _lib.PEG_WS_VF_VJP, 0), dtype=torch.uint8, device=cuda)
            g_y, g_flat = torch.empty_like(y0), torch.zeros_like(flat)
            g_xd = torch.empty((B, n, 2 * e), device=cuda)
            _lib.check(l.pegncde_vf_vjp(torch.cuda.current_stream().cuda_stream, dims, ctl.struct(), flat.data_ptr(), 0.9, y0.data_ptr(),
                                        gy.data_ptr(), g_y.data_ptr(), g_flat.data_ptr(), g_xd.data_ptr(), ws.data_ptr(), ws.numel()), "vjp")
            torch.cuda.synchronize()
            outs.append((g_y, g_xd))
        _assert_equal(outs[0], outs[1], f"{path} g_xdot")


@pytest.mark.gpu
def test_adj_light_means_nothing_for_a_static_control(cuda):
    n, h, B = 256, 32, 2
    ts = torch.arange(3.0, device=cuda)
    A = _graphs(B, n, 5, cuda)
    sc, dense = _pair(ts, A)
    g = torch.Generator(device="cpu").manual_seed(4)
    y0, gy = torch.randn((B, n, h), generator=g).to(cuda), torch.randn((B, n, h), generator=g).to(cuda)
    light = _vf(n, h, 0, 2, TC | _lib.PEG_FLAG_ADJ_LIGHT | OFF_SMALL).to(cuda)
    exact = _vf(n, h, 0, 2, TC | OFF_SMALL).to(cuda)
    _assert_equal_to_reference(_eval_vjp(light, sc, h, 0, y0, gy), _eval_vjp(exact, dense, h, 0, y0, gy), "ADJ_LIGHT")


# ---------------------------------------------------------------------------------------------------
# GPU 3: solves
# ---------------------------------------------------------------------------------------------------
def _solve(vf, ctl, y0, gy, e, h, saveat, store, controller=None, dt0=0.25):
    vf.zero_grad(set_to_none=True)
    vf.store_stages = store
    y = y0.clone().requires_grad_(True)
    sol = P.diffeqsolve(P.ODETerm(vf), P.Tsit5(), 0.0, 2.5, dt0, y, ctl, saveat=saveat,
                        stepsize_controller=controller if controller is not None else P.ConstantStepSize())
    (sol.ys * gy).sum().backward()
    return sol.ys.detach(), y.grad, [q.grad.clone() for q in vf.parameters()]


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["fp16x2", "ffma", "cluster_resident"])
@pytest.mark.parametrize("save", ["t1", "steps", "ts"])
@pytest.mark.parametrize("store", [True, False])
def test_fixed_step_solve_and_adjoint_equal_the_replicated_control(cuda, path, save, store):
    n, flags, _ = PATHS[path]
    B, h, L, e = 2, 32, 2, 0       # e > 0 solves: the three models below
    ts = torch.tensor([0.0, 0.7, 1.5, 2.5], device=cuda)
    A = _graphs(B, n, 11, cuda)
    g = torch.Generator(device="cpu").manual_seed(5)
    x_t = None
    y0 = torch.randn((B, n, h), generator=g).to(cuda)
    saveat = {"t1": P.SaveAt(t1=True), "steps": P.SaveAt(steps=True), "ts": P.SaveAt(ts=torch.tensor([0.3, 1.1, 2.5]))}[save]
    sc, dense = _pair(ts, A, x_t)
    vf = _vf(n, h, e, L, flags).to(cuda)
    nsave = {"t1": 1, "steps": 11, "ts": 3}[save]
    gy = torch.randn((nsave, B, n, h), generator=g).to(cuda)
    ref = _solve(vf, dense, y0, gy, e, h, saveat, store)
    got = _solve(vf, sc, y0, gy, e, h, saveat, store)
    _assert_equal_to_reference(got, ref, f"{path} {save} store={store}")


@pytest.mark.gpu
def test_batched_adaptive_solve_equals_the_replicated_control(cuda):
    n, h, B, e = 256, 32, 3, 0
    ts = torch.tensor([0.0, 0.7, 1.5, 2.5], device=cuda)
    A = _graphs(B, n, 13, cuda)
    g = torch.Generator(device="cpu").manual_seed(6)
    y0 = torch.randn((B, n, h), generator=g).to(cuda)
    sc, dense = _pair(ts, A)
    vf = _vf(n, h, e, 2, TC).to(cuda)
    gy = torch.randn((3, B, n, h), generator=g).to(cuda)
    saveat = P.SaveAt(ts=torch.tensor([0.3, 1.1, 2.5]))
    ctrl = P.PIDController(rtol=1e-3, atol=1e-6)
    ref = _solve(vf, dense, y0, gy, e, h, saveat, True, ctrl, None)
    got = _solve(vf, sc, y0, gy, e, h, saveat, True, ctrl, None)
    _assert_equal_to_reference(got, ref, "adaptive")


@pytest.mark.gpu
def test_batch_of_different_graphs_equals_each_graph_alone(cuda):
    n, h, B = 256, 32, 3
    ts = torch.tensor([0.0, 1.0, 2.5], device=cuda)
    A = _graphs(B, n, 17, cuda)
    g = torch.Generator(device="cpu").manual_seed(7)
    y0 = torch.randn((B, n, h), generator=g).to(cuda)
    vf = _vf(n, h, 0, 2, TC).to(cuda)
    sc = P.build_static_control(ts, A)
    yT = P.diffeqsolve(P.ODETerm(vf), P.Tsit5(), 0.0, 2.5, 0.25, y0, sc).ys[-1]
    for b in range(B):
        alone = P.diffeqsolve(P.ODETerm(vf), P.Tsit5(), 0.0, 2.5, 0.25, y0[b:b + 1], P.build_static_control(ts, A[b])).ys[-1]
        assert torch.equal(yT[b], alone[0]), b


# ---------------------------------------------------------------------------------------------------
# GPU 4: the three models
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_models_on_static_controls_equal_the_replicated_control(cuda):
    n, h, e, T = 130, 16, 3, 5
    ts = torch.arange(T, dtype=torch.float32, device=cuda)
    A = _graphs(1, n, 19, cuda)
    g = torch.Generator().manual_seed(9)
    x0 = torch.randn(n, 1, generator=g).to(cuda)
    sc, dense = _pair(ts, A)

    def run(make, call, what):
        res = []
        for ctl in (dense, sc):
            model = make().to(cuda)
            out = call(model, ctl)
            out.square().mean().backward()
            res.append((out.detach(), [q.grad.clone() for q in model.parameters()]))
        _assert_equal_to_reference(res[1], res[0], what, nstate=1)

    run(lambda: P.GraphNeuralCDE(16, P.PermEquivGraphVectorField(16, 16, 16, 2, 0, n, key=1), seed=3, dt0=0.25,
                                 controller=P.ConstantStepSize()),
        lambda m, ctl: m(ts, ctl, x0), "GraphNeuralCDE")
    xco = tuple(torch.randn((T - 1, n, e, 2), generator=g).to(cuda) for _ in range(4))
    x2 = torch.randn(n, 2, generator=g).to(cuda)
    run(lambda: P.PGTGraphNeuralCDE(h, 2, 3, P.PermEquivGraphVectorField(h, h, 2 * h * e, 2, e, n, key=2), seed=1, dt0=0.1),
        lambda m, ctl: m(ts, ctl, P.CubicInterpolation(ts, xco), x2), "PGTGraphNeuralCDE")
    x_data = torch.randn(T, n, n, generator=g).to(cuda)
    xt0 = torch.randn(n, n, generator=g).to(cuda)
    run(lambda: P.TGBGraphNeuralCDE(h, P.PermEquivGraphVectorField(h, h, 2 * h * 4, 2, 4, n, key=3), use_mlps=True, seed=2, dt0=0.05),
        lambda m, ctl: m(ts, ctl, x_data, xt0, None), "TGBGraphNeuralCDE")


# ---------------------------------------------------------------------------------------------------
# GPU 5: a large graph, and the fp64 oracle
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_large_graph_evaluation_and_vjp_equal_the_replicated_control(cuda, tmp_path):
    n, h, B = 16384, 128, 1
    ts = torch.tensor([0.0, 1.0], device=cuda)
    import bench
    A = bench.synth_adjacency(n, 1, 21, cuda)
    g = torch.Generator(device=cuda).manual_seed(8)
    y0, gy = torch.randn((B, n, h), generator=g, device=cuda), torch.randn((B, n, h), generator=g, device=cuda)
    vf = _vf(n, h, 0, 2, TC).to(cuda)
    dense = P.build_control(ts, A.expand(2, n, n).contiguous())
    ref = _eval_vjp(vf, dense, h, 0, y0, gy)
    del dense
    torch.cuda.empty_cache()
    got, names = _kernel_names(lambda: _eval_vjp(vf, P.build_static_control(ts, A[0]), h, 0, y0, gy), tmp_path)
    assert any("k_tc_contract<0, 2, true>" in s for s in names) and any("k_tc_contract<1, 2, true>" in s for s in names)
    _assert_equal_to_reference(got, ref, "n=16384")


@pytest.mark.gpu
@pytest.mark.parametrize("n, flags", [(37, None), (200, TC | OFF_SMALL)])
def test_static_evaluation_against_the_fp64_oracle(cuda, n, flags):
    """One evaluation on the static control of the oracle problem's first adjacency plane against the fp64 oracle on the constant path
    (b = c = d = 0).  A sanity anchor; the bit-identity with the replicated control above is the contract."""
    p = R.make_problem(n=n, h=16, e=0, L=2, T=4, t1=3, dt0=0.25, seed=2)
    vf, _, _ = device_model(p, cuda, flags=flags)
    a = p.coeffs_adj[3][0, :, :, 1].to(torch.float64)
    coeffs = [torch.zeros_like(p.coeffs_adj[0], dtype=torch.float64) for _ in range(3)]
    coeffs[2][..., 0] = 1.0                       # the time channel X_time(t) = t: b = 1 (what the static builder's tch_coef says)
    const = p.coeffs_adj[3].to(torch.float64).clone()
    const[..., 1] = a
    ts64 = p.ts.to(torch.float64)
    layers = R.params_to(p.layers, torch.float64)
    t = float(p.ts[1]) + 0.3
    ref = R.perm_equiv_vector_field(t, p.y0.to(torch.float64), R.CubicInterpolation(ts64, (coeffs[0], coeffs[1], coeffs[2], const)), layers)
    sc = P.build_static_control(p.ts.to(torch.float32).to(cuda), a.to(torch.float32).to(cuda))
    dy = vf(t, p.y0.to(torch.float32).to(cuda), sc)
    assert rel_err(dy[0].double().cpu() if dy.dim() == 3 else dy.double().cpu(), ref) < 2e-5
