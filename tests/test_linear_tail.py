"""The adjoint's Linear tail: solve_fwd keeps each layer's M = Linear(RMSNorm(Z)) and its column sums in the stage store, the
tensor-core adjoint reads them back instead of recomputing them, and k_tc_linear_bwd adds the Linear's weight and bias
gradient itself for 128-wide layers (k_tc_weight_grad keeps the other shapes)."""
import pytest
import torch

import bench
import perm_equiv_graph_neural_cdes_b200 as P
from perm_equiv_graph_neural_cdes_b200 import _lib
from oracle import reference_path as R
from tests.helpers import device_model, product_grads_as_oracle, rel_err


def _dims(B, n, h, e, L, T):
    return _lib.PegDims(B=B, n=n, h=h, e=e, L=L, T=T, ldn=(n + 31) // 32 * 32, flags=0)


@pytest.mark.parametrize("B,n,h,e,L", [(9, 2048, 128, 0, 3), (18, 1024, 128, 8, 3), (2, 100, 64, 3, 2), (1, 40, 16, 0, 1)])
def test_stage_store_bytes_follow_the_layout(B, n, h, e, L):
    """Per step and stage: L layer inputs [B,n,h], then M and its [B][2][h] column sums of every h-wide layer (all of them
    unless e > 0, whose last layer is 2he wide)."""
    l = _lib.lib()
    st = B * n * h
    kept = L - 1 if e > 0 else L
    per_stage = (L + kept) * st + kept * B * 2 * h
    for steps in (1, 3, 81):
        assert l.pegncde_stage_store_bytes(_dims(B, n, h, e, L, 9), steps) == 4 * steps * 6 * per_stage
    assert l.pegncde_stage_store_bytes(_dims(B, n, h, e, L, 9), 0) == 0


def _solve(cuda, wl, store):
    """A reduced flagship solve (forward + adjoint) with or without the stage store; returns y(t1), dloss/dy0, the 16 fusion-scalar
    gradients per layer and the other parameter gradients."""
    n, h, e, L = wl["n"], wl["h"], wl["e"], wl["L"]
    vf = P.PermEquivGraphVectorField(h, h, 2 * h * e if e > 0 else h, L, e, n, key=1234,
                                     flags=_lib.PEG_FLAG_TENSOR_CORES | _lib.PEG_FLAG_NO_FUSED_SMALL).to(cuda)
    vf.store_stages = store
    term = P.ODETerm(P.CDEWrapperVectorField(vf, h) if e > 0 else vf)
    ts, cadj, xco, y0, gy, _, snaps, x_t = bench.make_inputs(wl, 1234, cuda, host_copy=False)
    pc = P.pack_control(ts, cadj, xco) if cadj is not None else P.build_control(ts, snaps, x_t)
    y = y0.detach().clone().requires_grad_(True)
    sol = P.diffeqsolve(term, P.Tsit5(), 0.0, wl["t1"], wl["dt0"], y, [pc, None] if e > 0 else pc,
                        stepsize_controller=P.ConstantStepSize(), saveat=P.SaveAt(t1=True))
    (sol.ys[-1] * gy).sum().backward()
    torch.cuda.synchronize()
    fus = [torch.stack([getattr(layer, f"param{i}").grad for i in range(1, 9)]).clone() for layer in vf.gnn_layers]
    rest = [[t.clone() for t in g[1:]] for g in product_grads_as_oracle(vf)]
    return sol.ys[-1].detach().clone(), y.grad.clone(), fus, rest


@pytest.mark.gpu
@pytest.mark.parametrize("e", [0, 8], ids=["flagship", "control-e8"])
def test_kept_m_and_recompute_give_the_same_adjoint(cuda, e):
    """n = 2048, h = 128, B = 5, two steps: the solve with the stage store (M read back) against the checkpoint-and-recompute
    solve.  M and 1^T M are bit-identical either way, so y(t1) and dloss/dy0 are too.  (B = 5 keeps every contraction grid at
    least half the GPU: smaller grids take split-K, whose atomics make the solve itself vary in the last bits from run to run.)
    Parameter gradients are sums of per-CTA atomics, whose order differs from run to run: two solves of the same kind differ by up
    to 3e-6 relative here, so the bound is 1e-5."""
    wl = dict(n=2048, h=128, e=e, L=3, T=3, t1=0.5, dt0=0.25, B=5)
    yk, gk, fk, rk = _solve(cuda, wl, True)
    yr, gr, fr, rr = _solve(cuda, wl, False)
    assert torch.isfinite(gk).all() and float(gk.abs().max()) > 0
    assert torch.equal(yk, yr)
    assert torch.equal(gk, gr)
    for l, (a, b) in enumerate(zip(fk, fr)):
        assert rel_err(a, b) < 1e-5, ("fusion", l, rel_err(a, b))
    for l, (la, lb) in enumerate(zip(rk, rr)):
        for name, a, b in zip(("W", "b", "nw", "nb"), la, lb):
            assert rel_err(a, b) < 1e-5, (name, l, rel_err(a, b))


@pytest.mark.gpu
@pytest.mark.parametrize("n,e", [(1000, 0), (640, 2)])
def test_fused_weight_gradient_against_fp64(cuda, n, e):
    """One evaluation + VJP with h = 128 on the tcgen05 path (3xTF32 operands): the Linear gradients of the 128-wide layers come
    from k_tc_linear_bwd (n = 1000 leaves a partial last block of 128 nodes), the 2he-wide last layer of the control model from
    k_tc_weight_grad.  Both against fp64 autograd through the oracle."""
    p = R.make_problem(n=n, h=128, e=e, L=3, T=3, t1=2, dt0=0.5, seed=7)
    p64 = R.problem_to(p, torch.float64)
    vf, term, args = device_model(p, cuda, flags=_lib.PEG_FLAG_TENSOR_CORES | _lib.PEG_FLAG_TF32X3)
    t = 1.3
    y = p.y0.to(cuda).requires_grad_(True)
    (term(t, y, args) * p.gyT.to(cuda)).sum().backward()
    layers = R.params_to(p64.layers, requires_grad=True)
    q = R.Problem(p64.n, p64.h, p64.e, p64.L, p64.ts, p64.coeffs_adj, p64.x_coeffs, p64.y0, layers, p64.step_ts, p64.gyT)
    ca = R.CubicInterpolation(q.ts, q.coeffs_adj)
    if e > 0:
        ref = R.cde_wrapper_vector_field(t, q.y0, ca, R.CubicInterpolation(q.ts, q.x_coeffs), q.layers, q.h, q.e)
    else:
        ref = R.perm_equiv_vector_field(t, q.y0, ca, q.layers)
    (ref * p64.gyT).sum().backward()
    for l, (got, lp) in enumerate(zip(product_grads_as_oracle(vf), layers)):
        ref_t = lp.tensors()
        for name, g, r in (("W", got[1], ref_t[1]), ("b", got[2], ref_t[2])):
            assert rel_err(g, r.grad) < 2e-5, (l, name, rel_err(g, r.grad))
