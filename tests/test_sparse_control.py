"""Sparse (CSR) adjacency controls (PegSparse in include/pegncde.h): the pattern builder and the C-ABI checks on the host, and on
the GPU the sparse builders, solves, vector fields and models against the dense path on the densified graph and against the oracle.
"""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

import perm_equiv_graph_neural_cdes_b200 as P
from perm_equiv_graph_neural_cdes_b200 import _lib
from oracle import reference_path as R
from tests.helpers import GOLDEN_CASES, device_model, per_operator, product_grads_as_oracle, rel_err, sparse_of_coeffs, union_pattern

GOLD = os.path.join(os.path.dirname(__file__), "golden")
TC = _lib.PEG_FLAG_TENSOR_CORES


# ---------------------------------------------------------------------------------------------------
# host side
# ---------------------------------------------------------------------------------------------------
def test_peg_sparse_layout_matches_the_ctypes_mirror(tmp_path):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cls = _lib.PegSparse
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "pegncde.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(PegSparse));', '  printf("ctl.sparse %zu\\n", offsetof(PegControl, sparse));']
    lines += [f'  printf("{f} %zu\\n", offsetof(PegSparse, {f}));' for f, _ in cls._fields_] + ['  return 0;', '}']
    src, exe = tmp_path / "sp.c", tmp_path / "sp"
    src.write_text("\n".join(lines))
    subprocess.run(["gcc", "-std=c99", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(got["size"]) == ctypes.sizeof(cls)
    assert int(got["ctl.sparse"]) == _lib.PegControl.sparse.offset
    for f, _ in cls._fields_:
        assert int(got[f]) == getattr(cls, f).offset, f


def _csr_reference(ei, n):
    """coalesced pattern of one graph with numpy: dense count matrix -> CSR of it and of its transpose"""
    M = np.zeros((n, n), dtype=np.int64)
    np.add.at(M, (ei[0], ei[1]), 1)
    rows, cols = np.nonzero(M)
    rows_t, cols_t = np.nonzero(M.T)
    rp = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=n))])
    rpt = np.concatenate([[0], np.cumsum(np.bincount(rows_t, minlength=n))])
    return rp, cols, rpt, cols_t, rows


def test_sparse_pattern_coalesces_sorts_and_transposes():
    g = torch.Generator().manual_seed(3)
    n = 23
    graphs = []
    for E in (60, 1, 140):
        ei = torch.randint(0, n, (2, E), generator=g)
        graphs.append(torch.cat([ei, ei[:, : E // 3]], dim=1))        # duplicates
    pat = P.sparse_pattern(graphs, n)
    assert pat.B == 3 and pat.row_ptr.dtype == torch.int32 and pat.row_ptr.shape == (3, n + 1)
    base = 0
    for b, ei in enumerate(graphs):
        rp, cols, rpt, cols_t, rows = _csr_reference(ei.numpy(), n)
        assert np.array_equal(pat.row_ptr[b].numpy(), rp + base)
        assert np.array_equal(pat.row_ptr_t[b].numpy(), rpt + base)
        m = len(cols)
        assert np.array_equal(pat.col[base:base + m].numpy(), cols)
        assert np.array_equal(pat.col_t[base:base + m].numpy(), cols_t)
        # perm_t scatters entry e to its place in the transposed order: same (row, col) seen from the other side
        perm = pat.perm_t[base:base + m].numpy() - base
        assert sorted(perm.tolist()) == list(range(m))
        assert np.array_equal(cols_t[perm], rows) and np.array_equal(np.repeat(np.arange(n), np.diff(rpt))[perm], cols)
        # coalescing: edge weights summed into their entry equal index_put_(accumulate=True) into a dense matrix
        w = torch.rand(ei.shape[1], generator=g, dtype=torch.float64)
        dense = torch.zeros((n, n), dtype=torch.float64).index_put_((ei[0], ei[1]), w, accumulate=True)
        vals = torch.zeros(pat.nnz, dtype=torch.float64).index_add_(0, pat.edge_map[b], w)
        assert torch.allclose(vals[base:base + m], dense[torch.from_numpy(rows), torch.from_numpy(cols)], rtol=0, atol=1e-15)
        base += m
    assert pat.nnz == base


@pytest.mark.parametrize("bad", [torch.tensor([[0, 1], [2, 23]]), torch.tensor([[0, -1], [2, 3]]), torch.zeros((3, 4), dtype=torch.int64),
                                 torch.zeros((2, 3), dtype=torch.float32), torch.zeros(5, dtype=torch.int64), "not a tensor"],
                         ids=["col-out-of-range", "negative", "three-rows", "float", "1-d", "type"])
def test_sparse_pattern_rejects_malformed_input(bad):
    with pytest.raises(ValueError):
        P.sparse_pattern(bad, 23)


def _host_call(sparse=None, shard=None, n=64):
    """pegncde_vf_fwd with fake (never dereferenced) device pointers: the argument checks return before anything is enqueued"""
    fake = 4096
    dims = _lib.PegDims(1, n, (n + 31) // 32 * 32, 8, 0, 1, 3, 0)
    ctl = _lib.PegControl(fake, None, fake, fake, fake, fake, None, None, None,
                          ctypes.pointer(shard) if shard is not None else None, ctypes.pointer(sparse) if sparse is not None else None)
    return _lib.lib().pegncde_vf_fwd(None, dims, ctl, fake, 0.5, fake, fake, fake, 1 << 30)


def test_c_abi_checks_sparse_controls_without_a_device():
    full = dict(nnz=10, nnz_stride=10, row_ptr=4096, col=4096, coef=4096, row_ptr_t=4096, col_t=4096, coef_t=4096)
    for missing in ("row_ptr", "col", "coef", "row_ptr_t", "col_t", "coef_t"):
        sp = _lib.PegSparse(**{**full, missing: None})
        assert _host_call(sp) == 2, missing                       # PEG_ERR_NULL_POINTER
    assert _host_call(_lib.PegSparse(**{**full, "nnz_stride": 5})) == 1       # PEG_ERR_BAD_DIMS
    assert _host_call(_lib.PegSparse(**{**full, "coef": 4100})) == 6          # PEG_ERR_ALIGNMENT
    sh = _lib.PegShard(0, 1, 64, 0)
    assert _host_call(_lib.PegSparse(**full), shard=sh) == 5                  # PEG_ERR_UNSUPPORTED
    # neither a dense nor a sparse adjacency path
    assert _host_call(None) == 2
    for fn in ("pegncde_build_adj_sparse", "pegncde_pack_adj_sparse"):
        dims = _lib.PegDims(1, 64, 64, 4, 0, 1, 3, 0)
        nargs = len(_lib.SIGNATURES[fn][1])
        args = [None, dims, ctypes.pointer(_lib.PegSparse(**{**full, "col_t": None}))] + [4096] * (nargs - 3)
        assert getattr(_lib.lib(), fn)(*args) == 2, fn


# ---------------------------------------------------------------------------------------------------
# GPU: helpers
# ---------------------------------------------------------------------------------------------------
def _sparse_model(p, cuda, flags):
    """device_model with the adjacency control replaced by its sparse form"""
    vf, term, _ = device_model(p, cuda, flags=flags)
    ts = p.ts.to(torch.float32).to(cuda)
    co = tuple(c.to(torch.float32).to(cuda) for c in p.coeffs_adj)
    xc = None if p.e == 0 else tuple(c.to(torch.float32).to(cuda) for c in p.x_coeffs)
    sc = sparse_of_coeffs(ts, co)
    args = sc if p.e == 0 else [sc, P.CubicInterpolation(ts, xc)]
    return vf, term, args


def _snapshot_edges(A):
    """snapshots [T, n, n] -> (edge_index [2, E], edge_weight [T, E]) on the union of nonzeros"""
    ei = union_pattern(A)
    return ei, A[:, ei[0], ei[1]].contiguous()


# ---------------------------------------------------------------------------------------------------
# GPU 1: the builder against the dense builder
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [37, 130, 1000])
def test_sparse_builder_matches_the_dense_builder(cuda, n):
    T = 5
    ts = torch.tensor([0.0, 0.7, 1.1, 2.5, 3.0], device=cuda)
    A = torch.from_numpy(R.synthetic_graph_path(n, T, seed=n)).to(torch.float32).to(cuda)
    ei, w = _snapshot_edges(A)
    dense = P.build_control(ts, A).ensure_colsums()
    sc = P.build_sparse_control(ts, ei, w, n)
    planes = dense.dense_planes()[0]                                # [T-1, 4, n, n]
    at_pattern = planes[:, :, ei[0], ei[1]].permute(0, 2, 1)        # [T-1, E, 4]
    assert torch.equal(sc.coef, at_pattern)                          # bit for bit: the same Hermite arithmetic
    assert torch.equal(sc.coef_t[:, sc.pattern.perm_t.long()], sc.coef)
    assert torch.equal(sc.dense_planes(), dense.dense_planes())
    assert torch.equal(sc.adj_diag, dense.adj_diag)
    # the sums run in another order than the dense pre-pass: compared relative to the sum of the magnitudes they add (the rows of
    # the b, c, d planes of a row-normalised path sum to ~0, so a plain relative error would measure cancellation)
    mag = planes.abs().double()
    for name, scale in (("adj_rowsum", mag.sum(-1)), ("adj_colsum", mag.sum(-2)), ("adj_total", mag.sum((-1, -2)))):
        err = float(((getattr(sc, name)[0].double() - getattr(dense, name)[0].double()).abs() / scale.clamp_min(1e-30)).max())
        assert err < 1e-6, (name, err)
    assert torch.equal(sc.tch_coef, dense.tch_coef)


# ---------------------------------------------------------------------------------------------------
# GPU 2: every golden case, solved on its sparse control
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, TC], ids=["ffma", "tcgen05-linear"])
@pytest.mark.parametrize("case", list(GOLDEN_CASES))
def test_sparse_solve_against_goldens(cuda, case, flags):
    g = np.load(os.path.join(GOLD, f"{case}.npz"))
    kw = GOLDEN_CASES[case]
    p = R.make_problem(**kw)
    vf, term, args = _sparse_model(p, cuda, flags)
    y0 = p.y0.to(cuda).requires_grad_(True)
    sol = P.diffeqsolve(P.ODETerm(term), P.Tsit5(), float(p.ts[0]), float(p.ts[-1]), kw["dt0"], y0, args,
                        stepsize_controller=P.ConstantStepSize(), saveat=P.SaveAt(t1=True))
    assert sol.stats["num_steps"] == int(g["steps"])
    yT = sol.ys[-1]
    assert rel_err(yT.detach(), g["yT64"]) < 1e-4 + 4.0 * float(g["rel32"]), case
    (yT * p.gyT.to(cuda)).sum().backward()
    flat = torch.cat([t.reshape(-1) for layer in product_grads_as_oracle(vf) for t in layer]).cpu().double()
    if float(g["cond"]) >= 50:     # the stiff case: kink-aware bound of test_solve_against_goldens
        ref_y = torch.from_numpy(g["gy0_64"])
        assert float((y0.grad.cpu().double() - ref_y).norm() / ref_y.norm()) < 2e-2
        ref = torch.from_numpy(g["gparams64"])
        assert float((flat - ref).norm() / ref.norm()) < 2e-2
        return
    assert rel_err(y0.grad, g["gy0_64"]) < 1e-3, case
    flat, ref, off = flat.numpy(), g["gparams64"], 0
    for layer in vf.gnn_layers:
        cl = layer.conv_layer
        for name, numel in (("fusion", 16), ("W", cl.linear.weight.numel()), ("b", cl.linear.bias.numel()),
                            ("nw", cl.norm.weight.numel()), ("nb", cl.norm.bias.numel())):
            a, b = flat[off:off + numel], ref[off:off + numel]
            assert np.abs(a - b).max() <= 1e-3 * max(np.abs(b).max(), 1e-12) + 1e-7, (case, name)
            off += numel


# ---------------------------------------------------------------------------------------------------
# GPU 3: one evaluation + VJP against the fp64 oracle
# ---------------------------------------------------------------------------------------------------
def _vf_oracle(p64, t, y):
    ca = R.CubicInterpolation(p64.ts, p64.coeffs_adj)
    if p64.e > 0:
        return R.cde_wrapper_vector_field(t, y, ca, R.CubicInterpolation(p64.ts, p64.x_coeffs), p64.layers, p64.h, p64.e)
    return R.perm_equiv_vector_field(t, y, ca, p64.layers)


@pytest.mark.gpu
@pytest.mark.parametrize("n,h,e,L", [(1000, 64, 16, 3), (1000, 64, 0, 3), (515, 32, 0, 2), (300, 32, 3, 2), (129, 64, 8, 3)])
def test_sparse_vector_field_and_vjp_against_oracle(cuda, n, h, e, L):
    p = R.make_problem(n=n, h=h, e=e, L=L, T=3, t1=2, dt0=0.5, seed=21)
    p64 = R.problem_to(p, torch.float64)
    vf, term, args = _sparse_model(p, cuda, TC)
    t = 1.3
    y = p.y0.to(cuda).requires_grad_(True)
    dy = term(t, y, args)
    (dy * p.gyT.to(cuda)).sum().backward()
    layers = R.params_to(p64.layers, requires_grad=True)
    q = R.Problem(p64.n, p64.h, p64.e, p64.L, p64.ts, p64.coeffs_adj, p64.x_coeffs, p64.y0, layers, p64.step_ts, p64.gyT)
    y64 = p64.y0.clone().requires_grad_(True)
    ref = _vf_oracle(q, t, y64)
    (ref * p64.gyT).sum().backward()
    assert rel_err(dy.detach(), ref.detach()) < 2e-5
    assert rel_err(y.grad, y64.grad) < 5e-5
    for l, (got, lp) in enumerate(zip(product_grads_as_oracle(vf), layers)):
        for name, g, r in zip(("fusion", "W", "b", "nw", "nb"), got, lp.tensors()):
            assert rel_err(g, r.grad) < 3e-4, (l, name)


# ---------------------------------------------------------------------------------------------------
# GPU 4: the directed field and the sibling fields on sparse controls
# ---------------------------------------------------------------------------------------------------
DIR_FIELDS = ("param1", "param2", "param3", "param4", "param4_prime", "param5", "param5_prime", "param6", "param6_prime", "param7", "param8")


@pytest.mark.gpu
def test_sparse_directed_vector_field_against_oracle(cuda):
    p = R.make_problem(n=140, h=32, e=0, L=2, T=4, t1=3, dt0=0.75, seed=29)
    vf = P.PermEquivDirGraphVectorField(p.h, p.h, p.h, p.L, 0, p.n, key=4)
    with torch.no_grad():
        for mine, lp in zip(vf.gnn_layers, p.layers):
            mine.conv_layer.linear.weight.copy_(lp.weight); mine.conv_layer.linear.bias.copy_(lp.bias)
            mine.conv_layer.norm.weight.copy_(lp.norm_weight); mine.conv_layer.norm.bias.copy_(lp.norm_bias)
    fus64 = [torch.stack([getattr(m, f).detach().double() for f in DIR_FIELDS]).requires_grad_(True) for m in vf.gnn_layers]
    vf = vf.to(cuda)
    vf.flags = per_operator(TC)
    ts = p.ts.to(torch.float32).to(cuda)
    sc = sparse_of_coeffs(ts, tuple(c.to(cuda) for c in p.coeffs_adj))
    y0 = p.y0.to(cuda).requires_grad_(True)
    dy = vf(1.3, y0, sc)
    p64 = R.problem_to(p, torch.float64)
    layers = R.params_to(p64.layers, requires_grad=True)
    c64 = R.CubicInterpolation(p64.ts, p64.coeffs_adj)
    assert rel_err(dy, R.perm_equiv_dir_vector_field(1.3, p64.y0, c64, layers, fus64)) < 2e-5
    sol = P.diffeqsolve(P.ODETerm(vf), P.Tsit5(), 0.0, 3.0, 0.75, y0, sc)
    (sol.ys[-1] * p.gyT.to(cuda)).sum().backward()
    y64 = p64.y0.clone().requires_grad_(True)
    yT = R.tsit5_solve_fixed(lambda t, y: R.perm_equiv_dir_vector_field(t, y, c64, layers, fus64), y64, R.constant_step_table(0.0, 3.0, 0.75))
    (yT * p64.gyT).sum().backward()
    assert rel_err(sol.ys[-1], yT) < 1e-4
    assert rel_err(y0.grad, y64.grad) < 1e-3
    for mine, lp, f64 in zip(vf.gnn_layers, layers, fus64):
        assert rel_err(torch.stack([getattr(mine, f).grad for f in DIR_FIELDS]), f64.grad) < 1e-3
        assert rel_err(mine.conv_layer.linear.weight.grad, lp.weight.grad) < 1e-3
        assert rel_err(mine.conv_layer.norm.weight.grad, lp.norm_weight.grad) < 1e-3


@pytest.mark.gpu
@pytest.mark.parametrize("cls,with_derivative", [("GraphVectorField", True), ("GNODEVectorField", False)])
def test_sparse_sibling_vector_fields_against_oracle(cuda, cls, with_derivative):
    p = R.make_problem(n=140, h=32, e=0, L=3, T=4, t1=3, dt0=0.75, seed=19)
    vf = getattr(P, cls)(p.h, p.h, p.h, p.L, 0, p.n, key=0)
    with torch.no_grad():
        for mine, lp in zip(vf.gnn_layers, p.layers):
            mine.linear.weight.copy_(lp.weight); mine.linear.bias.copy_(lp.bias)
            mine.norm.weight.copy_(lp.norm_weight); mine.norm.bias.copy_(lp.norm_bias)
    vf = vf.to(cuda)
    vf.flags = per_operator(TC)
    ts = p.ts.to(torch.float32).to(cuda)
    sc = sparse_of_coeffs(ts, tuple(c.to(cuda) for c in p.coeffs_adj))
    y0 = p.y0.to(cuda).requires_grad_(True)
    sol = P.diffeqsolve(P.ODETerm(vf), P.Tsit5(), 0.0, 3.0, 0.75, y0, sc)
    (sol.ys[-1] * p.gyT.to(cuda)).sum().backward()
    p64 = R.problem_to(p, torch.float64)
    layers = R.params_to(p64.layers, requires_grad=True)
    c64 = R.CubicInterpolation(p64.ts, p64.coeffs_adj)
    y64 = p64.y0.clone().requires_grad_(True)
    yT = R.tsit5_solve_fixed(lambda t, y: R.plain_graph_vector_field(t, y, c64, layers, with_derivative), y64, R.constant_step_table(0.0, 3.0, 0.75))
    (yT * p64.gyT).sum().backward()
    assert rel_err(sol.ys[-1], yT) < 1e-4
    assert rel_err(y0.grad, y64.grad) < 1e-3
    for mine, lp in zip(vf.gnn_layers, layers):
        assert rel_err(mine.linear.weight.grad, lp.weight.grad) < 1e-3
        assert rel_err(mine.norm.weight.grad, lp.norm_weight.grad) < 1e-3


# ---------------------------------------------------------------------------------------------------
# GPU 5: sparse against dense at the benchmarked shape
# ---------------------------------------------------------------------------------------------------
def _synth_batch(n, T, seeds, device):
    import bench
    return torch.stack([bench.synth_adjacency(n, T, s, device) for s in seeds])


@pytest.mark.gpu
def test_sparse_matches_dense_at_the_benchmarked_shape(cuda):
    """n = 2048, h = 128, B = 3, one evaluation + VJP on identical inputs, with the kink-aware rule of
    test_benchmarked_instantiations_one_evaluation_and_vjp for the cotangent"""
    n, h, T, B = 2048, 128, 3, 3
    ts = torch.arange(T, dtype=torch.float32, device=cuda)
    A = _synth_batch(n, T, [31, 32, 33], cuda)
    dense = P.build_control(ts, A)
    sc = P.build_sparse_control(ts, [_snapshot_edges(A[b])[0] for b in range(B)], [_snapshot_edges(A[b])[1] for b in range(B)], n)
    vf = P.PermEquivGraphVectorField(h, h, h, 3, 0, n, key=5).to(cuda)
    g = torch.Generator(device=cuda).manual_seed(1)
    y0, gy = torch.randn((B, n, h), generator=g, device=cuda), torch.randn((B, n, h), generator=g, device=cuda)
    out = []
    for ctl in (dense, sc):
        vf.zero_grad()
        y = y0.clone().requires_grad_(True)
        dy = vf(1.3, y, ctl)
        (dy * gy).sum().backward()
        out.append((dy.detach(), y.grad, [q.grad.clone() for q in vf.parameters()]))
    (dyd, gyd, gpd), (dys, gys, gps) = out
    for b in range(B):
        assert rel_err(dys[b], dyd[b]) < 2e-5, b
        err = (gys[b] - gyd[b]).abs().double() / gyd[b].abs().max().double()
        bad_rows = int((err.max(dim=1).values > 5e-5).sum())
        assert float(err.flatten().median()) < 5e-6 and float(err.flatten().float().quantile(0.9)) < 5e-5, b
        assert bad_rows <= 0.15 * n and rel_err(gys[b], gyd[b]) < 2e-2, (b, bad_rows)
    for a, r in zip(gps, gpd):
        assert rel_err(a, r) < 5e-3


# ---------------------------------------------------------------------------------------------------
# GPU 6: the models on sparse controls equal the same calls on dense controls
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_models_on_sparse_controls_match_dense_controls(cuda):
    # adaptive GraphNeuralCDE, SaveAt(ts): the same accepted-step count
    p = R.make_problem(n=150, h=16, e=0, L=2, T=6, t1=5, dt0=0.1, seed=8)
    ts = p.ts.to(torch.float32).to(cuda)
    co = tuple(c.to(torch.float32).to(cuda) for c in p.coeffs_adj)
    vf, term, _ = device_model(p, cuda)
    stats = [P.diffeqsolve(P.ODETerm(vf), P.Tsit5(), float(ts[0]), float(ts[-1]), None, p.y0.to(cuda), ctl,
                           stepsize_controller=P.PIDController(rtol=1e-3, atol=1e-6), saveat=P.SaveAt(ts=ts)).stats
             for ctl in (P.pack_control(ts, co), sparse_of_coeffs(ts, co))]
    print(f"\nadaptive solve, dense / sparse control: {stats[0]} / {stats[1]}")
    assert stats[0]["num_steps"] == stats[1]["num_steps"], stats
    # The step sizes themselves follow y_err, a difference of nearly equal stage sums: the 1e-7 relative rounding difference of the
    # two contractions moves them by ~1e-4 relative (measured: step 2 is 0.12686639 / 0.12687518), and the dense-output samples by
    # the controller's local error (rtol = 1e-3).  So the adaptive model is compared within that tolerance, and the model plumbing
    # to 1e-4 / 1e-3 on fixed steps, where both controls take the same step table.
    assert np.allclose(stats[0]["step_ts"], stats[1]["step_ts"], rtol=2e-2, atol=0)
    x0 = torch.randn(150, 1, generator=torch.Generator().manual_seed(1)).to(cuda)
    for controller, tol_y, tol_g in ((None, 1e-2, 2e-2), (P.ConstantStepSize(), 1e-4, 1e-3)):
        res = []
        for ctl in (P.pack_control(ts, co), sparse_of_coeffs(ts, co)):
            vf, _, _ = device_model(p, cuda)
            model = P.GraphNeuralCDE(16, vf, seed=3, dt0=None if controller is None else 0.25, controller=controller).to(cuda)
            out = model(ts, ctl, x0)
            out.square().mean().backward()
            res.append((out.detach(), [q.grad.clone() for q in model.parameters()]))
        assert rel_err(res[1][0], res[0][0]) < tol_y, controller
        if controller is None:    # different step tables: the gradients are compared as a whole (measured 2.5e-2 on one leaf)
            flat = [torch.cat([g.reshape(-1) for g in r[1]]).double() for r in res]
            assert float((flat[1] - flat[0]).norm() / flat[0].norm()) < tol_g
            continue
        for a, r in zip(res[1][1], res[0][1]):
            assert rel_err(a, r) < tol_g, controller

    # PGT (cubic and linear interpolation) and TGB (data encoder included), forward + backward
    n, h, e, T = 130, 16, 3, 5
    p = R.make_problem(n=n, h=h, e=e, L=2, T=T, t1=T - 1, dt0=0.1, seed=23)
    ts = p.ts.to(torch.float32).to(cuda)
    co = tuple(c.to(torch.float32).to(cuda) for c in p.coeffs_adj)
    # knot values of the path (what interpolation="linear" takes): a at every knot, the end of the last cubic piece at the last one
    dt = ts[-1] - ts[-2]
    ys = torch.cat([co[3], co[3][-1:] + dt * (co[2][-1:] + dt * (co[1][-1:] + dt * co[0][-1:]))], dim=0)
    lin = P.LinearInterpolation(ts, ys)
    g = torch.Generator().manual_seed(9)
    x0 = torch.randn(n, 2, generator=g).to(cuda)
    xco = tuple(c.to(torch.float32).to(cuda) for c in p.x_coeffs)
    for interp, dense_in, coeffs in (("cubic", co, co), ("linear", ys, (lin.d, lin.c, lin.b, lin.a))):
        res = []
        for sparse in (False, True):
            vf, _, _ = device_model(p, cuda)
            model = P.PGTGraphNeuralCDE(h, 2, 3, vf, interpolation=interp, seed=1, dt0=0.1).to(cuda)
            cadj = sparse_of_coeffs(ts, coeffs) if sparse else dense_in
            out = model(ts, cadj, P.CubicInterpolation(ts, xco), x0)
            out.square().sum().backward()
            res.append((out.detach(), [q.grad.clone() for q in model.parameters()]))
        assert rel_err(res[1][0], res[0][0]) < 1e-4, interp
        for a, r in zip(res[1][1], res[0][1]):
            assert rel_err(a, r) < 1e-3, interp
    x_data = torch.randn(T, n, n, generator=g).to(cuda)
    xt0 = torch.randn(n, n, generator=g).to(cuda)
    res = []
    for sparse in (False, True):
        vf = P.PermEquivGraphVectorField(h, h, 2 * h * 4, 2, 4, n, key=3).to(cuda)
        model = P.TGBGraphNeuralCDE(h, vf, use_mlps=True, seed=2, dt0=0.05).to(cuda)
        cadj = sparse_of_coeffs(ts, co) if sparse else P.pack_control(ts, co)
        out = model(ts, cadj, x_data, xt0, None)
        out.square().mean().backward()
        assert float(model.data_encoder.weight.grad.abs().max()) > 0
        res.append((out.detach(), [q.grad.clone() for q in model.parameters()]))
    assert rel_err(res[1][0], res[0][0]) < 1e-4
    # data_encoder.bias shifts the node signal by a constant, which X'(t) does not see: its exact gradient is 0 and both controls
    # give rounding noise (~1e-9).  Leaves are compared relative to max(their own scale, 1e-4 x the largest gradient entry).
    gmax = max(float(r.abs().max()) for r in res[0][1])
    for a, r in zip(res[1][1], res[0][1]):
        assert float((a - r).abs().max()) <= 1e-3 * max(float(r.abs().max()), 1e-4 * gmax)


# ---------------------------------------------------------------------------------------------------
# GPU 7: a batch of graphs with different patterns equals the graphs solved alone
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_batch_of_different_patterns_equals_graphs_alone(cuda):
    n, h, T = 300, 32, 4
    ts = torch.arange(T, dtype=torch.float32, device=cuda)
    eis, ws = [], []
    for b, density in enumerate((0.01, 0.05, 0.2)):
        A = torch.from_numpy(R.synthetic_graph_path(n, T, seed=40 + b, density=density)).to(torch.float32).to(cuda)
        ei, w = _snapshot_edges(A)
        eis.append(ei); ws.append(w)
    batch = P.build_sparse_control(ts, eis, ws, n)
    assert len({int(batch.row_ptr[b, -1] - batch.row_ptr[b, 0]) for b in range(3)}) == 3
    vf = P.PermEquivGraphVectorField(h, h, h, 2, 0, n, key=8).to(cuda)
    y0 = torch.randn((3, n, h), generator=torch.Generator().manual_seed(4)).to(cuda)
    def run(ctl, y):
        vf.zero_grad()
        y = y.clone().requires_grad_(True)
        yT = P.diffeqsolve(P.ODETerm(vf), P.Tsit5(), 0.0, 3.0, 0.25, y, ctl).ys[-1]
        yT.square().sum().backward()
        return yT.detach(), y.grad
    yb, gb = run(batch, y0)
    for b in range(3):
        ya, ga = run(P.build_sparse_control(ts, eis[b], ws[b], n), y0[b:b + 1])
        assert rel_err(yb[b], ya[0]) < 1e-6 and rel_err(gb[b], ga[0]) < 1e-6, b
        ys, _ = run(batch.select(b), y0[b:b + 1])      # the no-copy view of one graph
        assert torch.equal(ys, ya)


# ---------------------------------------------------------------------------------------------------
# GPU 8: the size the dense layout cannot hold, against an fp64 torch.sparse restatement of the field
# ---------------------------------------------------------------------------------------------------
def _sparse_vf64(t, y, ts, rows, cols, coef, layers, n):
    """PermEquivGraphVectorField (perm_equiv_graph_vector_field.py:85-129, time channel = t) restated with torch.sparse, fp64.
    coef [T-1, E, 4] (a,b,c,d) on entries (rows, cols); layers: (fusion [8,2], W, b, nw, nb) per layer."""
    T = ts.numel()
    iv = int(min(max(int(torch.searchsorted(ts, torch.tensor(t, dtype=ts.dtype), right=False)) - 1, 0), T - 2))
    s = t - float(ts[iv])
    c = coef[iv]
    a_val = c @ torch.tensor([1.0, s, s * s, s ** 3], dtype=c.dtype)
    d_val = c @ torch.tensor([0.0, 1.0, 2 * s, 3 * s * s], dtype=c.dtype)
    idx = torch.stack([rows, cols])
    A = torch.sparse_coo_tensor(idx, a_val, (n, n)).coalesce()
    D = torch.sparse_coo_tensor(idx, d_val, (n, n)).coalesce()
    At, Dt = A.t().coalesce(), D.t().coalesce()
    rsA = torch.zeros(n, dtype=c.dtype).index_add_(0, rows, a_val)
    rsD = torch.zeros(n, dtype=c.dtype).index_add_(0, rows, d_val)
    on = rows == cols
    dgA = torch.zeros(n, dtype=c.dtype).index_add_(0, rows[on], a_val[on])
    dgD = torch.zeros(n, dtype=c.dtype).index_add_(0, rows[on], d_val[on])
    totA, totD = a_val.sum(), d_val.sum()
    z = y
    for li, (p, W, bias, nw, nb) in enumerate(layers):
        m = R.rms_norm(z, nw, nb) @ W.t() + bias
        colm = m.sum(dim=0, keepdim=True)
        fused = ((1 + p[0, 0]) * torch.sparse.mm(A, m) + (1 + p[0, 1]) * torch.sparse.mm(D, m) + p[1, 0] * torch.sparse.mm(At, m)
                 + p[1, 1] * torch.sparse.mm(Dt, m) + (p[2, 0] * dgA + p[2, 1] * dgD)[:, None] * m
                 + ((p[3, 0] * rsA + p[3, 1] * rsD) / n)[:, None] * colm
                 + (((p[4, 0] * rsA + p[4, 1] * rsD) / n)[:, None] * m).sum(dim=0, keepdim=True)
                 + ((p[5, 0] * rsA + p[5, 1] * rsD) / n)[:, None] * m
                 + (p[6, 0] + p[6, 1]) / n ** 2 * totA * colm
                 + (p[7, 0] * totA + p[7, 1] * totD) / n ** 2 * m)
        z = m + fused
        if li < len(layers) - 1:
            z = torch.relu(z)
    return z


@pytest.mark.parametrize("n", [37, 300])
def test_fp64_sparse_restatement_equals_the_oracle(n):
    """pins _sparse_vf64 to the oracle's dense vector field (CPU, fp64) on the union pattern of a synthetic path"""
    p = R.problem_to(R.make_problem(n=n, h=16, e=0, L=3, T=4, t1=3, dt0=0.5, seed=5), torch.float64)
    adj = torch.stack([c[..., 1] for c in p.coeffs_adj])        # [4(d,c,b,a), T-1, n, n]
    ei = union_pattern(adj)
    coef = torch.stack([adj[3], adj[2], adj[1], adj[0]], dim=-1)[:, ei[0], ei[1]]   # [T-1, E, 4] (a,b,c,d)
    layers = [(lp.fusion, lp.weight, lp.bias, lp.norm_weight, lp.norm_bias) for lp in p.layers]
    for t in (0.3, 1.0, 2.7):
        ref = R.perm_equiv_vector_field(t, p.y0, R.CubicInterpolation(p.ts, p.coeffs_adj), p.layers)
        got = _sparse_vf64(t, p.y0, p.ts, ei[0], ei[1], coef, layers, n)
        assert rel_err(got, ref) < 1e-12, t


def _large_sparse_path(n, T, deg, seed, device):
    """about `deg` random edges per row + a unit self-loop, LogNormal weights, 10 % of the weights redrawn per knot (a redrawn
    edge is absent at that knot with probability 1/2), rows normalised per knot -> (edge_index, edge_weight [T, E])"""
    g = torch.Generator(device=device).manual_seed(seed)
    rows = torch.cat([torch.arange(n, device=device).repeat_interleave(deg), torch.arange(n, device=device)])
    cols = torch.cat([torch.randint(0, n, (n * deg,), generator=g, device=device), torch.arange(n, device=device)])
    E = rows.numel()
    w = torch.exp(torch.randn(E, generator=g, device=device))
    out = []
    for k in range(T):
        if k > 0:
            redraw = torch.rand(E, generator=g, device=device) < 0.10
            w = torch.where(redraw, torch.exp(torch.randn(E, generator=g, device=device)) * (torch.rand(E, generator=g, device=device) < 0.5), w)
        wk = torch.where(rows == cols, torch.ones_like(w), w)
        out.append(wk / torch.zeros(n, device=device).index_add_(0, rows, wk)[rows])
    return torch.stack([rows, cols]), torch.stack(out)


@pytest.mark.gpu
def test_sparse_control_past_the_dense_ceiling(cuda):
    """n = 65536, h = 64, L = 2, ~16 edges per row: one piece of dense planes would be 68.7 GB.  One evaluation + VJP against the fp64
    restatement (kink-aware rule for the cotangent), then a 2-step fixed solve forward + backward."""
    n, h, L, T = 65536, 64, 2, 3
    ei, w = _large_sparse_path(n, T, 16, 3, cuda)
    ts = torch.arange(T, dtype=torch.float32, device=cuda)
    sc = P.build_sparse_control(ts, ei, w, n)
    vf = P.PermEquivGraphVectorField(h, h, h, L, 0, n, key=6).to(cuda)
    g = torch.Generator(device=cuda).manual_seed(2)
    y0, gy = torch.randn((n, h), generator=g, device=cuda), torch.randn((n, h), generator=g, device=cuda)
    y = y0.clone().requires_grad_(True)
    t = 1.3
    dy = vf(t, y, sc)
    (dy * gy).sum().backward()
    # fp64 restatement on the same coefficients
    ent = sc.row_ptr[0].long()
    rows = torch.repeat_interleave(torch.arange(n, device=cuda), ent[1:] - ent[:-1]).cpu()
    cols = sc.col.long().cpu()
    layers = []
    for layer in vf.gnn_layers:
        cl = layer.conv_layer
        layers.append([x.detach().double().cpu().requires_grad_(True) for x in
                       (layer.fusion_params().reshape(8, 2), cl.linear.weight, cl.linear.bias, cl.norm.weight, cl.norm.bias)])
    y64 = y0.double().cpu().requires_grad_(True)
    ref = _sparse_vf64(t, y64, ts.double().cpu(), rows, cols, sc.coef.double().cpu(), layers, n)
    (ref * gy.double().cpu()).sum().backward()
    assert rel_err(dy.detach(), ref.detach()) < 2e-5
    err = (y.grad.double().cpu() - y64.grad).abs() / y64.grad.abs().max()
    bad_rows = int((err.max(dim=1).values > 5e-5).sum())
    print(f"\n[n={n}] dy {rel_err(dy.detach(), ref.detach()):.1e}  cotangent max {float(err.max()):.1e}  rows above 5e-5: {bad_rows}")
    assert float(err.flatten().median()) < 5e-6 and float(err.flatten().float().quantile(0.9)) < 5e-5
    assert bad_rows <= 0.15 * n and rel_err(y.grad, y64.grad) < 2e-2
    tol_p = 3e-4 if bad_rows == 0 else 5e-3
    for layer, ref_l in zip(vf.gnn_layers, layers):
        cl = layer.conv_layer
        got = [torch.cat([getattr(layer, f"param{i}").grad for i in range(1, 9)]).reshape(8, 2), cl.linear.weight.grad, cl.linear.bias.grad,
               cl.norm.weight.grad, cl.norm.bias.grad]
        for a, r in zip(got, ref_l):
            assert rel_err(a, r.grad) < tol_p
    # a fixed-step solve, forward + adjoint
    vf.zero_grad()
    y = y0.clone().requires_grad_(True)
    yT = P.diffeqsolve(P.ODETerm(vf), P.Tsit5(), 0.0, 2.0, 1.0, y, sc).ys[-1]
    (yT * gy).sum().backward()
    assert torch.isfinite(yT).all() and torch.isfinite(y.grad).all()
    assert all(torch.isfinite(q.grad).all() for q in vf.parameters())


# ---------------------------------------------------------------------------------------------------
# GPU 9: reproducibility and CUDA-graph replay
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_sparse_solve_is_reproducible_and_replays_as_a_cuda_graph(cuda):
    n, h, T, B = 1000, 64, 4, 2
    ts = torch.arange(T, dtype=torch.float32, device=cuda)
    A = _synth_batch(n, T, [5, 6], cuda)
    sc = P.build_sparse_control(ts, [_snapshot_edges(A[b])[0] for b in range(B)], [_snapshot_edges(A[b])[1] for b in range(B)], n)
    vf = P.PermEquivGraphVectorField(h, h, h, 3, 0, n, key=2).to(cuda)
    g = torch.Generator(device=cuda).manual_seed(3)
    y0, gy = torch.randn((B, n, h), generator=g, device=cuda), torch.randn((B, n, h), generator=g, device=cuda)
    params = list(vf.parameters())

    def step():
        for q in params:
            q.grad = None
        y = y0.detach().requires_grad_(True)
        yT = P.diffeqsolve(P.ODETerm(vf), P.Tsit5(), 0.0, 3.0, 0.5, y, sc, stepsize_controller=P.ConstantStepSize(),
                           saveat=P.SaveAt(t1=True)).ys[-1]
        (yT * gy).sum().backward()
        return yT.detach(), y.grad, torch.cat([q.grad.reshape(-1) for q in params])

    eager = [tuple(x.clone() for x in step()) for _ in range(2)]
    assert torch.equal(eager[0][0], eager[1][0]) and torch.equal(eager[0][1], eager[1][1])
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = step()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out[0], eager[0][0]) and torch.equal(out[1], eager[0][1])
    # the parameter gradients sum per-CTA partials with float atomics (as the dense path does): equal up to that order
    assert rel_err(out[2], eager[0][2]) < 1e-5
