"""The small-graph cluster kernels (k_small_fwd / k_small_vjp, csrc/peg_small.cuh) against the fp64 oracle.

They are the product default below n = 128 (and up to n = 256 with PEG_FLAG_FUSED_SMALL): a cluster of C CTAs owns one graph,
every phase deals its work items to the ranks in contiguous ranges, and `small_plan` (pegncde.cu) picks C in {16, 8, 4, 2, 1}
from the batch, the SM count and the item count of the last layer.  Up to n = 128 the interpolated adjacency A_s / A'_s stays in
shared memory ("resident"), above that the contraction streams the cubic planes ("streamed").  The tests here reach every C in
both modes, the shape edges (n = 1, L = 1, h = 128, L = 8, partial 64-column blocks, the largest n of each mode) and the
boundaries of the selection rule.

Every test first calls the C-ABI directly and counts launches: one evaluation on the small path is exactly one launch and its VJP
exactly two, while the per-operator path needs at least three.  `small_plan` falls back to the per-operator path silently, so a
test that did not count could pass without running the kernels it is about.  The workspace, dy, g_y and g_xdot are filled
with NaN before each call: a row that no rank writes, or scratch read before it is written, shows up as a non-finite output.
"""
import json
import math

import pytest
import torch

import perm_equiv_graph_neural_cdes_b200 as P
from perm_equiv_graph_neural_cdes_b200 import _lib
from oracle import reference_path as R
from tests.helpers import FUSED, device_model, per_operator, product_grads_as_oracle, rel_err, sparse_of_coeffs

pytestmark = pytest.mark.gpu
TOL_Y = 1e-4
TOL_G = 1e-3
B200_SMS = 148
LEAVES = ("fusion", "W", "b", "nw", "nb")


# ---------------------------------------------------------------------------------------------------
# mirror of small_plan (pegncde.cu) and of small_smem_floats (peg_small.cuh)
# ---------------------------------------------------------------------------------------------------
def small_smem_bytes(n, L):
    nv, n16 = (n + 3) // 4 * 4, (n + 15) // 16 * 16
    resident = 2 * n16 * (n16 + 1) + 4 if n <= 128 else 0
    return 4 * ((3 * L + 1) * nv + 4 * nv + n16 * 64 + 5632 + 5 * 64 + 160 + resident)


def small_plan(B, n, h, e, L, flags, sms, max_cluster=16, sparse=False):
    """(C, mode) of the small-graph kernels for this call, or None when it runs on the per-operator path.  max_cluster is 16 when
    the non-portable cluster-size opt-in succeeds on the device and 8 (the portable limit) when it does not."""
    if flags & (_lib.PEG_FLAG_NO_FUSED_SMALL | _lib.PEG_FLAG_DIRECTED) or sparse:
        return None
    max_n = 256 if flags & _lib.PEG_FLAG_FUSED_SMALL else 127
    if n > max_n or h > 128 or small_smem_bytes(n, L) > 220 * 1024:
        return None
    d_last = 2 * h * e if e > 0 else h
    items = math.ceil(n / 64) * math.ceil(d_last / 64)
    C = next(c for c in (16, 8, 4, 2, 1) if c <= max_cluster and ((B * c <= sms and c <= items) or c == 1))
    return C, ("resident" if n <= 128 else "streamed")


def flags_of(flags):
    """the PegDims flags device_model(flags=...) gives the vector field"""
    if flags is None:
        return _lib.PEG_FLAG_TENSOR_CORES
    if flags == FUSED:
        return _lib.PEG_FLAG_TENSOR_CORES | _lib.PEG_FLAG_FUSED_SMALL
    return per_operator(flags)


def plan_id(B, n, h, e, L, flags):
    C, mode = small_plan(B, n, h, e, L, flags_of(flags), B200_SMS)
    return f"C{C}-{mode}"


def device_sms(cuda):
    return torch.cuda.get_device_properties(cuda).multi_processor_count


# ---------------------------------------------------------------------------------------------------
# direct C-ABI calls with the launch-count witness and NaN sentinels
# ---------------------------------------------------------------------------------------------------
def setup(ps, cuda, flags=None, repeat=1, vf=None):
    """(vf, packed control, dims) for the batch of graphs ps (one parameter set, the first problem's), each repeated `repeat` times"""
    p0 = ps[0]
    if vf is None:
        vf, _, _ = device_model(p0, cuda, flags=flags)
    ts = p0.ts.to(torch.float32).to(cuda)

    def stack(coeffs):
        out = []
        for i in range(4):
            c = torch.stack([cs[i] for cs in coeffs]).to(torch.float32).to(cuda)
            out.append(c.repeat_interleave(repeat, dim=0) if repeat > 1 else c)
        return tuple(out)

    cadj = P.CubicInterpolation(ts, stack([p.coeffs_adj for p in ps]))
    cx = P.CubicInterpolation(ts, stack([p.x_coeffs for p in ps])) if p0.e > 0 else None
    pc = P.vector_field.resolve_control(cadj, cx, cuda)
    return vf, pc, vf.dims_for(pc, with_wrapper=p0.e > 0)


def evaluate(vf, pc, dims, t, y, g_dy):
    """pegncde_vf_fwd then pegncde_vf_vjp (with g_xdot when e > 0).  Returns dy, g_y, the flat parameter gradient, g_xdot and the
    launches of each call."""
    l = _lib.lib()
    st = torch.cuda.current_stream(y.device).cuda_stream
    flat = vf.checked_flat_params(dims).detach().contiguous()
    ctl = pc.struct()
    ws = torch.empty(l.pegncde_workspace_bytes(dims, _lib.PEG_WS_VF_VJP, 0), dtype=torch.uint8, device=y.device)
    nan = float("nan")
    ws.fill_(0xFF)
    dy = torch.full_like(y, nan)
    c0 = l.pegncde_launch_count()
    _lib.check(l.pegncde_vf_fwd(st, dims, ctl, flat.data_ptr(), float(t), y.data_ptr(), dy.data_ptr(), ws.data_ptr(), ws.numel()),
               "pegncde_vf_fwd")
    c1 = l.pegncde_launch_count()
    ws.fill_(0xFF)
    g_y = torch.full_like(y, nan)
    g_flat = torch.zeros_like(flat)
    g_xd = torch.full((dims.B, dims.n, 2 * dims.e), nan, device=y.device) if dims.e > 0 else None
    _lib.check(l.pegncde_vf_vjp(st, dims, ctl, flat.data_ptr(), float(t), y.data_ptr(), g_dy.data_ptr(), g_y.data_ptr(), g_flat.data_ptr(),
                                g_xd.data_ptr() if g_xd is not None else None, ws.data_ptr(), ws.numel()), "pegncde_vf_vjp")
    c2 = l.pegncde_launch_count()
    torch.cuda.synchronize()
    return dy, g_y, g_flat, g_xd, (c1 - c0, c2 - c1)


def assert_path(launches, small):
    fwd, vjp = launches
    if small:
        assert (fwd, vjp) == (1, 2), f"expected the small-graph kernels (1 + 2 launches), got {fwd} + {vjp}"
    else:
        assert fwd >= 3 and vjp >= 3, f"expected the per-operator path (>= 3 launches per call), got {fwd} + {vjp}"


def leaf_grads(vf, dims, g_flat):
    """the flat parameter gradient as (fusion, W, b, nw, nb) per layer, through the packing's own autograd"""
    vf.zero_grad(set_to_none=True)
    vf.checked_flat_params(dims).backward(g_flat)
    return [[g.detach().clone() for g in layer] for layer in product_grads_as_oracle(vf)]


def batch_inputs(ps, cuda, repeat=1):
    y = torch.stack([p.y0 for p in ps]).to(torch.float32).to(cuda)
    g = torch.stack([p.gyT for p in ps]).to(torch.float32).to(cuda)
    if repeat > 1:
        y, g = y.repeat_interleave(repeat, dim=0), g.repeat_interleave(repeat, dim=0)
    return y.contiguous(), g.contiguous()


# ---------------------------------------------------------------------------------------------------
# the fp64 oracle
# ---------------------------------------------------------------------------------------------------
def oracle_eval(p64, t):
    """dy, d<gyT, dy>/dy, the per-layer parameter leaves (with .grad) and the x coefficients (d, c, b, a) (with .grad) or None"""
    layers = R.params_to(p64.layers, requires_grad=True)
    y = p64.y0.clone().requires_grad_(True)
    ca = R.CubicInterpolation(p64.ts, p64.coeffs_adj)
    xs = None
    if p64.e > 0:
        xs = tuple(c.clone().requires_grad_(True) for c in p64.x_coeffs)
        dy = R.cde_wrapper_vector_field(t, y, ca, R.CubicInterpolation(p64.ts, xs), layers, p64.h, p64.e)
    else:
        dy = R.perm_equiv_vector_field(t, y, ca, layers)
    (dy * p64.gyT).sum().backward()
    return dy.detach(), y.grad, layers, xs


def xcoef_cotangent(p64, t, g_xd):
    """g_xdot [n, 2e] -> the cotangent of the x coefficients (d, c, b): X'(t) = b + 2 s c + 3 s^2 d on the piece that holds t"""
    iv, s = R.CubicInterpolation(p64.ts, p64.x_coeffs)._interpret_t(t)
    s = float(s)
    gx = g_xd.detach().double().cpu().reshape(p64.n, p64.e, 2)
    out = []
    for scale in (3.0 * s * s, 2.0 * s, 1.0):
        g = torch.zeros_like(p64.x_coeffs[0])
        g[iv] = scale * gx
        out.append(g)
    return out


def check_against_oracle(p64, t, dy, g_y, grads, g_xd, tol_p=2e-4):
    assert torch.isfinite(dy).all() and torch.isfinite(g_y).all(), "non-finite output: a row nobody wrote or uninitialised scratch"
    ref, ref_gy, layers, xs = oracle_eval(p64, t)
    assert rel_err(dy, ref) < 2e-5, ("dy", t, rel_err(dy, ref))
    assert rel_err(g_y, ref_gy) < 5e-5, ("g_y", t, rel_err(g_y, ref_gy))
    for l, (got, lp) in enumerate(zip(grads or [], layers)):
        for name, g, r in zip(LEAVES, got, lp.tensors()):
            assert rel_err(g, r.grad) < tol_p, (t, l, name, rel_err(g, r.grad))
    if xs is not None:
        assert torch.isfinite(g_xd).all()
        for name, g, r in zip("dcb", xcoef_cotangent(p64, t, g_xd), xs[:3]):
            assert rel_err(g, r.grad) < 2e-4, (t, "x coefficient " + name, rel_err(g, r.grad))


def times_of(p):
    t_lo, t_hi = float(p.ts[0]), float(p.ts[-1])
    return [t_lo + 0.37 * (t_hi - t_lo), float(p.ts[1]), t_lo, t_hi + 0.25]   # interior, exact knot, t0, past t1 (index clipping)


# ---------------------------------------------------------------------------------------------------
# 1. the mirror against the grid of the kernels that actually run
# ---------------------------------------------------------------------------------------------------
def kernel_grids(fn, path):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    prof.export_chrome_trace(str(path))
    events = json.loads(path.read_text())["traceEvents"]
    return {k: [e["args"]["grid"] for e in events if e.get("cat") == "kernel" and k in e.get("name", "")] for k in ("k_small_fwd", "k_small_vjp")}


def test_cluster_width_mirror_matches_the_launched_grid(cuda, tmp_path):
    """grid = B * C of k_small_fwd and k_small_vjp, as the profiler records it, for shapes the mirror gives different C.  The
    first shape settles whether the device took the non-portable 16-CTA cluster (C = 16) or not (C = 8)."""
    cases = [(1, 120, 64, 8, 3, None), (1, 60, 64, 4, 3, None), (1, 127, 128, 0, 3, None), (1, 100, 32, 0, 3, None),
             (50, 100, 32, 3, 3, None), (80, 256, 64, 2, 3, FUSED)]
    sms = device_sms(cuda)
    seen = []
    for k, (B, n, h, e, L, flags) in enumerate(cases):
        p = R.make_problem(n=n, h=h, e=e, L=L, T=4, t1=3, dt0=0.25, seed=3)
        vf, pc, dims = setup([p], cuda, flags, repeat=B)
        y, g = batch_inputs([p], cuda, repeat=B)
        out = {}
        grids = kernel_grids(lambda: out.setdefault("r", evaluate(vf, pc, dims, 1.3, y, g)), tmp_path / f"case{k}.json")
        assert_path(out["r"][4], True)
        # the evaluation, then the VJP: a forward over the first L - 1 layers and the backward kernel
        assert len(grids["k_small_fwd"]) == 2 and len(grids["k_small_vjp"]) == 1, grids
        assert all(gr[1:] == [1, 1] and gr[0] % B == 0 for gr in grids["k_small_fwd"] + grids["k_small_vjp"]), grids
        Cs = {gr[0] // B for gr in grids["k_small_fwd"] + grids["k_small_vjp"]}
        assert len(Cs) == 1, grids
        seen.append(Cs.pop())
    max_cluster = seen[0]
    print(f"\nn = 120, h = 64, e = 8, B = 1 runs with C = {max_cluster}; C seen per case: {seen}")
    assert max_cluster in (16, 8)
    for (B, n, h, e, L, flags), C in zip(cases, seen):
        assert small_plan(B, n, h, e, L, flags_of(flags), sms, max_cluster)[0] == C, (B, n, h, e, L, C)


# ---------------------------------------------------------------------------------------------------
# 2. shape matrix: one evaluation and its VJP against the fp64 oracle, on the small path and on the per-operator FFMA path
# ---------------------------------------------------------------------------------------------------
# (n, h, e, L, seed): what each covers is in the comment
SHAPES = [
    (1, 4, 0, 1, 1),        # one node, L = 1
    (2, 4, 1, 1, 1),        # L = 1 behind the CDE wrapper: the VJP's forward runs no layer
    (3, 8, 0, 2, 1),        # n < 4: rounding of the vector pitch
    (100, 32, 0, 3, 1),
    (127, 128, 0, 3, 1),    # largest n of the default rule; h = SG_MAX_DIN
    (60, 64, 4, 3, 1),
    (120, 64, 8, 3, 1),     # England width below n = 128: ~191 KB of shared memory per CTA
    (64, 128, 4, 8, 1),     # PEG_MAX_LAYERS
    (128, 32, 0, 2, 1),     # largest resident n (PEG_FLAG_FUSED_SMALL)
    (130, 16, 0, 2, 1),     # three row blocks on two ranks
    (256, 32, 0, 3, 1),     # four full row blocks
    (200, 20, 3, 2, 1),     # 52-row blocks, a 56-wide last column block, h not a multiple of 32
    (256, 64, 2, 3, 1),     # top of the fused range
    (255, 128, 1, 3, 1),    # h = 128, short last row block
]


def small_flags(n):
    return FUSED if n >= 128 else None


def shape_params():
    out = []
    for n, h, e, L, seed in SHAPES:
        sid = f"n{n}_h{h}_e{e}_L{L}"
        out.append(pytest.param(n, h, e, L, seed, small_flags(n), id=f"{sid}-{plan_id(1, n, h, e, L, small_flags(n))}"))
        out.append(pytest.param(n, h, e, L, seed, 0, id=f"{sid}-ffma"))
    return out


@pytest.mark.parametrize("n,h,e,L,seed,flags", shape_params())
def test_evaluation_and_vjp_against_fp64_oracle(cuda, n, h, e, L, seed, flags):
    p = R.make_problem(n=n, h=h, e=e, L=L, T=4, t1=3, dt0=0.25, seed=seed)
    p64 = R.problem_to(p, torch.float64)
    vf, pc, dims = setup([p], cuda, flags)
    small = flags != 0
    if small:
        assert small_plan(1, n, h, e, L, dims.flags, device_sms(cuda)) == small_plan(1, n, h, e, L, dims.flags, B200_SMS)
    y, g = batch_inputs([p], cuda)
    for t in times_of(p):
        dy, g_y, g_flat, g_xd, launches = evaluate(vf, pc, dims, t, y, g)
        assert_path(launches, small)
        check_against_oracle(p64, t, dy[0], g_y[0], leaf_grads(vf, dims, g_flat), None if g_xd is None else g_xd[0])


# ---------------------------------------------------------------------------------------------------
# 3. cluster-width invariance and batches
# ---------------------------------------------------------------------------------------------------
# No atomics touch dy, g_y or g_xdot, and every work item computes the same arithmetic whichever rank owns it: those outputs
# must be the same bits at every C and at every batch position.  The parameter gradients are atomicAdd sums (fusion scalars,
# RMSNorm affine, Linear weight and bias) whose order changes with C and from run to run; the fusion scalars' sums cancel, so
# their rounding relative to the leaf's largest entry can be far above fp32 epsilon.  On a B200 (1000 W) the worst leaf differed
# from B x the single graph's by 3.0e-5 (the n = 120 replicated batch, the same in each of five runs of this module) and from the
# sum of the graphs' by 1.5e-6; TOL_ATOMIC is ten times the former.  A work item dropped or counted twice moves a leaf by its
# whole share of the sum, 1/32 or more here, a hundred times TOL_ATOMIC.
TOL_ATOMIC = 3e-4


def _invariance_id(n, h, e, L, flags, batches):
    C = [small_plan(B, n, h, e, L, flags_of(flags), B200_SMS) for B in batches]
    return f"n{n}_h{h}_e{e}-{C[0][1]}-B{'.'.join(map(str, batches))}-C{'.'.join(str(c[0]) for c in C)}"


INVARIANCE = [(120, 64, 8, 3, None, (1, 10, 20, 40, 80)), (256, 64, 2, 3, FUSED, (1, 9, 80))]


@pytest.mark.parametrize("n,h,e,L,flags,batches", INVARIANCE, ids=[_invariance_id(*c) for c in INVARIANCE])
def test_every_cluster_width_gives_the_same_bits(cuda, n, h, e, L, flags, batches):
    """one graph replicated B times: every copy at every C gives the bits of the graph alone, the parameter gradient is B times
    the graph's"""
    p = R.make_problem(n=n, h=h, e=e, L=L, T=4, t1=3, dt0=0.25, seed=1)
    vf = None
    ref = None
    worst = 0.0
    for B in batches:
        vf, pc, dims = setup([p], cuda, flags, repeat=B, vf=vf)
        y, g = batch_inputs([p], cuda, repeat=B)
        dy, g_y, g_flat, g_xd, launches = evaluate(vf, pc, dims, 1.11, y, g)
        assert_path(launches, True)
        assert torch.isfinite(dy).all() and torch.isfinite(g_y).all() and (g_xd is None or torch.isfinite(g_xd).all())
        grads = leaf_grads(vf, dims, g_flat)
        if ref is None:
            ref = (dy[0], g_y[0], None if g_xd is None else g_xd[0], grads)
            continue
        for b in range(B):
            assert torch.equal(dy[b], ref[0]), (B, b, "dy")
            assert torch.equal(g_y[b], ref[1]), (B, b, "g_y")
            if g_xd is not None:
                assert torch.equal(g_xd[b], ref[2]), (B, b, "g_xdot")
        for l, (got, want) in enumerate(zip(grads, ref[3])):
            for name, a, r in zip(LEAVES, got, want):
                err = rel_err(a, B * r)
                worst = max(worst, err)
                assert err < TOL_ATOMIC, (B, l, name, err)
    print(f"\nparameter gradients against B x the single graph's, worst leaf: {worst:.1e}")


# (n, h, e, L, B, flags, seed of graph 0): the SIR benchmark shape (resident, C = 2 in the batch, C = 4 alone) and a streamed
# batch (C = 1 in the batch, C = 16 alone); every graph has its own control path, so a slip in a per-graph offset shows
DIFFERENT = [(100, 32, 3, 3, 50, None, 100), (256, 64, 2, 3, 80, FUSED, 200)]


@pytest.mark.parametrize("n,h,e,L,B,flags,seed", DIFFERENT,
                         ids=[f"n{c[0]}_h{c[1]}_e{c[2]}_B{c[4]}-{plan_id(c[4], *c[:4], c[5])}-alone-{plan_id(1, *c[:4], c[5])}" for c in DIFFERENT])
def test_batch_of_different_graphs(cuda, n, h, e, L, B, flags, seed):
    """The first, middle and last graph against the oracle; every graph against itself evaluated alone: dy, g_y and g_xdot bit
    for bit, the batch's parameter gradient = the sum of the graphs' within TOL_ATOMIC."""
    ps = [R.make_problem(n=n, h=h, e=e, L=L, T=4, t1=3, dt0=0.25, seed=seed + b) for b in range(B)]
    for q in ps[1:]:
        q.layers = ps[0].layers
    sms = device_sms(cuda)
    assert small_plan(B, n, h, e, L, flags_of(flags), sms) != small_plan(1, n, h, e, L, flags_of(flags), sms)
    t = 1.11
    vf, pc, dims = setup(ps, cuda, flags)
    y, g = batch_inputs(ps, cuda)
    dy, g_y, g_flat, g_xd, launches = evaluate(vf, pc, dims, t, y, g)
    assert_path(launches, True)
    batch_grads = leaf_grads(vf, dims, g_flat)
    for b in (0, B // 2, B - 1):
        check_against_oracle(R.problem_to(ps[b], torch.float64), t, dy[b], g_y[b], None, g_xd[b])   # parameters: summed over the batch
    acc = torch.zeros_like(g_flat)
    for b, q in enumerate(ps):
        _, pc1, dims1 = setup([q], cuda, vf=vf)
        y1, g1 = batch_inputs([q], cuda)
        dy1, g_y1, g_flat1, g_xd1, launches1 = evaluate(vf, pc1, dims1, t, y1, g1)
        assert_path(launches1, True)
        assert torch.equal(dy[b], dy1[0]), b
        assert torch.equal(g_y[b], g_y1[0]), b
        assert torch.equal(g_xd[b], g_xd1[0]), b
        acc += g_flat1
    worst = 0.0
    for l, (got, want) in enumerate(zip(batch_grads, leaf_grads(vf, dims, acc))):
        for name, a, r in zip(LEAVES, got, want):
            worst = max(worst, rel_err(a, r))
            assert rel_err(a, r) < TOL_ATOMIC, (l, name, rel_err(a, r))
    print(f"\nparameter gradients against the sum of the graphs', worst leaf: {worst:.1e}")


# ---------------------------------------------------------------------------------------------------
# 4. solves on the small path
# ---------------------------------------------------------------------------------------------------
SOLVES = [(127, 128, 0, 3, None), (120, 64, 8, 3, None), (256, 64, 2, 3, FUSED)]


@pytest.mark.parametrize("n,h,e,L,flags", SOLVES, ids=[f"n{c[0]}_h{c[1]}_e{c[2]}-{plan_id(1, *c)}" for c in SOLVES])
def test_fixed_step_solve_and_adjoint(cuda, n, h, e, L, flags):
    """diffeqsolve over [0, 3] at dt0 = 0.25 (12 steps) and its exact adjoint against the fp64 oracle: y(t1), dloss/dy0, every
    parameter leaf and (e > 0) the x coefficients.  With and without the stage store: y(t1) and dloss/dy0 bit for bit."""
    p = R.make_problem(n=n, h=h, e=e, L=L, T=4, t1=3, dt0=0.25, seed=1)
    vf, pc, dims = setup([p], cuda, flags)
    y, g = batch_inputs([p], cuda)
    assert_path(evaluate(vf, pc, dims, 0.5, y, g)[4], True)
    ts = p.ts.to(torch.float32).to(cuda)
    runs = []
    for store in (True, False):
        vf, _, _ = device_model(p, cuda, flags=flags)
        vf.store_stages = store
        cadj = P.CubicInterpolation(ts, tuple(c.to(cuda) for c in p.coeffs_adj))
        xco = tuple(c.to(cuda).requires_grad_(True) for c in p.x_coeffs) if e > 0 else None
        term = P.CDEWrapperVectorField(vf, h) if e > 0 else vf
        args = [cadj, P.CubicInterpolation(ts, xco)] if e > 0 else cadj
        y0 = p.y0.to(cuda).requires_grad_(True)
        sol = P.diffeqsolve(P.ODETerm(term), P.Tsit5(), 0.0, 3.0, 0.25, y0, args)
        assert sol.stats["num_steps"] == 12
        (sol.ys[-1] * p.gyT.to(cuda)).sum().backward()
        runs.append((sol.ys[-1].detach(), y0.grad, product_grads_as_oracle(vf), None if xco is None else [c.grad for c in xco]))
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
    p64 = R.problem_to(p, torch.float64)
    layers = R.params_to(p64.layers, requires_grad=True)
    x64 = tuple(c.clone().requires_grad_(True) for c in p64.x_coeffs) if e > 0 else None
    y64 = p64.y0.clone().requires_grad_(True)
    yT = R.solve_cde(p64.step_ts, p64.ts, p64.coeffs_adj, x64, y64, layers, h, e)
    (yT * p64.gyT).sum().backward()
    for yT_got, gy0, grads, xg in runs:
        assert rel_err(yT_got, yT) < TOL_Y, rel_err(yT_got, yT)
        assert rel_err(gy0, y64.grad) < TOL_G, rel_err(gy0, y64.grad)
        for l, (got, lp) in enumerate(zip(grads, layers)):
            for name, a, r in zip(LEAVES, got, lp.tensors()):
                assert rel_err(a, r.grad) < TOL_G, (l, name, rel_err(a, r.grad))
        if e > 0:
            for name, a, r in zip("dcb", xg[:3], x64[:3]):
                assert rel_err(a, r.grad) < TOL_G, ("x coefficient " + name, rel_err(a, r.grad))


def test_tsit5_step_and_error_estimate(cuda):
    """one Tsit5 step at n = 120, e = 8 (C = 16) against the oracle's stages"""
    p = R.make_problem(n=120, h=64, e=8, L=3, T=4, t1=3, dt0=0.25, seed=1)
    p64 = R.problem_to(p, torch.float64)
    vf, term, args = device_model(p, cuda)
    _, pc, dims = setup([p], cuda, vf=vf)
    y, g = batch_inputs([p], cuda)
    assert_path(evaluate(vf, pc, dims, 0.4, y, g)[4], True)
    t, dt = 0.4, 0.3
    y1, yerr, k7 = P.tsit5_step(P.ODETerm(term), t, dt, p.y0.to(cuda), args)
    ca, cx = R.CubicInterpolation(p64.ts, p64.coeffs_adj), R.CubicInterpolation(p64.ts, p64.x_coeffs)
    f = lambda tt, yy: R.cde_wrapper_vector_field(tt, yy, ca, cx, p64.layers, p64.h, p64.e)
    ks = [f(t, p64.y0)]
    for i in range(1, 7):
        ks.append(f(t + R.TSIT5_C[i] * dt, p64.y0 + dt * sum(ks[j] * R.TSIT5_A[i][j] for j in range(i))))
    y1_ref = p64.y0 + dt * sum(ks[j] * R.TSIT5_B[j] for j in range(6))
    err_ref = dt * sum(ks[j] * R.TSIT5_BERR[j] for j in range(7))
    assert rel_err(y1, y1_ref) < 2e-5
    assert rel_err(k7, ks[6]) < 5e-5
    assert rel_err(k7, f(t + dt, y1.cpu().double())) < 2e-6
    assert float((yerr.cpu().double() - err_ref).abs().max()) < 1e-5 * float(y1_ref.abs().max())


# ---------------------------------------------------------------------------------------------------
# 5. selection boundaries (the rule include/pegncde.h documents for PEG_FLAG_NO_FUSED_SMALL / PEG_FLAG_FUSED_SMALL)
# ---------------------------------------------------------------------------------------------------
BOUNDARIES = [
    pytest.param(127, 32, None, "dense", True, id="n127-default-small"),
    pytest.param(128, 32, None, "dense", False, id="n128-default-per-operator"),
    pytest.param(128, 32, FUSED, "dense", True, id="n128-fused-small"),
    pytest.param(256, 32, FUSED, "dense", True, id="n256-fused-small"),
    pytest.param(257, 32, FUSED, "dense", False, id="n257-fused-per-operator"),
    pytest.param(100, 132, None, "dense", False, id="n100_h132-per-operator"),
    pytest.param(100, 32, _lib.PEG_FLAG_TENSOR_CORES, "dense", False, id="n100-no-fused-small-per-operator"),
    pytest.param(100, 32, None, "directed", False, id="n100-directed-per-operator"),
    pytest.param(100, 32, None, "sparse", False, id="n100-sparse-per-operator"),
]
DIR_FIELDS = ("param1", "param2", "param3", "param4", "param4_prime", "param5", "param5_prime", "param6", "param6_prime", "param7", "param8")


@pytest.mark.parametrize("n,h,flags,kind,small", BOUNDARIES)
def test_selection_boundary(cuda, n, h, flags, kind, small):
    """which path one evaluation takes, by launch count, and that it matches the oracle either way (parameter leaves within 3e-4,
    the bound of the per-operator tensor-core tests)"""
    p = R.make_problem(n=n, h=h, e=0, L=2, T=4, t1=3, dt0=0.25, seed=1)
    p64 = R.problem_to(p, torch.float64)
    t = 1.11
    y, g = batch_inputs([p], cuda)
    if kind == "directed":
        vf = P.PermEquivDirGraphVectorField(h, h, h, 2, 0, n, key=4)
        with torch.no_grad():
            for mine, lp in zip(vf.gnn_layers, p.layers):
                mine.conv_layer.linear.weight.copy_(lp.weight); mine.conv_layer.linear.bias.copy_(lp.bias)
                mine.conv_layer.norm.weight.copy_(lp.norm_weight); mine.conv_layer.norm.bias.copy_(lp.norm_bias)
        fus64 = [torch.stack([getattr(m, f).detach().double() for f in DIR_FIELDS]) for m in vf.gnn_layers]
        vf, pc, dims = setup([p], cuda, vf=vf.to(cuda))
    else:
        vf, pc, dims = setup([p], cuda, flags)
    if kind == "sparse":
        pc = sparse_of_coeffs(p.ts.to(torch.float32).to(cuda), tuple(c.to(cuda) for c in p.coeffs_adj))
        dims = vf.dims_for(pc, with_wrapper=False)
    assert (small_plan(1, n, h, 0, 2, dims.flags, device_sms(cuda), sparse=kind == "sparse") is not None) == small
    dy, g_y, g_flat, _, launches = evaluate(vf, pc, dims, t, y, g)
    assert_path(launches, small)
    if kind == "directed":
        assert torch.isfinite(dy).all() and torch.isfinite(g_y).all()
        y64 = p64.y0.clone().requires_grad_(True)
        ref = R.perm_equiv_dir_vector_field(t, y64, R.CubicInterpolation(p64.ts, p64.coeffs_adj), p64.layers, fus64)
        (ref * p64.gyT).sum().backward()
        assert rel_err(dy[0], ref) < 2e-5
        assert rel_err(g_y[0], y64.grad) < 5e-5
        return
    check_against_oracle(p64, t, dy[0], g_y[0], leaf_grads(vf, dims, g_flat), None, tol_p=3e-4)
