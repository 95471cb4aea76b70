"""CPU: host logic of the product package and the C-ABI surface (no compute calls without a GPU)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import perm_equiv_graph_neural_cdes_b200 as P
from perm_equiv_graph_neural_cdes_b200 import _lib
from oracle import reference_path as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "pegncde.h")).read()
    declared = set(re.findall(r"\b(pegncde_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    l = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(l, name), name


def test_strerror_and_version():
    l = _lib.lib()
    assert b"sm_100a" in l.pegncde_version()
    assert l.pegncde_strerror(0) == b"ok"
    assert b"workspace" in l.pegncde_strerror(3)
    assert b"unknown" in l.pegncde_strerror(99)


@pytest.mark.parametrize("n,h,e,L", [(129, 64, 8, 3), (1000, 64, 16, 3), (100, 32, 3, 3), (400, 16, 0, 2)])
def test_param_count_matches_reference_pytree(n, h, e, L):
    d = _lib.PegDims(1, n, (n + 31) // 32 * 32, h, e, L, 4, 0)
    widths = R.layer_widths(h, L, e, e > 0)
    expect = sum(widths[i + 1] * widths[i] + widths[i + 1] + 2 * widths[i] + 16 for i in range(L))
    assert _lib.lib().pegncde_param_count(d) == expect
    vf = P.PermEquivGraphVectorField(h, h, widths[-1], L, e, n, key=0)
    assert vf.flat_params().numel() == expect
    off = (ctypes.c_int64 * (5 * L))()
    assert _lib.lib().pegncde_param_offsets(d, off) == 0
    assert off[0] == 0 and off[4] == widths[1] * widths[0] + widths[1] + 2 * widths[0]


def test_bad_dims_are_rejected_without_touching_the_gpu():
    l = _lib.lib()
    good = dict(B=1, n=10, ldn=32, h=8, e=0, L=2, T=4, flags=0)
    for k, v in [("ldn", 10), ("ldn", 12), ("ldn", 64), ("h", 6), ("h", 512), ("L", 0), ("L", 9), ("T", 1), ("B", 0), ("n", 0)]:
        d = _lib.PegDims(**{**good, k: v})
        assert l.pegncde_param_count(d) == 0, (k, v)
        assert l.pegncde_workspace_bytes(d, 0, 1) == 0
    assert l.pegncde_workspace_bytes(_lib.PegDims(**good), 99, 1) == 0
    # a compute entry point validates before any CUDA call
    rc = l.pegncde_solve_fwd(None, _lib.PegDims(**{**good, "h": 6}), _lib.PegControl(), None, None, 1, None, None, None, None, None, 0)
    assert rc == 1
    rc = l.pegncde_solve_fwd(None, _lib.PegDims(**good), _lib.PegControl(), None, None, 1, None, None, None, None, None, 0)
    assert rc == 2  # null pointers


def test_workspace_grows_with_problem():
    l = _lib.lib()
    a = l.pegncde_workspace_bytes(_lib.PegDims(1, 100, 128, 32, 3, 3, 12, 0), _lib.PEG_WS_SOLVE_BWD, 10)
    b = l.pegncde_workspace_bytes(_lib.PegDims(4, 100, 128, 32, 3, 3, 12, 0), _lib.PEG_WS_SOLVE_BWD, 10)
    assert 0 < a < b


def test_step_table_matches_oracle():
    for rule in ("state", "prev_diff"):
        for (t1, dt) in [(3, 0.1), (1, 0.1), (1, 0.01), (8, 0.1), (2, 0.01), (5, 0.3)]:
            assert np.array_equal(P.constant_step_table(0.0, t1, dt, rule), R.constant_step_table(0.0, t1, dt, rule))


def test_hermite_coefficients_match_oracle():
    ts = torch.tensor([0.0, 0.5, 1.5, 2.0])
    ys = torch.randn(4, 5, 5, 2, generator=torch.Generator().manual_seed(0))
    for a, b in zip(P.backward_hermite_coefficients(ts, ys), R.backward_hermite_coefficients(ts, ys)):
        assert torch.equal(a, b)


def test_flat_params_layout_and_grad_routing():
    vf = P.PermEquivGraphVectorField(8, 8, 8, 2, 0, 5, key=3)
    flat = vf.flat_params()
    l0 = vf.gnn_layers[0]
    assert torch.equal(flat[:64], l0.conv_layer.linear.weight.reshape(-1))
    assert torch.equal(flat[64 + 8 + 16: 64 + 8 + 16 + 2], l0.param1)
    (flat * torch.arange(flat.numel())).sum().backward()
    assert torch.equal(l0.param2.grad, torch.tensor([64 + 8 + 16 + 2.0, 64 + 8 + 16 + 3.0]))


def test_cpu_tensors_are_refused():
    vf = P.PermEquivGraphVectorField(8, 8, 8, 2, 0, 5, key=3)
    ts = torch.arange(4.0)
    A = torch.rand(4, 5, 5)
    co = R.reference_layout_coeffs(ts, A)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        P.diffeqsolve(P.ODETerm(vf), P.Tsit5(), 0.0, 3.0, 0.1, torch.zeros(5, 8), P.CubicInterpolation(ts, co))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "perm_equiv_graph_neural_cdes_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cc", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("load_oracle_layers", ""), os.path.join(dirpath, f)


def test_tiled_layout_is_a_permutation_with_contiguous_warp_loads():
    """The 32x32-tiled plane layout: a bijection onto [0, 4*npad^2), 16-KB tiles, and every (g, plane, m) warp
    row of 32 lanes x 4 floats is 512 contiguous bytes."""
    from perm_equiv_graph_neural_cdes_b200.control import tiled_offsets

    npad = 96
    off = tiled_offsets(npad)
    assert sorted(off.reshape(-1).tolist()) == list(range(4 * npad * npad))
    tile = off[:, 32:64, 64:96]  # tile (1, 2)
    assert int(tile.min()) == (1 * 3 + 2) * 4096 and int(tile.max()) == (1 * 3 + 2) * 4096 + 4095
    # elements of one micro-tile row are 4 consecutive floats
    assert torch.equal(off[2, 5, 8:12] - off[2, 5, 8], torch.arange(4))


# ---- adaptive path: controller / dense-output host logic against the oracle's restatement ----
def test_pid_controller_matches_oracle_restatement():
    c = P.PIDController(rtol=1e-3, atol=1e-6)
    for err in [0.0, 1e-12, 1e-4, 0.3, 0.999999, 1.0, 1.0000001, 1.7, 50.0, 1e9, float("inf")]:
        for dt in [1e-4, 0.037, 0.5]:
            assert c.adapt(err, np.float32(dt)) == R.pid_adapt(err, np.float32(dt)), (err, dt)
    keep, dt = c.adapt(0.5, np.float32(0.1))
    assert keep and dt >= np.float32(0.1)          # an accepted step never shrinks the next one
    keep, dt = c.adapt(1e6, np.float32(0.1))
    assert not keep and np.isclose(dt, 0.02)       # factormin
    keep, dt = c.adapt(1e-30, np.float32(0.1))
    assert keep and np.isclose(dt, 1.0)            # factormax
    with pytest.raises(NotImplementedError):
        P.PIDController(1e-3, 1e-6, pcoeff=0.4)


def test_clip_to_end_matches_oracle_restatement():
    for tprev, tnext, keep in [(0.0, 0.5, True), (4.9, 5.0000005, True), (4.9, 4.9999995, True), (4.0, 5.2, False), (4.0, 4.5, False)]:
        assert P.clip_to_end(tprev, tnext, 5.0, keep) == R.clip_to_end(tprev, tnext, 5.0, keep)
    assert P.clip_to_end(4.0, 5.2, 5.0, False) == np.float32(4.5)
    assert P.clip_to_end(4.9, 4.9999995, 5.0, True) == np.float32(5.0)


def test_dense_output_weights():
    """Host helper of the C-ABI (expanded Horner form) against the oracle's factored form (diffrax's)."""
    for theta in np.linspace(0.0, 1.0, 21):
        assert np.allclose(P.dense_weights(theta), np.asarray(R.tsit5_dense_weights(theta)), atol=2e-6), theta
    assert np.allclose(P.dense_weights(1.0), np.asarray(R.TSIT5_B), atol=1e-7)
    assert np.allclose(P.dense_weights(0.0), 0.0)


def test_oracle_adaptive_solver_on_a_known_ode():
    """Restated PID + dense output: y' = -(1 + sin(t)/2) y has y = exp(-(t + (1 - cos t)/2))."""
    f = lambda t, y: -y * (1.0 + 0.5 * np.sin(t))
    ts = np.linspace(0, 5, 11).astype(np.float32)
    ys, table, stats = R.tsit5_solve_adaptive(f, torch.ones(3, 2, dtype=torch.float64), 0.0, 5.0, save_ts=ts)
    exact = np.exp(-(ts + 0.5 * (1 - np.cos(ts))))
    assert np.abs(ys[:, 0, 0].numpy() - exact).max() < 2e-3
    assert table[0] == 0 and table[-1] == 5 and np.all(np.diff(table) > 0)
    assert stats["num_accepted_steps"] == len(table) - 1
    # forcing the accepted table reproduces the run
    ys2, table2, _ = R.tsit5_solve_adaptive(f, torch.ones(3, 2, dtype=torch.float64), 0.0, 5.0, save_ts=ts, forced_steps=table)
    assert np.array_equal(table, table2) and torch.allclose(ys, ys2, atol=1e-12)


def test_new_entry_points_validate_before_touching_the_gpu():
    """build_adj / tsit5_dense / scaled_sumsq / step_fwd / solve_bwd: bad dims -> 1, missing pointers -> 2 (no CUDA call made)."""
    l = _lib.lib()
    good = _lib.PegDims(1, 10, 32, 8, 0, 2, 4, 0)
    bad = _lib.PegDims(1, 10, 32, 6, 0, 2, 4, 0)
    assert l.pegncde_build_adj(None, bad, None, None, None, None, None, None, None) in (1, 2)
    assert l.pegncde_build_adj(None, good, None, None, None, None, None, None, None) == 2
    assert l.pegncde_tsit5_dense(None, bad, 0.1, 0.5, None, None, None, None, None) == 1
    assert l.pegncde_tsit5_dense(None, good, 0.1, 0.5, None, None, None, None, None) == 2
    assert l.pegncde_scaled_sumsq(None, bad, None, None, None, None, 1e-3, 1e-6, None) == 1
    assert l.pegncde_scaled_sumsq(None, good, None, None, None, None, 1e-3, 1e-6, None) == 2
    assert l.pegncde_step_fwd(None, good, _lib.PegControl(), None, 0.0, 0.1, None, None, 0, None, None, None, None, None, 0) == 2
    assert l.pegncde_solve_bwd(None, good, _lib.PegControl(), None, None, 1, None, None, None, None, None, None, None, None, None, 0) == 2
    # g_xcoef without a node-signal control is a dimension error, not a crash (needs every other pointer non-null to reach the check)
    w = (ctypes.c_float * 7)()
    l.pegncde_tsit5_dense_weights(0.5, w)
    assert abs(sum(w) - 0.5) < 1e-6      # sum_i b_i(theta) = theta (the interpolant reproduces y' = const exactly)


def test_packed_control_select_is_a_view():
    """PackedControl.select(b) (adaptive solves step each trajectory alone) must not copy: same storage, B = 1."""
    pc = P.PackedControl.__new__(P.PackedControl)
    pc.B, pc.n, pc.T, pc.e, pc.ldn = 3, 5, 4, 0, 32
    for name, shape in (("ts", (3, 4)), ("adj_coef", (3, 3, 4 * 32 * 32)), ("adj_rowsum", (3, 3, 4, 5)), ("adj_diag", (3, 3, 4, 5)),
                        ("adj_total", (3, 3, 4)), ("tch_coef", (3, 3, 3, 5)), ("adj_absmax", (3, 3, 4))):
        setattr(pc, name, torch.zeros(shape))
    pc.x_coef = None
    pc._adj = {"colsum": None, "pending": None, "host_ts": None}
    v = pc.select(1)
    assert v.B == 1 and v.n == 5 and v.adj_coef.data_ptr() == pc.adj_coef[1].data_ptr() and v.ts.shape == (1, 4)
    assert v.dims(8, 2).B == 1


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (CPU arm, no GPU needed): one JSON line with the contract's keys, config matching our arm's."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--workload", "england", "--steps", "1",
                          "--warmup", "1", "--cpu-sample-steps", "1"], capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["value"] > 0 and line["higher_is_better"] is True
    assert line["config"]["workload"] == "england" and line["config"]["n"] == 129 and line["config"]["solver_steps"] == 30
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_bench_reference_arm_is_silent_on_nonzero_ranks():
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--workload", "england", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=root, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_bench_dump_outputs_samples_past_the_budget_at_fixed_positions(tmp_path):
    """`bench.py --dump-outputs` writes float32 arrays; past the byte budget every array keeps the same share of its elements, at
    positions that depend only on the array's size, so two runs (or two builds) write comparable samples."""
    import bench

    a = torch.arange(1000, dtype=torch.float32)
    b = torch.arange(3000, dtype=torch.float64).reshape(30, 100)
    for d in ("x", "y"):
        bench.dump_outputs(str(tmp_path / d), {"a": a, "b": b}, budget=1600)
    xa, xb = np.load(tmp_path / "x" / "a.npy"), np.load(tmp_path / "x" / "b.npy")
    assert xa.dtype == xb.dtype == np.float32 and xa.shape == (100,) and xb.shape == (300,)
    assert np.array_equal(xa, np.load(tmp_path / "y" / "a.npy")) and np.array_equal(xb, np.load(tmp_path / "y" / "b.npy"))
    assert np.all(np.diff(xa) > 0) and xa[-1] < 1000 and np.all(xa == np.round(xa))   # a sorted subset of the elements
    bench.dump_outputs(str(tmp_path / "z"), {"b": b}, budget=4 * 3000)                # within the budget: whole, shape kept
    assert np.array_equal(np.load(tmp_path / "z" / "b.npy"), b.numpy().astype(np.float32))


def test_bench_rejects_zero_timed_steps():
    import subprocess
    import sys

    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode != 0 and "--steps" in out.stderr


def test_c_abi_dense_weights_satisfy_the_continuous_order_conditions():
    """pegncde_tsit5_dense_weights (fp32, expanded Horner form) against the order-4 conditions of the interpolant -- a check that
    does not go through the oracle's (factored) restatement of the same polynomials."""
    from tests.test_oracle import _tsit5_trees

    A, c, trees = _tsit5_trees()
    for theta in (0.0, 0.1, 0.35, 0.5, 0.77, 1.0):
        w = P.dense_weights(theta).astype(np.float64)
        for order, phi, gamma in trees:
            if order <= 4:
                assert abs(w @ phi - theta**order / gamma) < 3e-6, (theta, order, gamma)


def test_jax_ffi_shim_type_checks_against_the_c_abi():
    """jax_ffi/pegncde_ffi.cc cannot be built for real here (no XLA FFI headers), but it must stay consistent with
    include/pegncde.h: compiled (syntax + types only) against tests/mock_xla_ffi, whose XLA_FFI_DEFINE_HANDLER_SYMBOL
    static_asserts that every handler is invocable with exactly the types its binding declares."""
    import shutil
    import subprocess

    if shutil.which("g++") is None:
        pytest.skip("no g++")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    if not os.path.exists(os.path.join(cuda_inc, "cuda_runtime_api.h")):
        pytest.skip("no CUDA headers")
    src = os.path.join(root, "perm_equiv_graph_neural_cdes_b200", "jax_ffi", "pegncde_ffi.cc")
    cmd = ["g++", "-std=c++17", "-fsyntax-only", "-Wall", "-I" + os.path.join(root, "tests", "mock_xla_ffi"), "-I" + os.path.join(root, "include"),
           "-I" + cuda_inc, src]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-3000:]
    # ... and the mock does reject a binding that disagrees with its handler
    bad = open(src).read().replace('.Attr<int32_t>("B")', '.Attr<float>("B")', 1)
    assert bad != open(src).read()
    out = subprocess.run(cmd[:-1] + ["-x", "c++", "-"], input=bad, capture_output=True, text=True, timeout=300)
    assert out.returncode != 0 and "does not match its binding" in out.stderr


def test_jax_wrapper_operands_match_the_shim_bindings(monkeypatch):
    """jax_ffi/pegncde_jax.py cannot run for real here (no jax).  Imported on recording stand-ins for jax / equinox / diffrax, every
    ffi_call it makes -- control pre-pass, the vector field and its VJP (through the Equinox module), the whole solve and its adjoint
    (through fused_diffeqsolve with the diffrax call-site signature) -- must hand the handler exactly as many operands / results /
    attributes as the binding in pegncde_ffi.cc declares, with vmap_method="broadcast_all"."""
    import importlib.util
    import sys
    import types

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cc = open(os.path.join(root, "perm_equiv_graph_neural_cdes_b200", "jax_ffi", "pegncde_ffi.cc")).read()
    dim_attrs = "".join(f'.Attr<int32_t>("{k}")' for k in ("B", "n", "h", "e", "L", "T", "flags"))
    cc = cc.replace(".PEG_DIM_ATTRS()", dim_attrs).replace(".PEG_CONTROL_ARGS()", ".Arg<x>()" * 9)
    bindings = {}
    for m in re.finditer(r"XLA_FFI_DEFINE_HANDLER_SYMBOL\((\w+),\s*\w+,(.*?)\);", cc, flags=re.S):
        body = m.group(2)
        bindings[m.group(1)] = (body.count(".Arg<"), body.count(".Ret<"), sorted(re.findall(r'\.Attr<[^>]*>+\("(\w+)"\)', body)))
    handlers = {"PegSolveFwd", "PegSolveBwd", "PegPackAdj", "PegPackX", "PegVfFwd", "PegVfVjp", "PegStepFwd"}
    assert set(bindings) == handlers

    calls, targets = [], {}

    class Struct:
        def __init__(self, shape, dtype):
            self.shape, self.dtype = tuple(shape), dtype

    def ffi_call(name, out_types, vmap_method=None):
        assert vmap_method == "broadcast_all"      # the batching rule: one custom call for the whole jax.vmap batch

        def run(*args, **attrs):
            calls.append((name, len(args), len(out_types), sorted(attrs)))
            return tuple(np.zeros(o.shape, o.dtype) for o in out_types)
        return run

    jax = types.ModuleType("jax")
    jnp = types.ModuleType("jax.numpy")
    for nm in ("asarray", "zeros", "zeros_like", "broadcast_to", "concatenate", "ndim", "float32", "uint8"):
        setattr(jnp, nm, getattr(np, nm))
    jax.numpy = jnp
    jax.ShapeDtypeStruct = Struct
    jax.ffi = types.SimpleNamespace(register_ffi_target=lambda name, capsule, platform=None: targets.__setitem__(name, capsule),
                                    pycapsule=lambda sym: sym, ffi_call=ffi_call)
    jax.tree_util = types.SimpleNamespace(tree_map=lambda f, t: tuple(f(x) for x in t))

    class custom_vjp:
        def __init__(self, fn):
            self.fn = fn

        def defvjp(self, fwd, bwd):
            self.fwd, self.bwd = fwd, bwd

        def __call__(self, *a):
            out, self.res = self.fwd(*a)      # run the forward rule, keep the residuals so the test can drive the backward rule
            return out

    jax.custom_vjp = custom_vjp
    eqx = types.ModuleType("equinox")
    eqx.Module = object
    eqx.field = lambda **k: None
    dfx = types.ModuleType("diffrax")
    for nm in ("ConstantStepSize", "Tsit5", "PIDController"):
        setattr(dfx, nm, type(nm, (), {}))
    dfx.SaveAt = type("SaveAt", (), {"__init__": lambda self, t1=False, steps=False, ts=None: self.__dict__.update(t1=t1, steps=steps, ts=ts)})
    dfx.ODETerm = type("ODETerm", (), {"__init__": lambda self, vector_field: setattr(self, "vector_field", vector_field)})
    dfx.diffeqsolve = lambda *a, **k: (_ for _ in ()).throw(AssertionError("the fused combination must not fall back to diffrax"))
    for name, mod_ in (("jax", jax), ("jax.numpy", jnp), ("equinox", eqx), ("diffrax", dfx)):
        monkeypatch.setitem(sys.modules, name, mod_)
    real_cdll = ctypes.CDLL
    monkeypatch.setattr(ctypes, "CDLL", lambda path, *a, **k: types.SimpleNamespace(**{h: h for h in handlers})
                        if str(path).endswith("libpegncde_ffi.so") else real_cdll(path, *a, **k))
    spec = importlib.util.spec_from_file_location("pegncde_jax_under_test", os.path.join(root, "perm_equiv_graph_neural_cdes_b200", "jax_ffi", "pegncde_jax.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    assert set(targets.values()) == handlers and targets["peg_vf_fwd"] == "PegVfFwd" and targets["peg_step_fwd"] == "PegStepFwd"

    f = lambda *s: np.zeros(s, np.float32)
    n, h, e, L, T, B = 40, 8, 3, 2, 4, 2
    pc = mod.fused_control(np.arange(T), [f(B, T - 1, n, n, 2)] * 4, [f(B, T - 1, n, e, 2)] * 4, hidden_dim=h, num_layers=L)
    control = pc.control
    assert pc.dims == dict(B=B, n=n, h=h, e=e, L=L, T=T, flags=1)
    assert len(control) == 8 and control[0].shape == (B, T) and control[1].shape == (B, T - 1, 4 * 64 * 64) and control[6].shape == (B, T - 1, 3, n, 2 * e)
    assert control[7].shape == (B, T - 1, 4)

    # the Equinox module: leaves built by the (stand-in) reference class, __call__ = peg_vf_fwd, its VJP = peg_vf_vjp
    def ref_layer(din, dout):
        cl = types.SimpleNamespace(linear=types.SimpleNamespace(weight=f(dout, din), bias=f(dout)), norm=types.SimpleNamespace(weight=f(din), bias=f(din)))
        return types.SimpleNamespace(conv_layer=cl, **{f"param{i}": f(2) for i in range(1, 9)})
    ref_cls = lambda **kw: types.SimpleNamespace(gnn_layers=[ref_layer(h, h), ref_layer(h, 2 * h * e)])
    vf = mod.FusedPermEquivGraphVectorField(h, h, 2 * h * e, L, e, n, key=0, reference_cls=ref_cls)
    nparams = mod.pack_params(vf).shape[0]
    assert nparams == _lib.lib().pegncde_param_count(_lib.PegDims(B, n, 64, h, e, L, T, 1))
    dy = vf(0.5, f(B, n, h), [pc])
    assert dy.shape == (B, n, h) and vf(0.5, f(n, h), pc).shape == (n, h)

    # the diffrax call site of pgt_graph_neural_cde.py:119-129
    sol = mod.fused_diffeqsolve(terms=dfx.ODETerm(types.SimpleNamespace(vector_field=vf)), solver=dfx.Tsit5(), t0=0.0, t1=3.0, dt0=0.1, y0=f(B, n, h),
                                args=[pc, None], stepsize_controller=dfx.ConstantStepSize(), saveat=dfx.SaveAt(t1=True))
    assert sol.ys.shape == (1, B, n, h) and sol.stats["num_steps"] == 30
    solve = mod.make_fused_solve(pc.dims, np.linspace(0, 3, 31))
    y_ckpt = solve(f(nparams), control, f(B, n, h))
    assert y_ckpt.shape == (31, B, n, h)
    g_params, g_control, g_y0 = solve.bwd(solve.res, np.zeros_like(y_ckpt))
    assert g_params.shape == (nparams,) and g_y0.shape == (B, n, h) and len(g_control) == 8
    # backward rule of the vector field
    vfun = mod.make_fused_vf(pc.dims)
    seen_before = len(calls)
    vfun(0.25, f(nparams), control, f(B, n, h))
    assert calls[seen_before][0] == "peg_vf_fwd"
    seen = {}
    for name, nargs, nouts, attrs in calls:
        seen[targets[name]] = (nargs, nouts, attrs)
    # drive the VJP rule of the vector field and the step handler's operand list by hand (no tracer here)
    mod._call("peg_vf_vjp", (Struct((B, n, h), np.float32), Struct((nparams,), np.float32), Struct((16,), np.uint8)), f(nparams), *control, f(B, n, h), f(B, n, h),
              t=np.float32(0.1), **mod._attrs(pc.dims))
    mod._call("peg_step_fwd", tuple(Struct((B, n, h), np.float32) for _ in range(4)) + (Struct((5, B, n, h), np.float32), Struct((16,), np.uint8)),
              f(nparams), *control, f(B, n, h), f(B, n, h), t=np.float32(0.1), dt=np.float32(0.05), k1_valid=np.int32(1), **mod._attrs(pc.dims))
    for name, nargs, nouts, attrs in calls:
        seen[targets[name]] = (nargs, nouts, attrs)
    assert seen == bindings, (seen, bindings)


def test_integration_doc_quotes_the_committed_file():
    """INTEGRATION.md's reference-side "after" snippet is the literal body of jax_ffi/reference_integration.py."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    body = open(os.path.join(root, "perm_equiv_graph_neural_cdes_b200", "jax_ffi", "reference_integration.py")).read()
    code = body[body.index("import diffrax"):].rstrip("\n")
    doc = open(os.path.join(root, "INTEGRATION.md")).read()
    assert code in doc
    # and the file is valid Python (it cannot be imported here: jax / diffrax / the reference tree are absent)
    compile(body, "reference_integration.py", "exec")


def test_ctypes_mirror_has_the_layout_and_flag_values_of_the_header(tmp_path):
    """Every struct of include/pegncde.h: size and the offset of every field as gcc lays them out == the ctypes mirror in _lib.py
    (a field added to one side only would shift everything behind it silently); same for the PEG_FLAG_* / PEG_WS_* values."""
    import subprocess

    from perm_equiv_graph_neural_cdes_b200 import _lib

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    structs = {"PegDims": _lib.PegDims, "PegShard": _lib.PegShard, "PegControl": _lib.PegControl, "PegAdaptState": _lib.PegAdaptState}
    enums = [k for k in dir(_lib) if k.startswith(("PEG_FLAG_", "PEG_WS_"))]
    assert "PEG_FLAG_FUSED_SMALL" in enums and "PEG_WS_SOLVE_BWD" in enums
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "pegncde.h"', 'int main(void) {']
    for name, cls in structs.items():
        lines.append(f'  printf("{name} %zu\\n", sizeof({name}));')
        for field, _ in cls._fields_:
            lines.append(f'  printf("{name}.{field} %zu\\n", offsetof({name}, {field}));')
    for k in enums:
        lines.append(f'  printf("{k} %d\\n", (int){k});')
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for name, cls in structs.items():
        assert int(got[name]) == ctypes.sizeof(cls), name
        for field, _ in cls._fields_:
            assert int(got[f"{name}.{field}"]) == getattr(cls, field).offset, (name, field)
    for k in enums:
        assert int(got[k]) == getattr(_lib, k), k
