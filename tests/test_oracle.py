"""CPU: the oracle against the committed goldens and against the mathematical identities the CUDA
path relies on (matrix-free fusion, permutation equivariance, Hermite interpolation properties)."""
import os

import numpy as np
import pytest
import torch

from oracle import reference_path as R
from oracle.make_goldens import input_checksum
from tests.helpers import GOLDEN_CASES

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("name", ["tiny_nocontrol", "tiny_control", "ragged_n"])
def test_oracle_reproduces_goldens(name):
    g = np.load(os.path.join(GOLD, f"{name}.npz"))
    p = R.make_problem(**GOLDEN_CASES[name])
    assert abs(input_checksum(p) - float(g["in_checksum"])) < 1e-6 * max(1.0, abs(float(g["in_checksum"])))
    yT, gy0, grads = R.run_forward_backward(R.problem_to(p, torch.float64))
    assert np.allclose(yT.numpy(), g["yT64"], rtol=0, atol=1e-10)
    assert np.allclose(gy0.numpy(), g["gy0_64"], rtol=0, atol=1e-9)
    flat = np.concatenate([t.numpy().reshape(-1) for layer in grads for t in layer])
    assert np.allclose(flat, g["gparams64"], rtol=0, atol=1e-8)
    assert len(p.step_ts) - 1 == int(g["steps"])


def test_goldens_are_well_conditioned():
    for name in GOLDEN_CASES:
        g = np.load(os.path.join(GOLD, f"{name}.npz"))
        assert float(g["rel32"]) < 5e-5, (name, float(g["rel32"]))


def test_matrix_free_identity():
    """(I + Abar) M == M + E M + G^T M + v*M + r (1^T M) + 1 (c^T M) + kappa 1 (1^T M)  (SURVEY Q11)."""
    torch.manual_seed(0)
    n, d = 23, 7
    A = torch.randn(n, n, dtype=torch.float64)
    D = torch.randn(n, n, dtype=torch.float64)
    p = torch.randn(8, 2, dtype=torch.float64) / 3
    M = torch.randn(n, d, dtype=torch.float64)
    ref = M + R.fusion(A, D, p) @ M
    E = (1 + p[0, 0]) * A + (1 + p[0, 1]) * D
    G = p[1, 0] * A + p[1, 1] * D
    rA, rD = A.sum(1), D.sum(1)
    v = p[2, 0] * A.diag() + p[2, 1] * D.diag() + (p[5, 0] * rA + p[5, 1] * rD) / n + (p[7, 0] * A.sum() + p[7, 1] * D.sum()) / n**2
    r = (p[3, 0] * rA + p[3, 1] * rD) / n
    c = (p[4, 0] * rA + p[4, 1] * rD) / n
    kappa = (p[6, 0] + p[6, 1]) * A.sum() / n**2  # reference quirk: both coefficients use sum(A)
    s = M.sum(0, keepdim=True)
    mf = M + E @ M + G.t() @ M + v[:, None] * M + r[:, None] * s + (c @ M)[None, :] + kappa * s
    assert torch.allclose(ref, mf, atol=1e-12)


def test_permutation_equivariance():
    """f(P Z, P A P^T) = P f(Z, A) for the undirected layer stack."""
    p = R.problem_to(R.make_problem(n=15, h=8, e=2, L=3, T=4, t1=3, dt0=0.1, seed=2), torch.float64)
    perm = torch.randperm(p.n, generator=torch.Generator().manual_seed(1))
    ca = R.CubicInterpolation(p.ts, p.coeffs_adj)
    cx = R.CubicInterpolation(p.ts, p.x_coeffs)
    t = 1.37
    out = R.cde_wrapper_vector_field(t, p.y0, ca, cx, p.layers, p.h, p.e)
    cap = R.CubicInterpolation(p.ts, tuple(c[:, perm][:, :, perm] for c in p.coeffs_adj))
    cxp = R.CubicInterpolation(p.ts, tuple(c[:, perm] for c in p.x_coeffs))
    outp = R.cde_wrapper_vector_field(t, p.y0[perm], cap, cxp, p.layers, p.h, p.e)
    assert torch.allclose(outp, out[perm], atol=1e-10)


def test_backward_hermite_interpolates_knots_and_is_c1():
    ts = torch.tensor([0.0, 0.7, 1.0, 2.5, 3.0], dtype=torch.float64)
    ys = torch.randn(5, 3, dtype=torch.float64, generator=torch.Generator().manual_seed(0))
    ci = R.CubicInterpolation(ts, R.backward_hermite_coefficients(ts, ys))
    for k in range(5):
        assert torch.allclose(ci.evaluate(float(ts[k])), ys[k], atol=1e-12)
    eps = 1e-9
    for k in range(1, 4):  # derivative continuous across interior knots
        assert torch.allclose(ci.derivative(float(ts[k]) - eps), ci.derivative(float(ts[k]) + eps), atol=1e-6)
    # first piece is linear (b_0 = m_0  =>  c = d = 0)
    assert float(ci.c[0].abs().max()) == 0.0 and float(ci.d[0].abs().max()) == 0.0


def test_time_channel_gradient_is_one():
    p = R.make_problem(n=6, h=4, e=0, L=1, T=4, t1=3, dt0=0.1, seed=0, dtype=torch.float64)
    ca = R.CubicInterpolation(p.ts, p.coeffs_adj)
    assert torch.allclose(ca.derivative(1.3)[..., 0], torch.ones(6, 6, dtype=torch.float64))


def test_step_table_rules():
    for (t1, dt, n_state) in [(3, 0.1, 30), (1, 0.1, 10), (1, 0.01, 100), (8, 0.01, 800)]:
        tab = R.constant_step_table(0.0, t1, dt)
        assert len(tab) - 1 == n_state and tab[0] == 0 and tab[-1] == np.float32(t1)
        assert np.all(np.diff(tab) > 0)
    with pytest.raises(RuntimeError):
        R.constant_step_table(0.0, 100.0, 0.001)


def test_tsit5_order_on_linear_ode():
    """y' = -y: 10 steps of 0.1 must reproduce exp(-1) to 5th-order accuracy."""
    y0 = torch.ones(1, 1, dtype=torch.float64)
    yT = R.tsit5_solve_fixed(lambda t, y: -y, y0, np.linspace(0, 1, 11))
    assert abs(float(yT) - np.exp(-1.0)) < 2e-8
    yT2 = R.tsit5_solve_fixed(lambda t, y: -y, y0, np.linspace(0, 1, 21))
    assert abs(float(yT2) - np.exp(-1.0)) < abs(float(yT) - np.exp(-1.0)) / 16


def test_directed_fusion_matrix_free_identity():
    """(I + A_bar_dir) M with the directed layer's 11 terms equals the matrix-free form the kernels use: E M + G^T M + v.M +
    r (1^T M) + 1 (c^T M) + kappa 1 (1^T M), with v, r, c built from row sums, COLUMN sums, diagonals and totals (k_stage_prep)."""
    g = torch.Generator().manual_seed(2)
    n, d = 9, 5
    A = torch.rand(n, n, generator=g, dtype=torch.float64)
    D = torch.randn(n, n, generator=g, dtype=torch.float64)
    M = torch.randn(n, d, generator=g, dtype=torch.float64)
    p = torch.randn(11, 2, generator=g, dtype=torch.float64) / 3
    lit = M + R.fusion_directed(A, D, p) @ M
    rA, rD, cA, cD = A.sum(1), D.sum(1), A.sum(0), D.sum(0)
    E = (1 + p[0, 0]) * A + (1 + p[0, 1]) * D
    G = p[1, 0] * A + p[1, 1] * D
    v = p[2, 0] * torch.diag(A) + p[2, 1] * torch.diag(D) + (p[7, 0] * cA + p[7, 1] * cD) / n + (p[8, 0] * rA + p[8, 1] * rD) / n \
        + (p[10, 0] * A.sum() + p[10, 1] * D.sum()) / n**2
    r = (p[3, 0] * cA + p[3, 1] * cD) / n
    c = (p[4, 0] * rA + p[4, 1] * cD) / n + (p[5, 0] * cA + p[5, 1] * cD) / n + (p[6, 0] * rA + p[6, 1] * rD) / n
    kappa = (p[9, 0] + p[9, 1]) * A.sum() / n**2
    ones = torch.ones(n, dtype=torch.float64)
    mf = M + E @ M + G.t() @ M + v[:, None] * M + r[:, None] * (ones @ M)[None, :] + ones[:, None] * (c @ M)[None, :] + kappa * ones[:, None] * (ones @ M)[None, :]
    assert torch.allclose(lit, mf, atol=1e-12)


# ---------------------------------------------------------------------------------------------------
# the restatement against the reference's OWN source files (fixtures made by oracle/pin_reference_source.py)
# ---------------------------------------------------------------------------------------------------
from oracle import pin_reference_source as PIN  # noqa: E402

REFSRC_TOL = 1e-11   # fp64 restatement vs fp64 execution of the reference source: different summation orders only


def _close(got, ref, what):
    ref = np.asarray(ref)
    err = float(np.abs(np.asarray(got) - ref).max() / max(float(np.abs(ref).max()), 1e-300))
    assert err < REFSRC_TOL, (what, err)


def _oracle_outputs_for_refsrc(name):
    """What oracle/pin_reference_source.py records, computed by the oracle's restatement instead of the reference files."""
    kw = PIN.REFSRC_CASES[name]
    p = R.problem_to(R.make_problem(**kw), torch.float64)
    ca = R.CubicInterpolation(p.ts, p.coeffs_adj)
    dir_tables = PIN.directed_fusion_tables(p.L, kw["seed"])
    return p, ca, dir_tables


@pytest.mark.parametrize("name", list(PIN.REFSRC_CASES))
def test_oracle_matches_reference_source_fixtures(name):
    g = np.load(os.path.join(GOLD, f"refsrc_{name}.npz"))
    p, ca, dir_tables = _oracle_outputs_for_refsrc(name)
    assert abs(input_checksum(R.make_problem(**PIN.REFSRC_CASES[name])) - float(g["in_checksum"])) < 1e-6 * max(1.0, abs(float(g["in_checksum"])))
    # layer level: ConvEquivFusionLayer._fusion / ConvEquivFusionDirectedLayer._fusion (layers.py:102-160, 256-345)
    t1 = PIN.EVAL_TIMES[1]
    adj, dadj = ca.evaluate(t1)[..., -1], ca.derivative(t1)[..., -1]
    fus, fus_dir = R.fusion(adj, dadj, p.layers[0].fusion).numpy(), R.fusion_directed(adj, dadj, dir_tables[0]).numpy()
    wgt = np.cos(np.arange(p.n * p.n, dtype=np.float64)).reshape(p.n, p.n)
    scale = float(np.abs(fus).sum())
    assert abs(float((fus * wgt).sum()) - float(g["fusion_t1_wsum"])) < REFSRC_TOL * scale
    assert abs(float((fus_dir * wgt).sum()) - float(g["fusion_dir_t1_wsum"])) < REFSRC_TOL * scale
    if "fusion_t1" in g:
        _close(fus, g["fusion_t1"], "fusion")
        _close(fus_dir, g["fusion_dir_t1"], "fusion_directed")
    # field level: every reference __call__ on the path and its siblings (behind CDEWrapperVectorField on control shapes)
    times = [float(t) for t in g["times"]]
    if p.e > 0:
        cx = R.CubicInterpolation(p.ts, p.x_coeffs)
        wrap = lambda out, t: torch.einsum("nmlk,nlk->nm", out.reshape(-1, p.h, p.e, 2), cx.derivative(t))   # cde_wrapper_vector_field.py:21-25
        _close(torch.stack([R.cde_wrapper_vector_field(t, p.y0, ca, cx, p.layers, p.h, p.e) for t in times]), g["vf_perm_equiv"], "wrapper")
    else:
        wrap = lambda out, t: out
        _close(torch.stack([R.perm_equiv_vector_field(t, p.y0, ca, p.layers) for t in times]), g["vf_perm_equiv"], "perm_equiv")
        _close(torch.stack([R.plain_graph_vector_field(t, p.y0, ca, p.layers, False) for t in times]), g["vf_gnode"], "gnode")
    _close(torch.stack([wrap(R.perm_equiv_dir_vector_field(t, p.y0, ca, p.layers, dir_tables), t) for t in times]), g["vf_perm_equiv_dir"], "directed")
    _close(torch.stack([wrap(R.plain_graph_vector_field(t, p.y0, ca, p.layers, True), t) for t in times]), g["vf_graph"], "graph")
    # the whole fixed-step solve over the reference's callable
    assert len(p.step_ts) - 1 == int(g["steps"])
    _close(R.run_forward(p), g["yT"], "yT")


@pytest.mark.skipif(not os.path.isdir(os.path.join(PIN.REFERENCE_SRC, "models", "vector_fields")),
                    reason="needs the reference project's source tree (PEG_REFERENCE_SRC)")
def test_reference_source_fixtures_are_reproducible_from_the_reference_tree():
    """Re-executes the unmodified reference files (numpy stand-ins for jax / equinox) and compares with the committed fixtures."""
    mods = PIN.load_reference_vector_fields()
    try:
        assert mods["layers"].__file__.startswith(PIN.REFERENCE_SRC)     # the code under test is the reference's file
        Wrapper = mods["cde_wrapper_vector_field"].CDEWrapperVectorField
        for name, kw in PIN.REFSRC_CASES.items():
            if kw["n"] > 40:
                continue
            g = np.load(os.path.join(GOLD, f"refsrc_{name}.npz"))
            p, ca, dir_tables = _oracle_outputs_for_refsrc(name)
            pe, pd, gv, gn = PIN.build_reference_fields(mods, p, dir_tables)
            nca = PIN.NumpyControl(ca)
            y = p.y0.numpy()
            if p.e > 0:
                ncx = PIN.NumpyControl(R.CubicInterpolation(p.ts, p.x_coeffs))
                fields = {"perm_equiv": Wrapper(pe, p.h), "perm_equiv_dir": Wrapper(pd, p.h), "graph": Wrapper(gv, p.h)}
                args = [nca, ncx]
            else:
                fields = {"perm_equiv": pe, "perm_equiv_dir": pd, "graph": gv, "gnode": gn}
                args = nca
            for k, t in enumerate(float(t) for t in g["times"]):
                for key, field in fields.items():
                    assert np.array_equal(field(t, y, args), g[f"vf_{key}"][k]), (name, key, t)
    finally:
        PIN.uninstall_shims()
    import sys
    assert "jax" not in sys.modules


# ---------------------------------------------------------------------------------------------------
# model level: the reference's solve wrappers (pgt_ / tgb_ / graph_neural_cde.py) executed unmodified, diffrax backed by the oracle
# ---------------------------------------------------------------------------------------------------
def _model_fixture(name):
    g = np.load(os.path.join(GOLD, f"refsrc_model_{name}.npz"))
    kind, kw, extra = PIN.MODEL_CASES[name]
    p = R.problem_to(R.make_problem(**kw), torch.float64)
    tt = lambda a: torch.from_numpy(np.asarray(a, dtype=np.float64))
    stack = lambda pre: [(tt(g[f"{pre}_W{i}"]), tt(g[f"{pre}_b{i}"])) for i in range(sum(k.startswith(f"{pre}_W") for k in g.files))]
    inp = {k: tt(v) for k, v in PIN.model_inputs(name).items()}
    return g, kind, p, stack("enc"), stack("dec"), inp, tt


@pytest.mark.parametrize("name", list(PIN.MODEL_CASES))
def test_oracle_models_match_reference_source_fixtures(name):
    g, kind, p, enc, dec, inp, tt = _model_fixture(name)
    extra = PIN.MODEL_CASES[name][2]
    ev = bool(extra.get("evolving_out"))
    if kind == "pgt":
        cadj, cx = p.coeffs_adj, p.x_coeffs
        if extra.get("interpolation") == "linear":   # piecewise-linear control = cubic pieces with c = d = 0 (unit knot spacing)
            A_k, X_k = tt(g["adj_knots"]), tt(g["x_knots"])
            cadj = (torch.zeros_like(cadj[0]), torch.zeros_like(cadj[0]), A_k[1:] - A_k[:-1], A_k[:-1])
            cx = (torch.zeros_like(cx[0]), torch.zeros_like(cx[0]), X_k[1:] - X_k[:-1], X_k[:-1])
        _close(R.pgt_graph_neural_cde(p.ts, cadj, cx, inp["x0"], enc, dec, p.layers, p.h, p.e, evolving_out=ev), g["out_global"], "pgt global")
        _close(R.pgt_graph_neural_cde(p.ts, cadj, cx, inp["x0"], enc, dec, p.layers, p.h, p.e, global_readout=False, evolving_out=ev), g["out_nodes"], "pgt nodes")
        assert g["out_global"].shape == (extra["feature_dim"],) and g["out_nodes"].shape == (p.n, extra["feature_dim"])
    elif kind == "tgb":
        seq = bool(extra.get("return_sequence"))
        out = R.tgb_graph_neural_cde(p.ts, p.coeffs_adj, inp["x_data"], inp["x0"], enc, dec, (tt(g["data_encoder_W"]), tt(g["data_encoder_b"])), p.layers, p.h, p.e,
                                     evolving_out=ev, return_sequence=seq)
        _close(out, g["out"], "tgb")
        assert g["out"].shape == ((p.ts.numel(), p.n, p.n) if seq else (p.n, p.n))
    else:
        out, table = R.graph_neural_cde(p.ts, p.coeffs_adj, inp["x0"], enc[0], dec[0], p.layers)
        _close(out, g["out"], "dyn")
        assert len(table) - 1 == int(g["accepted_steps"]) and g["out"].shape == (p.ts.numel(), p.n, 1)


@pytest.mark.skipif(not os.path.isdir(os.path.join(PIN.REFERENCE_SRC, "models", "vector_fields")),
                    reason="needs the reference project's source tree (PEG_REFERENCE_SRC)")
def test_reference_model_fixture_is_reproducible_from_the_reference_tree():
    """Re-runs the unmodified reference PGTGraphNeuralCDE on the stand-ins and requires the committed fixture bit for bit."""
    import types

    g, kind, p, enc, dec, inp, tt = _model_fixture("pgt")
    kind, kw, extra = PIN.MODEL_CASES["pgt"]
    mods = PIN.load_reference_models()
    try:
        import jax.random as jr   # the stand-in

        widths = R.layer_widths(p.h, p.L, p.e, True)
        vf = mods["perm_equiv_graph_vector_field"].PermEquivGraphVectorField(
            input_dim=p.h, hidden_dim=p.h, output_dim=widths[-1], num_layers=p.L, data_embed_dim=p.e, num_nodes=p.n, key=jr.PRNGKey(0))
        for l, lp in enumerate(p.layers):
            for i in range(8):
                setattr(vf.gnn_layers[l], f"param{i + 1}", lp.fusion[i].numpy().copy())
            PIN._set_conv(vf.gnn_layers[l].conv_layer, lp)
        cfg = types.SimpleNamespace(data_dim=extra["data_dim"], hidden_dim=p.h, feature_dim=extra["feature_dim"], method="Tsit5", return_sequence=False)
        model = mods["pgt_graph_neural_cde"].PGTGraphNeuralCDE(cfg, vf, "cubic", jr.PRNGKey(kw["seed"]))
        assert mods["pgt_graph_neural_cde"].__file__.startswith(PIN.REFERENCE_SRC)
        out = model(np.arange(kw["T"], dtype=np.int32), np.stack([c.numpy() for c in p.coeffs_adj]),
                    np.stack([c.numpy() for c in p.x_coeffs]), inp["x0"].numpy())
        assert np.array_equal(out, g["out_global"])
    finally:
        PIN.uninstall_shims()
    import sys
    assert "jax" not in sys.modules and "diffrax" not in sys.modules


# ---------------------------------------------------------------------------------------------------
# data side of the boundary: the reference's control-path builders (src/configs/dataset_configs.py, executed unmodified)
# ---------------------------------------------------------------------------------------------------
def test_reference_layout_matches_reference_source_fixture():
    """What the trainers hand to the models (trainer_pgt.py:201-207): PGTDataSetCfg.process_window -> graph_path_coeffs /
    x_coeffs as (d, c, b, a), each [T-1, n, n|e, 2] with the last axis (time, value); ODEDataSetCfg for float time stamps."""
    g = np.load(os.path.join(GOLD, "refsrc_dataset.npz"))
    window = PIN.dataset_window()
    ts = torch.arange(len(window) - 1)
    A = torch.stack([w.adj for w in window[:-1]])
    x_t = torch.stack([w.x for w in window[:-1]])
    assert np.array_equal(g["t"], ts.numpy()) and np.array_equal(g["true_y"], window[-1].y.numpy()) and np.array_equal(g["true_y0"], window[0].x.numpy())
    for nm, mine_g, mine_x in zip("dcba", R.reference_layout_coeffs(ts, A), R.reference_layout_xcoeffs(ts, x_t)):
        assert g[f"graph_{nm}"].shape == (len(window) - 2, PIN.DATASET_CASE["n"], PIN.DATASET_CASE["n"], 2)
        assert np.array_equal(mine_g.numpy(), g[f"graph_{nm}"]), nm
        assert np.array_equal(mine_x.numpy(), g[f"x_{nm}"]), nm
    assert np.array_equal(g["graph_a"][..., 0], np.broadcast_to(np.arange(3.0)[:, None, None], (3, 11, 11)))   # time channel
    ts_f = torch.from_numpy(np.linspace(0.0, 5.0, 6))
    A_f = torch.from_numpy(R.synthetic_graph_path(9, 6, PIN.DATASET_CASE["seed"] + 1))
    for nm, mine in zip("dcba", R.reference_layout_coeffs(ts_f, A_f)):
        assert np.allclose(mine.numpy(), g[f"ode_graph_{nm}"], rtol=0, atol=1e-12), nm


def test_product_hermite_builder_matches_reference_source_fixture():
    """The product's host-side builder (control.backward_hermite_coefficients, used by TGBGraphNeuralCDE) on the same window."""
    import perm_equiv_graph_neural_cdes_b200 as P

    g = np.load(os.path.join(GOLD, "refsrc_dataset.npz"))
    window = PIN.dataset_window()
    ts = torch.arange(len(window) - 1, dtype=torch.float64)
    x_t = torch.stack([w.x for w in window[:-1]])
    x_path = torch.stack([ts[:, None, None].expand_as(x_t), x_t], dim=-1)
    for nm, mine in zip("dcba", P.backward_hermite_coefficients(ts, x_path)):
        assert np.allclose(mine.numpy(), g[f"x_{nm}"], rtol=0, atol=1e-12), nm


@pytest.mark.skipif(not os.path.isdir(os.path.join(PIN.REFERENCE_SRC, "models", "vector_fields")),
                    reason="needs the reference project's source tree (PEG_REFERENCE_SRC)")
def test_reference_dataset_fixture_is_reproducible_from_the_reference_tree():
    import types

    g = np.load(os.path.join(GOLD, "refsrc_dataset.npz"))
    mod = PIN.load_reference_dataset_configs()
    try:
        assert mod.__file__.startswith(PIN.REFERENCE_SRC)
        cfg = types.SimpleNamespace(interpolation="cubic")
        cfg.get_interpolation_coeffs = lambda ts, sig: mod.PGTDataSetCfg.get_interpolation_coeffs(cfg, ts, sig)
        d = mod.PGTDataSetCfg.process_window(cfg, PIN.dataset_window())
        for i, nm in enumerate("dcba"):
            assert np.array_equal(d["graph_path_coeffs"][i].numpy(), g[f"graph_{nm}"])
            assert np.array_equal(d["x_coeffs"][i].numpy(), g[f"x_{nm}"])
    finally:
        PIN.uninstall_shims()
    import sys
    assert "jax" not in sys.modules and "torch_geometric" not in sys.modules


def test_pgt_mse_loss_matches_reference_source_fixture():
    """mse_loss of src/engine/trainer_pgt.py:45-66 (compiled from the reference's own lines): the (1,1) - (n,) broadcast is kept."""
    g = np.load(os.path.join(GOLD, "refsrc_dataset.npz"))
    y_pred, label = torch.from_numpy(g["loss_y_pred"]), torch.from_numpy(g["loss_label"])
    mine = R.pgt_mse_loss(torch.ones(1, 1, dtype=torch.float64), y_pred.reshape(1, 1), label)
    assert abs(float(mine) - float(g["loss"])) < 1e-14
    assert abs(float(g["loss"]) - float(((y_pred.reshape(1, 1) - label) ** 2).mean())) < 1e-14
    if os.path.isdir(os.path.join(PIN.REFERENCE_SRC, "engine")):
        try:
            mse = PIN.reference_pgt_mse_loss()
            assert float(mse(lambda t, a, x, x0: g["loss_y_pred"], (None, None, None, None, g["loss_label"]))) == float(g["loss"])
        finally:
            PIN.uninstall_shims()


# ---------------------------------------------------------------------------------------------------
# third-party arithmetic pinned against mathematics: the Tsit5 constants must satisfy the Runge-Kutta order conditions
# ---------------------------------------------------------------------------------------------------
def _tsit5_trees():
    """Elementary weights Phi(tree) and densities gamma(tree) of the 17 rooted trees up to order 5, for weights w: sum_i w_i Phi_i."""
    A = np.zeros((7, 7))
    for i, row in enumerate(R.TSIT5_A):
        A[i, :len(row)] = row
    c = np.array(R.TSIT5_C)
    Ac, Ac2 = A @ c, A @ (c * c)
    AAc = A @ Ac
    one = np.ones(7)
    trees = [  # (order, Phi, gamma)
        (1, one, 1), (2, c, 2), (3, c**2, 3), (3, Ac, 6),
        (4, c**3, 4), (4, c * Ac, 8), (4, Ac2, 12), (4, AAc, 24),
        (5, c**4, 5), (5, c * c * Ac, 10), (5, c * Ac2, 15), (5, c * AAc, 30), (5, Ac * Ac, 20),
        (5, A @ c**3, 20), (5, A @ (c * Ac), 40), (5, A @ Ac2, 60), (5, A @ AAc, 120),
    ]
    return A, c, trees


def test_tsit5_tableau_satisfies_the_order_conditions():
    """The restated tableau (diffrax.Tsit5 = Tsitouras 2011) is a 5th-order method with a 4th-order embedded estimate:
    all 17 order-5 conditions for b, all 8 order-4 conditions for b_hat = b - b_err, row sums = c, FSAL row = b."""
    A, c, trees = _tsit5_trees()
    b, berr = np.array(R.TSIT5_B), np.array(R.TSIT5_BERR)
    assert np.abs(A.sum(1) - c).max() < 2e-15
    assert np.array_equal(A[6, :6], b[:6]) and b[6] == 0.0                       # FSAL: the 7th stage is evaluated at y1
    for order, phi, gamma in trees:
        assert abs(b @ phi - 1.0 / gamma) < 3e-15, (order, gamma)
        if order <= 4:
            assert abs((b - berr) @ phi - 1.0 / gamma) < 3e-15, ("embedded", order, gamma)
    # ... and the embedded weights are genuinely 4th order only (the estimate does not vanish)
    assert max(abs((b - berr) @ phi - 1.0 / gamma) for order, phi, gamma in trees if order == 5) > 1e-4


def test_tsit5_dense_output_satisfies_the_continuous_order_conditions():
    """b_i(theta) of the interpolant: sum_i b_i(theta) Phi_i(tree) = theta^order / gamma(tree) for every tree up to order 4,
    b_i(0) = 0 and b_i(1) = b_i."""
    A, c, trees = _tsit5_trees()
    assert np.abs(np.array(R.tsit5_dense_weights(0.0), dtype=float)).max() == 0.0
    assert np.abs(np.array(R.tsit5_dense_weights(1.0), dtype=float) - np.array(R.TSIT5_B)).max() < 5e-15
    for theta in (0.05, 0.1, 0.35, 0.5, 0.77, 0.9, 1.0):
        w = np.array(R.tsit5_dense_weights(theta), dtype=float)
        for order, phi, gamma in trees:
            if order <= 4:
                assert abs(w @ phi - theta**order / gamma) < 5e-15, (theta, order, gamma)


def test_initial_step_heuristic_matches_scipy():
    """diffrax picks dt0=None steps with Hairer-Norsett-Wanner's starting-step algorithm (II.4); scipy.integrate ships an
    independent implementation of the same published algorithm (order + 1 = error_order = 5 for a 5(4) pair)."""
    from scipy.integrate._ivp.common import select_initial_step as scipy_select

    rng = np.random.default_rng(0)
    for trial in range(4):
        M = torch.from_numpy(rng.standard_normal((6, 6)) * (0.3 + 0.4 * trial))
        f = lambda t, y: torch.tanh(y @ M) * (1 + 0.1 * t)
        y0 = torch.from_numpy(rng.standard_normal((4, 6)))
        f0 = f(0.0, y0)
        mine = float(R.select_initial_step(f, 0.0, y0, f0, 1e-3, 1e-6))
        theirs = float(scipy_select(lambda t, y: f(t, torch.from_numpy(y.reshape(4, 6))).numpy().reshape(-1), 0.0, y0.numpy().reshape(-1),
                                    5.0, np.inf, f0.numpy().reshape(-1), 1.0, 4, 1e-3, 1e-6))
        assert abs(mine - theirs) < 2e-6 * theirs, (trial, mine, theirs)      # the oracle follows diffrax and works in fp32


def test_hermite_path_matches_scipy_cubic_hermite_spline():
    """backward_hermite_coefficients + CubicInterpolation == the cubic Hermite spline through the knots whose slope at knot k is the
    backward difference m_{k-1} (m_0 at the first knot), evaluated by scipy's independent implementation."""
    from scipy.interpolate import CubicHermiteSpline

    rng = np.random.default_rng(3)
    ts = np.array([0.0, 0.6, 1.0, 2.5, 3.0, 4.2])
    ys = rng.standard_normal((6, 5))
    m = (ys[1:] - ys[:-1]) / (ts[1:] - ts[:-1])[:, None]
    spline = CubicHermiteSpline(ts, ys, np.concatenate([m[:1], m], axis=0))
    ci = R.CubicInterpolation(torch.from_numpy(ts), R.backward_hermite_coefficients(torch.from_numpy(ts), torch.from_numpy(ys)))
    for t in (0.0, 0.3, 0.6, 0.61, 1.7, 2.5, 2.9, 3.0, 4.0, 4.2):
        assert np.allclose(ci.evaluate(t).numpy(), spline(t), rtol=0, atol=1e-13), t
        if t not in ts:     # at a knot scipy returns the right-hand piece's derivative, diffrax's lookup the left-hand one (they agree: C1)
            assert np.allclose(ci.derivative(t).numpy(), spline(t, 1), rtol=0, atol=1e-12), t


def test_rms_norm_matches_torch_rms_norm():
    """equinox.nn.RMSNorm arithmetic (x * rsqrt(mean(x^2) + eps) * weight, then + bias) against torch's independent rms_norm."""
    g = torch.Generator().manual_seed(0)
    x = torch.randn(7, 16, generator=g, dtype=torch.float64)
    w, b = torch.randn(16, generator=g, dtype=torch.float64), torch.randn(16, generator=g, dtype=torch.float64)
    ref = torch.nn.functional.rms_norm(x, (16,), weight=w, eps=1e-5) + b
    assert torch.allclose(R.rms_norm(x, w, b), ref, rtol=0, atol=1e-14)


def test_fp16x2_block_floating_point_scheme_reaches_fp32_accuracy():
    """CPU emulation (numpy) of the default operand format of the tensor-core contraction (csrc/peg_tc.cu, DESIGN.md "Operand formats"):
    V^T is stored as V * 2^e_J with one power-of-two exponent per 128-node block and split hi + lo into two fp16 numbers; the
    interpolated adjacency gets one power-of-two scale, is aligned to the smallest block exponent by an exact factor 2^(E - e_J) per
    K block, and is split with the symmetric rounding ((bits + 0x1000) & 0xffffe000); the products hi*hi + lo*hi + hi*lo accumulate in
    fp32 and the scales are divided out (exactly) at the end.  The scheme must reproduce the fp64 product to fp32-level accuracy on
    operands with England's dynamic range and block magnitudes that differ by 1e6, where single-pass fp16 is off by > 1e-4."""
    rng = np.random.default_rng(5)
    n, m, d, VEXP_MAX = 512, 96, 24, 60

    def block_exponent(amax):
        if not amax > 0:
            return VEXP_MAX
        e = 14 - (int((np.float32(amax).view(np.uint32) >> 23) & 0xFF) - 127)
        return max(-VEXP_MAX, min(VEXP_MAX, e))

    A = (rng.lognormal(0.0, 2.0, (m, n)) * (rng.random((m, n)) < 0.1) * rng.choice([-1.0, 1.0], (m, n))).astype(np.float32)     # sparse-ish, 1e4 range
    V = rng.standard_normal((n, d)).astype(np.float32)
    V *= np.repeat(np.float32(10.0) ** rng.integers(-3, 4, n // 128), 128)[:, None]                     # block magnitudes 1e-3 .. 1e3
    V[128:256] = 0.0                                                                                   # an all-zero block never wins the minimum
    ref = A.astype(np.float64) @ V.astype(np.float64)
    # V side: per-block exponents, hi = rn_f16(v 2^e), lo = rn_f16(v 2^e - hi)
    eJ = np.array([block_exponent(np.abs(V[j * 128:(j + 1) * 128]).max()) for j in range(n // 128)])
    Vs = V * np.repeat(np.exp2(eJ.astype(np.float64)), 128)[:, None].astype(np.float32)                 # exact: power of two
    assert np.abs(Vs).max() < 65504
    v_hi = Vs.astype(np.float16)
    v_lo = (Vs - v_hi.astype(np.float32)).astype(np.float16)
    # A side: one scale for the launch, aligned per K block to the smallest exponent
    E = int(eJ.min())
    eA = block_exponent(np.abs(A).max())
    As = A * np.float32(np.exp2(eA)) * np.repeat(np.exp2((E - eJ).astype(np.float64)), 128)[None, :].astype(np.float32)
    bits = As.view(np.uint32)
    a_hi32 = ((bits + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)
    a_hi = a_hi32.astype(np.float16)
    big = np.abs(As) >= 2.0 ** -14                  # hi is exact in fp16 wherever it is a normal fp16 number
    assert np.array_equal(a_hi.astype(np.float32)[big], a_hi32[big])
    a_lo = (As - a_hi32).astype(np.float16)
    f32 = lambda x: x.astype(np.float32)
    acc = f32(a_hi) @ f32(v_hi) + f32(a_lo) @ f32(v_hi) + f32(a_hi) @ f32(v_lo)                         # fp32 accumulation
    got = acc.astype(np.float64) * np.exp2(-float(eA)) * np.exp2(-float(E))
    scale = np.abs(ref).max()
    err3 = np.abs(got - ref).max() / scale
    err1 = np.abs((f32(a_hi) @ f32(v_hi)).astype(np.float64) * np.exp2(-float(eA)) * np.exp2(-float(E)) - ref).max() / scale
    assert err3 < 5e-6, err3
    assert err1 > 1e-4, err1        # the split is what buys the accuracy
    # column-wise too (every column of V has its own magnitude profile): no column is worse than 2e-5 of its own maximum
    col = np.abs(got - ref).max(axis=0) / np.abs(ref).max(axis=0)
    assert col.max() < 2e-5, col.max()
