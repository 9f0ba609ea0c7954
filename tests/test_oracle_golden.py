"""CPU: the oracle restatement against the golden vectors frozen from the live reference
(tests/golden/make_golden.py), and its closed-form backward against autograd."""
import numpy as np
import pytest
import torch

import ign_oracle as O
from helpers import MODES, assert_close, load_golden, t

LAYER_CASES = ["layer_l1", "layer_l1_stride", "layer_cosine", "layer_pearson", "layer_cosine_stride",
               "layer_l1_struct", "layer_lts", "layer_l1_min", "layer_pearson_k12", "layer_sql2"]


@pytest.mark.parametrize("name", LAYER_CASES)
def test_oracle_layer_matches_reference_golden(name):
    g = load_golden(name)
    mode = MODES[str(g["dfunc"])][0]
    pool = str(g["pool"])
    thr = t(g["threshold"]) if "threshold" in g else None
    xn, W, up = t(g["xn"]), t(g["W"]), t(g["g"])
    out = O.shapelet_forward(xn, W, int(g["stride"]), float(g["eps"]), mode, pool, thr)
    # forward: same ops in the same order as the reference -> bit-exact on the same CPU build,
    # 1e-6 relative allowed for a different BLAS/vectorisation width
    assert_close(out.p, t(g["p"]).reshape(out.p.shape), 1e-6, 1e-7, name + " p")
    assert_close(out.dmin, t(g["dmin"]).reshape(out.dmin.shape), 1e-6, 1e-7, name + " dmin")
    dW, dthr = O.shapelet_backward_formula(xn.double(), W.double(), up.double(), int(g["stride"]), float(g["eps"]),
                                           mode, pool, None if thr is None else thr.double())
    assert_close(dW, t(g["dW"]), 2e-5, 2e-6, name + " dW (closed form vs reference autograd, fp32 reference)")
    if dthr is not None:
        assert_close(dthr, t(g["dthreshold"]), 2e-5, 2e-6, name + " dthreshold")


def test_oracle_known_answers():
    """SURVEY.md §8c table: x=[0..4], L=3, eps=1."""
    g = load_golden("kat")
    x = torch.tensor([[[0., 1., 2., 3., 4.]]])
    expect = {"euclidean": (0.6411804, 0.6666667, [-0.3164448, -0.0052398, 0.3089988]),
              "cosine": (0.9987689, 0.0350987, [-6.5409709e-03, 3.7e-09, 6.5409727e-03]),
              "pearson": (0.9996753, 0.0180196, [-0.0016847, 0.0025270, -0.0008423])}
    for flag, (p_e, d_e, dW_e) in expect.items():
        W = t(g[flag + "_W"]).reshape(1, 1, 3)
        out = O.shapelet_forward(x, W, 1, 1.0, MODES[flag][0])
        assert abs(float(out.p) - p_e) < 2e-7 and abs(float(out.dmin) - d_e) < 2e-7
        assert abs(float(out.p) - float(g[flag + "_p"].ravel()[0])) < 1e-7
        dW, _ = O.shapelet_backward_formula(x.double(), W.double(), torch.ones(1, 1, 1, dtype=torch.double),
                                            1, 1.0, MODES[flag][0])
        np.testing.assert_allclose(dW.flatten().numpy(), np.array(dW_e), atol=2e-7)
        np.testing.assert_allclose(dW.flatten().numpy(), g[flag + "_dW"].flatten(), atol=2e-7)
    # exact 3-way tie of the pearson case resolves to the first index
    out = O.shapelet_forward(x, torch.tensor([[[1., 2., 4.]]]), 1, 1.0, O.DIST_PEARSON)
    assert int(out.argmin_d) == 0


@pytest.mark.parametrize("mode", [O.DIST_L1, O.DIST_SQL2, O.DIST_COS, O.DIST_PEARSON])
@pytest.mark.parametrize("pool", [O.POOL_RBF_MAX, O.POOL_LTS_MIN])
@pytest.mark.parametrize("stride", [1, 3])
def test_closed_form_backward_equals_autograd(mode, pool, stride):
    if pool == O.POOL_LTS_MIN and mode in (O.DIST_COS, O.DIST_PEARSON):
        pytest.skip("DistThresholdShapelet ignores distance_func (Shapelet.py:100-103)")
    torch.manual_seed(11)
    B, M, T, K, L = 2, 3, 41, 4, 7
    xn = torch.randn(B, M, T, dtype=torch.double)
    W = torch.randn(K, M, L, dtype=torch.double)
    g = torch.randn(B, K, M, dtype=torch.double)
    thr = torch.rand(1, K, M, dtype=torch.double) if pool == O.POOL_LTS_MIN else None
    dWf, dtf = O.shapelet_backward_formula(xn, W, g, stride, 0.9, mode, pool, thr)
    dWa, dta, _ = O.shapelet_backward_autograd(xn, W, g, stride, 0.9, mode, pool, thr)
    assert float((dWf - dWa).abs().max()) < 1e-13
    if thr is not None:
        assert float((dtf - dta).abs().max()) < 1e-13


@pytest.mark.parametrize("gv", [None, 0.0, 0.3, 1.0])
def test_gate_closed_form(gv):
    torch.manual_seed(3)
    s = torch.randn(6, 5, dtype=torch.double, requires_grad=True)
    z = torch.randn(6, 5, dtype=torch.double, requires_grad=True)
    go, ge = torch.randn(6, 5, dtype=torch.double), torch.randn(6, 1, dtype=torch.double)
    out, eta = O.gate_forward(s, z, gv)
    ((out * go).sum() + (eta * ge).sum()).backward()
    gs, gz = O.gate_backward_formula(s.detach(), z.detach(), go, ge, gv)
    assert float((gs - s.grad).abs().max()) < 1e-13 and float((gz - z.grad).abs().max()) < 1e-13
    if gv == 1.0:    # eta <= 1 always: gating at 1 never fires (SURVEY.md §8c invariants)
        out0, _ = O.gate_forward(s, z, None)
        assert torch.equal(out0, out)
    if gv == 0.0:    # eta > 0 unless softmax is exactly uniform: gate fires, out == sbm_out
        assert torch.allclose(out, s)


MODEL_CASES = ["model_jv_interpgn", "model_jv_interpgn_gate", "model_jv_interpgn_cos", "model_jv_sbm",
               "model_jv_lts", "model_small_chisco", "model_small_transformer"]


@pytest.mark.parametrize("name", MODEL_CASES)
def test_oracle_model_matches_reference_golden(name):
    g = load_golden(name)
    cfg = dict(zip(g["cfg_keys"].tolist(), g["cfg_vals"].tolist()))
    T = int(cfg["seq_len"])
    mode = MODES[cfg.get("distance_func", "euclidean")][0]
    prefix = "sd::sbm." if any(k.startswith("sd::sbm.") for k in g) else "sd::"
    lts = name.endswith("lts")
    Ws = [t(g[f"{prefix}shapelets.{i}.weights"]) for i in range(4)]
    thr = [t(g[f"{prefix}shapelets.{i}.threshold"]) for i in range(4)] if lts else None
    Wc = t(g[f"{prefix}output_layer.weight"])
    lens = O.shapelet_lengths(T, [0.1, 0.2, 0.3, 0.5])
    assert lens == [w.shape[-1] for w in Ws]
    strides = [O.shapelet_stride(T, L) for L in lens]
    logits, probs, dists = O.sbm_forward(t(g["x"]), Ws, strides, Wc, 1.0, mode,
                                         O.POOL_LTS_MIN if lts else O.POOL_RBF_MAX, thr)
    assert_close(probs, t(g["p"]), 1e-6, 1e-7, name + " p")
    assert_close(dists, t(g["d"]), 1e-6, 1e-7, name + " d")
    assert_close(logits, t(g["shapelet_preds"]), 1e-5, 1e-6, name + " shapelet logits")
    assert_close(O.sbm_loss(Wc, Ws, 0.1, 0.1).reshape(1), t(g["reg_loss"]), 1e-6, 1e-8, name + " regulariser")
    if "eta" in g:
        gv = None if np.isnan(g["gating_value"]) else float(g["gating_value"])
        out, eta = O.gate_forward(t(g["shapelet_preds"]), t(g["dnn_preds"]), gv)
        assert_close(out, t(g["logits"]), 1e-6, 1e-7, name + " gated logits")
        assert_close(eta, t(g["eta"]), 1e-6, 1e-7, name + " eta")


def test_oracle_against_live_reference_if_mounted():
    """Only with IGN_REFERENCE_ROOT set: run the unmodified reference modules side by side."""
    import ref_shim
    if not ref_shim.available():
        pytest.skip("IGN_REFERENCE_ROOT does not name a reference checkout")
    ns = ref_shim.load_reference()
    torch.manual_seed(5)
    for flag in ("euclidean", "cosine", "pearson"):
        layer = ns.Shapelet(3, 8, 4, stride=2, eps=1.1, distance_func=flag)
        xn = torch.randn(2, 3, 50)
        p, dm = layer(xn)
        out = O.shapelet_forward(xn, layer.weights.detach(), 2, 1.1, MODES[flag][0])
        assert torch.equal(out.p, p.detach()) and torch.equal(out.dmin, dm.detach())


def test_shape_rules():
    assert O.shapelet_lengths(29, [0.1, 0.2, 0.3, 0.5]) == [3, 6, 9, 15]
    assert O.shapelet_lengths(1000, [0.1, 0.2, 0.3, 0.5]) == [100, 200, 300, 500]
    assert [O.shapelet_stride(4000, L) for L in (400, 800, 1200, 2000)] == [8, 9, 10, 10]
    assert O.shapelet_stride(2999, 1500) == 1
    with pytest.raises(RuntimeError):
        O.num_windows(5, 6, 1)


@pytest.mark.parametrize("name", ["model_chisco_full", "model_chisco_full_cos", "model_chisco39_transformer"])
def test_oracle_at_the_baseline_shapes_matches_live_reference_golden(name):
    """BASELINE configs 2 and 5 at full width (125 ch x T=1000, default shapelet set, B=2): the fixture holds the live
    reference's outputs; weights and batch are regenerated from its seed (helpers.seeded_fill / seeded_batch)."""
    from types import SimpleNamespace
    from helpers import seeded_batch, seeded_fill
    from models.InterpGN import InterpGN          # host-side construction only (state-dict layout); no kernels run
    g = load_golden(name)
    kw = dict(zip(g["cfg_keys"].tolist(), g["cfg_vals"].tolist()))
    cfg = SimpleNamespace(epsilon=1., distance_func=kw.get("distance_func", "euclidean"), memory_efficient=False,
                          sbm_cls="linear", dropout=0., lambda_reg=0.1, lambda_div=0.1, dnn_type="FCN",
                          enc_in=int(kw["enc_in"]), num_class=int(kw["num_class"]), seq_len=int(kw["seq_len"]))
    seed, B = int(g["seed"]), int(g["B"])
    model = InterpGN(cfg).sbm                      # the FCN placeholder expert is not used: only sbm.* names matter
    # seeded_fill derives every tensor's stream from (seed, parameter name): fill under the InterpGN names
    holder = torch.nn.Module()
    holder.sbm = model
    seeded_fill(holder, seed)
    x, y = seeded_batch(B, cfg.seq_len, cfg.enc_in, cfg.num_class, seed)
    assert abs(float(x.double().abs().sum()) - float(g["x_checksum"])) <= 1e-9 * float(g["x_checksum"])
    Ws = [s.weights.detach() for s in model.shapelets]
    Wc = model.output_layer.weight.detach()
    mode = MODES[cfg.distance_func][0]
    logits, probs, dists = O.sbm_forward(x, Ws, [1, 1, 1, 1], Wc, 1.0, mode)
    assert_close(probs, t(g["p"]), 1e-6, 1e-7, name + " p")
    assert_close(dists, t(g["d"]), 1e-6, 1e-7, name + " d")
    assert_close(logits, t(g["shapelet_preds"]), 1e-5, 1e-6, name + " shapelet logits")
    out, eta = O.gate_forward(t(g["shapelet_preds"]), t(g["dnn_preds"]))
    assert_close(out, t(g["logits"]), 1e-6, 1e-7, name + " gated logits")
    assert_close(eta, t(g["eta"]), 1e-6, 1e-7, name + " eta")
    assert_close(O.sbm_loss(Wc, Ws, 0.1, 0.1).reshape(1), t(g["reg_loss"]), 1e-6, 1e-8, name + " regulariser")
