"""GPU parity of the whole models against golden vectors frozen from the reference (same weights via
load_state_dict, same inputs): logits, eta, predicates, regulariser, loss and parameter gradients."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from helpers import assert_close, load_golden, sample_indices, seeded_batch, seeded_fill, t

pytestmark = pytest.mark.gpu
DEV = "cuda"


def build(name):
    from models.InterpGN import InterpGN
    from models.Shapelet import DistThresholdSBM, ShapeBottleneckModel
    g = load_golden(name)
    kw = dict(zip(g["cfg_keys"].tolist(), g["cfg_vals"].tolist()))
    cfg = SimpleNamespace(epsilon=1., distance_func=kw.get("distance_func", "euclidean"), memory_efficient=False,
                          sbm_cls=kw.get("sbm_cls", "linear"), dropout=0., lambda_reg=0.1, lambda_div=0.1,
                          dnn_type=kw.get("dnn_type", "FCN"),
                          enc_in=int(kw["enc_in"]), num_class=int(kw["num_class"]), seq_len=int(kw["seq_len"]))
    for key in ("task_name", "embed", "freq", "activation"):
        if key in kw:
            setattr(cfg, key, kw[key])
    for key in ("pred_len", "label_len", "d_model", "factor", "n_heads", "d_ff", "e_layers"):
        if key in kw:
            setattr(cfg, key, int(kw[key]))
    cfg.output_attention = False
    cls = DistThresholdSBM if name.endswith("lts") else ShapeBottleneckModel if "_sbm" in name else InterpGN
    model = cls(cfg)
    model.load_state_dict({k[4:]: torch.as_tensor(v) for k, v in g.items() if k.startswith("sd::")})
    return model.to(DEV).train(), g


@pytest.mark.parametrize("name", ["model_jv_interpgn", "model_jv_interpgn_gate", "model_jv_interpgn_cos",
                                  "model_jv_sbm", "model_jv_lts", "model_small_chisco", "model_small_transformer",
                                  # alternate heads (Shapelet.py:170-177, 199-205): forward AND gradients on the GPU
                                  "model_jv_sbm_bilinear", "model_jv_sbm_attention", "model_jv_interpgn_attention"])
def test_model_matches_reference_golden(name):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.set_float32_matmul_precision("highest")
    model, g = build(name)
    x, y = t(g["x"], DEV), torch.as_tensor(g["y"]).to(DEV)
    mask = torch.ones(x.shape[0], x.shape[1], device=DEV)
    is_ign = "eta" in g
    if is_ign:
        gv = None if np.isnan(g["gating_value"]) else float(g["gating_value"])
        logits, info = model(x, mask, None, None, gating_value=gv)
    else:
        logits, info = model(x, mask, None, None)
    loss = torch.nn.functional.cross_entropy(logits, y) + info.loss.mean()
    if is_ign:
        loss = loss + torch.nn.functional.cross_entropy(info.shapelet_preds, y)
    loss.backward()
    torch.cuda.synchronize()
    assert_close(info.p, t(g["p"]), 2e-5, 2e-6, name + " p")
    assert_close(info.d, t(g["d"]), 2e-5, 2e-6, name + " d")
    assert_close(info.shapelet_preds, t(g["shapelet_preds"]), 1e-4, 1e-5, name + " shapelet logits")
    assert_close(logits, t(g["logits"]), 1e-4, 2e-5, name + " logits")
    assert torch.equal(logits.argmax(-1).cpu(), torch.as_tensor(g["logits"]).argmax(-1)), "predicted classes"
    assert_close(info.loss, t(g["reg_loss"]), 1e-5, 1e-7, name + " regulariser")
    assert_close(loss.reshape(()), t(g["loss"]).reshape(()), 1e-4, 1e-5, name + " loss")
    if is_ign:
        assert_close(info.eta, t(g["eta"]), 1e-4, 1e-6, name + " eta")
        assert_close(info.dnn_preds, t(g["dnn_preds"]), 1e-3, 1e-4, name + " deep logits (cuDNN)")
    for k, p in model.named_parameters():
        if "grad::" + k in g:
            ref = t(g["grad::" + k])
            assert_close(p.grad, ref, 1e-3, 2e-4 * float(ref.abs().max()) + 1e-7, name + " grad " + k)
        elif "gradsum::" + k in g:
            s, a = g["gradsum::" + k]
            assert abs(float(p.grad.double().abs().sum()) - a) <= 2e-2 * a + 1e-4, name + " |grad| checksum " + k


def test_eval_path_with_test_time_gating_and_amp():
    """test() calls forward with gating_value (experiment_classification.py:974); under bf16 autocast the
    shapelet maths stays fp32 as in the reference (SURVEY.md §7.3-7)."""
    model, g = build("model_jv_interpgn")
    model.eval()
    x = t(g["x"], DEV)
    with torch.no_grad():
        out1, info1 = model(x, None, None, None, gating_value=1.0)
        out0, info0 = model(x, None, None, None, gating_value=None)
        assert torch.allclose(out1, out0)                       # eta <= 1: gate at 1.0 never fires
        outg, infog = model(x, None, None, None, gating_value=0.0)
        assert torch.allclose(outg, infog.shapelet_preds, atol=1e-6) and bool((infog.eta == 1).all())
        with torch.autocast("cuda", dtype=torch.bfloat16):
            outa, infoa = model(x, None, None, None)
        assert infoa.p.dtype == torch.float32 and infoa.d.dtype == torch.float32
        assert_close(infoa.p, info0.p, 1e-6, 1e-7, "p under autocast")


def test_training_reduces_loss_and_pos_weight_step():
    model, g = build("model_jv_interpgn")
    x, y = t(g["x"], DEV), torch.as_tensor(g["y"]).to(DEV)
    opt = torch.optim.Adam(model.parameters(), lr=5e-3)
    losses = []
    for _ in range(12):
        logits, info = model(x, None, None, None)
        loss = torch.nn.functional.cross_entropy(logits, y) + info.loss.mean() + \
            torch.nn.functional.cross_entropy(info.shapelet_preds, y)
        opt.zero_grad()
        loss.backward()
        opt.step()
        model.step()
        losses.append(float(loss))
    assert losses[-1] < losses[0]
    assert float(model.sbm.output_layer.weight.min()) >= 0.0


# ---------------------------------------------------------------------------------------------------------------------
# Whole models at the BASELINE shapes, against fixtures frozen from the LIVE reference at exactly those shapes
# (tests/golden/make_golden.py full_model_case): config 2 = 125 ch x T=1000, 3 classes, default shapelet set, FCN expert,
# B=2, seed 42 (euclidean and cosine); config 5 = 39 classes with the Transformer expert (d_model 512, 2 layers).
# Weights and batch are regenerated from the seed (helpers.seeded_fill / seeded_batch; checksums are in the fixture).
# ---------------------------------------------------------------------------------------------------------------------
FULL_CASES = [
    # fixture, shapelet precision, (p/d rtol, atol)
    ("model_chisco_full", "fp32", 2e-5, 2e-6),
    ("model_chisco_full_cos", "fp32", 2e-5, 2e-6),
    ("model_chisco_full_cos", "3xtf32", 2e-5, 2e-6),          # the tcgen05 engine, fp32-equivalent operand split
    ("model_chisco_full_cos", "tf32", 3e-3, 3e-3),            # single-pass TF32: its own, looser tolerance
    ("model_chisco39_transformer", "fp32", 2e-5, 2e-6),
]


@pytest.mark.parametrize("name,precision,rtol,atol", FULL_CASES)
def test_full_size_model_matches_live_reference_golden(name, precision, rtol, atol):
    from models.InterpGN import InterpGN
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.set_float32_matmul_precision("highest")
    g = load_golden(name)
    kw = dict(zip(g["cfg_keys"].tolist(), g["cfg_vals"].tolist()))
    cfg = SimpleNamespace(epsilon=1., distance_func=kw.get("distance_func", "euclidean"), memory_efficient=False,
                          sbm_cls="linear", dropout=0., lambda_reg=0.1, lambda_div=0.1, dnn_type=kw.get("dnn_type", "FCN"),
                          enc_in=int(kw["enc_in"]), num_class=int(kw["num_class"]), seq_len=int(kw["seq_len"]),
                          shapelet_precision=precision, output_attention=False)
    for key in ("task_name", "embed", "freq", "activation"):
        if key in kw:
            setattr(cfg, key, kw[key])
    for key in ("pred_len", "label_len", "d_model", "factor", "n_heads", "d_ff", "e_layers"):
        if key in kw:
            setattr(cfg, key, int(kw[key]))
    seed, B = int(g["seed"]), int(g["B"])
    torch.manual_seed(seed)
    model = InterpGN(cfg)
    wsum = seeded_fill(model, seed)
    assert abs(wsum - float(g["weight_checksum"])) <= 1e-9 * abs(wsum), "seeded weights differ from the fixture's"
    x, y = seeded_batch(B, cfg.seq_len, cfg.enc_in, cfg.num_class, seed)
    assert abs(float(x.double().abs().sum()) - float(g["x_checksum"])) <= 1e-9 * float(g["x_checksum"])
    assert torch.equal(y, torch.as_tensor(g["y"]))
    model = model.to(DEV).train()
    x, y = x.to(DEV), y.to(DEV)
    logits, info = model(x, torch.ones(B, cfg.seq_len, device=DEV), None, None)
    loss = torch.nn.functional.cross_entropy(logits, y) + info.loss.mean() + \
        torch.nn.functional.cross_entropy(info.shapelet_preds, y)
    loss.backward()
    torch.cuda.synchronize()
    tag = "%s/%s" % (name, precision)
    assert_close(info.p, t(g["p"]), rtol, atol, tag + " p")                       # 2500 predicates per sample
    assert_close(info.d, t(g["d"]), rtol, atol, tag + " d")
    loose = 30.0 if precision == "tf32" else 1.0
    assert_close(info.shapelet_preds, t(g["shapelet_preds"]), 1e-4 * loose, 1e-5 * loose, tag + " shapelet logits")
    assert_close(info.dnn_preds, t(g["dnn_preds"]), 2e-3, 2e-4, tag + " deep logits (cuDNN / SDPA)")
    assert_close(info.eta, t(g["eta"]), 1e-3 * loose, 1e-6 * loose, tag + " eta")
    assert_close(logits, t(g["logits"]), 2e-3, 2e-4, tag + " logits")
    assert torch.equal(logits.argmax(-1).cpu(), torch.as_tensor(g["logits"]).argmax(-1)), "predicted classes"
    assert torch.equal(info.shapelet_preds.argmax(-1).cpu(), torch.as_tensor(g["shapelet_preds"]).argmax(-1))
    assert_close(info.loss, t(g["reg_loss"]), 1e-5, 1e-7, tag + " regulariser")
    assert_close(loss.reshape(()), t(g["loss"]).reshape(()), 1e-4 * loose, 1e-5, tag + " loss")
    n_sample = int(g["n_sample"])
    for k, p in model.named_parameters():
        if not k.startswith("sbm."):
            continue
        s, a, l2 = g["gradnorm::" + k]
        gd = p.grad.double().flatten()
        gtol = 1e-3 if precision != "tf32" else 3e-2
        assert abs(float(gd.pow(2).sum().sqrt()) - l2) <= gtol * l2, tag + " |grad|_2 of " + k
        assert abs(float(gd.abs().sum()) - a) <= gtol * a, tag + " |grad|_1 of " + k
        if "grad::" + k in g:
            ref = t(g["grad::" + k])
            assert_close(p.grad, ref, 10 * gtol, gtol * float(ref.abs().max()), tag + " grad " + k)
        else:
            idx = sample_indices(gd.numel(), n_sample, seed + 17)
            ref = t(g["gradsample::" + k])
            got = p.grad.flatten()[idx.to(DEV)]
            # shapelet gradients at 8192 seeded positions of each [5,125,L] tensor
            if precision == "tf32":
                # single-pass TF32 flips a few near-tie arg-maxes (SURVEY.md 7.3-4: ~0.1 %), which moves the hard one-hot
                # of those (sample, shapelet, channel) rows: bound the NUMBER of affected positions, not their size
                bad = (got.cpu().double() - ref.double()).abs() > 10 * gtol * ref.double().abs() + gtol * float(ref.abs().max())
                assert int(bad.sum()) <= 0.01 * bad.numel(), tag + " sampled grad %s: %d outliers" % (k, int(bad.sum()))
            else:
                assert_close(got, ref, 10 * gtol, gtol * float(ref.abs().max()), tag + " sampled grad " + k)


def test_overlapped_experts_give_identical_gradients():
    """The deep expert on its side stream is the same arithmetic as on the main stream: bit-identical gradients."""
    model, g = build("model_small_chisco")
    x, y = t(g["x"], DEV), torch.as_tensor(g["y"]).to(DEV)

    def grads():
        model.zero_grad(set_to_none=True)
        logits, info = model(x, None, None, None)
        (torch.nn.functional.cross_entropy(logits, y) + info.loss.mean()
         + torch.nn.functional.cross_entropy(info.shapelet_preds, y)).backward()
        torch.cuda.synchronize()
        return [p.grad.clone() for p in model.sbm.parameters()]

    model.overlap_experts = True
    overlapped = grads()
    model.overlap_experts = False
    serial = grads()
    for a, b in zip(overlapped, serial):
        assert torch.equal(a, b)


@pytest.mark.parametrize("name", ["model_jv_interpgn", "model_jv_interpgn_cos", "model_small_chisco"])
def test_saliency_input_gradient_through_the_whole_model(name):
    """dLoss/dx of the raw batch through instance norm, all length groups, the head, the gate and the deep expert —
    against autograd through the oracle restatement of the shapelet expert (fp64) with the same deep-expert gradient."""
    import ign_oracle as O
    from helpers import MODES
    model, g = build(name)
    model.overlap_experts = False
    x = t(g["x"], DEV).requires_grad_(True)
    y = torch.as_tensor(g["y"]).to(DEV)
    logits, info = model(x, torch.ones(x.shape[0], x.shape[1], device=DEV), None, None)
    # isolate the shapelet expert's path: its logits only (the deep expert's input gradient is plain cuDNN autograd)
    loss = torch.nn.functional.cross_entropy(info.shapelet_preds, y)
    loss.backward()
    torch.cuda.synchronize()
    kw = dict(zip(g["cfg_keys"].tolist(), g["cfg_vals"].tolist()))
    mode = MODES[kw.get("distance_func", "euclidean")][0]
    xr = t(g["x"]).double().requires_grad_(True)
    Ws = [s.weights.detach().cpu().double() for s in model.sbm.shapelets]
    Wc = model.sbm.output_layer.weight.detach().cpu().double()
    ref_logits, _, _ = O.sbm_forward(xr, Ws, [s.stride for s in model.sbm.shapelets], Wc, 1.0, mode)
    torch.nn.functional.cross_entropy(ref_logits, torch.as_tensor(g["y"])).backward()
    assert_close(x.grad, xr.grad, 1e-3, 2e-4 * float(xr.grad.abs().max()), name + " dLoss/dx")
