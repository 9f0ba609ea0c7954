"""Generate golden vectors from the UNMODIFIED live reference.

    IGN_REFERENCE_ROOT=<InterpretGatedNetwork checkout> python tests/golden/make_golden.py

Imports the reference's model/{Shapelet,InterpGN,FullyConvNet}.py through oracle/ref_shim.py, runs them
on seeded CPU inputs and freezes inputs + outputs + gradients into tests/golden/*.npz.  The reference
has no tests/golden vectors of its own (SURVEY.md §4), so these files are the parity pin for
oracle/ign_oracle.py and (through it, and directly) for the CUDA path.  The repository does not carry
the reference; the .npz files are what the tests compare against.
"""
import os
import sys
from types import SimpleNamespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "..", "oracle"))
sys.path.insert(0, os.path.join(HERE, ".."))
import ref_shim  # noqa: E402
from helpers import sample_indices, seeded_batch, seeded_fill  # noqa: E402

ns = ref_shim.load_reference()
torch.set_num_threads(4)


def np_(t):
    return t.detach().cpu().numpy()


def layer_case(name, cls, M, L, K, T, B, stride, eps, dfunc, seed, structured=False):
    torch.manual_seed(seed)
    layer = cls(M, L, K, stride=stride, eps=eps, distance_func=dfunc)
    if structured:
        t = torch.arange(T, dtype=torch.float32)
        xn = torch.sin(t[None, None, :] * (0.05 + 0.03 * torch.rand(B, M, 1)) + 6.28 * torch.rand(B, M, 1))
        xn = xn + 0.1 * torch.randn(B, M, T)
    else:
        xn = torch.randn(B, M, T)
    g = torch.randn(B, K, M)
    p, dmin = layer(xn)
    (p.view(B, K, M) * g).sum().backward()
    out = dict(xn=np_(xn), W=np_(layer.weights), g=np_(g), p=np_(p), dmin=np_(dmin),
               dW=np_(layer.weights.grad), stride=stride, eps=eps, dfunc=dfunc,
               pool="lts_min" if cls is ns.DistThresholdShapelet else "rbf_max")
    if hasattr(layer, "threshold"):
        out["threshold"] = np_(layer.threshold)
        out["dthreshold"] = np_(layer.threshold.grad)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, p.shape)


def kat_cases():
    """Known-answer vectors of SURVEY.md §8c (x=[0..4], L=3, eps=1, single channel/shapelet)."""
    rows = {}
    for dfunc, w in (("euclidean", [1., 1., 1.]), ("cosine", [1., 1., 1.]), ("pearson", [1., 2., 4.])):
        s = ns.Shapelet(1, 3, 1, distance_func=dfunc)
        with torch.no_grad():
            s.weights.copy_(torch.tensor([[w]]))
        x = torch.tensor([[[0., 1., 2., 3., 4.]]])
        p, dmin = s(x)
        p.sum().backward()
        rows[dfunc + "_W"] = np.array(w, dtype=np.float32)
        rows[dfunc + "_p"] = np_(p)
        rows[dfunc + "_dmin"] = np_(dmin)
        rows[dfunc + "_dW"] = np_(s.weights.grad)
    np.savez_compressed(os.path.join(HERE, "kat.npz"), **rows)
    print("kat", {k: v.ravel().tolist() for k, v in rows.items()})


def sql2_case():
    """memory_efficient arithmetic (Shapelet.py:28,34-39): the reference's shape plumbing is broken
    when called from Shapelet.forward (SURVEY.md §0), so the Function is driven directly on the
    [B,M,T] series (its own slicing convention), then pooled by the reference lines 77-84 verbatim
    through a Shapelet whose distance is pre-computed."""
    torch.manual_seed(7)
    B, M, T, K, L, eps = 3, 4, 37, 5, 8, 0.9
    xn = torch.randn(B, M, T)
    W = torch.randn(K, M, L, requires_grad=True)
    d = ns.ShapeletDistanceFunc.apply(xn, W)             # [B,T',K,M]
    p = torch.exp(-torch.pow(eps * d, 2))
    hard = torch.zeros_like(p).scatter_(1, p.argmax(dim=1, keepdim=True), 1.)
    soft = torch.softmax(p, dim=1)
    max_p = torch.sum((hard + soft - soft.detach()) * p, dim=1)
    g = torch.randn(B, K, M)
    (max_p * g).sum().backward()
    np.savez_compressed(os.path.join(HERE, "layer_sql2.npz"), xn=np_(xn), W=np_(W), g=np_(g),
                        p=np_(max_p.flatten(1)), dmin=np_(d.min(dim=1).values.flatten(1)),
                        dW=np_(W.grad), stride=1, eps=eps, dfunc="sql2", pool="rbf_max")
    print("layer_sql2", max_p.shape)


def model_case(name, cfg_kw, B, seed, gating_value=None, cls="InterpGN"):
    cfg = SimpleNamespace(epsilon=1., distance_func="euclidean", memory_efficient=False,
                          sbm_cls="linear", dropout=0., lambda_reg=0.1, lambda_div=0.1, dnn_type="FCN")
    for k, v in cfg_kw.items():
        setattr(cfg, k, v)
    keep_deep_grads = cfg.dnn_type != "FCN"      # small expert: keep its gradients too
    torch.manual_seed(seed)
    model = getattr(ns, cls)(cfg)
    model.train()
    x = torch.randn(B, cfg.seq_len, cfg.enc_in)
    y = torch.randint(0, cfg.num_class, (B,))
    mask = torch.ones(B, cfg.seq_len)
    if cls == "InterpGN":
        logits, info = model(x, mask, None, None, gating_value=gating_value)
    else:
        logits, info = model(x, mask, None, None)
    loss = torch.nn.functional.cross_entropy(logits, y) + info.loss.mean()
    if cls == "InterpGN":
        loss = loss + 1.0 * torch.nn.functional.cross_entropy(info.shapelet_preds, y)
    loss.backward()
    out = dict(x=np_(x), y=np_(y), logits=np_(logits), p=np_(info.p), d=np_(info.d),
               reg_loss=np_(info.loss), loss=np_(loss), shapelet_preds=np_(info.shapelet_preds),
               gating_value=np.array(np.nan if gating_value is None else gating_value),
               cfg_keys=np.array(list(cfg_kw.keys())), cfg_vals=np.array([str(v) for v in cfg_kw.values()]))
    if cls == "InterpGN":
        out["eta"] = np_(info.eta)
        out["dnn_preds"] = np_(info.dnn_preds)
    for k, v in model.state_dict().items():
        out["sd::" + k] = np_(v)
    for k, v in model.named_parameters():
        if v.grad is None:                    # e.g. the unused temporal embedding of the Transformer expert
            continue
        if k.startswith("deep_model.") and not keep_deep_grads:      # not our kernels' gradients: keep a checksum only
            out["gradsum::" + k] = np.array([float(v.grad.double().sum()), float(v.grad.double().abs().sum())])
        else:
            out["grad::" + k] = np_(v.grad)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, logits.shape, float(loss.detach()))


def full_model_case(name, cfg_kw, B, seed, n_sample=8192):
    """Whole models at the BASELINE shapes (config 2: 125 ch x T=1000, 3 classes; config 5: 39 classes, Transformer
    expert d_model 512).  The state dict (4-100 MB) and the batch are NOT stored: both are regenerated from `seed` by
    tests/helpers.py (seeded_fill / seeded_batch) and the fixture keeps checksums of them, the reference's outputs,
    and its parameter gradients as (sum, sum|.|, L2) plus the values at `n_sample` seeded positions per tensor
    (output head in full)."""
    cfg = SimpleNamespace(epsilon=1., distance_func="euclidean", memory_efficient=False,
                          sbm_cls="linear", dropout=0., lambda_reg=0.1, lambda_div=0.1, dnn_type="FCN")
    for k, v in cfg_kw.items():
        setattr(cfg, k, v)
    torch.manual_seed(seed)
    model = ns.InterpGN(cfg)
    model.train()
    wsum = seeded_fill(model, seed)
    x, y = seeded_batch(B, cfg.seq_len, cfg.enc_in, cfg.num_class, seed)
    mask = torch.ones(B, cfg.seq_len)
    logits, info = model(x, mask, None, None)
    loss = torch.nn.functional.cross_entropy(logits, y) + info.loss.mean() \
        + 1.0 * torch.nn.functional.cross_entropy(info.shapelet_preds, y)
    loss.backward()
    out = dict(seed=np.array(seed), B=np.array(B), weight_checksum=np.array(wsum),
               x_checksum=np.array(float(x.double().abs().sum())), y=np_(y),
               logits=np_(logits), p=np_(info.p), d=np_(info.d), reg_loss=np_(info.loss), loss=np_(loss),
               shapelet_preds=np_(info.shapelet_preds), eta=np_(info.eta), dnn_preds=np_(info.dnn_preds),
               n_sample=np.array(n_sample),
               cfg_keys=np.array(list(cfg_kw.keys())), cfg_vals=np.array([str(v) for v in cfg_kw.values()]))
    for k, v in model.named_parameters():
        if v.grad is None:
            continue
        gd = v.grad.double().flatten()
        out["gradnorm::" + k] = np.array([float(gd.sum()), float(gd.abs().sum()), float(gd.pow(2).sum().sqrt())])
        if k.startswith("sbm."):
            if k.endswith("output_layer.weight"):
                out["grad::" + k] = np_(v.grad)
            else:
                idx = sample_indices(gd.numel(), n_sample, seed + 17)
                out["gradsample::" + k] = np_(v.grad.flatten()[idx])
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, logits.shape, float(loss.detach()))


TRANSFORMER_KW = dict(dnn_type="Transformer", task_name="classification", pred_len=0, label_len=0, output_attention=False,
                      d_model=512, embed="timeF", freq="h", factor=1, n_heads=8, d_ff=2048, activation="gelu", e_layers=2,
                      dec_in=7, c_out=7, d_layers=1)


def new_cases():
    """Round-2 additions (kept separate so the round-1 fixtures are not rewritten)."""
    jv = dict(enc_in=12, num_class=9, seq_len=29)
    model_case("model_jv_sbm_bilinear", dict(enc_in=4, num_class=9, seq_len=29, sbm_cls="bilinear"), B=4, seed=3,
               cls="ShapeBottleneckModel")
    model_case("model_jv_sbm_attention", dict(jv, sbm_cls="attention"), B=4, seed=4, cls="ShapeBottleneckModel")
    model_case("model_jv_interpgn_attention", dict(jv, sbm_cls="attention"), B=4, seed=5)
    chisco = dict(enc_in=125, num_class=3, seq_len=1000)
    full_model_case("model_chisco_full", chisco, B=2, seed=42)
    full_model_case("model_chisco_full_cos", dict(chisco, distance_func="cosine"), B=2, seed=42)
    full_model_case("model_chisco39_transformer", dict(enc_in=125, num_class=39, seq_len=1000, **TRANSFORMER_KW), B=2, seed=7)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "new":
        new_cases()
        sys.exit(0)
    kat_cases()
    S, D = ns.Shapelet, ns.DistThresholdShapelet
    layer_case("layer_l1", S, M=4, L=9, K=5, T=40, B=3, stride=1, eps=1.3, dfunc="euclidean", seed=1)
    layer_case("layer_l1_stride", S, M=3, L=11, K=7, T=64, B=2, stride=3, eps=1.0, dfunc="euclidean", seed=2)
    layer_case("layer_cosine", S, M=4, L=9, K=5, T=40, B=3, stride=1, eps=1.3, dfunc="cosine", seed=3)
    layer_case("layer_pearson", S, M=4, L=9, K=5, T=40, B=3, stride=1, eps=1.3, dfunc="pearson", seed=4)
    layer_case("layer_cosine_stride", S, M=3, L=12, K=6, T=70, B=2, stride=3, eps=0.8, dfunc="cosine", seed=5)
    layer_case("layer_l1_struct", S, M=5, L=32, K=5, T=160, B=2, stride=1, eps=1.0, dfunc="euclidean", seed=6,
               structured=True)
    layer_case("layer_lts", D, M=4, L=9, K=5, T=40, B=3, stride=1, eps=1.0, dfunc="euclidean", seed=8)
    layer_case("layer_l1_min", S, M=1, L=3, K=1, T=3, B=1, stride=1, eps=1.0, dfunc="euclidean", seed=9)
    layer_case("layer_pearson_k12", S, M=2, L=20, K=12, T=96, B=2, stride=1, eps=1.0, dfunc="pearson", seed=10)
    sql2_case()
    jv = dict(enc_in=12, num_class=9, seq_len=29)
    model_case("model_jv_interpgn", jv, B=4, seed=0)
    model_case("model_jv_interpgn_gate", jv, B=4, seed=42, gating_value=0.3)
    model_case("model_jv_interpgn_cos", dict(jv, distance_func="cosine"), B=4, seed=1234)
    model_case("model_jv_sbm", jv, B=4, seed=0, cls="ShapeBottleneckModel")
    model_case("model_jv_lts", jv, B=4, seed=0, cls="DistThresholdSBM")
    model_case("model_small_chisco", dict(enc_in=7, num_class=3, seq_len=120), B=2, seed=42)
    # Transformer deep expert (BASELINE config 5 in miniature): run.py defaults scaled down
    model_case("model_small_transformer", dict(enc_in=7, num_class=5, seq_len=64, dnn_type="Transformer",
               task_name="classification", pred_len=0, label_len=0, output_attention=False, d_model=32, embed="timeF",
               freq="h", factor=1, n_heads=4, d_ff=64, activation="gelu", e_layers=2, dec_in=7, c_out=7, d_layers=1),
               B=3, seed=7)
    new_cases()
