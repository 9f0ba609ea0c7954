"""CPU: the oracle's deep-expert restatements (oracle/ign_oracle_experts.py, used by bench.py's reference arm) against
the golden vectors frozen from the live reference — same state dict (identical parameter names), same inputs."""
from types import SimpleNamespace

import pytest
import torch

import ign_oracle_experts as E
from helpers import assert_close, load_golden, t


def _cfg(g):
    kw = dict(zip(g["cfg_keys"].tolist(), g["cfg_vals"].tolist()))
    c = SimpleNamespace(enc_in=int(kw["enc_in"]), num_class=int(kw["num_class"]), seq_len=int(kw["seq_len"]), dropout=0.0,
                        activation=kw.get("activation", "gelu"))
    for k in ("d_model", "n_heads", "d_ff", "e_layers"):
        if k in kw:
            setattr(c, k, int(kw[k]))
    return c, kw.get("dnn_type", "FCN")


@pytest.mark.parametrize("name", ["model_jv_interpgn", "model_small_chisco", "model_small_transformer"])
def test_expert_restatement_matches_reference_golden(name):
    g = load_golden(name)
    cfg, kind = _cfg(g)
    net = E.build_expert(kind, cfg).train()
    sd = {k[len("sd::deep_model."):]: torch.as_tensor(v) for k, v in g.items() if k.startswith("sd::deep_model.")}
    missing, unexpected = net.load_state_dict(sd, strict=True)
    x = t(g["x"])
    out = net(x, torch.ones(x.shape[0], x.shape[1]))
    assert_close(out, t(g["dnn_preds"]), 1e-5, 1e-6, name + " deep expert logits")


def test_expert_restatement_against_live_reference_if_mounted():
    import ref_shim
    if not ref_shim.available():
        pytest.skip("IGN_REFERENCE_ROOT does not name a reference checkout")
    ns = ref_shim.load_reference()
    torch.manual_seed(3)
    cfg = SimpleNamespace(enc_in=5, num_class=4, seq_len=40, dropout=0.0, activation="gelu", d_model=16, n_heads=2,
                          d_ff=32, e_layers=2, task_name="classification", pred_len=0, label_len=0, output_attention=False,
                          embed="timeF", freq="h", factor=1)
    x = torch.randn(3, 40, 5)
    for kind, ref in (("FCN", ns.FullyConvNetwork(cfg)), ("Transformer", ns.Transformer(cfg))):
        mine = E.build_expert(kind, cfg)
        mine.load_state_dict(ref.state_dict(), strict=True)
        a = ref(x, torch.ones(3, 40), None, None)
        b = mine(x, torch.ones(3, 40))
        assert_close(b, a, 1e-6, 1e-6, kind)
