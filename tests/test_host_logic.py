"""CPU: host-side mirror of the reference interface — construction, naming, flag dispatch, loud failure."""
from types import SimpleNamespace

import pytest
import torch

from helpers import load_golden


def cfg(**kw):
    base = dict(enc_in=12, num_class=9, seq_len=29, epsilon=1., distance_func='euclidean', memory_efficient=False,
                sbm_cls='linear', dropout=0., lambda_reg=0.1, lambda_div=0.1, dnn_type='FCN')
    base.update(kw)
    return SimpleNamespace(**base)


def test_flag_dispatch_matches_reference():
    from layers.shapelet_ops import resolve_dist
    assert resolve_dist("euclidean", False) == "l1"          # Shapelet.py:74
    assert resolve_dist("euclidean", True) == "sql2"         # Shapelet.py:72 -> :28
    assert resolve_dist("cosine", True) == "cosine"          # memory_efficient only consulted in the else branch
    assert resolve_dist("pearson", False) == "pearson"
    assert resolve_dist("anything-else", False) == "l1"      # the reference's `else:`


def test_interpgn_shapes_and_state_dict_keys_match_reference():
    from models.InterpGN import InterpGN
    torch.manual_seed(0)
    m = InterpGN(cfg())
    assert m.sbm.shapelet_len == [3, 6, 9, 15] and m.sbm.total_shapelets == 240
    assert sum(p.numel() for p in m.sbm.parameters()) == 4140           # SURVEY.md §8c
    assert sum(p.numel() for p in m.parameters()) == 281269
    g = load_golden("model_jv_interpgn")
    ref_keys = sorted(k[4:] for k in g if k.startswith("sd::"))
    assert sorted(m.state_dict().keys()) == ref_keys
    for k, v in m.state_dict().items():
        assert tuple(v.shape) == tuple(g["sd::" + k].shape), k
    # same initialiser / RNG consumption as the reference for the shapelets (seed 0)
    assert torch.allclose(m.sbm.shapelets[0].weights.detach(), torch.as_tensor(g["sd::sbm.shapelets.0.weights"]))


def test_chisco_shapes():
    from models.Shapelet import ShapeBottleneckModel
    m = ShapeBottleneckModel(cfg(enc_in=125, num_class=3, seq_len=1000))
    assert m.shapelet_len == [100, 200, 300, 500] and m.total_shapelets == 2500
    assert sum(p.numel() for p in m.parameters()) == 695000
    assert [s.stride for s in m.shapelets] == [1, 1, 1, 1]
    big = ShapeBottleneckModel(cfg(enc_in=2, num_class=3, seq_len=4000))
    assert [(s.length, s.stride) for s in big.shapelets] == [(400, 8), (800, 9), (1200, 10), (2000, 10)]


def test_lts_keys_and_doubled_length_list():
    from models.Shapelet import DistThresholdSBM
    m = DistThresholdSBM(cfg())
    assert m.shapelet_len == [3, 6, 9, 15, 3, 6, 9, 15]
    keys = set(m.state_dict().keys())
    assert {"shapelets.0.weights", "shapelets.0.threshold", "output_layer.weight"} <= keys
    assert m.shapelets[0].threshold.shape == (1, 5, 12)


@pytest.mark.parametrize("cls", ["bilinear", "attention"])
def test_alternate_heads_construct(cls):
    from models.Shapelet import ShapeBottleneckModel
    m = ShapeBottleneckModel(cfg(sbm_cls=cls))
    assert ("output_bilinear.weight" in m.state_dict()) == (cls == "bilinear")
    assert ("attention.q_proj.weight" in m.state_dict()) == (cls == "attention")


def test_regulariser_matches_reference_golden_on_cpu():
    """loss() touches parameters only, so it is checkable without a GPU."""
    from models.Shapelet import ShapeBottleneckModel
    g = load_golden("model_jv_sbm")
    m = ShapeBottleneckModel(cfg())
    m.load_state_dict({k[4:]: torch.as_tensor(v) for k, v in g.items() if k.startswith("sd::")})
    assert abs(float(m.loss()) - float(g["reg_loss"][0])) < 1e-7
    m.step()
    assert float(m.output_layer.weight.min()) >= 0.0


def test_cpu_tensors_fail_loudly():
    from models.InterpGN import InterpGN
    m = InterpGN(cfg())
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.randn(2, 29, 12), torch.ones(2, 29))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.sbm.shapelets[0](torch.randn(2, 12, 29))


def test_unknown_dnn_type_is_rejected():
    from models.InterpGN import InterpGN
    with pytest.raises(ValueError):
        InterpGN(cfg(dnn_type="TimesNet"))


def test_product_code_never_imports_the_oracle():
    import os
    import re
    root = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "speech-imagery-eeg_b200")
    for dp, _, files in os.walk(root):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(import|from)\s+(ign_oracle|ref_shim|oracle)\b", src, re.M), f


def test_transformer_expert_matches_reference_golden_on_cpu():
    """The deep expert is plain PyTorch (SDPA instead of the reference's materialised attention), so its parity
    against the reference's outputs is checkable without a GPU."""
    from models.Transformer import Model
    g = load_golden("model_small_transformer")
    kw = dict(zip(g["cfg_keys"].tolist(), g["cfg_vals"].tolist()))
    c = cfg(enc_in=int(kw["enc_in"]), num_class=int(kw["num_class"]), seq_len=int(kw["seq_len"]), task_name="classification",
            d_model=int(kw["d_model"]), embed="timeF", freq="h", n_heads=int(kw["n_heads"]), d_ff=int(kw["d_ff"]),
            activation="gelu", e_layers=int(kw["e_layers"]))
    m = Model(c)
    sd = {k[len("sd::deep_model."):]: torch.as_tensor(v) for k, v in g.items() if k.startswith("sd::deep_model.")}
    assert sorted(sd) == sorted(m.state_dict())
    m.load_state_dict(sd)
    x = torch.as_tensor(g["x"])
    with torch.no_grad():
        out = m(x, torch.ones(x.shape[0], x.shape[1]), None, None)
    assert torch.allclose(out, torch.as_tensor(g["dnn_preds"]), rtol=1e-4, atol=1e-5)


def test_bench_dump_outputs_keeps_its_size_limit_and_samples_the_same_positions_every_run(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float32 / float64 .npy files; past the size limit, a sample at positions fixed by name."""
    import os
    import numpy as np
    import bench
    g = torch.Generator().manual_seed(0)
    arrays = {"loss": torch.tensor(1.5), "model.w": torch.randn(300, 40, generator=g), "model.n": torch.tensor(7),
              "model.h": torch.randn(1000, generator=g).half()}
    bench.dump_outputs(str(tmp_path / "full"), arrays)
    full = {k: np.load(tmp_path / "full" / (k + ".npy")) for k in arrays}
    assert [full[k].dtype for k in arrays] == [np.float32, np.float32, np.float64, np.float32]
    assert np.array_equal(full["model.w"], arrays["model.w"].numpy()) and float(full["model.n"]) == 7.0
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4 * 1024 + 20000)        # 20000 payload bytes for 52012
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays)
    assert sum(os.path.getsize(p) for p in (tmp_path / "a").iterdir()) <= bench.DUMP_LIMIT_BYTES
    for k in arrays:
        a, b = np.load(tmp_path / "a" / (k + ".npy")), np.load(tmp_path / "b" / (k + ".npy"))
        assert np.array_equal(a, b) and np.isin(a, full[k]).all()
    assert 0 < np.load(tmp_path / "a" / "model.w.npy").size < 300 * 40


def test_reference_arm_line_contract():
    """`bench.py --impl reference` (the oracle port timed on the host cores): one JSON line with the bench contract's keys
    on rank 0, silence and exit 0 on the other ranks of a torchrun launch."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0 and out.stdout.strip() == ""
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "train samples/sec" and line["unit"] == "samples/s"
    assert line["value"] > 0 and line["steps"] == 1 and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["config"]["workload"].startswith("InterpGN(FCN)") and line["data"] == "synthetic"
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    e2e = line["e2e"]
    assert e2e["value"] == line["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
