"""GPU: the product API end to end, as a user drives it — run.py's main() in-process (the reference's entry point,
run.py:490-692 -> Experiment.train()/test(), experiment_classification.py:295-378, :828-1138), leave-one-subject-out
fold batching, the real-data path on a generated UEA archive, and (on >= 2 GPUs) NCCL data parallelism."""
import os
import pickle
import subprocess
import sys

import pytest
import torch

from helpers import load_golden

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "speech-imagery-eeg_b200")


def _run_main(argv, tmp_path, monkeypatch):
    import run
    monkeypatch.chdir(tmp_path)                      # checkpoints/ and results go under the test's directory
    return run, run.main(argv)


def test_run_py_trains_tests_and_checkpoints_with_reference_keys(tmp_path, monkeypatch):
    """run_uea.sh's flag set on JapaneseVowels-shaped synthetic series (BASELINE config 1), 6 epochs."""
    argv = ["--model", "InterpGN", "--dnn_type", "FCN", "--dataset", "JapaneseVowels", "--train_epochs", "6",
            "--batch_size", "32", "--lr", "5e-3", "--dropout", "0.", "--num_shapelet", "10", "--lambda_div", "0.1",
            "--lambda_reg", "0.1", "--epsilon", "1", "--beta_schedule", "constant", "--seed", "0", "--gating_value", "1",
            "--amp", "--log_interval", "1", "--syn_train", "256", "--syn_val", "64", "--syn_test", "64", "--cuda_graph"]
    run, results = _run_main(argv, tmp_path, monkeypatch)
    assert len(results) == 1
    loss, acc = results[0]
    assert loss == loss and loss < 10 and 0.0 <= acc <= 1.0
    ckpts = [os.path.join(dp, f) for dp, _, fs in os.walk(tmp_path / "checkpoints") for f in fs if f == "checkpoint.pth"]
    assert len(ckpts) == 1 and "JapaneseVowels-synthetic" in ckpts[0]          # the data source is part of the path
    sd = torch.load(ckpts[0], map_location="cpu")
    g = load_golden("model_jv_interpgn")
    ref_keys = sorted(k[4:] for k in g if k.startswith("sd::"))                  # the live reference's state-dict keys
    assert sorted(sd.keys()) == ref_keys
    for k in ref_keys:
        assert tuple(sd[k].shape) == tuple(g["sd::" + k].shape), k
    pk = os.path.join(os.path.dirname(ckpts[0]), "test_results.pkl")
    with open(pk, "rb") as f:
        res = pickle.load(f)
    assert res["args"]["data_source"] == "synthetic" and res["test_metrics"].p.shape[1] == 240
    # a second invocation finds the checkpoint and only tests (run.py:582-585)
    _, again = _run_main(argv, tmp_path, monkeypatch)
    assert abs(again[0][0] - loss) < 1e-4


def test_experiment_train_reduces_the_loss_and_learns_the_synthetic_classes(tmp_path, monkeypatch):
    import run
    from exp.experiment_classification import Experiment
    monkeypatch.chdir(tmp_path)
    args = run.get_args(["--dataset", "BasicMotions", "--dnn_type", "FCN", "--train_epochs", "12", "--batch_size", "32",
                         "--seed", "0", "--amp", "--syn_train", "256", "--syn_val", "64", "--syn_test", "64", "--pos_weight"])
    run.set_seed(0)
    exp = Experiment(args)
    exp.train()
    first, last = exp.history[0], exp.history[-1]
    assert last[1] < first[1], exp.history                     # training loss went down through the product's _loss
    loss, res, _ = exp.test()
    assert res.accuracy > 1.5 / args.num_class                 # better than chance on class-conditional synthetic series
    assert float(exp.model.sbm.output_layer.weight.min()) >= 0.0           # --pos_weight clamp ran after every step
    assert res.eta.shape == (64, 1) and res.d.shape == res.p.shape == (64, exp.model.sbm.total_shapelets)


def test_loso_fold_batching_runs_on_the_gpu(tmp_path, monkeypatch):
    argv = ["--loso", "--syn_subjects", "3", "--dataset", "JapaneseVowels", "--dnn_type", "FCN", "--train_epochs", "3",
            "--batch_size", "32", "--seed", "0", "--amp", "--syn_train", "192", "--syn_val", "32", "--syn_test", "32"]
    run, merged = _run_main(argv, tmp_path, monkeypatch)
    assert sorted(v[0] for v in merged.values()) == [0, 1, 2]                   # one fold per held-out subject
    assert all(v[2] is not None and 0.0 <= v[2] <= 1.0 for v in merged.values())
    results = [os.path.join(dp, f) for dp, _, fs in os.walk(tmp_path / "checkpoints") for f in fs if f == "fold_result.json"]
    assert len(results) == 3                                                     # each fold's result is on disk


def test_real_uea_archive_with_longer_test_series_and_transformer_expert(tmp_path, monkeypatch):
    """Variable-length archive whose TEST series are longer than its TRAIN series, default Transformer expert
    (Linear(d_model * seq_len)): every split is padded to one length, so validation and test do not crash."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import make_toy_uea as mk
    from data_provider.data_factory import SyntheticSeries
    d = tmp_path / "uea" / "Toy"
    d.mkdir(parents=True)
    gen = torch.Generator().manual_seed(0)
    tr, te = SyntheticSeries(6, 60, 4, 96, 11), SyntheticSeries(6, 60, 4, 48, 33)
    tr.x = tr.x[:, :50]                                  # train series at most 50 steps, test series up to 60
    mk.write(str(d / "Toy_TRAIN.ts"), tr, gen)
    mk.write(str(d / "Toy_TEST.ts"), te, gen)
    argv = ["--data", "UEA", "--data_root", str(tmp_path / "uea"), "--dataset", "Toy", "--dnn_type", "Transformer",
            "--d_model", "32", "--n_heads", "4", "--d_ff", "64", "--train_epochs", "2", "--batch_size", "16", "--seed", "0",
            "--amp"]
    run, results = _run_main(argv, tmp_path, monkeypatch)
    assert results[0][0] == results[0][0] and results[0][1] is not None


NCCL_SCRIPT = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %(pkg)r)
from types import SimpleNamespace
from exp.parallel import FlatGradAllReduce, init_distributed
from models.InterpGN import InterpGN
rank, local, world = init_distributed()
dev = torch.device("cuda", local); torch.cuda.set_device(dev)
cfg = SimpleNamespace(enc_in=12, num_class=9, seq_len=29, epsilon=1., distance_func="euclidean", memory_efficient=False,
                      sbm_cls="linear", dropout=0., lambda_reg=0.1, lambda_div=0.1, dnn_type="FCN")
def build():
    torch.manual_seed(0)
    m = InterpGN(cfg).to(dev).train()
    m.deep_model.eval()          # BatchNorm uses running statistics: the deep expert no longer depends on the batch split
    return m
def loss_of(m, x, y):
    out, info = m(x, torch.ones(x.shape[0], x.shape[1], device=dev), None, None)
    return torch.nn.functional.cross_entropy(out, y) + info.loss.mean() + torch.nn.functional.cross_entropy(info.shapelet_preds, y)
g = torch.Generator().manual_seed(5)
X = torch.randn(16 * world, 29, 12, generator=g).to(dev); Y = torch.randint(0, 9, (16 * world,), generator=g).to(dev)
# data parallel: every rank takes its shard, gradients averaged by the flat NCCL all-reduce
m = build()
pl = FlatGradAllReduce(m, world)
pl.zero_grad(); pl.arm()
loss_of(m, X[rank * 16:(rank + 1) * 16], Y[rank * 16:(rank + 1) * 16]).backward()
pl.finish()
# single process, full batch
ref = build()
loss_of(ref, X, Y).backward()
worst = 0.0
for (n, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
    scale = float(q.grad.abs().max()) + 1e-12
    worst = max(worst, float((p.grad - q.grad).abs().max()) / scale)
flat = pl.flat.clone()
dist.all_reduce(flat, op=dist.ReduceOp.MAX)
same = bool(torch.equal(flat, pl.flat))
dist.barrier()
if rank == 0:
    print("NCCL_GRAD_CHECK worst_rel=%%.3e identical_across_ranks=%%s world=%%d" %% (worst, same, world))
dist.destroy_process_group()
'''


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_nccl_two_rank_gradients_equal_full_batch_gradients(tmp_path):
    """N-rank averaged gradients == single-process full-batch gradients for InterpGN (shapelet expert, gate, head and
    deep expert), through the product's FlatGradAllReduce on NCCL."""
    script = tmp_path / "nccl_check.py"
    script.write_text(NCCL_SCRIPT % {"pkg": PKG})
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29531", str(script)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-4000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("NCCL_GRAD_CHECK")][0]
    worst = float(line.split("worst_rel=")[1].split()[0])
    assert worst < 2e-4, line
    assert "identical_across_ranks=True" in line


def test_cuda_graph_replay_is_the_same_training_as_the_eager_step(tmp_path, monkeypatch):
    """--cuda_graph replays forward + backward + Adam (+ clamp, gradient reset) of a full batch from one captured graph.
    Same kernels, same order: the parameters after N steps equal those of the eager loop (which here repeats the
    capture's three warm-up steps on the first batch, as the graphed path does; the capture pass itself only records)."""
    import copy
    import run
    from exp.experiment_classification import Experiment
    monkeypatch.chdir(tmp_path)
    base = run.get_args(["--dataset", "JapaneseVowels", "--dnn_type", "FCN", "--batch_size", "32", "--seed", "0", "--amp",
                         "--syn_train", "64", "--syn_val", "32", "--syn_test", "32", "--pos_weight"])
    torch.backends.cudnn.deterministic = True
    gen = torch.Generator().manual_seed(3)
    batches = [(torch.randn(32, 29, 12, generator=gen).cuda(), torch.randint(0, 9, (32,), generator=gen).cuda(),
                torch.ones(32, 29).cuda()) for _ in range(5)]
    params = {}
    for mode in ("eager", "graph"):
        args = copy.copy(base)
        args.cuda_graph = mode == "graph"
        run.set_seed(0)
        exp = Experiment(args)
        exp.model.train()
        exp.grads.zero_grad()
        losses = []
        for i, (x, y, m) in enumerate(batches):
            if mode == "eager" and i == 0:
                for _ in range(3):                           # the 3 warm-up steps of the graphed path
                    exp.train_step(x, y, m, 0, 1)
            losses.append(float(exp.train_step(x, y, m, 0, i + 1)))
        if mode == "graph":
            assert exp._graph is not None
            # a ragged batch falls back to the eager step and keeps training the same parameters
            exp.train_step(batches[0][0][:7], batches[0][1][:7], batches[0][2][:7], 0, 9)
        params[mode] = ([p.detach().clone() for p in exp.model.parameters()], losses)
    for le, lg in zip(params["eager"][1], params["graph"][1]):
        assert abs(le - lg) <= 1e-4 * abs(le) + 1e-6, (params["eager"][1], params["graph"][1])


def test_bench_line_contract_of_our_arm(tmp_path):
    """`python bench.py` on one GPU (small batch, few steps, no extras): ONE JSON line with every key the measurement
    contract names — whole-job value, end-to-end object with its copy sizes, launch count, clocks, a roofline for the
    dominant kernel with live timing, per-kernel entries, engines as the library reported them — and the last timed
    step's outputs as .npy files."""
    import json
    import numpy as np
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    dump = tmp_path / "outputs"
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "3", "--warmup", "3", "--batch", "16",
                          "--no_extras", "--no_cpu_baseline", "--dump-outputs", str(dump)],
                         capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [ln for ln in out.stdout.strip().splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["metric"] == "train samples/sec" and d["unit"] == "samples/s" and d["n_gpus"] == 1
    assert d["steps"] == 3 and d["warmup"] == 3 and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and d["dtype"] == "f32"
    assert d["value"] > 0 and abs(d["value"] - 16 * 1e3 / d["ms_per_step"]) < 1e-6 * d["value"]
    assert d["config"]["workload"].startswith("InterpGN(FCN)") and "model" not in d["config"]
    e = d["e2e"]
    assert e["value"] > 0 and e["unit"] == "samples/s" and e["d2h_bytes_per_step"] == 4
    assert e["h2d_bytes_per_step"] == 16 * 1000 * 125 * 4 + 16 * 8 + 16 * 1000
    assert e["value"] != d["value"]
    assert d["gpu_launches"] > 0 and "sm_mhz" in d["clocks"] and isinstance(d["clocks"]["reasons"], list)
    r = d["roofline"]
    assert r["kernel"] == "bwd.contraction" and r["bound"] == "fp32_alu" and r["unit"] == "TFLOP/s"
    assert 0 < r["frac"] < 1 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["avg_ms"] > 0
    names = {k["kernel"] for k in d["rooflines"]}
    assert {"shapelet_fwd", "shapelet_bwd", "bwd.pool_bwd", "bwd.tie_check", "bwd.contraction", "instnorm"} <= names
    assert set(d["engines"].values()) == {"fp32"}               # the default L1 distance has no tensor-core form
    files = {p.name: np.load(p) for p in dump.iterdir()}
    assert files["loss.npy"].shape == () and np.isfinite(files["loss.npy"])
    assert files["model.sbm.shapelets.0.weights.npy"].shape == (5, 125, 100)
    assert files["adam.exp_avg.sbm.shapelets.3.weights.npy"].shape == (5, 125, 500)
    assert all(v.dtype in (np.float32, np.float64) and np.isfinite(v).all() for v in files.values())
    assert sum(p.stat().st_size for p in dump.iterdir()) <= 64 * 10 ** 6
