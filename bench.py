"""Contract benchmark: InterpGN training throughput on synthetic CHISCO-shaped EEG (BASELINE.json config 2:
125 channels, T=1000, 3 classes, default shapelet set K=5 x L in {100,200,300,500}, FCN deep expert).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A step is one full training step (forward, backward, gradient all-reduce when N>1, Adam) on a per-GPU batch
of --batch samples (weak scaling).  Rank 0 prints ONE JSON line:
  value        samples/s, whole job, inputs already resident in HBM, CUDA events, max over ranks
  e2e          the same step through the public Experiment API with the batch copied from pinned host
               memory every step and the loss read back every step (host clock, max over ranks)
  roofline     the dominant kernel of the step, timed live with CUDA events on the launching stream
  rooflines    the same for every kernel family of the hot path
  cpu_baseline the CPU restatement of the reference path (oracle/, "port") timed on this box's host cores on a
               bounded sample (N=1 only)
`--impl reference` times that CPU path alone under the same contract (rank 0 only).
`--dump-outputs DIR` writes what the last timed step left (see last_step_arrays) as DIR/<name>.npy, so that two builds
run with the same arguments, hence on the same seeded inputs, can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "speech-imagery-eeg_b200"))

import torch  # noqa: E402

CONFIG2 = dict(enc_in=125, seq_len=1000, num_class=3)          # BASELINE.json configs[1]
LENGTH_FRACS = [0.1, 0.2, 0.3, 0.5]
K_PER_LEN = 5
FP32_LANES_PER_SM = 128
DUMP_LIMIT_BYTES = 64 * 10 ** 6


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of every mode of the workload")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="samples per GPU per step")
    ap.add_argument("--dnn_type", default="FCN")
    ap.add_argument("--distance_func", default="euclidean")
    ap.add_argument("--memory_efficient", action="store_true")
    ap.add_argument("--precision", default="fp32")
    ap.add_argument("--num_class", type=int, default=3)
    ap.add_argument("--cpu_batch", type=int, default=2)
    ap.add_argument("--no_cpu_baseline", action="store_true")
    ap.add_argument("--cuda_graph", action="store_true", help="replay each step from one captured CUDA graph (N=1)")
    ap.add_argument("--no_extras", action="store_true", help="skip the cosine/3xtf32 mode, the same-GPU eager comparator "
                    "and the config-1 / config-5 lines (they run at N=1 only)")
    ap.add_argument("--amp", action="store_true", help="bf16 autocast for the deep expert (reference default is fp32 in its scripts)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the loss, model state and Adam moments after the last "
                    "timed step as DIR/<name>.npy (rank 0; at most 64 MB in all, larger outputs as a seeded sample)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return a


def model_args(a):
    from types import SimpleNamespace
    return SimpleNamespace(
        model="InterpGN", dnn_type=a.dnn_type, dataset="CHISCO-synthetic", data="synthetic",
        enc_in=CONFIG2["enc_in"], seq_len=CONFIG2["seq_len"], num_class=a.num_class, c_out=a.num_class,
        epsilon=1.0, distance_func=a.distance_func, memory_efficient=a.memory_efficient, sbm_cls="linear",
        dropout=0.0, lambda_reg=0.1, lambda_div=0.1, num_shapelet=10, shapelet_precision=a.precision,
        lr=5e-3, train_epochs=500, gradient_accumulation_steps=1, gradient_clip=0, pos_weight=False,
        beta_schedule="constant", amp=a.amp, gating_value=None, batch_size=a.batch, patience=50, seed=0,
        num_workers=0, log_interval=20, min_epochs=0, lr_decay=False,
        # Transformer expert (run.py defaults)
        task_name="classification", pred_len=0, label_len=0, output_attention=False, d_model=512, embed="timeF",
        freq="h", factor=1, n_heads=8, d_ff=2048, activation="gelu", e_layers=2, cuda_graph=getattr(a, "cuda_graph", False))


def algorithmic_elements(B, M, T, K, fracs):
    """E = B*M*sum_g K*T'_g*L_g window-shapelet-lag elements (SURVEY.md §8d)."""
    import math
    out = {}
    for f in fracs:
        L = max(3, math.ceil(f * T))
        out[L] = B * M * K * (T - L + 1) * L
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines, self.first = index, None, [], 0

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def mark(self):
        """Samples taken before this call (process start-up, idle clocks) are not part of the timed region."""
        self.first = len(self.lines)

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines[self.first:]:
            f = [v.strip() for v in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return (d.get("hbm_gbs", 6650.0), d.get("sm_max_mhz", 1965.0), d.get("bf16_tflops_sustained", 1365.9),
                "measured (MEASURED_PEAKS.json)")
    return 6650.0, 1965.0, 2250.0, "fallback (B200_PROFILING.md)"


def traffic_from_profiles(kernel):
    """dram bytes per launch of `kernel` from the committed ncu --set full summary, if one exists."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.isfile(p):
        return json.load(open(p)).get(kernel)
    return None


# ----------------------------------------------------------------------------------------------------
# CPU restatement of the reference step (oracle) — the cpu_baseline leg and the --impl reference arm
# ----------------------------------------------------------------------------------------------------
class CpuReferenceStep:
    """One InterpGN(FCN) training step exactly as the reference computes it on CPU: eager unfold/broadcast
    distance (Shapelet.py:61-84) through oracle/ign_oracle.py, FCN expert, Gini gate, CE + regulariser +
    beta*CE(shapelet_preds), Adam lr 5e-3 (experiment_classification.py:313-343), fp32, AMP off."""

    def __init__(self, a):
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import ign_oracle as O
        import ign_oracle_experts as OE          # CPU restatement of the deep experts: nothing from the product package
        self.O = O
        cfg = model_args(a)
        torch.manual_seed(0)
        T, M, C = cfg.seq_len, cfg.enc_in, cfg.num_class
        self.lens = O.shapelet_lengths(T, LENGTH_FRACS)
        self.strides = [O.shapelet_stride(T, L) for L in self.lens]
        self.Ws = [torch.normal(0, 1, (K_PER_LEN, M, L)).requires_grad_(True) for L in self.lens]
        self.Wc = (torch.randn(C, K_PER_LEN * M * len(self.lens)) * 0.02).requires_grad_(True)
        self.fcn = OE.build_expert(a.dnn_type, cfg).train()
        self.mode = O.resolve_mode(a.distance_func, a.memory_efficient)
        self.opt = torch.optim.Adam(self.Ws + [self.Wc] + list(self.fcn.parameters()), lr=5e-3)
        self.cfg = cfg

    def step(self, x, y):
        O = self.O
        sbm_out, probs, dists = O.sbm_forward(x, self.Ws, self.strides, self.Wc, 1.0, self.mode)
        deep_out = self.fcn(x, torch.ones(x.shape[0], x.shape[1], device=x.device), None, None)
        out, eta = O.gate_forward(sbm_out, deep_out)
        loss = torch.nn.functional.cross_entropy(out, y) + O.sbm_loss(self.Wc, self.Ws, 0.1, 0.1) \
            + torch.nn.functional.cross_entropy(sbm_out, y)
        self.opt.zero_grad()
        loss.backward()
        self.opt.step()
        return float(loss)


def time_cpu_reference(a, steps, warmup, batch, budget_s=None):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ref = CpuReferenceStep(a)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(batch, ref.cfg.seq_len, ref.cfg.enc_in, generator=g)
    y = torch.randint(0, ref.cfg.num_class, (batch,), generator=g)
    tw = time.perf_counter()
    for i in range(warmup):          # the same warm-up count as the GPU arm, but never more than a minute of it
        ref.step(x, y)
        if budget_s is not None and time.perf_counter() - tw > 60.0:
            break
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        ref.step(x, y)
        done += 1
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return batch * done / dt, dt / done * 1e3, done, cores


def run_reference_arm(a):
    """The reference's own CPU implementation of the path (oracle port: the reference is pure Python and its
    modules cannot travel to the GPU box; oracle/ign_oracle.py restates them line by line and is pinned to
    their outputs by tests/golden).  Rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    # bounded sample: a.cpu_batch (2) CHISCO-shaped samples per step (the reference's eager path needs ~4 GB per
    # sample), the same warm-up count as the GPU arm, timed steps capped at 240 s
    warm = max(a.warmup, 3)
    sps, ms, done, cores = time_cpu_reference(a, a.steps, warm, a.cpu_batch, budget_s=240.0)
    line = {
        "impl": "reference", "metric": "train samples/sec", "value": sps, "unit": "samples/s", "n_gpus": a.gpus,
        "steps": done, "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(a, a.cpu_batch, 1),
        "cpu_baseline": {"value": sps, "unit": "samples/s", "cores": cores, "kind": "port",
                         "sample": "InterpGN(%s) full train step, batch %d of the config-2 workload, %d timed steps after %d warm-up"
                                   % (a.dnn_type, a.cpu_batch, done, warm)},
        "e2e": {"value": sps, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def workload_config(a, per_gpu_batch, world):
    return {"workload": "InterpGN(%s) train step on synthetic CHISCO-shaped EEG: 125 ch x T=1000, %d classes, "
                        "shapelets K=5 x L={100,200,300,500}, distance_func=%s%s" % (
                            a.dnn_type, a.num_class, a.distance_func, "+memory_efficient" if a.memory_efficient else ""),
            "baseline_config": "configs[1]", "per_gpu_batch": per_gpu_batch, "global_batch": per_gpu_batch * world,
            "parallelism": "dp%d" % world, "precision": a.precision, "amp": bool(a.amp),
            "l2": "inputs larger than L2 (x 128 MB + saved distances 1.9 GB per step)"}


# ----------------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def emit(line):
    """The contract is ONE JSON line on stdout; libraries (NCCL, cuDNN) may print to fd 1, so main() points
    fd 1 at stderr for the whole run and the result line goes to the saved descriptor."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def last_step_arrays(exp, loss):
    """What a training step hands its caller, copied to the host: the loss and the model's state after the optimiser
    step, plus Adam's moments, which carry that step's gradients (the step zeroes the gradients themselves)."""
    out = {"loss": loss}
    for k, v in exp.model.state_dict().items():
        out["model." + k] = v
    names = {p: n for n, p in exp.model.named_parameters()}
    for p, st in exp.optimizer.state.items():
        for k, v in st.items():
            if k != "step":
                out["adam.%s.%s" % (k, names[p])] = v
    return {k: v.detach().cpu() for k, v in out.items()}


def dump_outputs(out_dir, arrays):
    """Writes each tensor as out_dir/<name>.npy, in float32 (float64 for float64 and integer tensors).  When they come
    to more than DUMP_LIMIT_BYTES, each is cut to the same fraction of its elements, flattened, at positions drawn
    from a generator seeded by its name: runs with the same arguments write the same positions."""
    os.makedirs(out_dir, exist_ok=True)
    arrs = {k: v.to(torch.float32 if v.is_floating_point() and v.dtype != torch.float64 else torch.float64).numpy()
            for k, v in arrays.items()}
    budget = DUMP_LIMIT_BYTES - 1024 * len(arrs)        # 1 KiB a file for the .npy header
    total = sum(a.nbytes for a in arrs.values())
    for k, a in arrs.items():
        if total > budget:
            keep = max(1, a.size * budget // total)
            idx = np.random.default_rng(zlib.crc32(k.encode())).choice(a.size, keep, replace=False)
            a = a.reshape(-1)[np.sort(idx)]
        np.save(os.path.join(out_dir, k + ".npy"), a)


def run_ours(a, primary=True):
    """One measurement of this repo's training step under the contract: W warm-up, K timed steps with inputs resident
    (CUDA events, max over ranks), per-kernel rooflines from a second instrumented pass, and (primary only) the clock
    sampler, the end-to-end region with pinned host batches and the CPU baseline.  Returns the JSON line as a dict."""
    import torch.distributed as dist
    from exp.experiment_classification import Experiment
    from layers.shapelet_ops import STATS

    cfg = model_args(a)
    torch.manual_seed(0)
    exp = Experiment(cfg, load_data=False)          # also initialises torch.distributed from torchrun's env
    rank, world, dev = exp.rank, exp.world, exp.device
    exp.model.train()
    torch.set_float32_matmul_precision("medium")    # experiment_classification.py:297
    B, T, M, C = a.batch, cfg.seq_len, cfg.enc_in, cfg.num_class
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    x = torch.randn(B, T, M, device=dev, generator=gen)
    y = torch.randint(0, C, (B,), device=dev, generator=gen)
    mask = torch.ones(B, T, device=dev)
    exp.grads.zero_grad()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    step_no = 0
    for _ in range(max(a.warmup, 3)):
        step_no += 1
        exp.train_step(x, y, mask, 0, step_no)
    # ---------------- device-resident timed region ----------------
    sampler = ClockSampler(exp.local_rank)
    if rank == 0 and primary:
        sampler.start()
    # nvidia-smi needs ~0.5 s to start (its launch cost 2-5 ms of step 1 when it overlapped the timed region).  The GPU
    # is kept busy with untimed steps meanwhile — an idle half second let the clocks drop and the first timed step
    # then took up to 39 ms instead of 24.  Same count on every rank (the step contains the gradient all-reduce).
    for _ in range(20):
        step_no += 1
        exp.train_step(x, y, mask, 0, step_no)
    torch.cuda.synchronize()
    barrier()
    sampler.mark()
    STATS.reset(timing=False)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    marks = []
    e0.record()
    for _ in range(a.steps):
        step_no += 1
        loss = exp.train_step(x, y, mask, 0, step_no)
        marks.append(torch.cuda.Event(enable_timing=True)); marks[-1].record()
    e1.record()
    barrier()
    last_step = last_step_arrays(exp, loss) if (primary and rank == 0 and a.dump_outputs) else None
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    if rank == 0:      # per-step spread of the timed region (diagnostic, stderr)
        prev, per = e0, []
        for mk in marks:
            per.append(prev.elapsed_time(mk)); prev = mk
        sys.stderr.write("per-step ms: " + " ".join("%.2f" % v for v in per) + "\n")
    clocks = sampler.stop() if (rank == 0 and primary) else None
    launches = STATS.launches
    engines = STATS.engine_summary()
    # per-kernel durations for the rooflines: the same steps once more with a CUDA-event pair around every C-ABI
    # call, on the stream the kernels run on (kept out of the timed region above so that it is unperturbed)
    ksteps = min(a.steps, 5)
    import ctypes
    from layers import ign_cabi as CABI
    CABI.check(CABI.lib.ign_debug_bwd_phase_timing(1), "ign_debug_bwd_phase_timing")     # events around the phases inside ign_shapelet_backward
    STATS.reset(timing=True)
    # per-kernel durations are taken with the deep expert back on the main stream: in the timed region above it runs on
    # a side stream and shares the SMs with the shapelet kernels, which would charge its work to their event pairs
    overlap_was = getattr(exp.model, "overlap_experts", None)
    if overlap_was is not None:
        exp.model.overlap_experts = False
    from layers import shapelet_ops as _ops
    prep_was, _ops.OVERLAP_BWD_PREPARE = _ops.OVERLAP_BWD_PREPARE, False     # and the backward's phases in stream order
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k0.record()
    for _ in range(ksteps):
        step_no += 1
        exp.train_step(x, y, mask, 0, step_no)
    k1.record()
    barrier()
    if overlap_was is not None:
        exp.model.overlap_experts = overlap_was
    _ops.OVERLAP_BWD_PREPARE = prep_was
    ms_kernel_region = k0.elapsed_time(k1)
    kern = STATS.summary()
    STATS.reset(timing=False)
    ph_ms, ph_n = (ctypes.c_float * 4)(), (ctypes.c_int32 * 4)()
    CABI.check(CABI.lib.ign_debug_bwd_phase_read(ph_ms, ph_n), "ign_debug_bwd_phase_read")
    CABI.check(CABI.lib.ign_debug_bwd_phase_timing(0), "ign_debug_bwd_phase_timing")
    for i, name in enumerate(("bwd.pool_bwd", "bwd.tie_check", "bwd.contraction", "bwd.finalize")):
        if ph_n[i]:
            kern[name] = (int(ph_n[i]), float(ph_ms[i]))
    value = world * B * a.steps / (ms_total * 1e-3)

    e2e = None
    if primary:
        # ---------------- end-to-end region: pinned host batch in, loss out, every step ----------------
        xh = torch.randn(B, T, M).pin_memory()
        yh = torch.randint(0, C, (B, 1)).pin_memory()
        mh = torch.ones(B, T, dtype=torch.bool).pin_memory()
        from exp.parallel import DevicePrefetcher
        for xd, yd, md in DevicePrefetcher(((xh, yh, mh) for _ in range(2)), dev):   # warm-up of the same path
            step_no += 1
            float(exp.train_step(xd, yd, md, 0, step_no))
        barrier()
        t0 = time.perf_counter()
        # the public training loop's own batch path (Experiment.train): every step's batch is copied from pinned host
        # memory inside the timed region, one batch ahead on a side stream; the first copy is not overlapped
        for xd, yd, md in DevicePrefetcher(((xh, yh, mh) for _ in range(a.steps)), dev):
            step_no += 1
            loss = exp.train_step(xd, yd, md, 0, step_no)
            loss_host = float(loss)                    # D2H read of the step's result
        barrier()
        e2e_s = max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": world * B * a.steps / e2e_s, "unit": "samples/s",
               "h2d_bytes_per_step": xh.numel() * 4 + yh.numel() * 8 + mh.numel(), "d2h_bytes_per_step": 4,
               "ms_per_step": e2e_s / a.steps * 1e3, "last_loss": loss_host}
    nbytes_allreduce = exp.grads.nbytes() if world > 1 else 0
    del exp
    torch.cuda.empty_cache()
    if last_step is not None:
        dump_outputs(a.dump_outputs, last_step)
    if rank != 0:
        return None

    # ---------------- rooflines from the live per-kernel CUDA-event times ----------------
    hbm_peak, sm_max_mhz, bf16_peak, peak_src = measured_peaks()
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    alu_peak = sms * FP32_LANES_PER_SM * sm_max_mhz * 1e6 / 1e12        # T FP32 instr/s (FADD/FSETP: 1 op each)
    E = algorithmic_elements(B, M, T, K_PER_LEN, LENGTH_FRACS)
    l1 = (a.distance_func not in ("cosine", "pearson")) and not a.memory_efficient
    tensor_mode = (not l1) and a.precision in ("3xtf32", "tf32", "bf16")
    mma_passes = {"3xtf32": 3, "tf32": 1, "bf16": 1}.get(a.precision, 1)
    fams = {}
    for tag, (n, ms) in kern.items():
        fam = tag.split("/")[0]
        L = int(tag.rsplit("L", 1)[1]) if "/L" in tag else None
        f = fams.setdefault(fam, {"launches": 0, "ms": 0.0, "ops": 0.0, "bytes": 0.0})
        f["launches"] += n; f["ms"] += ms
        if fam == "shapelet_fwd":
            f["ops"] += n * 2.0 * E[L]                      # 2 flop per element (SURVEY.md §8d)
        elif fam == "shapelet_bwd":
            # SURVEY.md §8d counts 4E (recompute d + contraction); this implementation stores d in the forward,
            # so the backward EXECUTES 2E (L1: FSETP + predicated FADD per element; dot modes: one FFMA).
            f["ops"] += n * 2.0 * E[L]
            f["alg"] = f.get("alg", 0.0) + n * 4.0 * E[L]
        elif fam == "bwd.pool_bwd":
            # one read of the saved distances + one write of the coefficients per (sample, channel, shapelet, window);
            # every group is launched once per step, so n launches = n/len(E) steps
            f["bytes"] += (n / len(E)) * sum(8.0 * B * M * K_PER_LEN * ((T - L_ + 1 + 3) // 4 * 4) for L_ in E)
        elif fam == "bwd.contraction":
            f["ops"] += (n / len(E)) * 2.0 * sum(E.values())
        elif fam == "instnorm":
            f["bytes"] += n * (2.0 * B * T * M * 4)
        elif fam == "window_stats":
            # reads the normalised series once, writes one fp32 statistic per window and group (two for pearson)
            nst = 2 if a.distance_func == "pearson" else 1
            f["bytes"] += n * (B * M * T * 4.0 + nst * sum(4.0 * B * M * ((T - L_ + 1 + 15) // 16 * 16) for L_ in E))
        elif fam == "window_prefix":
            f["bytes"] += n * (B * M * T * 4 + 2.0 * B * M * (T + 1) * 8)
    rooflines = []
    for fam, f in sorted(fams.items(), key=lambda kv: -kv[1]["ms"]):
        avg_ms = f["ms"] / max(1, f["launches"])
        r = {"kernel": fam, "launches": f["launches"], "avg_ms": avg_ms, "share_of_step": f["ms"] / ms_kernel_region}
        if f["ops"]:
            ach = f["ops"] / (f["ms"] * 1e-3) / 1e12
            if fam in ("shapelet_fwd", "shapelet_bwd", "bwd.contraction") and tensor_mode:
                # cross term (forward) / coefficient contraction (backward, incl. its HBM-bound pooling pass) on the
                # tcgen05 pipe: algorithmic 2E flop against the TF32 peak (= half the measured bf16 cuBLAS rate); the
                # 3xTF32 split executes three MMAs per algorithmic multiply-add
                peak = bf16_peak if a.precision == "bf16" else bf16_peak / 2.0
                r.update(bound="tensor", achieved=ach, peak=peak, unit="TFLOP/s", frac=ach / peak,
                         mma_passes=mma_passes, frac_executed=mma_passes * ach / peak,
                         peak_source="%s dense = bf16_tflops_sustained%s (%s)" % (
                             "bf16" if a.precision == "bf16" else "TF32", "" if a.precision == "bf16" else " / 2", peak_src),
                         traffic=None)
            else:
                # executed FP32-pipe work: L1 issues 1 op per flop (no FMA): peak = lanes*clock; dot modes are FFMA
                peak = alu_peak if l1 else 2.0 * alu_peak
                r.update(bound="fp32_alu", achieved=ach, peak=peak, unit="TFLOP/s", frac=ach / peak,
                         peak_source="%d SMs x %d FP32 lanes x %.0f MHz (%s)" % (sms, FP32_LANES_PER_SM, sm_max_mhz, peak_src),
                         traffic=traffic_from_profiles(fam))
            if "alg" in f:
                r["algorithmic_tflops_4E"] = f["alg"] / (f["ms"] * 1e-3) / 1e12
        elif f["bytes"]:
            ach = f["bytes"] / (f["ms"] * 1e-3) / 1e9
            r.update(bound="hbm", achieved=ach, peak=hbm_peak, unit="GB/s", frac=ach / hbm_peak,
                     peak_source=peak_src, traffic=traffic_from_profiles(fam))
        rooflines.append(r)
    # the dominant KERNEL: the backward op as a whole is an aggregate of four kernels (pooling backward, tie pre-check,
    # contraction, finalize), reported for continuity; its phases are the entries named "bwd.*"
    have_phases = any(r["kernel"] == "bwd.contraction" for r in rooflines)
    for r in rooflines:
        if r["kernel"] == "shapelet_bwd" and have_phases:
            r["aggregate_of"] = ["bwd.pool_bwd", "bwd.tie_check", "bwd.contraction", "bwd.finalize"]
    dominant = next((r for r in rooflines if "bound" in r and "aggregate_of" not in r), None)

    cpu = None
    if primary and world == 1 and not a.no_cpu_baseline:
        sps, ms, done, cores = time_cpu_reference(a, 1, 0, a.cpu_batch)
        cpu = {"value": sps, "unit": "samples/s", "cores": cores, "kind": "port",
               "sample": "1 full InterpGN(%s) train step on %d CHISCO-shaped samples (oracle/ign_oracle.py restatement "
                         "of the reference's eager path, fp32, %d threads)" % (a.dnn_type, a.cpu_batch, cores),
               "ms_per_step": ms}

    return {
        "metric": "train samples/sec", "value": value, "unit": "samples/s", "n_gpus": world, "steps": a.steps,
        "warmup": max(a.warmup, 3), "ms_per_step": ms_total / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(a, B, world),
        "untimed_steps_before_region": max(a.warmup, 3) + 20,   # W warm-up + 20 while the clock sampler starts
        "kernel_timing_pass": {"steps": ksteps, "ms_per_step": ms_kernel_region / ksteps,
                               "note": "separate instrumented pass after the timed region: CUDA-event pair around every "
                                       "C-ABI call, deep expert serialised on the main stream (it overlaps the shapelet "
                                       "kernels on a side stream in the timed region)"},
        "e2e": e2e, "gpu_launches": launches, "engines": engines, "clocks": clocks,
        "roofline": dominant, "rooflines": rooflines, "cpu_baseline": cpu,
        "shapelet_layer": {"fwd_tflops": fams.get("shapelet_fwd", {}).get("ops", 0) / max(1e-9, fams.get("shapelet_fwd", {}).get("ms", 0) * 1e-3) / 1e12,
                           "bwd_tflops": fams.get("shapelet_bwd", {}).get("alg", 0) / max(1e-9, fams.get("shapelet_bwd", {}).get("ms", 0) * 1e-3) / 1e12,
                           "share_of_step": sum(f["ms"] for k, f in fams.items() if k.startswith("shapelet")) / ms_kernel_region},
        "allreduce_bytes_per_step": nbytes_allreduce,
    }


def gpu_eager_reference(a, budget_s=60.0):
    """Same-box comparator (SURVEY.md §8d, BASELINE.md §3): the reference's EAGER PyTorch path — the oracle port of
    Shapelet.py:61-84 / InterpGN.py:44-52 with the restated FCN expert, autograd backward, Adam — moved to this B200,
    at the largest batch that fits (the eager path keeps ~4 GB of 5-D temporaries per sample for backward)."""
    dev = torch.device("cuda", 0)
    batch, err = 32, None
    while batch >= 1:
        try:
            ref = CpuReferenceStep(a)
            ref.fcn.to(dev)
            ref.Ws = [w.detach().to(dev).requires_grad_(True) for w in ref.Ws]
            ref.Wc = ref.Wc.detach().to(dev).requires_grad_(True)
            ref.opt = torch.optim.Adam(ref.Ws + [ref.Wc] + list(ref.fcn.parameters()), lr=5e-3)
            ref.dev = dev
            g = torch.Generator(device=dev).manual_seed(0)
            x = torch.randn(batch, ref.cfg.seq_len, ref.cfg.enc_in, device=dev, generator=g)
            y = torch.randint(0, ref.cfg.num_class, (batch,), device=dev, generator=g)
            for _ in range(2):
                ref.step(x, y)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0, done = time.perf_counter(), 0
            e0.record()
            while done < 5 and time.perf_counter() - t0 < budget_s:
                ref.step(x, y)
                done += 1
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / done
            peak = torch.cuda.max_memory_allocated(dev) / 2 ** 30
            del ref, x, y
            torch.cuda.empty_cache()
            return {"value": batch / (ms * 1e-3), "unit": "samples/s", "batch": batch, "ms_per_step": ms, "steps": done,
                    "peak_mem_gib": peak,
                    "what": "reference eager PyTorch path (oracle port, fp32, allow_tf32 off) on the same B200"}
        except torch.OutOfMemoryError as e:            # halve the batch and retry
            err = str(e)[:80]
            ref = x = y = None
            torch.cuda.empty_cache()
            batch //= 2
    return {"unavailable": err}


def extra_config_lines(a):
    """BASELINE.json configs[0] and configs[4] through the same train step (short runs; N=1 only):
    config 1 = JapaneseVowels-shaped InterpGN(FCN), B=32 — launch-latency-bound, reported as microseconds per step;
    config 5 = 39-class CHISCO-shaped InterpGN(Transformer d_model 512, 2 layers), per-fold batch 64."""
    import copy
    from exp.experiment_classification import Experiment
    out = {}
    for name, kw, batch, steps, graph in (
            ("config1_jv_fcn_b32", dict(enc_in=12, seq_len=29, num_class=9, dnn_type="FCN"), 32, 50, False),
            # the same step replayed from one captured CUDA graph (run.py --cuda_graph): config 1 is launch-latency-bound
            ("config1_jv_fcn_b32_cuda_graph", dict(enc_in=12, seq_len=29, num_class=9, dnn_type="FCN"), 32, 200, True),
            ("config5_chisco39_transformer_b64", dict(enc_in=125, seq_len=1000, num_class=39, dnn_type="Transformer"), 64, 10, False)):
        cfg = model_args(a)
        for k, v in kw.items():
            setattr(cfg, k, v)
        cfg.c_out, cfg.batch_size, cfg.cuda_graph = cfg.num_class, batch, graph
        torch.manual_seed(0)
        exp = Experiment(cfg, load_data=False)
        exp.model.train()
        dev = exp.device
        x = torch.randn(batch, cfg.seq_len, cfg.enc_in, device=dev)
        y = torch.randint(0, cfg.num_class, (batch,), device=dev)
        mask = torch.ones(batch, cfg.seq_len, device=dev)
        exp.grads.zero_grad()
        for i in range(5):
            exp.train_step(x, y, mask, 0, i + 1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            exp.train_step(x, y, mask, 0, i + 6)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out[name] = {"samples_per_s": batch / (ms * 1e-3), "step_us": ms * 1e3, "batch": batch, "steps": steps,
                     "dnn_type": cfg.dnn_type, "num_class": cfg.num_class, "distance_func": cfg.distance_func,
                     "precision": cfg.shapelet_precision, "cuda_graph": graph}
        del exp, x, y, mask
        torch.cuda.empty_cache()
    return out


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    a = parse()
    if a.impl == "reference":
        return run_reference_arm(a)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    import copy
    import torch.distributed as dist
    line = run_ours(a, primary=True)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world == 1 and not a.no_extras:
        # the tensor-core engine in the same record: cosine distance, 3xTF32 operands (fp32-equivalent), same workload
        b = copy.copy(a)
        b.distance_func, b.precision = "cosine", "3xtf32"
        m = run_ours(b, primary=False)
        line["modes"] = {"cosine_3xtf32": {k: m[k] for k in ("value", "unit", "ms_per_step", "steps", "warmup", "config",
                                                               "gpu_launches", "engines", "roofline", "rooflines",
                                                               "shapelet_layer")}}
        try:
            line["gpu_eager_reference"] = gpu_eager_reference(a)
        except Exception as e:                     # a comparator must never take the bench line down
            line["gpu_eager_reference"] = {"unavailable": repr(e)[:200]}
        try:
            line["extra_configs"] = extra_config_lines(a)
        except Exception as e:
            line["extra_configs"] = {"unavailable": repr(e)[:200]}
    if line is not None:
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
