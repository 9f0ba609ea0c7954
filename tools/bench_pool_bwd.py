"""Per-group timing of the backward's phases (pooling backward, tie check, contraction, finalize) through
ign_debug_bwd_phase_timing.  Default: config 2.  Each group is timed twice: with the gradient of the pooled output only
(the training path), then with a gradient on the reported min distance as well (ign_shapelet_backward_dmin, "+dmin").
   python tools/bench_pool_bwd.py [l1|cosine] [precision] [T] [K] [L,L,...]"""
import ctypes, math, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "speech-imagery-eeg_b200"))
import torch
from layers import ign_cabi as C
from layers.shapelet_ops import instance_norm, shapelet_transform
dist = sys.argv[1] if len(sys.argv) > 1 else "l1"
prec = sys.argv[2] if len(sys.argv) > 2 else "fp32"
T = int(sys.argv[3]) if len(sys.argv) > 3 else 1000
K = int(sys.argv[4]) if len(sys.argv) > 4 else 5
Ls = [int(v) for v in sys.argv[5].split(",")] if len(sys.argv) > 5 else [math.ceil(f * T) for f in (0.1, 0.2, 0.3, 0.5)]
B, M = 256, 125
x = torch.randn(B, T, M, device="cuda"); pack = instance_norm(x)
for L in Ls:
    stride = 1 if T < 3000 else max(1, int(math.log2(L)))
    Tw = (T - L) // stride + 1
    W = torch.randn(K, M, L, device="cuda", requires_grad=True)
    p, dmin, _ = shapelet_transform(pack, W, stride, 1.0, dist, precision=prec); g = torch.randn_like(p)
    gd = torch.randn_like(dmin)
    for outs, grads, tag in (([p], [g], ""), ([p, dmin], [g, gd], " +dmin")):
        for _ in range(3):
            W.grad = None; torch.autograd.backward(outs, grads, retain_graph=True)
        torch.cuda.synchronize()
        C.lib.ign_debug_bwd_phase_timing(1)
        n = 10
        for _ in range(n):
            W.grad = None; torch.autograd.backward(outs, grads, retain_graph=True)
        torch.cuda.synchronize()
        ms, cnt = (ctypes.c_float * 4)(), (ctypes.c_int32 * 4)()
        C.lib.ign_debug_bwd_phase_read(ms, cnt); C.lib.ign_debug_bwd_phase_timing(0)
        Ts = (Tw + 3) // 4 * 4
        gb = 8.0 * B * M * K * Ts / 1e9
        E = B * M * K * Tw * L
        print("%s/%s%s T=%d L=%d s=%d T'=%d K=%d  pool_bwd %.3f ms (%.0f GB/s algorithmic)  tie %.3f  contraction %.3f (%.1f TFLOP/s 2E)  finalize %.3f" % (
            dist, prec, tag, T, L, stride, Tw, K, ms[0] / n, gb / (ms[0] / n) * 1e3, ms[1] / max(1, cnt[1]), ms[2] / n,
            2 * E / (ms[2] / n) / 1e9, ms[3] / n), flush=True)
    del W, p, dmin, g, gd
