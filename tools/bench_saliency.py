"""Time of one saliency pass of the shapelet layer: forward + backward with the input series requiring grad and the
shapelets frozen, so the backward gives dLoss/dx only.  Each length group runs alone; CUDA events on torch's current
stream, 256 MB written between passes to flush L2, median of --iters passes after three warm-up passes.

  config 2 (B 256, M 125, T 1000, K 5, L 100/200/300/500): stored-distance backward (the default budget) against the
  recompute backward, forced by the largest budget that recomputes (2 x dstore bytes - 1); "fwd" is the forward alone
  (no grad), for comparing the extra cost of the recompute with one forward.
  --corner: K = 1000, L = 100, which only the recompute backward can run (the stored mode would keep 2 x 116 GB).

Usage: python tools/bench_saliency.py [--dists l1,cosine,pearson] [--precision fp32] [--corner] [--json out.json]"""
import argparse
import json
import os
import subprocess
import sys
from ctypes import byref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "speech-imagery-eeg_b200"))

import torch  # noqa: E402

from layers import ign_cabi as C  # noqa: E402
from layers import shapelet_ops  # noqa: E402
from layers.shapelet_ops import SeriesPack, shapelet_transform  # noqa: E402


def timeit(fn, iters, flush):
    fn(); fn(); fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=256)
    ap.add_argument("--M", type=int, default=125)
    ap.add_argument("--T", type=int, default=1000)
    ap.add_argument("--K", type=int, default=5)
    ap.add_argument("--Ls", default="100,200,300,500")
    ap.add_argument("--dists", default="l1,cosine,pearson")
    ap.add_argument("--precision", default="fp32")
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--corner", action="store_true", help="also time K = 1000, L = 100 (recompute only)")
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    dev = "cuda"
    print("card, power limit, max SM clock:", card())
    torch.manual_seed(0)
    x = torch.randn(a.B, a.M, a.T, device=dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    default_budget = shapelet_ops.STORE_BUDGET_BYTES
    rows = []

    def saliency(W, gp, dist, budget):
        def run():
            shapelet_ops.STORE_BUDGET_BYTES = budget
            xd = x.detach().requires_grad_(True)
            p, _, _ = shapelet_transform(SeriesPack.from_channel_major(xd), W, 1, 1.0, dist, precision=a.precision)
            p.backward(gp)
            return xd.grad
        return run

    def forward(W, dist):
        def run():
            with torch.no_grad():
                shapelet_transform(SeriesPack.from_channel_major(x), W, 1, 1.0, dist, precision=a.precision)
        return run

    cases = [(a.K, L) for L in (int(v) for v in a.Ls.split(","))] + ([(1000, 100)] if a.corner else [])
    for dist in a.dists.split(","):
        for K, L in cases:
            W = torch.randn(K, a.M, L, device=dev)
            gp = torch.randn(a.B, K, a.M, device=dev)
            desc = C.ShapeletDesc(a.B, a.M, a.T, C.padded_len(a.T), K, L, 1, 1.0, C.DIST[dist], C.POOL["rbf_max"],
                                  C.PRECISION[a.precision])
            stored_bytes = 2 * int(C.lib.ign_shapelet_dstore_bytes(byref(desc)))
            can_store = stored_bytes <= default_budget
            rec_budget = min(default_budget, stored_bytes - 1)
            ws = int(C.lib.ign_shapelet_backward_recompute_input_workspace(byref(desc), rec_budget))
            tf = timeit(forward(W, dist), a.iters, flush)
            ts = timeit(saliency(W, gp, dist, default_budget), a.iters, flush) if can_store else None
            tr = timeit(saliency(W, gp, dist, rec_budget), a.iters, flush)
            shapelet_ops.STORE_BUDGET_BYTES = default_budget
            if ts is not None:
                dx_s = saliency(W, gp, dist, default_budget)()
                dx_r = saliency(W, gp, dist, rec_budget)()
                same = bool(torch.equal(dx_s, dx_r))
                shapelet_ops.STORE_BUDGET_BYTES = default_budget
            extra = "" if ts is None else (f" | stored {ts:9.3f} ms | recompute - stored {tr - ts:8.3f} ms = "
                                           f"{(tr - ts) / tf:5.2f} fwd | dx bit-identical {same}")
            print(f"{dist:8s} K={K:4d} L={L:4d} fwd {tf:9.3f} ms | recompute {tr:9.3f} ms (workspace "
                  f"{ws / 2 ** 30:6.2f} GiB){extra}", flush=True)
            rows.append(dict(dist=dist, K=K, L=L, precision=a.precision, fwd_ms=tf, stored_ms=ts, recompute_ms=tr,
                             recompute_ws_bytes=ws, stored_bytes=stored_bytes,
                             dx_bit_identical=None if ts is None else same))
            del W, gp
            torch.cuda.empty_cache()
    if a.json:
        json.dump(dict(card=card(), rows=rows), open(a.json, "w"), indent=1)


if __name__ == "__main__":
    main()
