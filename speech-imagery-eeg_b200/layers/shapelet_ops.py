"""torch.autograd glue over the C ABI (include/ign_b200.h).  PyTorch owns every buffer; the kernels are
launched on torch's current CUDA stream through ctypes.  CUDA-only: CPU tensors raise.

Replaces the eager op chains of the reference:
  instance_norm      <- Shapelet.py:186-187
  shapelet_transform <- Shapelet.py:61-84 (Shapelet.forward) and :97-111 (DistThresholdShapelet.forward)
  gini_gate          <- InterpGN.py:44-52
"""
from __future__ import annotations

import os
from ctypes import byref, c_int32, c_void_p
from typing import Optional

import torch

from . import ign_cabi as C

_DIST_OF_FLAG = {"cosine": "cosine", "pearson": "pearson"}

# Memory the backward may spend per length group on the window distances it keeps from the forward plus the
# coefficient workspace of the same size (stored-distance mode: fastest, 2 x 4*B*M*K*T' bytes).  Above it the layer
# switches to the recompute backward (nothing saved, shapelets walked in chunks inside a workspace of at most this
# size): config 2 at B=256 needs 1.2 GB per group and stores, so do the K = 100 points of the config-4 sweep (23 GB);
# the K = 1000 points would need 232 GB and recompute.  The saved distances of every stored group are live from the
# forward until the backward; the backward allocates one group's workspace at a time and releases it before the next
# group's.  Four groups at the limit keep 4 x 16 GiB of distances plus one 16 GiB workspace: under 80 GiB of the 180.
STORE_BUDGET_BYTES = int(float(os.environ.get("IGN_BWD_STORE_BUDGET_GB", "32")) * 2 ** 30)


def resolve_dist(distance_func: str, memory_efficient: bool) -> str:
    """Flag -> arithmetic exactly as Shapelet.forward dispatches (Shapelet.py:64-74):
    'cosine' / 'pearson' by name; anything else is the L1 mean ('euclidean' in the reference's
    vocabulary) unless memory_efficient selects the squared-L2 arithmetic of Shapelet.py:28."""
    if distance_func in _DIST_OF_FLAG:
        return _DIST_OF_FLAG[distance_func]
    return "sql2" if memory_efficient else "l1"


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _require_cuda(t: torch.Tensor, name: str):
    if not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor: the ign_b200 hot path has no CPU fallback "
                           "(got device %s)" % (name, t.device))


_checked_devices = set()


class KernelStats:
    """Launch counter + optional CUDA-event timing of every C-ABI call, on the stream the kernels run on.
    bench.py enables it around the timed region to obtain per-kernel durations for the roofline."""

    def __init__(self):
        self.launches = 0          # kernels launched through the C ABI since the last reset
        self.timing = False
        self.records = []          # (tag, start_event, end_event)
        self.engines = {}          # tag -> engine the library reported for that call ("fp32" | "tcgen05")

    def reset(self, timing=False):
        self.launches, self.timing, self.records, self.engines = 0, timing, [], {}

    def note_engine(self, tag, desc, backward):
        """Record which engine the library runs this call on (asked, not assumed: ign_shapelet_engine)."""
        self.engines[tag] = C.ENGINE.get(int(C.lib.ign_shapelet_engine(byref(desc), int(backward))), "?")

    def engine_summary(self):
        return dict(sorted(self.engines.items()))

    def call(self, tag, nkernels, fn):
        self.launches += nkernels
        if not self.timing:
            return fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        self.records.append((tag, e0, e1))
        return out

    def summary(self):
        """{tag: (calls, total_ms)}; call after torch.cuda.synchronize()."""
        agg = {}
        for tag, e0, e1 in self.records:
            n, t = agg.get(tag, (0, 0.0))
            agg[tag] = (n + 1, t + e0.elapsed_time(e1))
        return agg


STATS = KernelStats()


def _check_device(dev: torch.device):
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    if idx not in _checked_devices:
        C.check(C.lib.ign_device_check(idx), "ign_device_check")
        _checked_devices.add(idx)


class SeriesPack:
    """Instance-normalised series in the kernels' layout: xn [B,M,Tp] fp32 (time contiguous, zero padded
    to a multiple of 4) plus the lazily built window statistics of each length group."""

    def __init__(self, xn: torch.Tensor, T: int, xn_var: Optional[torch.Tensor] = None):
        self.xn = xn               # the kernels' buffer (never tracked by autograd)
        self.xn_var = xn_var       # the same values as an autograd variable when the caller wants dLoss/dx, else None
        self.T = T
        self._stats = {}

    @property
    def B(self):
        return self.xn.shape[0]

    @property
    def M(self):
        return self.xn.shape[1]

    @property
    def Tp(self):
        return self.xn.shape[2]

    def prepare_stats(self, dist: str, groups):
        """One fused prefix + window-difference pass for several (L, stride) groups (ign_window_stats).
        ShapeBottleneckModel calls this once per batch so the series is scanned once for all its layers."""
        if dist == "l1":
            return
        todo = [(int(L), int(s)) for (L, s) in groups if (dist, int(L), int(s)) not in self._stats]
        todo = list(dict.fromkeys(todo))
        B, M, T = self.B, self.M, self.T
        for i in range(0, len(todo), 8):
            part = todo[i:i + 8]
            G = len(part)
            st0, st1 = [], []
            for (L, s) in part:
                sp = C.lib.ign_stats_pitch(T, L, s)
                buf = torch.empty((2 if dist == "pearson" else 1, B, M, sp), dtype=torch.float32, device=self.xn.device)
                st0.append(buf[0]); st1.append(buf[1] if dist == "pearson" else None)
            Ls = (c_int32 * G)(*[L for L, _ in part])
            Ss = (c_int32 * G)(*[s for _, s in part])
            p0 = (c_void_p * G)(*[t.data_ptr() for t in st0])
            p1 = (c_void_p * G)(*[(t.data_ptr() if t is not None else None) for t in st1])
            with torch.cuda.device(self.xn.device):
                C.check(STATS.call("window_stats", 1, lambda: C.lib.ign_window_stats(
                    _ptr(self.xn), B, M, T, G, Ls, Ss, C.DIST[dist], p0, p1 if dist == "pearson" else None,
                    _stream())), "ign_window_stats")
            for (L, s), a0, a1 in zip(part, st0, st1):
                self._stats[(dist, L, s)] = (a0, a1)

    def window_stats(self, dist: str, L: int, stride: int):
        """(st0, st1) fp32 [B,M,SP] for one group; computed on demand if prepare_stats was not called."""
        if dist == "l1":
            return None, None
        key = (dist, int(L), int(stride))
        if key not in self._stats:
            self.prepare_stats(dist, [(L, stride)])
        return self._stats[key]

    @staticmethod
    def from_channel_major(x: torch.Tensor) -> "SeriesPack":
        """Wrap an already-normalised [B,M,T] tensor (what Shapelet.forward receives, Shapelet.py:60)."""
        _require_cuda(x, "x")
        B, M, T = x.shape
        Tp = C.padded_len(T)
        if x.requires_grad and torch.is_grad_enabled():      # input gradients wanted: keep a differentiable view
            var = torch.nn.functional.pad(x.to(torch.float32), (0, Tp - T)).contiguous()
            if var is x:
                var = x.view_as(x)
            return SeriesPack(var.detach(), T, xn_var=var)
        xn = x.detach().to(torch.float32)
        if Tp != T or not xn.is_contiguous():
            buf = torch.zeros((B, M, Tp), dtype=torch.float32, device=x.device)
            buf[:, :, :T] = xn
            xn = buf
        return SeriesPack(xn, T)


class _InstanceNorm(torch.autograd.Function):
    """Instance norm with a gradient, for callers that ask for dLoss/dx (saliency, gradcheck).  The training loop never
    does (experiment_classification.py:315) and takes the plain path of instance_norm() below."""

    @staticmethod
    def forward(ctx, x):
        xc = x.detach().to(torch.float32).contiguous()
        B, T, M = xc.shape
        xn = torch.empty((B, M, C.padded_len(T)), dtype=torch.float32, device=xc.device)
        stat = torch.empty((2, B, M), dtype=torch.float32, device=xc.device)      # mean, 1 / (std + 1e-8)
        with torch.cuda.device(xc.device):
            C.check(STATS.call("instnorm", 1, lambda: C.lib.ign_instnorm_forward(
                _ptr(xc), _ptr(xn), _ptr(stat[0]), _ptr(stat[1]), B, T, M, _stream())), "ign_instnorm_forward")
        ctx.save_for_backward(xn, stat)
        ctx.T = T
        ctx.in_dtype = x.dtype
        return xn

    @staticmethod
    def backward(ctx, g):
        xn, stat = ctx.saved_tensors
        T = ctx.T
        # xn = (x - mu) r,  r = 1 / (sigma + 1e-8),  sigma = unbiased std over T   (Shapelet.py:187)
        # dx_j = r (g_j - mean g) - xn_j * sum_i(g_i xn_i) / ((T - 1) sigma)
        g = g[:, :, :T].to(torch.float32)
        z = xn[:, :, :T]
        r = stat[1].unsqueeze(-1)
        sigma = 1.0 / r - 1e-8
        dx = r * (g - g.mean(dim=-1, keepdim=True)) - z * (g * z).sum(dim=-1, keepdim=True) / ((T - 1) * sigma)
        return dx.transpose(1, 2).contiguous().to(ctx.in_dtype)


def instance_norm(x: torch.Tensor) -> SeriesPack:
    """x [B,T,M] -> SeriesPack(xn [B,M,Tp]).  Shapelet.py:186-187.  In the reference's training loop the raw batch never
    requires grad (experiment_classification.py:315); when it does (saliency), the pack carries an autograd variable
    and the shapelet transform returns dLoss/dxn through ign_shapelet_backward_input (stored-distance groups) or
    ign_shapelet_backward_recompute_input (recompute groups)."""
    _require_cuda(x, "x")
    if x.dim() != 3:
        raise RuntimeError("instance_norm expects [B,T,M], got %s" % (tuple(x.shape),))
    _check_device(x.device)
    if x.requires_grad and torch.is_grad_enabled():
        with torch.autocast(device_type="cuda", enabled=False):
            var = _InstanceNorm.apply(x)
        return SeriesPack(var.detach(), x.shape[1], xn_var=var)
    x = x.detach().to(torch.float32).contiguous()
    B, T, M = x.shape
    xn = torch.empty((B, M, C.padded_len(T)), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        C.check(STATS.call("instnorm", 1, lambda: C.lib.ign_instnorm_forward(
            _ptr(x), _ptr(xn), None, None, B, T, M, _stream())), "ign_instnorm_forward")
    return SeriesPack(xn, T)


# Has no effect; kept because bench.py saves and restores it around its per-kernel timing.
OVERLAP_BWD_PREPARE = False


class _Group:
    """One length group's forward state (what the backward needs)."""
    __slots__ = ("desc", "dist", "pool", "stored", "thr_shape", "needs")   # needs: (any, W, threshold)


def _forward_group(pack: SeriesPack, W, threshold, stride, eps, dist, pool, precision, need_grad):
    """Launch one group's forward.  Returns (group record, outputs (p, dmin, idx), the 4 tensors or Nones to save for
    backward)."""
    xn = pack.xn
    B, M, T, Tp = pack.B, pack.M, pack.T, pack.Tp
    K, M2, L = W.shape
    if M2 != M:
        raise RuntimeError("shapelet channels %d != series channels %d" % (M2, M))
    Wc = W.detach().to(torch.float32).contiguous()
    thr = None
    if pool == "lts_min":
        thr = threshold.detach().to(torch.float32).reshape(K, M).contiguous()
    desc = C.ShapeletDesc(B, M, T, Tp, K, L, int(stride), float(eps), C.DIST[dist], C.POOL[pool], C.PRECISION[precision])
    st0, _ = pack.window_stats(dist, L, stride)
    dev = xn.device
    out = torch.empty((2, B, K, M), dtype=torch.float32, device=dev)     # p, dmin
    idx = torch.empty((B, K, M), dtype=torch.int32, device=dev)         # argmin_t d
    dstore = None
    # stored-distance backward while distances + coefficients fit the budget, recompute backward beyond it
    store = need_grad and 2 * int(C.lib.ign_shapelet_dstore_bytes(byref(desc))) <= STORE_BUDGET_BYTES
    if store:
        Tw = C.padded_windows(T, L, int(stride))
        dstore = torch.empty((B, M, K, Tw), dtype=torch.float32, device=dev)
    fws_bytes = int(C.lib.ign_shapelet_forward_workspace(byref(desc)))
    fws = torch.empty((fws_bytes,), dtype=torch.uint8, device=dev) if fws_bytes else None
    tag = "shapelet_fwd/%s/L%d" % (dist, L)
    STATS.note_engine(tag, desc, False)
    with torch.cuda.device(dev):
        C.check(STATS.call(tag, 2 if fws_bytes else 1, lambda: C.lib.ign_shapelet_forward(
            byref(desc), _ptr(xn), _ptr(st0), _ptr(Wc), _ptr(thr), _ptr(out[0]), _ptr(out[1]),
            _ptr(idx), _ptr(dstore), _ptr(fws), fws_bytes, _stream())), "ign_shapelet_forward")
    rec = _Group()
    rec.desc, rec.dist, rec.pool, rec.stored = desc, dist, pool, bool(store)
    rec.thr_shape = None if threshold is None else threshold.shape
    saved = (Wc, out, idx, dstore if store else thr) if need_grad else (None,) * 4
    return rec, (out[0], out[1], idx), saved


def _backward_group(rec: _Group, pack: SeriesPack, saved, g_p, g_dmin, need_dx):
    """Host side of one group's backward: returns (dW or None, dthreshold or None, launch or None).  launch(dxn)
    allocates the group's workspace, runs the library (adding dLoss/dxn into dxn unless it is None) and releases the
    workspace on return: every launch is on the current stream, so the next group gets the same block in stream order.
    g_p or g_dmin may be None (no gradient on that output), not both."""
    Wc, out, idx, extra = saved
    dstore, thr = (extra, None) if rec.stored else (None, extra)
    desc = rec.desc
    _, need_w, need_thr = rec.needs
    # min_t d is the hard minimum (Shapelet.py:84 | :111): its gradient goes to the argmin window, inside the library
    gd = None if g_dmin is None else g_dmin.to(torch.float32).contiguous()
    g = torch.zeros_like(out[0]) if g_p is None else g_p.to(torch.float32).contiguous()
    dthr = None
    if rec.pool == "lts_min" and g_p is not None:     # min_t d does not depend on the threshold
        p = out[0]
        sig = p * (1.0 - p)                         # d sigmoid(thr - min_d)
        if need_thr:
            dthr = (g * sig).sum(dim=0).reshape(rec.thr_shape)
        g = (-g * sig).contiguous()                 # dLoss/d(min_d)
    if not need_w and not need_dx:
        return None, dthr, None
    st0, st1 = pack.window_stats(rec.dist, desc.L, desc.stride)
    if rec.stored:
        nbytes = C.lib.ign_shapelet_backward_workspace(byref(desc))
    elif need_dx:   # recompute mode with dx: one call per group, as no chunk's coefficients outlive the chunk
        nbytes = C.lib.ign_shapelet_backward_recompute_input_workspace(byref(desc), STORE_BUDGET_BYTES)
    else:       # recompute mode: the library walks the shapelets in chunks inside this bounded workspace
        nbytes = C.lib.ign_shapelet_backward_recompute_workspace(byref(desc), STORE_BUDGET_BYTES)
    dW = torch.empty_like(Wc) if need_w else None      # None: the library only prepares the coefficients for dxn
    tag = "shapelet_bwd/%s/L%d" % (rec.dist, desc.L)
    STATS.note_engine(tag, desc, True)

    def launch(dxn):
        ws = torch.empty((max(int(nbytes), 16),), dtype=torch.uint8, device=g.device)
        head = (byref(desc), _ptr(pack.xn), _ptr(st0), _ptr(st1), _ptr(Wc), _ptr(thr), _ptr(g))
        tail = (_ptr(dstore), _ptr(out[1]), _ptr(idx), _ptr(dW), _ptr(ws), int(nbytes), _stream())
        with torch.cuda.device(g.device):
            if dxn is not None and not rec.stored:
                C.check(STATS.call(tag, 3 if need_w else 2, lambda: C.lib.ign_shapelet_backward_recompute_input(
                    *head, _ptr(gd), _ptr(dW), _ptr(dxn), _ptr(ws), int(nbytes), _stream())),
                    "ign_shapelet_backward_recompute_input")
                return
            if gd is None:
                C.check(STATS.call(tag, 2 if need_w else 1, lambda: C.lib.ign_shapelet_backward(*head, *tail)),
                        "ign_shapelet_backward")
            else:
                C.check(STATS.call(tag, 2 if need_w else 1, lambda: C.lib.ign_shapelet_backward_dmin(
                    *head, _ptr(gd), *tail)), "ign_shapelet_backward_dmin")
            if dxn is not None:
                C.check(STATS.call("shapelet_bwd_input/%s/L%d" % (rec.dist, desc.L), 1, lambda: C.lib.ign_shapelet_backward_input(
                    byref(desc), _ptr(pack.xn), _ptr(st0), _ptr(st1), _ptr(Wc), _ptr(dstore), _ptr(dxn), _ptr(ws),
                    int(nbytes), _stream())), "ign_shapelet_backward_input")
    return dW, dthr, launch


def shapelet_transform(pack: SeriesPack, W: torch.Tensor, stride: int = 1, eps: float = 1.0, dist: str = "l1",
                       pool: str = "rbf_max", threshold: Optional[torch.Tensor] = None, precision: str = "fp32"):
    """Returns (p [B,K,M], dmin [B,K,M], argmin_t d [B,K,M] int32)."""
    _require_cuda(W, "shapelet weights")
    _check_device(W.device)
    if pool == "lts_min" and threshold is None:
        raise RuntimeError("lts_min pooling needs a threshold")
    track = torch.is_grad_enabled()
    # fp32 in / fp32 out regardless of autocast: the reference's distance math stays fp32 under bf16
    # autocast as well (SURVEY.md §7.3-7).
    with torch.autocast(device_type="cuda", enabled=False):
        outs = _SbmTransform.apply(pack, ((stride, eps, dist, pool, precision),), track, pack.xn_var, W, threshold)
    return outs[0], outs[1], outs[2]


class _SbmTransform(torch.autograd.Function):
    """All length groups of a ShapeBottleneckModel as ONE autograd node (the python loop of Shapelet.py:191-194).  The
    backward launches the groups one after another, each with its own workspace (_backward_group)."""

    @staticmethod
    def forward(ctx, pack: SeriesPack, cfgs, track, xn_var, *params):      # params = W_0, thr_0, W_1, thr_1, ...
        # Grad mode is always off inside Function.forward and needs_input_grad mirrors requires_grad even under
        # torch.no_grad(), so the caller's grad mode is passed in: evaluation loops must not pay for the 1.9 GB of
        # saved window distances.
        need_dx = bool(track and xn_var is not None and ctx.needs_input_grad[3])
        recs, outs, saved_all = [], [], []
        for gi, (stride, eps, dist, pool, precision) in enumerate(cfgs):
            W, thr = params[2 * gi], params[2 * gi + 1]
            nW, nT = bool(ctx.needs_input_grad[4 + 2 * gi]), bool(ctx.needs_input_grad[5 + 2 * gi])
            need = bool(track and (nW or nT or need_dx))
            rec, o, saved = _forward_group(pack, W, thr, stride, eps, dist, pool, precision, need)
            rec.needs = (need, nW, nT)
            recs.append(rec); outs.extend(o); saved_all.extend(saved)
        ctx.set_materialize_grads(False)
        ctx.recs, ctx.pack, ctx.need_dx = recs, pack, need_dx
        ctx.save_for_backward(*saved_all)
        ctx.mark_non_differentiable(*outs[2::3])
        return tuple(outs)

    @staticmethod
    def backward(ctx, *gs):
        recs, pack = ctx.recs, ctx.pack
        saved = ctx.saved_tensors
        grads = [None] * (2 * len(recs))
        launches = []
        for gi, rec in enumerate(recs):
            g_p, g_dmin = gs[3 * gi], gs[3 * gi + 1]
            if (g_p is None and g_dmin is None) or not rec.needs[0]:
                continue
            grads[2 * gi], grads[2 * gi + 1], launch = _backward_group(rec, pack, saved[4 * gi:4 * gi + 4], g_p,
                                                                       g_dmin, ctx.need_dx)
            if launch is not None:
                launches.append(launch)
        # input gradients (saliency): each group adds dLoss/dxn from the coefficients its own backward call left
        dxn = torch.zeros_like(pack.xn) if ctx.need_dx else None
        # The host work of every group first, then the launches back to back, one workspace at a time.  Host work
        # between the launches shifts how the shapelet kernels overlap the deep expert's side stream: measured at
        # +0.3-0.6 % (L1) and +4 % (cosine / 3xTF32) per step at config 2 on a B200 at 1000 W, with the same kernel times.
        for launch in launches:
            launch(dxn)
        return (None, None, None, dxn) + tuple(grads)


def sbm_transform(pack: SeriesPack, layers):
    """[(p, dmin, idx)] for the Shapelet layers of one bottleneck model, as one autograd node."""
    cfgs, params = [], []
    for layer in layers:
        _require_cuda(layer.weights, "shapelet weights")
        if pack.T < layer.length:   # what x.unfold raises in Shapelet.py:61
            raise RuntimeError(f"maximum size for tensor at dimension 2 is {pack.T} but size is {layer.length}")
        cfgs.append((layer.stride, layer.eps, layer._dist(), layer.pool, layer.precision))
        params.extend((layer.weights, layer._threshold()))
    _check_device(pack.xn.device)
    track = torch.is_grad_enabled()
    with torch.autocast(device_type="cuda", enabled=False):
        outs = _SbmTransform.apply(pack, tuple(cfgs), track, pack.xn_var, *params)
    return [(outs[3 * i], outs[3 * i + 1], outs[3 * i + 2]) for i in range(len(layers))]


class _Diversity(torch.autograd.Function):
    """mean_{m, a != b} exp(-||w_b - w_a + 1e-6||) of one length group (Shapelet.py:223-230), one launch each way."""

    @staticmethod
    def forward(ctx, W):
        Wc = W.detach().to(torch.float32).contiguous()
        K, M, L = Wc.shape
        coef = torch.empty((M, K, K), dtype=torch.float32, device=Wc.device)
        part = torch.empty((M * int(C.lib.ign_diversity_partials(K)),), dtype=torch.float32, device=Wc.device)
        with torch.cuda.device(Wc.device):
            C.check(STATS.call("diversity_fwd", 1, lambda: C.lib.ign_diversity_forward(
                _ptr(Wc), _ptr(coef), _ptr(part), K, M, L, _stream())), "ign_diversity_forward")
        ctx.save_for_backward(Wc, coef)
        return part.sum() / float(M * K * K)

    @staticmethod
    def backward(ctx, gout):
        Wc, coef = ctx.saved_tensors
        K, M, L = Wc.shape
        g = gout.detach().to(torch.float32).reshape(1).contiguous()
        dW = torch.empty_like(Wc)
        with torch.cuda.device(Wc.device):
            C.check(STATS.call("diversity_bwd", 1, lambda: C.lib.ign_diversity_backward(
                _ptr(Wc), _ptr(coef), _ptr(g), _ptr(dW), K, M, L, _stream())), "ign_diversity_backward")
        return dW


def shapelet_diversity(W: torch.Tensor) -> torch.Tensor:
    """Diversity term of one Shapelet layer's weights [K,M,L] (scalar), fused CUDA path."""
    _require_cuda(W, "shapelet weights")
    _check_device(W.device)
    with torch.autocast(device_type="cuda", enabled=False):
        return _Diversity.apply(W)


class _GiniGate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, sbm_out, deep_out, gating_value):
        s = sbm_out.detach().to(torch.float32).contiguous()
        z = deep_out.detach().to(torch.float32).contiguous()
        B, Cn = s.shape
        out = torch.empty_like(s)
        eta = torch.empty((B, 1), dtype=torch.float32, device=s.device)
        use_gate = gating_value is not None
        gv = float(gating_value) if use_gate else 0.0
        with torch.cuda.device(s.device):
            C.check(STATS.call("gate_fwd", 1, lambda: C.lib.ign_gate_forward(
                _ptr(s), _ptr(z), _ptr(out), _ptr(eta), B, Cn, int(use_gate), gv, _stream())), "ign_gate_forward")
        ctx.save_for_backward(s, z)
        ctx.gate = (use_gate, gv)
        ctx.in_dtypes = (sbm_out.dtype, deep_out.dtype)
        return out, eta

    @staticmethod
    def backward(ctx, g_out, g_eta):
        s, z = ctx.saved_tensors
        B, Cn = s.shape
        go = g_out.to(torch.float32).contiguous()
        ge = None if g_eta is None else g_eta.to(torch.float32).contiguous()
        gs = torch.empty_like(s)
        gz = torch.empty_like(z)
        use_gate, gv = ctx.gate
        with torch.cuda.device(s.device):
            C.check(STATS.call("gate_bwd", 1, lambda: C.lib.ign_gate_backward(
                _ptr(s), _ptr(z), _ptr(go), _ptr(ge), _ptr(gs), _ptr(gz), B, Cn, int(use_gate), gv, _stream())),
                "ign_gate_backward")
        return gs.to(ctx.in_dtypes[0]), gz.to(ctx.in_dtypes[1]), None


def gini_gate(sbm_out: torch.Tensor, deep_out: torch.Tensor, gating_value: Optional[float] = None):
    """InterpGN.py:44-52 fused: returns (out [B,C], eta [B,1]); computed in fp32."""
    _require_cuda(sbm_out, "sbm_out")
    _require_cuda(deep_out, "deep_out")
    if sbm_out.shape != deep_out.shape or sbm_out.dim() != 2:
        raise RuntimeError("gini_gate expects two [B,C] tensors, got %s and %s"
                           % (tuple(sbm_out.shape), tuple(deep_out.shape)))
    _check_device(sbm_out.device)
    return _GiniGate.apply(sbm_out, deep_out, gating_value)
