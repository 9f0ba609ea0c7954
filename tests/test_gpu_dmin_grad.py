"""GPU: gradients through the shapelet layer's second output, the minimum window distance min_t d (Shapelet.py:84 for
Shapelet, :111 for DistThresholdShapelet; ShapeBottleneckModel reports it as ModelInfo.d).  It is the hard minimum
d.min(dim=time).values in both poolings, as the oracle restates it (ShapeletOut.dmin), so its gradient lands on one
window per row: argmin_t d, first index on ties.

Ground truth is fp64 autograd through oracle.shapelet_forward applied to sum(g_p * p) + sum(g_d * dmin).  Tolerances
are the layer tests': gradients 1e-4 relative to the largest entry, input gradients 2e-4."""
from ctypes import byref

import pytest
import torch

import ign_oracle as O
from helpers import MODES, assert_close, seeded_batch, seeded_fill

pytestmark = pytest.mark.gpu
DEV = "cuda"


def run_layer(xn, W, stride, eps, dist, pool, thr, gp, gd, precision="fp32", need_dx=False, train_w=True):
    """The library's layer on the GPU; returns (p, dmin, idx, dW, dthreshold, dx) for the loss sum(gp p) + sum(gd dmin)
    (either term may be None)."""
    from layers.shapelet_ops import SeriesPack, shapelet_transform
    Wd = W.detach().clone().to(DEV).requires_grad_(train_w)
    thd = None if thr is None else thr.detach().clone().to(DEV).requires_grad_(train_w)
    xd = xn.detach().clone().to(DEV).requires_grad_(need_dx)
    p, dmin, idx = shapelet_transform(SeriesPack.from_channel_major(xd), Wd, stride, eps, dist, pool, thd, precision)
    loss = 0.
    if gp is not None:
        loss = loss + (p * gp.to(DEV)).sum()
    if gd is not None:
        loss = loss + (dmin * gd.to(DEV)).sum()
    loss.backward()
    torch.cuda.synchronize()
    return p, dmin, idx, Wd.grad, None if thd is None else thd.grad, xd.grad


def oracle_grads(xn, W, stride, eps, mode, pool, thr, gp, gd, need_dx=False):
    """(dW, dthreshold, dx) by fp64 autograd through the oracle's forward."""
    Wv = W.double().requires_grad_(True)
    tv = None if thr is None else thr.double().requires_grad_(True)
    xv = xn.double().requires_grad_(need_dx)
    out = O.shapelet_forward(xv, Wv, stride, eps, mode, pool, tv)
    K, M = W.shape[0], W.shape[1]
    loss = 0.
    if gp is not None:
        loss = loss + (out.p.view(-1, K, M) * gp.double()).sum()
    if gd is not None:
        loss = loss + (out.dmin.view(-1, K, M) * gd.double()).sum()
    loss.backward()
    return Wv.grad, None if tv is None else tv.grad, xv.grad


def desc_of(B, M, T, K, L, stride, eps, dist, pool, precision):
    from layers import ign_cabi as C
    return C.ShapeletDesc(B, M, T, C.padded_len(T), K, L, stride, eps, C.DIST[dist], C.POOL[pool],
                          C.PRECISION[precision])


def check_grads(got, ref, what):
    dW, dthr = got
    dW_ref, dthr_ref = ref
    assert_close(dW, dW_ref, 1e-4, 1e-4 * float(dW_ref.abs().max()), what + " dW")
    if dthr_ref is None:
        assert dthr is None or float(dthr.abs().max()) == 0.0, what + " dthreshold"
    else:
        assert_close(dthr, dthr_ref, 1e-4, 1e-5, what + " dthreshold")


# (flag, pool, precision): every distance with rbf_max, on the CUDA-core engine and (cross-term modes) on tcgen05;
# lts_min takes L1 / squared L2 only (Shapelet.py:100-103)
LAYER_MODES = [("euclidean", "rbf_max", "fp32"), ("sql2", "rbf_max", "fp32"), ("cosine", "rbf_max", "fp32"),
               ("pearson", "rbf_max", "fp32"), ("sql2", "rbf_max", "3xtf32"), ("cosine", "rbf_max", "3xtf32"),
               ("pearson", "rbf_max", "3xtf32"), ("euclidean", "lts_min", "fp32"), ("sql2", "lts_min", "fp32"),
               ("sql2", "lts_min", "3xtf32")]
SHAPES = [(3, 4, 64, 5, 9, 1), (2, 3, 400, 4, 50, 3)]          # B, M, T, K, L, stride


@pytest.mark.parametrize("flag,pool,precision", LAYER_MODES)
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("terms", ["p_and_d", "d_only"])
def test_dmin_gradient_vs_oracle(flag, pool, precision, shape, terms):
    from layers import ign_cabi as C
    B, M, T, K, L, stride = shape
    mode, dist = MODES[flag]
    if precision != "fp32":
        d = desc_of(B, M, T, K, L, stride, 0.9, dist, pool, precision)
        assert C.ENGINE[C.lib.ign_shapelet_engine(byref(d), 1)] == "tcgen05"
    torch.manual_seed(500 + T + L + len(flag))
    xn, W = torch.randn(B, M, T), torch.randn(K, M, L)
    gp = torch.randn(B, K, M) if terms == "p_and_d" else None
    gd = torch.randn(B, K, M)
    thr = torch.rand(1, K, M) if pool == "lts_min" else None
    opool = O.POOL_LTS_MIN if pool == "lts_min" else O.POOL_RBF_MAX
    _, _, _, dW, dthr, _ = run_layer(xn, W, stride, 0.9, dist, pool, thr, gp, gd, precision)
    dW_ref, dthr_ref, _ = oracle_grads(xn, W, stride, 0.9, mode, opool, thr, gp, gd)
    check_grads((dW, dthr), (dW_ref, dthr_ref), f"{flag}/{pool}/{precision} {shape} {terms}")


def test_dmin_gradient_goes_to_the_argmin_not_to_the_p_argmax():
    """eps = 1000: every p = exp(-(eps d)^2) underflows to 0 in fp32, so the straight-through one-hot of p picks window 0
    while the minimum distance sits elsewhere.  The d gradient must follow the minimum."""
    B, M, T, K, L = 3, 4, 120, 5, 9
    torch.manual_seed(3)
    xn, W, gd = torch.randn(B, M, T), torch.randn(K, M, L), torch.randn(B, K, M)
    p, _, idx, dW, _, _ = run_layer(xn, W, 1, 1000.0, "l1", "rbf_max", None, torch.randn(B, K, M), gd)
    assert float(p.detach().abs().max()) == 0.0 and bool((idx != 0).float().mean() > 0.9)
    dW_ref, _, _ = oracle_grads(xn, W, 1, 1000.0, O.DIST_L1, O.POOL_RBF_MAX, None, None, gd)
    assert_close(dW, dW_ref, 1e-4, 1e-4 * float(dW_ref.abs().max()), "underflowed p: dW")


# Pooling backward row geometries: masked tails of the register-resident kernel (T' = 501: one masked float4 chunk;
# T' = 901: scalar sub-chunks) and the generic kernel above 1024 windows.
@pytest.mark.parametrize("flag", ["euclidean", "sql2", "cosine", "pearson", "lts"])
@pytest.mark.parametrize("Tw", [501, 901, 1025, 1500])
def test_dmin_gradient_row_geometries(flag, Tw):
    B, M, K, L = 2, 2, 3, 5
    T = Tw + L - 1
    torch.manual_seed(6000 + Tw)
    xn, W, gp, gd = torch.randn(B, M, T), torch.randn(K, M, L), torch.randn(B, K, M), torch.randn(B, K, M)
    # near copies of a shapelet in the last windows put the minimum of those rows inside the tail the kernels treat
    # apart (not exact copies: every distance is stationary there, and the d gradient would contribute nothing)
    xn[0, :, Tw - 1:Tw - 1 + L] = W[0] + 0.01 * torch.randn(M, L)
    xn[1, :, Tw - 3:Tw - 3 + L] = W[1] + 0.01 * torch.randn(M, L)
    pool = "lts_min" if flag == "lts" else "rbf_max"
    mode, dist = MODES["euclidean" if flag == "lts" else flag]
    thr = torch.rand(1, K, M) if flag == "lts" else None
    _, _, idx, dW, dthr, _ = run_layer(xn, W, 1, 0.9, dist, pool, thr, gp, gd)
    assert bool((idx[0, 0] == Tw - 1).all()) and bool((idx[1, 1] == Tw - 3).all())
    ref = oracle_grads(xn, W, 1, 0.9, mode, O.POOL_LTS_MIN if flag == "lts" else O.POOL_RBF_MAX, thr, gp, gd)
    check_grads((dW, dthr), ref[:2], f"{flag} Tw={Tw}")


# ---------------------------------------------------------------------------------------------------------------------
# Recompute backward: the shapelets are walked in chunks; each chunk's d gradient lands on the chunk's recomputed argmin
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def store_budget(monkeypatch):
    from layers import shapelet_ops
    def set_budget(nbytes):
        monkeypatch.setattr(shapelet_ops, "STORE_BUDGET_BYTES", int(nbytes))
    return set_budget


@pytest.mark.parametrize("flag,precision,pool", [("euclidean", "fp32", "rbf_max"), ("cosine", "fp32", "rbf_max"),
                                                 ("pearson", "3xtf32", "rbf_max"), ("sql2", "3xtf32", "rbf_max"),
                                                 ("euclidean", "fp32", "lts_min"), ("sql2", "fp32", "lts_min")])
# batches large enough that even the tcgen05 engine's chunk workspace for all K shapelets stays below what the
# stored mode would keep (the budget can then ask for one chunk)
@pytest.mark.parametrize("shape", [(16, 4, 200, 45, 20, 1), (48, 3, 400, 13, 50, 3)])
@pytest.mark.parametrize("chunks", ["one", "several"])
def test_dmin_gradient_recompute_mode(store_budget, flag, precision, pool, shape, chunks):
    from layers import ign_cabi as C
    B, M, T, K, L, stride = shape
    mode, dist = MODES[flag]
    torch.manual_seed(700 + K + L)
    xn, W, gp, gd = torch.randn(B, M, T), torch.randn(K, M, L), torch.randn(B, K, M), torch.randn(B, K, M)
    thr = torch.rand(1, K, M) if pool == "lts_min" else None
    stored = run_layer(xn, W, stride, 0.9, dist, pool, thr, gp, gd, precision)
    desc = desc_of(B, M, T, K, L, stride, 0.9, dist, pool, precision)
    ws_one = int(C.lib.ign_shapelet_backward_recompute_workspace(byref(desc), 2 ** 40))     # all K shapelets at once
    budget = ws_one if chunks == "one" else ws_one // 2
    assert 2 * int(C.lib.ign_shapelet_dstore_bytes(byref(desc))) > budget                 # the layer recomputes
    ws = int(C.lib.ign_shapelet_backward_recompute_workspace(byref(desc), budget))
    assert (ws == ws_one) if chunks == "one" else (ws < ws_one)
    store_budget(budget)
    rec = run_layer(xn, W, stride, 0.9, dist, pool, thr, gp, gd, precision)
    assert torch.equal(stored[2], rec[2])
    opool = O.POOL_LTS_MIN if pool == "lts_min" else O.POOL_RBF_MAX
    dW_ref, dthr_ref, _ = oracle_grads(xn, W, stride, 0.9, mode, opool, thr, gp, gd)
    what = f"{flag}/{precision}/{pool} {shape} recompute ({chunks} chunk)"
    check_grads(rec[3:5], (dW_ref, dthr_ref), what)
    scale = float(dW_ref.abs().max())
    assert_close(rec[3], stored[3], 1e-5, 1e-6 * scale, what + " vs stored dW")
    # the d gradient alone
    rec_d = run_layer(xn, W, stride, 0.9, dist, pool, thr, None, gd, precision)
    check_grads(rec_d[3:5], oracle_grads(xn, W, stride, 0.9, mode, opool, thr, None, gd)[:2], what + " d only")


# ---------------------------------------------------------------------------------------------------------------------
# Input gradients (stored mode): ign_shapelet_backward_input reads the coefficients, so the d term reaches dx unchanged
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("flag,pool", [("euclidean", "rbf_max"), ("cosine", "rbf_max"), ("pearson", "rbf_max"),
                                       ("euclidean", "lts_min")])
@pytest.mark.parametrize("shape", [(3, 4, 64, 5, 9, 1), (2, 3, 400, 4, 50, 3), (2, 2, 1000, 5, 300, 1)])
@pytest.mark.parametrize("terms", ["p_and_d", "d_only"])
def test_dmin_input_gradient(flag, pool, shape, terms):
    B, M, T, K, L, stride = shape
    mode, dist = MODES[flag]
    torch.manual_seed(800 + T + L)
    xn, W = torch.randn(B, M, T), torch.randn(K, M, L)
    gp = torch.randn(B, K, M) if terms == "p_and_d" else None
    gd = torch.randn(B, K, M)
    thr = torch.rand(1, K, M) if pool == "lts_min" else None
    opool = O.POOL_LTS_MIN if pool == "lts_min" else O.POOL_RBF_MAX
    dW_ref, dthr_ref, dx_ref = oracle_grads(xn, W, stride, 0.9, mode, opool, thr, gp, gd, need_dx=True)
    what = f"{flag}/{pool} {shape} {terms}"
    _, _, _, dW, dthr, dx = run_layer(xn, W, stride, 0.9, dist, pool, thr, gp, gd, need_dx=True)
    assert_close(dx, dx_ref, 2e-4, 2e-4 * float(dx_ref.abs().max()), what + " dx")
    check_grads((dW, dthr), (dW_ref, dthr_ref), what + " (with dx)")
    # weights frozen: only the pooling backward runs (dW == NULL), the input gradient is the same
    _, _, _, dW2, _, dx2 = run_layer(xn, W, stride, 0.9, dist, pool, thr, gp, gd, need_dx=True, train_w=False)
    assert dW2 is None and torch.equal(dx2, dx)


# ---------------------------------------------------------------------------------------------------------------------
# Modules: Shapelet.forward's second output and ModelInfo.d in a loss
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cls", ["Shapelet", "DistThresholdShapelet"])
def test_layer_second_output_backward(cls):
    import models.Shapelet as S
    torch.manual_seed(21)
    B, M, T, K, L = 4, 3, 90, 6, 12
    layer = getattr(S, cls)(M, L, K).to(DEV)
    x = torch.randn(B, M, T)
    p, d = layer(x.to(DEV))
    assert p.shape == d.shape == (B, K * M)
    d.sum().backward()
    torch.cuda.synchronize()
    W = layer.weights.detach().cpu()
    thr = layer.threshold.detach().cpu() if cls == "DistThresholdShapelet" else None
    dW_ref, _, _ = oracle_grads(x, W, 1, 1.0, O.DIST_L1, O.POOL_LTS_MIN if thr is not None else O.POOL_RBF_MAX, thr,
                                None, torch.ones(B, K, M))
    assert_close(layer.weights.grad, dW_ref, 1e-4, 1e-4 * float(dW_ref.abs().max()), cls + " dW of d.sum()")
    if thr is not None:
        assert layer.threshold.grad is None             # min_t d does not depend on the threshold


def _cfg(distance_func):
    from types import SimpleNamespace
    return SimpleNamespace(enc_in=12, num_class=9, seq_len=29, epsilon=1., distance_func=distance_func,
                           memory_efficient=False, sbm_cls="linear", dropout=0., lambda_reg=0.1, lambda_div=0.1,
                           dnn_type="FCN")


@pytest.mark.parametrize("model_cls,flag", [("ShapeBottleneckModel", "euclidean"), ("ShapeBottleneckModel", "cosine"),
                                            ("DistThresholdSBM", "euclidean")])
def test_bottleneck_model_loss_with_reported_distances(model_cls, flag):
    """(cross entropy + regulariser + info.d.sum()).backward() against the same loss on the oracle model in fp64."""
    import models.Shapelet as S
    model = getattr(S, model_cls)(_cfg(flag)).to(DEV).train()
    seeded_fill(model, 5)
    x, y = seeded_batch(6, 29, 12, 9, 5)
    out, info = model(x.to(DEV))
    loss = torch.nn.functional.cross_entropy(out, y.to(DEV)) + info.loss.mean() + info.d.sum()
    loss.backward()
    torch.cuda.synchronize()
    lts = model_cls == "DistThresholdSBM"
    Ws = [s.weights.detach().cpu().double().requires_grad_(True) for s in model.shapelets]
    thrs = [s.threshold.detach().cpu().double().requires_grad_(True) for s in model.shapelets] if lts else None
    Wc = model.output_layer.weight.detach().cpu().double().requires_grad_(True)
    logits, _, dists = O.sbm_forward(x.double(), Ws, [s.stride for s in model.shapelets], Wc, 1.0, MODES[flag][0],
                                     O.POOL_LTS_MIN if lts else O.POOL_RBF_MAX, thrs)
    ref_loss = torch.nn.functional.cross_entropy(logits, y) + O.sbm_loss(Wc, Ws, 0.1, 0.1) + dists.sum()
    ref_loss.backward()
    assert_close(info.d, dists, 2e-5, 2e-6, "ModelInfo.d")
    pairs = [(s.weights.grad, w.grad, "shapelets.%d.weights" % i) for i, (s, w) in enumerate(zip(model.shapelets, Ws))]
    if lts:
        pairs += [(s.threshold.grad, t.grad, "shapelets.%d.threshold" % i)
                  for i, (s, t) in enumerate(zip(model.shapelets, thrs))]
    pairs.append((model.output_layer.weight.grad, Wc.grad, "output_layer.weight"))
    for got, ref, name in pairs:
        assert_close(got, ref, 1e-3, 2e-4 * float(ref.abs().max()) + 1e-7, model_cls + " grad " + name)


def test_interpgn_loss_with_reported_distances():
    """InterpGN: adding info.d.sum() to the training loss changes the shapelet gradients by exactly the oracle's
    d(sum d)/dW and leaves every other parameter's gradient as it was."""
    from models.InterpGN import InterpGN
    model = InterpGN(_cfg("euclidean")).to(DEV).train()
    seeded_fill(model, 9)
    x, y = seeded_batch(6, 29, 12, 9, 9)
    x, y = x.to(DEV), y.to(DEV)
    mask = torch.ones(6, 29, device=DEV)
    grads = []
    for with_d in (False, True):
        model.zero_grad(set_to_none=True)
        out, info = model(x, mask, None, None)
        loss = torch.nn.functional.cross_entropy(out, y) + info.loss.mean() + \
            torch.nn.functional.cross_entropy(info.shapelet_preds, y)
        if with_d:
            loss = loss + info.d.sum()
        loss.backward()
        torch.cuda.synchronize()
        grads.append({k: p.grad.detach().clone() for k, p in model.named_parameters() if p.grad is not None})
    base, withd = grads
    assert base.keys() == withd.keys()
    Ws = [s.weights.detach().cpu().double().requires_grad_(True) for s in model.sbm.shapelets]
    _, _, dists = O.sbm_forward(x.cpu().double(), Ws, [s.stride for s in model.sbm.shapelets],
                                model.sbm.output_layer.weight.detach().cpu().double())
    dists.sum().backward()
    for k in base:
        if k.startswith("sbm.shapelets.") and k.endswith(".weights"):
            ref = Ws[int(k.split(".")[2])].grad
            scale = float(ref.abs().max()) + float(base[k].abs().max())
            assert_close(withd[k] - base[k], ref, 1e-4, 1e-4 * scale, "InterpGN d(sum d)/d " + k)
        else:
            assert_close(withd[k], base[k], 1e-5, 1e-6 * float(base[k].abs().max()) + 1e-9, "InterpGN grad " + k)


# ---------------------------------------------------------------------------------------------------------------------
# The C ABI: ign_shapelet_backward is ign_shapelet_backward_dmin with gdmin_dev = NULL
# ---------------------------------------------------------------------------------------------------------------------
def _c_forward(xn, W, stride, dist, pool, thr, precision, store=True):
    from layers import ign_cabi as C
    from layers.shapelet_ops import SeriesPack
    B, M, T = xn.shape
    K, _, L = W.shape
    desc = desc_of(B, M, T, K, L, stride, 0.9, dist, pool, precision)
    pack = SeriesPack.from_channel_major(xn.to(DEV))
    st0, st1 = pack.window_stats(dist, L, stride)
    out = torch.empty((2, B, K, M), device=DEV)
    idx = torch.empty((B, K, M), dtype=torch.int32, device=DEV)
    dstore = torch.empty((B, M, K, C.padded_windows(T, L, stride)), device=DEV) if store else None
    nf = int(C.lib.ign_shapelet_forward_workspace(byref(desc)))
    fws = torch.empty((max(nf, 16),), dtype=torch.uint8, device=DEV)
    ptr = lambda t: None if t is None else t.data_ptr()
    C.check(C.lib.ign_shapelet_forward(byref(desc), ptr(pack.xn), ptr(st0), ptr(W), ptr(thr), ptr(out[0]),
                                       ptr(out[1]), ptr(idx), ptr(dstore), ptr(fws), nf, None), "forward")
    return desc, pack, st0, st1, out, idx, dstore


@pytest.mark.parametrize("flag,pool,precision", [("euclidean", "rbf_max", "fp32"), ("cosine", "rbf_max", "3xtf32"),
                                                 ("pearson", "rbf_max", "fp32"), ("sql2", "lts_min", "fp32")])
@pytest.mark.parametrize("store", [True, False])
def test_backward_without_dmin_gradient_is_bit_identical(flag, pool, precision, store):
    from layers import ign_cabi as C
    torch.manual_seed(31)
    B, M, T, K, L = 3, 4, 300, 20, 40
    xn, W, g = torch.randn(B, M, T), torch.randn(K, M, L, device=DEV), torch.randn(B, K, M, device=DEV)
    thr = torch.rand(K, M, device=DEV) if pool == "lts_min" else None
    dist = MODES[flag][1]
    desc, pack, st0, st1, out, idx, dstore = _c_forward(xn, W, 1, dist, pool, thr, precision, store)
    nbytes = int(C.lib.ign_shapelet_backward_workspace(byref(desc)) if store else
                 C.lib.ign_shapelet_backward_recompute_workspace(byref(desc), 200_000))
    ptr = lambda t: None if t is None else t.data_ptr()
    dWs = []
    for fn in ("ign_shapelet_backward", "ign_shapelet_backward_dmin"):
        ws = torch.full((nbytes,), 255, dtype=torch.uint8, device=DEV)
        dW = torch.full_like(W, float("nan"))
        head = (byref(desc), ptr(pack.xn), ptr(st0), ptr(st1), ptr(W), ptr(thr), ptr(g))
        tail = (ptr(dstore), ptr(out[1]), ptr(idx), ptr(dW), ptr(ws), nbytes, None)
        args = head + tail if fn == "ign_shapelet_backward" else head + (None,) + tail
        C.check(getattr(C.lib, fn)(*args), fn)
        dWs.append(dW)
    torch.cuda.synchronize()
    assert bool(torch.isfinite(dWs[0]).all()) and torch.equal(dWs[0], dWs[1])


def test_dmin_gradient_needs_the_forward_argmin_in_stored_mode():
    from layers import ign_cabi as C
    B, M, T, K, L = 2, 2, 50, 3, 5
    xn, W = torch.randn(B, M, T), torch.randn(K, M, L, device=DEV)
    desc, pack, _, _, out, idx, dstore = _c_forward(xn, W, 1, "l1", "rbf_max", None, "fp32")
    nbytes = int(C.lib.ign_shapelet_backward_workspace(byref(desc)))
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=DEV)
    g, dW = torch.zeros(B, K, M, device=DEV), torch.empty_like(W)
    rc = C.lib.ign_shapelet_backward_dmin(byref(desc), pack.xn.data_ptr(), None, None, W.data_ptr(), None,
                                          g.data_ptr(), g.data_ptr(), dstore.data_ptr(), out[1].data_ptr(), None,
                                          dW.data_ptr(), ws.data_ptr(), nbytes, None)
    assert rc == 1 and "argmin" in C.last_error()
