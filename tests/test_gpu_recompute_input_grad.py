"""GPU: input gradients (dLoss/dx: saliency, gradcheck) of length groups that take the recompute backward, the bounded-
memory mode for shapes whose window distances the stored mode cannot keep.  There one library call per group
(ign_shapelet_backward_recompute_input) walks the shapelets in chunks: it recomputes each chunk's distances, runs the
pooling backward and the contraction, and adds the chunk's share of dx.

STORE_BUDGET_BYTES is lowered to force the recompute mode, and every case asserts that the stored mode would need more
(2 x dstore bytes > budget).  Ground truth is fp64 autograd through the oracle on sum(g_p * p) + sum(g_d * dmin).
Tolerances are those of the stored-mode input-gradient tests: dx 2e-4 relative to the largest entry, dW 1e-4."""
from ctypes import byref
from types import SimpleNamespace

import pytest
import torch

import ign_oracle as O
from helpers import MODES, assert_close, load_golden, t

pytestmark = pytest.mark.gpu
DEV = "cuda"
EPS = 0.9


@pytest.fixture
def store_budget(monkeypatch):
    from layers import shapelet_ops
    def set_budget(nbytes):
        monkeypatch.setattr(shapelet_ops, "STORE_BUDGET_BYTES", int(nbytes))
    return set_budget


def desc_of(B, M, T, K, L, stride, dist, pool, precision):
    from layers import ign_cabi as C
    return C.ShapeletDesc(B, M, T, C.padded_len(T), K, L, stride, EPS, C.DIST[dist], C.POOL[pool],
                          C.PRECISION[precision])


def run_layer(xn, W, stride, dist, pool, thr, gp, gd, precision, train_w=True):
    """The library's layer on the GPU: (dW, dthreshold, dx) of sum(gp p) + sum(gd dmin) (either term may be None)."""
    from layers.shapelet_ops import SeriesPack, shapelet_transform
    Wd = W.detach().clone().to(DEV).requires_grad_(train_w)
    thd = None if thr is None else thr.detach().clone().to(DEV).requires_grad_(train_w)
    xd = xn.detach().clone().to(DEV).requires_grad_(True)
    p, dmin, _ = shapelet_transform(SeriesPack.from_channel_major(xd), Wd, stride, EPS, dist, pool, thd, precision)
    loss = 0.
    if gp is not None:
        loss = loss + (p * gp.to(DEV)).sum()
    if gd is not None:
        loss = loss + (dmin * gd.to(DEV)).sum()
    loss.backward()
    torch.cuda.synchronize()
    return Wd.grad, None if thd is None else thd.grad, xd.grad


def oracle_grads(xn, W, stride, mode, pool, thr, gp, gd):
    """(dW, dthreshold, dx) by fp64 autograd through the oracle's forward."""
    Wv = W.double().requires_grad_(True)
    tv = None if thr is None else thr.double().requires_grad_(True)
    xv = xn.double().requires_grad_(True)
    out = O.shapelet_forward(xv, Wv, stride, EPS, mode, pool, tv)
    K, M = W.shape[0], W.shape[1]
    loss = 0.
    if gp is not None:
        loss = loss + (out.p.view(-1, K, M) * gp.double()).sum()
    if gd is not None:
        loss = loss + (out.dmin.view(-1, K, M) * gd.double()).sum()
    loss.backward()
    return Wv.grad, None if tv is None else tv.grad, xv.grad


def check_grads(dW, dthr, dx, ref, what):
    dW_ref, dthr_ref, dx_ref = ref
    if dx_ref is not None:
        assert_close(dx, dx_ref, 2e-4, 2e-4 * float(dx_ref.abs().max()), what + " dx")
    assert_close(dW, dW_ref, 1e-4, 1e-4 * float(dW_ref.abs().max()), what + " dW")
    if dthr_ref is None:
        assert dthr is None or float(dthr.abs().max()) == 0.0, what + " dthreshold"
    else:
        assert_close(dthr, dthr_ref, 1e-4, 1e-5, what + " dthreshold")


def force_recompute(store_budget, desc, chunks):
    """Sets a budget that makes the layer recompute with `chunks` ("several": fewer shapelets per chunk than K,
    "minimum": budget 1, the 8-shapelet minimum chunk) and returns it."""
    from layers import ign_cabi as C
    ws_all = int(C.lib.ign_shapelet_backward_recompute_input_workspace(byref(desc), 2 ** 40))   # one chunk of K
    stored = 2 * int(C.lib.ign_shapelet_dstore_bytes(byref(desc)))
    budget = min(ws_all // 3, stored - 1) if chunks == "several" else 1
    assert stored > budget                                                        # the layer recomputes
    assert int(C.lib.ign_shapelet_backward_recompute_input_workspace(byref(desc), budget)) < ws_all
    store_budget(budget)
    return budget


# (flag, pool, precision): L1 / cosine / pearson with rbf_max, L1 with lts_min (Shapelet.py:100-103); the cross-term
# modes on the CUDA-core engine and on tcgen05 (3xTF32)
DX_MODES = [("euclidean", "rbf_max", "fp32"), ("cosine", "rbf_max", "fp32"), ("pearson", "rbf_max", "fp32"),
            ("euclidean", "lts_min", "fp32"), ("cosine", "rbf_max", "3xtf32"), ("pearson", "rbf_max", "3xtf32")]
DX_SHAPES = [((3, 4, 200, 45, 20, 1), "several"),       # several chunks of 8..16 shapelets
             ((2, 3, 400, 13, 50, 3), "several"),       # strided windows, ragged last chunk
             ((2, 5, 130, 20, 16, 1), "minimum")]       # budget 1: chunks of the minimum size


@pytest.mark.parametrize("flag,pool,precision", DX_MODES)
@pytest.mark.parametrize("shape,chunks", DX_SHAPES)
@pytest.mark.parametrize("terms", ["p", "p_and_d", "d"])
def test_recompute_input_gradient_vs_oracle_and_stored(store_budget, flag, pool, precision, shape, chunks, terms):
    from layers import ign_cabi as C
    B, M, T, K, L, stride = shape
    mode, dist = MODES[flag]
    if precision != "fp32":
        assert C.ENGINE[C.lib.ign_shapelet_engine(byref(desc_of(B, M, T, K, L, stride, dist, pool, precision)), 0)] \
            == "tcgen05"
    torch.manual_seed(1300 + T + L + len(flag))
    xn, W = torch.randn(B, M, T), torch.randn(K, M, L)
    gp = torch.randn(B, K, M) if terms != "d" else None
    gd = torch.randn(B, K, M) if terms != "p" else None
    thr = torch.rand(1, K, M) if pool == "lts_min" else None
    opool = O.POOL_LTS_MIN if pool == "lts_min" else O.POOL_RBF_MAX
    what = f"{flag}/{pool}/{precision} {shape} {chunks} chunks, {terms}"
    stored = run_layer(xn, W, stride, dist, pool, thr, gp, gd, precision)
    force_recompute(store_budget, desc_of(B, M, T, K, L, stride, dist, pool, precision), chunks)
    dW, dthr, dx = run_layer(xn, W, stride, dist, pool, thr, gp, gd, precision)
    check_grads(dW, dthr, dx, oracle_grads(xn, W, stride, mode, opool, thr, gp, gd), what)
    if precision == "fp32":
        # the same kernels on the same distances, and each dxn row adds the shapelets in the same k order
        assert torch.equal(dx, stored[2]), what + ": recompute dx != stored dx"
    # weights frozen: the pooling backward and dx run, the contraction does not; dx is the same
    dW2, dthr2, dx2 = run_layer(xn, W, stride, dist, pool, thr, gp, gd, precision, train_w=False)
    assert dW2 is None and dthr2 is None
    assert torch.equal(dx2, dx), what + ": frozen-weight dx != trainable-weight dx"


@pytest.mark.parametrize("precision", ["fp32", "3xtf32"])
@pytest.mark.parametrize("shape,chunks", DX_SHAPES[:2])
def test_recompute_input_gradient_of_squared_l2_is_zero(store_budget, precision, shape, chunks):
    """The reference's ShapeletDistanceFunc returns zeros for its input (Shapelet.py:40); dW is still the oracle's."""
    B, M, T, K, L, stride = shape
    torch.manual_seed(1400 + T)
    xn, W, gp = torch.randn(B, M, T), torch.randn(K, M, L), torch.randn(B, K, M)
    force_recompute(store_budget, desc_of(B, M, T, K, L, stride, "sql2", "rbf_max", precision), chunks)
    dW, _, dx = run_layer(xn, W, stride, "sql2", "rbf_max", None, gp, None, precision)
    assert float(dx.abs().max()) == 0.0
    dW_ref, _, _ = oracle_grads(xn, W, stride, O.DIST_SQL2, O.POOL_RBF_MAX, None, gp, None)
    assert_close(dW, dW_ref, 1e-4, 1e-4 * float(dW_ref.abs().max()), f"sql2/{precision} {shape} recompute dW")


def test_recompute_input_gradient_at_k1000_bounded_memory(store_budget):
    """Config-4 corner K = 1000, B = 256, T = 1000, L = 100 on a channel subset: the stored mode would keep 7.4 GB here
    (232 GB at M = 125).  With a 1 GiB budget the memory the backward adds is its workspace, dxn and the gradients."""
    from layers import ign_cabi as C
    from layers.shapelet_ops import SeriesPack, shapelet_transform
    budget = 2 ** 30
    store_budget(budget)
    torch.manual_seed(15)
    B, M, T, K, L = 256, 4, 1000, 1000, 100
    xn = torch.randn(B, M, T, device=DEV)
    W = torch.randn(K, M, L, device=DEV)
    g = torch.zeros(B, K, M, device=DEV)
    bs = [7, 200]
    g[bs] = torch.randn(len(bs), K, M, device=DEV)          # only two samples carry gradient: the oracle can check them
    desc = desc_of(B, M, T, K, L, 1, "l1", "rbf_max", "fp32")
    assert 2 * int(C.lib.ign_shapelet_dstore_bytes(byref(desc))) > 6 * 2 ** 30
    ws = int(C.lib.ign_shapelet_backward_recompute_input_workspace(byref(desc), budget))
    assert 0 < ws <= budget
    xd = xn.clone().requires_grad_(True)
    Wd = W.clone().requires_grad_(True)
    p, _, _ = shapelet_transform(SeriesPack.from_channel_major(xd), Wd, 1, 1.0, "l1")
    loss = (p * g).sum()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    loss.backward()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    dxn_bytes = 4 * B * M * C.padded_len(T)
    grads = 4 * K * M * L + 4 * B * K * M + dxn_bytes      # dW, dLoss/dp and dLoss/dx
    assert peak < ws + dxn_bytes + grads + 8 * 2 ** 20, (peak, ws)
    # fp64 autograd through the oracle for the two samples, on the device: its L1 temporaries are 3 GB per sample
    Wr, _, dxr = O.shapelet_backward_autograd(xn[bs].double(), W.double(), g[bs].double(), 1, 1.0, O.DIST_L1,
                                              need_dx=True)
    assert_close(xd.grad[bs], dxr, 2e-4, 2e-4 * float(dxr.abs().max()), "K=1000 recompute dx")
    assert float(xd.grad[[b for b in range(B) if b not in bs]].abs().max()) == 0.0
    assert_close(Wd.grad, Wr, 1e-4, 1e-4 * float(Wr.abs().max()), "K=1000 recompute dW")


def build_model(name):
    """The golden model `name` (InterpGN) with the weights the reference ran."""
    from models.InterpGN import InterpGN
    g = load_golden(name)
    kw = dict(zip(g["cfg_keys"].tolist(), g["cfg_vals"].tolist()))
    cfg = SimpleNamespace(epsilon=1., distance_func=kw.get("distance_func", "euclidean"), memory_efficient=False,
                          sbm_cls=kw.get("sbm_cls", "linear"), dropout=0., lambda_reg=0.1, lambda_div=0.1,
                          dnn_type=kw.get("dnn_type", "FCN"), enc_in=int(kw["enc_in"]), num_class=int(kw["num_class"]),
                          seq_len=int(kw["seq_len"]))
    model = InterpGN(cfg)
    model.load_state_dict({k[4:]: torch.as_tensor(v) for k, v in g.items() if k.startswith("sd::")})
    return model.to(DEV).train(), g, kw


@pytest.mark.parametrize("name", ["model_jv_interpgn", "model_jv_interpgn_cos"])
def test_saliency_through_the_whole_model_in_recompute_mode(store_budget, name):
    """dLoss/dx of the raw batch through instance norm, every length group (each recomputing in minimum chunks) and the
    shapelet expert's head, against autograd through the oracle restatement in fp64."""
    store_budget(1)
    model, g, kw = build_model(name)
    model.overlap_experts = False
    x = t(g["x"], DEV).requires_grad_(True)
    y = torch.as_tensor(g["y"]).to(DEV)
    _, info = model(x, torch.ones(x.shape[0], x.shape[1], device=DEV), None, None)
    torch.nn.functional.cross_entropy(info.shapelet_preds, y).backward()
    torch.cuda.synchronize()
    xr = t(g["x"]).double().requires_grad_(True)
    Ws = [s.weights.detach().cpu().double() for s in model.sbm.shapelets]
    Wc = model.sbm.output_layer.weight.detach().cpu().double()
    mode = MODES[kw.get("distance_func", "euclidean")][0]
    ref_logits, _, _ = O.sbm_forward(xr, Ws, [s.stride for s in model.sbm.shapelets], Wc, 1.0, mode)
    torch.nn.functional.cross_entropy(ref_logits, torch.as_tensor(g["y"])).backward()
    assert_close(x.grad, xr.grad, 1e-3, 2e-4 * float(xr.grad.abs().max()), name + " dLoss/dx (recompute)")


# ---------------------------------------------------------------------------------------------------------------------
# The C ABI directly: writes stay inside dxn, dW and the workspace; invalid arguments return IGN_ERR_INVALID
# ---------------------------------------------------------------------------------------------------------------------
GUARD = 4096
FILL = 0xA5


def guarded(nbytes, zero=False):
    """(raw, body): `body` is nbytes inside a buffer with GUARD sentinel bytes on either side (128-byte aligned)."""
    raw = torch.full((GUARD + nbytes + GUARD,), FILL, dtype=torch.uint8, device=DEV)
    body = raw[GUARD:GUARD + nbytes]
    if zero:
        body.zero_()
    return raw, body


def assert_guards(raw, nbytes, what):
    assert bool((raw[:GUARD] == FILL).all()), what + ": write BEFORE the buffer"
    assert bool((raw[GUARD + nbytes:] == FILL).all()), what + ": write PAST the buffer"


def c_setup(shape, dist, pool, precision):
    from layers.shapelet_ops import SeriesPack
    B, M, T, K, L, stride = shape
    torch.manual_seed(1500 + T + L)
    pack = SeriesPack.from_channel_major(torch.randn(B, M, T, device=DEV))
    st0, st1 = pack.window_stats(dist, L, stride)
    W = torch.randn(K, M, L, device=DEV)
    thr = torch.rand(K, M, device=DEV) if pool == "lts_min" else None
    g, gd = torch.randn(B, K, M, device=DEV), torch.randn(B, K, M, device=DEV)
    return desc_of(B, M, T, K, L, stride, dist, pool, precision), pack, st0, st1, W, thr, g, gd


def ptr(x):
    return None if x is None else x.data_ptr()


@pytest.mark.parametrize("shape,dist,pool,precision", [
    ((2, 3, 600, 21, 120, 7), "l1", "rbf_max", "fp32"),          # strided, ragged last chunk
    ((3, 5, 250, 20, 25, 1), "cosine", "rbf_max", "3xtf32"),    # tcgen05 forward, ragged tile
    ((2, 2, 1031, 11, 5, 1), "pearson", "rbf_max", "fp32"),      # generic pooling backward (more than 1024 windows)
    ((2, 5, 333, 17, 37, 1), "l1", "lts_min", "fp32")])
@pytest.mark.parametrize("frozen", [False, True])
def test_recompute_input_call_writes_only_inside_its_buffers(shape, dist, pool, precision, frozen):
    from layers import ign_cabi as C
    desc, pack, st0, st1, W, thr, g, gd = c_setup(shape, dist, pool, precision)
    B, M, T, K, L, _ = shape
    nws = int(C.lib.ign_shapelet_backward_recompute_input_workspace(byref(desc), 1))     # minimum chunks
    ws_raw, ws = guarded(nws)
    dx_raw, dxb = guarded(4 * B * M * pack.Tp, zero=True)
    dW_raw, dWb = guarded(4 * K * M * L)
    dxn, dW = dxb.view(torch.float32), None if frozen else dWb.view(torch.float32)
    rc = C.lib.ign_shapelet_backward_recompute_input(byref(desc), ptr(pack.xn), ptr(st0), ptr(st1), ptr(W), ptr(thr),
                                                     ptr(g), ptr(gd), ptr(dW), ptr(dxn), ptr(ws), nws, None)
    assert rc == 0, C.last_error()
    torch.cuda.synchronize()
    what = f"{shape} {dist}/{pool}/{precision} frozen={frozen}"
    for raw, n, name in ((ws_raw, nws, "workspace"), (dx_raw, dxb.numel(), "dxn"), (dW_raw, dWb.numel(), "dW")):
        assert_guards(raw, n, what + " " + name)
    assert bool(torch.isfinite(dxn).all()) and float(dxn.abs().max()) > 0
    if not frozen:
        assert bool(torch.isfinite(dW).all())
    else:
        assert bool((dWb == FILL).all())                # frozen weights: dW is neither read nor written


def test_recompute_input_call_rejects_invalid_arguments():
    from layers import ign_cabi as C
    desc, pack, st0, st1, W, thr, g, _ = c_setup((2, 3, 200, 9, 20, 1), "pearson", "rbf_max", "fp32")
    nws = int(C.lib.ign_shapelet_backward_recompute_input_workspace(byref(desc), 2 ** 30))
    ws = torch.empty((nws + 256,), dtype=torch.uint8, device=DEV)
    dxn = torch.zeros_like(pack.xn)
    dW = torch.empty_like(W)

    def call(st1_=st1, dxn_=dxn, ws_ptr=ws.data_ptr(), nbytes=nws, thr_=None, d=desc):
        return C.lib.ign_shapelet_backward_recompute_input(byref(d), ptr(pack.xn), ptr(st0), ptr(st1_), ptr(W),
                                                           ptr(thr_), ptr(g), None, ptr(dW), ptr(dxn_), ws_ptr,
                                                           nbytes, None)
    assert call(dxn_=None) == 1 and "null pointer" in C.last_error()
    assert call(nbytes=1024) == 1 and "workspace" in C.last_error()
    assert call(ws_ptr=ws.data_ptr() + 16) == 1 and "aligned" in C.last_error()
    assert call(st1_=None) == 1 and "st1" in C.last_error()
    lts = desc_of(2, 3, 200, 9, 20, 1, "l1", "lts_min", "fp32")
    assert call(d=lts) == 1 and "threshold" in C.last_error()
    assert call() == 0, C.last_error()
    torch.cuda.synchronize()
    assert bool(torch.isfinite(dxn).all()) and float(dxn.abs().max()) > 0
