"""GPU parity: the CUDA shapelet layer (through the C ABI) against the CPU oracle and the golden vectors
frozen from the reference.  Tolerances: distances / probabilities within 1e-4 relative (north-star bound;
we assert 2e-5), gradients 1e-4 relative to the largest entry, indices bit-exact barring near-ties."""
import numpy as np
import pytest
import torch

import ign_oracle as O
from helpers import MODES, assert_close, index_parity, load_golden, t

pytestmark = pytest.mark.gpu
DEV = "cuda"

RTOL, ATOL = 2e-5, 2e-6          # forward values (fp32 path)


def run_layer(xn, W, stride, eps, dist, pool="rbf_max", thr=None, g=None, precision="fp32"):
    from layers.shapelet_ops import SeriesPack, shapelet_transform
    Wd = W.detach().clone().to(DEV).requires_grad_(g is not None)      # fresh leaf: .grad never accumulates across calls
    thd = None if thr is None else thr.detach().clone().to(DEV).requires_grad_(g is not None)
    pack = SeriesPack.from_channel_major(xn.to(DEV))
    p, dmin, idx = shapelet_transform(pack, Wd, stride, eps, dist, pool, thd, precision)
    dW = dthr = None
    if g is not None:
        (p * g.to(DEV)).sum().backward()
        dW = Wd.grad
        dthr = None if thd is None else thd.grad
    torch.cuda.synchronize()
    return p, dmin, idx, dW, dthr


LAYER_CASES = ["layer_l1", "layer_l1_stride", "layer_cosine", "layer_pearson", "layer_cosine_stride",
               "layer_l1_struct", "layer_lts", "layer_l1_min", "layer_pearson_k12", "layer_sql2"]


@pytest.mark.parametrize("name", LAYER_CASES)
def test_layer_matches_reference_golden(name):
    g = load_golden(name)
    dist = MODES[str(g["dfunc"])][1]
    thr = t(g["threshold"]) if "threshold" in g else None
    p, dmin, idx, dW, dthr = run_layer(t(g["xn"]), t(g["W"]), int(g["stride"]), float(g["eps"]), dist,
                                       str(g["pool"]), thr, t(g["g"]))
    B = g["xn"].shape[0]
    assert_close(p.reshape(B, -1), t(g["p"]).reshape(B, -1), RTOL, ATOL, name + " p")
    assert_close(dmin.reshape(B, -1), t(g["dmin"]).reshape(B, -1), RTOL, ATOL, name + " dmin")
    scale = float(np.abs(g["dW"]).max())
    assert_close(dW, t(g["dW"]), 1e-4, 1e-4 * scale, name + " dW")
    if dthr is not None:
        assert_close(dthr, t(g["dthreshold"]), 1e-4, 1e-5, name + " dthreshold")


def test_known_answer_vectors():
    g = load_golden("kat")
    x = torch.tensor([[[0., 1., 2., 3., 4.]]])
    for flag in ("euclidean", "cosine", "pearson"):
        W = t(g[flag + "_W"]).reshape(1, 1, 3)
        p, dmin, idx, dW, _ = run_layer(x, W, 1, 1.0, MODES[flag][1], g=torch.ones(1, 1, 1))
        assert abs(float(p) - float(g[flag + "_p"].ravel()[0])) < 2e-6, flag
        assert abs(float(dmin) - float(g[flag + "_dmin"].ravel()[0])) < 2e-6, flag
        np.testing.assert_allclose(dW.cpu().numpy().ravel(), g[flag + "_dW"].ravel(), atol=3e-6, err_msg=flag)
    # L1 case has exact ties x == w (sign(0) = 0 must hold); argmin of L1 is window 0
    p, dmin, idx, _, _ = run_layer(x, torch.ones(1, 1, 3), 1, 1.0, "l1")
    assert int(idx) == 0
    # cosine: best window is the last one
    p, dmin, idx, _, _ = run_layer(x, torch.ones(1, 1, 3), 1, 1.0, "cosine")
    assert int(idx) == 2


SHAPES = [
    # B, M, T, K, L, stride
    (3, 4, 64, 5, 9, 1),
    (2, 3, 200, 10, 37, 1),       # two k-chunks of 5, TT=8 path
    (2, 5, 130, 7, 16, 1),        # K not a multiple of 4 or 5
    (2, 2, 96, 3, 96, 1),         # T == L: a single window
    (1, 1, 17, 1, 3, 1),          # minimum sizes
    (2, 3, 400, 4, 50, 3),        # strided windows
    (2, 2, 600, 5, 120, 7),       # stride as used for seq_len >= 3000
    (2, 2, 300, 45, 20, 1),       # K > 40: several shapelet blocks per channel
    (5, 3, 120, 5, 30, 1),        # odd batch vs resident rows
]


@pytest.mark.parametrize("flag", ["euclidean", "sql2", "cosine", "pearson"])
@pytest.mark.parametrize("shape", SHAPES)
def test_layer_vs_oracle(flag, shape):
    B, M, T, K, L, stride = shape
    mode, dist = MODES[flag]
    torch.manual_seed(1234 + B + M + T)
    xn = torch.randn(B, M, T)
    W = torch.randn(K, M, L)
    g = torch.randn(B, K, M)
    eps = 0.8
    ref = O.shapelet_forward(xn, W, stride, eps, mode)
    p, dmin, idx, dW, _ = run_layer(xn, W, stride, eps, dist, g=g)
    assert_close(p.reshape(B, -1), ref.p, RTOL, ATOL, f"{flag} p")
    assert_close(dmin.reshape(B, -1), ref.dmin, RTOL, ATOL, f"{flag} dmin")
    index_parity(idx, ref.argmin_d, ref.d, False, L, f"{flag} argmin")
    dW_ref, _ = O.shapelet_backward_formula(xn.double(), W.double(), g.double(), stride, eps, mode)
    assert_close(dW, dW_ref, 1e-4, 1e-4 * float(dW_ref.abs().max()), f"{flag} dW")


@pytest.mark.parametrize("flag", ["euclidean", "sql2"])
@pytest.mark.parametrize("shape", [(3, 4, 64, 5, 9, 1), (2, 3, 300, 6, 40, 2)])
def test_lts_layer_vs_oracle(flag, shape):
    B, M, T, K, L, stride = shape
    mode, dist = MODES[flag]
    torch.manual_seed(99)
    xn, W, g = torch.randn(B, M, T), torch.randn(K, M, L), torch.randn(B, K, M)
    thr = torch.rand(1, K, M)
    ref = O.shapelet_forward(xn, W, stride, 1.0, mode, O.POOL_LTS_MIN, thr)
    p, dmin, idx, dW, dthr = run_layer(xn, W, stride, 1.0, dist, "lts_min", thr, g)
    assert_close(p.reshape(B, -1), ref.p, RTOL, ATOL, "lts p")
    assert_close(dmin.reshape(B, -1), ref.dmin, RTOL, ATOL, "lts dmin")
    dW_ref, dthr_ref = O.shapelet_backward_formula(xn.double(), W.double(), g.double(), stride, 1.0, mode,
                                                   O.POOL_LTS_MIN, thr.double())
    assert_close(dW, dW_ref, 1e-4, 1e-4 * float(dW_ref.abs().max()), "lts dW")
    assert_close(dthr, dthr_ref, 1e-4, 1e-5, "lts dthreshold")


# Pooling backward (pool_bwd_reg_kernel): the row is split into whole 128-window float4 chunks and a scalar tail of
# 32-window sub-chunks, with one instantiation per register budget (NCH = 2, 4, 6, 8) and the generic two-pass kernel
# above 1024 windows — cover every boundary of that split.
# The generic kernel walks float4 chunks with a masked last chunk: 1, 2, 3 valid windows in it (1025, 1026, 1027, 2047).
POOL_TW = [1, 31, 32, 33, 127, 128, 129, 256, 300, 512, 517, 768, 769, 1023, 1024, 1025, 1026, 1027, 1500, 2047, 2050]


@pytest.mark.parametrize("flag", ["euclidean", "sql2", "cosine", "pearson", "lts"])
@pytest.mark.parametrize("Tw", POOL_TW)
def test_pool_backward_row_geometries(flag, Tw):
    B, M, K, L = 2, 2, 3, 5
    T = Tw + L - 1
    torch.manual_seed(4000 + Tw)
    xn, W, g = torch.randn(B, M, T), torch.randn(K, M, L), torch.randn(B, K, M)
    if flag == "lts":
        mode, dist = MODES["euclidean"]
        thr = torch.rand(1, K, M)
        p, dmin, idx, dW, dthr = run_layer(xn, W, 1, 1.0, dist, "lts_min", thr, g)
        dW_ref, dthr_ref = O.shapelet_backward_formula(xn.double(), W.double(), g.double(), 1, 1.0, mode,
                                                       O.POOL_LTS_MIN, thr.double())
        assert_close(dthr, dthr_ref, 1e-4, 1e-5, "lts dthreshold Tw=%d" % Tw)
    else:
        mode, dist = MODES[flag]
        ref = O.shapelet_forward(xn, W, 1, 0.9, mode)
        p, dmin, idx, dW, _ = run_layer(xn, W, 1, 0.9, dist, g=g)
        assert_close(p.reshape(B, -1), ref.p, RTOL, ATOL, f"{flag} p Tw={Tw}")
        dW_ref, _ = O.shapelet_backward_formula(xn.double(), W.double(), g.double(), 1, 0.9, mode)
    assert_close(dW, dW_ref, 1e-4, 1e-4 * float(dW_ref.abs().max()), f"{flag} dW Tw={Tw}")


@pytest.mark.parametrize("flag", ["euclidean", "cosine"])
@pytest.mark.parametrize("K,L", [(5, 10), (5, 50), (5, 95), (5, 100), (5, 101), (5, 250), (8, 100), (10, 30), (3, 64)])
def test_backward_lag_tile_widths(flag, K, L):
    """The FP32 contraction gives each thread 8 or 10 lags, whichever wastes fewer lanes and padded lags for the
    (K, L) at hand (plan_bwd): shapelet lengths on and off both tile widths, block sizes that fill and do not fill."""
    torch.manual_seed(77 + K * 1000 + L)
    B, M, T = 3, 3, 300
    xn, W, g = torch.randn(B, M, T), torch.randn(K, M, L), torch.randn(B, K, M)
    mode, dist = MODES[flag]
    _, _, _, dW, _ = run_layer(xn, W, 1, 0.8, dist, g=g)
    dW_ref, _ = O.shapelet_backward_formula(xn.double(), W.double(), g.double(), 1, 0.8, mode)
    assert_close(dW, dW_ref, 1e-4, 1e-4 * float(dW_ref.abs().max()), f"{flag} dW K={K} L={L}")


def test_long_shapelet_needs_lag_blocks():
    """L = 2100 -> more lag tiles than threads: the backward splits the lag axis over CTAs."""
    torch.manual_seed(5)
    B, M, T, K, L = 2, 2, 2400, 5, 2100
    xn, W, g = torch.randn(B, M, T), torch.randn(K, M, L), torch.randn(B, K, M)
    for flag in ("euclidean", "cosine"):
        mode, dist = MODES[flag]
        ref = O.shapelet_forward(xn, W, 1, 1.0, mode)
        p, dmin, idx, dW, _ = run_layer(xn, W, 1, 1.0, dist, g=g)
        assert_close(p.reshape(B, -1), ref.p, RTOL, ATOL, flag + " p")
        dW_ref, _ = O.shapelet_backward_formula(xn.double(), W.double(), g.double(), 1, 1.0, mode)
        assert_close(dW, dW_ref, 1e-4, 1e-4 * float(dW_ref.abs().max()), flag + " dW")


@pytest.mark.parametrize("flag", ["euclidean", "cosine"])
def test_chisco_shaped_rows_vs_oracle(flag):
    """CHISCO geometry (T=1000, L in {100,200,300,500}, K=5) on a channel subset the oracle can afford."""
    mode, dist = MODES[flag]
    torch.manual_seed(42)
    B, M, T, K = 2, 6, 1000, 5
    xn = torch.randn(B, M, T)
    for L in (100, 200, 300, 500):
        W, g = torch.randn(K, M, L), torch.randn(B, K, M)
        ref = O.shapelet_forward(xn, W, 1, 1.0, mode)
        p, dmin, idx, dW, _ = run_layer(xn, W, 1, 1.0, dist, g=g)
        assert_close(p.reshape(B, -1), ref.p, RTOL, ATOL, f"{flag} L={L} p")
        assert_close(dmin.reshape(B, -1), ref.dmin, RTOL, ATOL, f"{flag} L={L} dmin")
        index_parity(idx, ref.argmin_d, ref.d, False, L, f"{flag} L={L} argmin")
        dW_ref, _ = O.shapelet_backward_formula(xn.double(), W.double(), g.double(), 1, 1.0, mode)
        assert_close(dW, dW_ref, 1e-4, 1e-4 * float(dW_ref.abs().max()), f"{flag} L={L} dW")


@pytest.mark.parametrize("flag", ["euclidean", "pearson"])
def test_full_size_properties(flag):
    """BASELINE config 2 at full size (B=256, M=125, T=1000): size-independent properties, determinism,
    batch-permutation equivariance, and a sampled row check against the oracle."""
    mode, dist = MODES[flag]
    torch.manual_seed(0)
    B, M, T, K, L = 256, 125, 1000, 5, 100
    xn = torch.randn(B, M, T, device=DEV)
    W = torch.randn(K, M, L, device=DEV)
    g = torch.randn(B, K, M, device=DEV)
    p, dmin, idx, dW, _ = run_layer(xn, W, 1, 1.0, dist, g=g)
    assert bool(((p > 0) & (p <= 1)).all())
    Tw = T - L + 1
    assert int(idx.min()) >= 0 and int(idx.max()) < Tw
    # where argmax p == argmin d (no ties), p_max == exp(-(dmin)^2) up to fp32 rounding
    assert_close(p, torch.exp(-dmin ** 2), 1e-6, 1e-7, "p_max == rbf(d_min)")
    # determinism: bit-identical on a second run
    p2, dmin2, idx2, dW2, _ = run_layer(xn, W, 1, 1.0, dist, g=g)
    assert torch.equal(p, p2) and torch.equal(dmin, dmin2) and torch.equal(idx, idx2) and torch.equal(dW, dW2)
    # permuting the batch permutes the outputs (samples are independent) and leaves dW unchanged up to order
    perm = torch.randperm(B, device=DEV)
    p3, dmin3, idx3, dW3, _ = run_layer(xn[perm], W, 1, 1.0, dist, g=g[perm])
    assert torch.equal(p3, p[perm]) and torch.equal(idx3, idx[perm])
    assert_close(dW3, dW, 1e-4, 1e-4 * float(dW.abs().max()), "dW under batch permutation")
    # linearity of the backward in the upstream gradient
    _, _, _, dW4, _ = run_layer(xn, W, 1, 1.0, dist, g=2.0 * g)
    assert_close(dW4, 2.0 * dW, 1e-5, 1e-6 * float(dW.abs().max()), "dW linear in g")
    # sampled (b, m) rows against the oracle
    bs, ms = [3, 200], [0, 77, 124]
    sub = xn[bs][:, ms].cpu()
    ref = O.shapelet_forward(sub, W[:, ms].cpu(), 1, 1.0, mode)
    assert_close(p[bs][:, :, ms].reshape(len(bs), -1), ref.p, RTOL, ATOL, "sampled p")
    assert_close(dmin[bs][:, :, ms].reshape(len(bs), -1), ref.dmin, RTOL, ATOL, "sampled dmin")


def test_error_behaviour_matches_reference():
    from layers.shapelet_ops import SeriesPack, shapelet_transform
    from models.Shapelet import Shapelet
    layer = Shapelet(3, 40, 4).to(DEV)
    with pytest.raises(RuntimeError, match="maximum size for tensor at dimension 2"):
        layer(torch.randn(2, 3, 30, device=DEV))           # T < L: unfold raises in the reference
    with pytest.raises(RuntimeError, match="channels"):
        shapelet_transform(SeriesPack.from_channel_major(torch.randn(2, 5, 64, device=DEV)),
                           torch.randn(4, 3, 8, device=DEV))


def test_gate_kernel_vs_oracle():
    from layers.shapelet_ops import gini_gate
    torch.manual_seed(8)
    for C in (3, 9, 39, 70):
        for gv in (None, 0.0, 0.3, 1.0):
            s = torch.randn(33, C)
            z = torch.randn(33, C)
            go, ge = torch.randn(33, C), torch.randn(33, 1)
            sd, zd = s.to(DEV).requires_grad_(True), z.to(DEV).requires_grad_(True)
            out, eta = gini_gate(sd, zd, gv)
            ((out * go.to(DEV)).sum() + (eta * ge.to(DEV)).sum()).backward()
            ro, re = O.gate_forward(s, z, gv)
            assert_close(out, ro, 1e-5, 1e-6, "gate out")
            assert_close(eta, re, 1e-5, 1e-6, "gate eta")
            gs, gz = O.gate_backward_formula(s.double(), z.double(), go.double(), ge.double(), gv)
            assert_close(sd.grad, gs, 1e-4, 1e-5, "gate d/ds")
            assert_close(zd.grad, gz, 1e-4, 1e-5, "gate d/dz")


# ---------------------------------------------------------------------------------------------------------
# tcgen05 engine (cross-term distances).  3xTF32 is the fp32-equivalent mode and is held to the same bound as
# the CUDA-core engine; single-pass TF32 is a separate mode with its own tolerance (SURVEY.md §7.3-4: 2e-4
# relative on d for unit-variance data, argmin flips ~0.1 %).
# ---------------------------------------------------------------------------------------------------------
TC_SHAPES = [
    (3, 4, 64, 5, 9),          # one k-block of 32, N = 80
    (2, 3, 200, 10, 37),       # K = 10 -> two shapelet blocks
    (2, 5, 130, 7, 16),        # N = 112
    (2, 2, 96, 3, 96),         # T == L: one window
    (1, 1, 17, 1, 3),          # minimum sizes
    (2, 2, 300, 45, 20),       # six shapelet blocks, last one ragged
    (5, 3, 120, 5, 30),        # odd batch vs samples per tile
    (3, 2, 1000, 5, 100),      # CHISCO geometry: 57 window groups, 2 samples per tile
    (5, 2, 1000, 5, 500),      # 32 window groups, 4 samples per tile, 17 k-blocks, ragged last tile
    (2, 1, 2100, 4, 100),      # 126 window groups: one sample per tile
]


@pytest.mark.parametrize("precision,rtol,atol", [("3xtf32", 2e-5, 2e-6), ("tf32", 3e-3, 3e-3)])
@pytest.mark.parametrize("flag", ["sql2", "cosine", "pearson"])
@pytest.mark.parametrize("shape", TC_SHAPES)
def test_tcgen05_forward_vs_oracle(precision, rtol, atol, flag, shape):
    B, M, T, K, L = shape
    mode, dist = MODES[flag]
    torch.manual_seed(4321 + B + M + T + K)
    xn, W = torch.randn(B, M, T), torch.randn(K, M, L)
    ref = O.shapelet_forward(xn, W, 1, 0.8, mode)
    p, dmin, idx, _, _ = run_layer(xn, W, 1, 0.8, dist, precision=precision)
    assert_close(dmin.reshape(B, -1), ref.dmin, rtol, atol, f"{precision} {flag} dmin")
    assert_close(p.reshape(B, -1), ref.p, rtol, atol, f"{precision} {flag} p")
    if precision == "3xtf32":
        index_parity(idx, ref.argmin_d, ref.d, False, L, f"{precision} {flag} argmin")


@pytest.mark.parametrize("flag", ["cosine", "pearson", "sql2"])
def test_tcgen05_training_path(flag):
    """tcgen05 forward feeds the saved distances to the backward kernels: gradients still match the oracle."""
    mode, dist = MODES[flag]
    torch.manual_seed(77)
    B, M, T, K, L = 4, 6, 1000, 5, 200
    xn, W, g = torch.randn(B, M, T), torch.randn(K, M, L), torch.randn(B, K, M)
    p, dmin, idx, dW, _ = run_layer(xn, W, 1, 1.0, dist, g=g, precision="3xtf32")
    ref = O.shapelet_forward(xn, W, 1, 1.0, mode)
    assert_close(p.reshape(B, -1), ref.p, RTOL, ATOL, flag + " p")
    dW_ref, _ = O.shapelet_backward_formula(xn.double(), W.double(), g.double(), 1, 1.0, mode)
    assert_close(dW, dW_ref, 1e-4, 1e-4 * float(dW_ref.abs().max()), flag + " dW")
    # the two engines agree with each other far inside the tolerance
    p32, d32, _, _, _ = run_layer(xn, W, 1, 1.0, dist)
    assert_close(dmin, d32, 2e-6, 2e-6, flag + " 3xtf32 vs fp32 engine")


def test_tcgen05_runs_strided_windows_and_reports_it():
    """stride > 1 (seq_len >= 3000 in the reference, Shapelet.py:162) runs on the tensor-core engine, forward and backward:
    residue r of series and shapelet is its own unit-stride cross term / contraction; `ign_shapelet_engine` says so."""
    from ctypes import byref
    from layers import ign_cabi as C
    torch.manual_seed(3)
    xn, W = torch.randn(2, 2, 400), torch.randn(4, 2, 50)
    a = run_layer(xn, W, 3, 1.0, "cosine", precision="3xtf32")
    b = run_layer(xn, W, 3, 1.0, "cosine")
    assert_close(a[1], b[1], 2e-6, 2e-6, "strided 3xtf32 vs fp32 engine dmin")
    desc = C.ShapeletDesc(2, 2, 400, 400, 4, 50, 3, 1.0, C.DIST["cosine"], 0, C.PRECISION["3xtf32"])
    assert C.ENGINE[C.lib.ign_shapelet_engine(byref(desc), 0)] == "tcgen05"
    assert C.ENGINE[C.lib.ign_shapelet_engine(byref(desc), 1)] == "tcgen05"
    l1 = C.ShapeletDesc(2, 2, 400, 400, 4, 50, 3, 1.0, C.DIST["l1"], 0, C.PRECISION["3xtf32"])
    assert C.ENGINE[C.lib.ign_shapelet_engine(byref(l1), 0)] == "fp32"              # L1 has no cross term


# Strided groups on the tcgen05 engine: residue r of series and shapelet is its own unit-stride cross term (forward: the
# residues' k-blocks concatenate into one tile) / contraction (backward: one item per residue).  Covers strides that do / do not divide L, ragged residues, a residue that ends exactly at a lag-block
# boundary (its second block has no tiles) and several shapelet blocks.
STRIDED_BWD = [
    # B, M, T,    K,  L,    stride
    (3, 2, 400, 4, 50, 3),
    (2, 2, 600, 5, 120, 7),
    (2, 3, 640, 13, 64, 8),
    (1, 1, 3900, 2, 3681, 10),     # L0 = 369 > 368: two lag blocks; residues 1..9 have 368 lags (block 2 empty)
    (2, 2, 4000, 10, 400, 8),
    (37, 5, 4000, 5, 2000, 10),    # 13 window groups per sample: 8 samples per tile, ragged last tile, many tiles per CTA
]


@pytest.mark.parametrize("flag", ["cosine", "pearson", "sql2"])
@pytest.mark.parametrize("shape", STRIDED_BWD)
def test_tcgen05_strided_forward_and_backward_vs_oracle(flag, shape):
    B, M, T, K, L, stride = shape
    mode, dist = MODES[flag]
    torch.manual_seed(5 + T + L)
    xn, W, g = torch.randn(B, M, T), torch.randn(K, M, L), torch.randn(B, K, M)
    p, dmin, idx, dW, _ = run_layer(xn, W, stride, 1.0, dist, g=g, precision="3xtf32")
    ref = O.shapelet_forward(xn, W, stride, 1.0, mode)
    assert_close(p.reshape(B, -1), ref.p, RTOL, ATOL, f"{flag} {shape} strided tcgen05 p")
    assert_close(dmin.reshape(B, -1), ref.dmin, RTOL, ATOL, f"{flag} {shape} strided tcgen05 dmin")
    index_parity(idx, ref.argmin_d, ref.d, False, L, f"{flag} {shape} strided tcgen05 argmin")
    dW_ref, _ = O.shapelet_backward_formula(xn.double(), W.double(), g.double(), stride, 1.0, mode)
    assert_close(dW, dW_ref, 1e-4, 1e-4 * float(dW_ref.abs().max()), f"{flag} {shape} strided tcgen05 dW")
    _, _, _, dW32, _ = run_layer(xn, W, stride, 1.0, dist, g=g)
    assert_close(dW, dW32, 1e-5, 2e-6 * float(dW_ref.abs().max()), f"{flag} {shape} tcgen05 vs fp32 engine dW")


# Multi-tile geometries: every CTA of the persistent tcgen05 kernel walks many tiles here (ring wrap-around, phase
# flips, rotating finaliser, cell-buffer reuse, resident and streaming B rings, runs that change channel inside a
# CTA's range, ragged last tiles), checked against the exact-fp32 engine, itself pinned to the oracle above.
TC_BIG = [
    # B,   M,   T,    K,  L
    (250, 125, 1000, 5, 100),     # resident B ring, 3 accumulators, 2 samples per tile
    (250, 125, 1000, 5, 200),     # resident, 7 k-blocks
    (250, 125, 1000, 5, 300),     # streaming B ring (10 k-blocks do not fit)
    (250, 125, 1000, 5, 500),     # streaming, 4 samples per tile, ragged last tile of every channel
    (301, 40, 200, 13, 50),       # two shapelet blocks (K > 8), 8 samples per tile (cap), ragged
    (517, 64, 64, 3, 8),          # short series: 4 window groups per sample, rows mostly idle
    (96, 125, 1500, 1, 700),      # single shapelet, 23 k-blocks, 51 window groups
]


@pytest.mark.parametrize("shape", TC_BIG)
def test_tcgen05_many_tiles_vs_fp32_engine(shape):
    B, M, T, K, L = shape
    torch.manual_seed(1000 + L + K)
    xn = torch.randn(B, M, T, device=DEV)
    W = torch.randn(K, M, L, device=DEV)
    g = torch.randn(B, K, M, device=DEV)
    for dist in ("cosine", "sql2"):
        p32, d32, i32, dW32, _ = run_layer(xn, W, 1, 0.9, dist, g=g)
        ptc, dtc, itc, dWtc, _ = run_layer(xn, W, 1, 0.9, dist, g=g, precision="3xtf32")
        assert_close(dtc, d32, 2e-5, 2e-6, f"{dist} {shape} dmin")
        assert_close(ptc, p32, 2e-5, 2e-6, f"{dist} {shape} p")
        Tw = T - L + 1
        assert int(itc.min()) >= 0 and int(itc.max()) < Tw
        # indices agree except at near-ties between two windows (the engines round the cross term differently)
        diff = itc != i32
        assert float(diff.float().mean()) < 2e-3, f"{dist} {shape}: {int(diff.sum())} argmin differences"
        # the saved distances drive the backward: same gradient from either engine's forward — except for the
        # shapelet rows of the few (sample, shapelet, channel) triples whose best window is a near-tie and flips
        # between the engines (the hard one-hot then moves to the other window): bound their number, not their size
        scale = float(dW32.abs().max())
        bad = (dWtc - dW32).abs() > 1e-4 * scale + 1e-4 * dW32.abs()
        assert int(bad.sum()) <= L * (int(diff.sum()) + 2), f"{dist} {shape} dW: {int(bad.sum())} elements differ"
        assert float((dWtc - dW32).abs().median()) < 1e-5 * scale
    # bit-determinism of the tensor-core engine
    ptc2, dtc2, itc2, dWtc2, _ = run_layer(xn, W, 1, 0.9, "sql2", g=g, precision="3xtf32")
    assert torch.equal(ptc, ptc2) and torch.equal(dtc, dtc2) and torch.equal(itc, itc2) and torch.equal(dWtc, dWtc2)


def test_tcgen05_lts_pooling_many_tiles():
    """DistThresholdShapelet pooling (sigmoid(threshold - min d)) through the tensor-core engine, squared-L2 arithmetic."""
    torch.manual_seed(5)
    B, M, T, K, L = 200, 30, 400, 6, 60
    xn, W = torch.randn(B, M, T, device=DEV), torch.randn(K, M, L, device=DEV)
    thr = torch.randn(1, K, M, device=DEV)
    a = run_layer(xn, W, 1, 1.0, "sql2", pool="lts_min", thr=thr)
    b = run_layer(xn, W, 1, 1.0, "sql2", pool="lts_min", thr=thr, precision="3xtf32")
    assert_close(b[1], a[1], 2e-5, 2e-6, "lts dmin")
    assert_close(b[0], a[0], 2e-5, 2e-6, "lts p")


@pytest.mark.parametrize("K,M,L", [(5, 12, 3), (5, 125, 100), (1, 3, 9), (37, 4, 50), (10, 7, 301)])
def test_diversity_regulariser_vs_reference_formula(K, M, L):
    """Fused diversity kernels against the reference's broadcast formula (Shapelet.py:223-230) and its autograd."""
    from layers.shapelet_ops import shapelet_diversity
    torch.manual_seed(K + M + L)
    W = torch.randn(K, M, L, dtype=torch.float64)
    Wr = W.clone().requires_grad_(True)
    w = Wr.permute(1, 0, 2)
    dist = (w.unsqueeze(1) - w.unsqueeze(2) + 1e-6).norm(dim=-1)
    ref = (torch.exp(-dist) * (1.0 - torch.eye(K, dtype=torch.float64))).mean()
    (3.0 * ref).backward()
    Wd = W.float().to(DEV).requires_grad_(True)
    out = shapelet_diversity(Wd)
    (3.0 * out).backward()
    torch.cuda.synchronize()
    assert abs(float(out) - float(ref)) <= 1e-5 * abs(float(ref)) + 1e-9
    scale = float(Wr.grad.abs().max())
    assert_close(Wd.grad, Wr.grad.float(), 1e-4, 1e-5 * scale + 1e-12, "diversity dW")
    out2 = shapelet_diversity(Wd.detach())
    assert float(out2) == float(out)          # deterministic


# ---------------------------------------------------------------------------------------------------------------------
# BASELINE config 4 (layer sweep: K = 10..1000 shapelets per length, L in {.1,.2,.3,.5} T, T up to 4000): ORACLE parity at
# the sweep's corner geometries, on a channel / batch subset the CPU oracle can afford.  The reference's stride rule
# (Shapelet.py:162: stride = int(log2 L) once seq_len >= 3000) gives T=4000 the pairs 400/8, 800/9, 1200/10, 2000/10.
# ---------------------------------------------------------------------------------------------------------------------
CONFIG4_POINTS = [
    # B, M, T,    K,    L,   stride
    (2, 3, 1000, 100, 100, 1),
    (2, 2, 1000, 100, 500, 1),
    (1, 2, 1000, 1000, 100, 1),
    (1, 2, 600, 1000, 500, 1),      # K = 1000 with the long shapelets of the sweep (T shortened: 101 windows)
    (2, 2, 2000, 10, 1000, 1),      # T = 2000, L = .5 T
    (1, 2, 2999, 10, 1500, 1),      # the largest unit-stride geometry (seq_len < 3000)
    (2, 2, 4000, 10, 400, 8),
    (2, 2, 4000, 10, 800, 9),
    (1, 2, 4000, 10, 1200, 10),
    (1, 2, 4000, 10, 2000, 10),
    (1, 2, 4000, 100, 400, 8),
]


@pytest.mark.parametrize("flag,precision", [("euclidean", "fp32"), ("cosine", "fp32"), ("cosine", "3xtf32"),
                                            ("sql2", "3xtf32"), ("pearson", "3xtf32")])
@pytest.mark.parametrize("shape", CONFIG4_POINTS)
def test_config4_sweep_points_vs_oracle(flag, precision, shape):
    B, M, T, K, L, stride = shape
    assert stride == O.shapelet_stride(T, L)
    mode, dist = MODES[flag]
    torch.manual_seed(31 + T + K + L)
    xn, W, g = torch.randn(B, M, T), torch.randn(K, M, L), torch.randn(B, K, M)
    ref = O.shapelet_forward(xn, W, stride, 1.0, mode)
    p, dmin, idx, dW, _ = run_layer(xn, W, stride, 1.0, dist, g=g, precision=precision)
    tag = f"{flag}/{precision} {shape}"
    assert_close(p.reshape(B, -1), ref.p, RTOL, ATOL, tag + " p")
    assert_close(dmin.reshape(B, -1), ref.dmin, RTOL, ATOL, tag + " dmin")
    index_parity(idx, ref.argmin_d, ref.d, False, L, tag + " argmin")
    del ref
    dW_ref, _ = O.shapelet_backward_formula(xn.double(), W.double(), g.double(), stride, 1.0, mode)
    assert_close(dW, dW_ref, 1e-4, 1e-4 * float(dW_ref.abs().max()), tag + " dW")


# ---------------------------------------------------------------------------------------------------------------------
# Recompute backward (nothing saved by the forward; the library walks the shapelets in chunks inside a bounded
# workspace) against the stored-distance backward and the oracle.
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def tiny_store_budget(monkeypatch):
    from layers import shapelet_ops
    def set_budget(nbytes):
        monkeypatch.setattr(shapelet_ops, "STORE_BUDGET_BYTES", int(nbytes))
    return set_budget


@pytest.mark.parametrize("flag,precision,pool", [("euclidean", "fp32", "rbf_max"), ("cosine", "fp32", "rbf_max"),
                                                 ("pearson", "3xtf32", "rbf_max"), ("sql2", "3xtf32", "rbf_max"),
                                                 ("euclidean", "fp32", "lts_min"), ("sql2", "fp32", "lts_min")])
@pytest.mark.parametrize("shape,budget", [((3, 4, 200, 45, 20, 1), 600_000),      # several chunks of 8..16 shapelets
                                          ((2, 3, 400, 13, 50, 3), 40_000),       # strided windows, ragged last chunk
                                          ((2, 5, 130, 7, 16, 1), 1)])            # budget too small: minimum chunk
def test_recompute_backward_matches_stored_backward_and_oracle(tiny_store_budget, flag, precision, pool, shape, budget):
    B, M, T, K, L, stride = shape
    mode, dist = MODES[flag]
    torch.manual_seed(900 + K + L)
    xn, W, g = torch.randn(B, M, T), torch.randn(K, M, L), torch.randn(B, K, M)
    thr = torch.rand(1, K, M) if pool == "lts_min" else None
    stored = run_layer(xn, W, stride, 0.9, dist, pool, thr, g, precision)
    tiny_store_budget(budget)
    from ctypes import byref
    from layers import ign_cabi as C
    desc = C.ShapeletDesc(B, M, T, C.padded_len(T), K, L, stride, 0.9, C.DIST[dist], C.POOL[pool], C.PRECISION[precision])
    assert 2 * C.lib.ign_shapelet_dstore_bytes(byref(desc)) > budget            # the layer really takes the recompute path
    rec = run_layer(xn, W, stride, 0.9, dist, pool, thr, g, precision)
    assert torch.equal(stored[0], rec[0]) and torch.equal(stored[1], rec[1]) and torch.equal(stored[2], rec[2])
    opool = O.POOL_LTS_MIN if pool == "lts_min" else O.POOL_RBF_MAX
    dW_ref, dthr_ref = O.shapelet_backward_formula(xn.double(), W.double(), g.double(), stride, 0.9, mode, opool,
                                                   None if thr is None else thr.double())
    scale = float(dW_ref.abs().max())
    assert_close(rec[3], dW_ref, 1e-4, 1e-4 * scale, f"{flag}/{precision}/{pool} recompute dW vs oracle")
    # the same kernels on the same distances, chunked differently: only the order of the per-chunk sums may differ
    assert_close(rec[3], stored[3], 1e-5, 1e-6 * scale, "recompute dW vs stored dW")
    if thr is not None:
        assert_close(rec[4], dthr_ref, 1e-4, 1e-5, "recompute dthreshold")


def test_recompute_backward_at_k1000_bounded_workspace(tiny_store_budget):
    """Config-4 corner K = 1000, B = 256, L = 100 on a channel subset: the stored mode would keep 2 x 4*B*M*K*T' bytes
    (7.4 GB here, 232 GB at M = 125); with a 1 GiB budget the backward recomputes in ~8 chunks.  Checked for linearity,
    determinism and against the oracle on sampled samples."""
    from ctypes import byref
    from layers import ign_cabi as C
    tiny_store_budget(2 ** 30)
    torch.manual_seed(12)
    B, M, T, K, L = 256, 4, 1000, 1000, 100
    xn = torch.randn(B, M, T, device=DEV)
    W = torch.randn(K, M, L, device=DEV)
    g = torch.zeros(B, K, M, device=DEV)
    bs = [5, 131]
    g[bs] = torch.randn(len(bs), K, M, device=DEV)          # only two samples carry gradient: the oracle can check them
    desc = C.ShapeletDesc(B, M, T, T, K, L, 1, 1.0, 0, 0, 0)
    assert 2 * C.lib.ign_shapelet_dstore_bytes(byref(desc)) > 6 * 2 ** 30
    assert C.lib.ign_shapelet_backward_recompute_workspace(byref(desc), 2 ** 30) <= 2 ** 30
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    p, dmin, idx, dW, _ = run_layer(xn, W, 1, 1.0, "l1", g=g)
    assert torch.cuda.max_memory_allocated() - base < 1.5 * 2 ** 30          # outputs + the bounded workspace
    p2, _, _, dW2, _ = run_layer(xn, W, 1, 1.0, "l1", g=g)
    assert torch.equal(dW, dW2) and torch.equal(p, p2)
    dW_ref, _ = O.shapelet_backward_formula(xn[bs].cpu().double(), W.cpu().double(), g[bs].cpu().double(), 1, 1.0, O.DIST_L1)
    assert_close(dW, dW_ref, 1e-4, 1e-4 * float(dW_ref.abs().max()), "K=1000 recompute dW")


@pytest.mark.parametrize("mode", ["stored", "recompute"])
def test_backward_holds_one_group_workspace_at_a_time(tiny_store_budget, mode):
    """Four length groups as one autograd node (sbm_transform, as ShapeBottleneckModel runs them): the backward allocates
    each group's workspace just before that group's call and releases it after, so the memory it adds is one workspace
    plus the gradients, not the sum of the four workspaces."""
    from ctypes import byref
    from layers import ign_cabi as C
    from layers.shapelet_ops import SeriesPack, sbm_transform
    from models.Shapelet import Shapelet
    B, M, T, K, Ls = 64, 16, 1000, 16, (50, 100, 150, 200)
    descs = [C.ShapeletDesc(B, M, T, C.padded_len(T), K, L, 1, 1.0, C.DIST["l1"], C.POOL["rbf_max"], C.PRECISION["fp32"])
             for L in Ls]
    dstore = [int(C.lib.ign_shapelet_dstore_bytes(byref(d))) for d in descs]
    if mode == "stored":
        ws = [int(C.lib.ign_shapelet_backward_workspace(byref(d))) for d in descs]
    else:
        budget = 3 * max(dstore) // 2
        assert all(2 * n > budget for n in dstore)          # every group takes the recompute backward
        tiny_store_budget(budget)
        ws = [int(C.lib.ign_shapelet_backward_recompute_workspace(byref(d), budget)) for d in descs]
    assert max(ws) < 1.5 * min(ws)                          # similar sizes: one workspace is well below their sum
    torch.manual_seed(41)
    layers = [Shapelet(M, L, K).to(DEV) for L in Ls]
    pack = SeriesPack.from_channel_major(torch.randn(B, M, T, device=DEV))
    gs = [torch.randn(B, K, M, device=DEV) for _ in Ls]
    loss = sum((p * g).sum() for (p, _, _), g in zip(sbm_transform(pack, layers), gs))
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    loss.backward()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    grads = sum(4 * K * M * L + 4 * B * K * M for L in Ls)     # dW and the upstream dLoss/dp of every group
    assert peak < max(ws) + grads + 2 * 2 ** 20, (peak, ws)
    assert peak < sum(ws), (peak, ws)
    assert all(float(layer.weights.grad.abs().sum()) > 0 for layer in layers)


def test_engine_report_matches_what_runs():
    """ign_shapelet_engine is what bench.py / tools/sweep.py label their rows with."""
    from layers.shapelet_ops import STATS
    STATS.reset()
    xn, W = torch.randn(2, 2, 400), torch.randn(4, 2, 50)
    run_layer(xn, W, 1, 1.0, "cosine", g=torch.randn(2, 4, 2), precision="3xtf32")
    run_layer(xn, W, 1, 1.0, "l1", g=torch.randn(2, 4, 2), precision="3xtf32")
    run_layer(xn, torch.randn(4, 2, 60), 1, 1.0, "cosine", g=torch.randn(2, 4, 2), precision="fp32")
    e = STATS.engine_summary()
    assert e["shapelet_fwd/cosine/L50"] == "tcgen05" and e["shapelet_bwd/cosine/L50"] == "tcgen05"
    assert e["shapelet_fwd/l1/L50"] == "fp32" and e["shapelet_bwd/l1/L50"] == "fp32"
    assert e["shapelet_fwd/cosine/L60"] == "fp32"


# ---------------------------------------------------------------------------------------------------------------------
# Input gradients (saliency / gradcheck): what autograd gives the reference's user for L1 / cosine / pearson
# (Shapelet.py:64-74); the memory_efficient squared-L2 Function returns zeros for its input (Shapelet.py:40).
# ---------------------------------------------------------------------------------------------------------------------
DX_SHAPES = [(3, 4, 64, 5, 9, 1), (2, 3, 200, 10, 37, 1), (2, 2, 96, 3, 96, 1), (2, 3, 400, 4, 50, 3),
             (2, 2, 1000, 5, 300, 1), (1, 2, 17, 1, 3, 1)]


@pytest.mark.parametrize("flag,pool", [("euclidean", "rbf_max"), ("cosine", "rbf_max"), ("pearson", "rbf_max"),
                                       ("euclidean", "lts_min")])
@pytest.mark.parametrize("shape", DX_SHAPES)
def test_input_gradient_vs_oracle_autograd(flag, pool, shape):
    from layers.shapelet_ops import SeriesPack, shapelet_transform
    B, M, T, K, L, stride = shape
    mode, dist = MODES[flag]
    torch.manual_seed(77 + T + L)
    xn, W, g = torch.randn(B, M, T), torch.randn(K, M, L), torch.randn(B, K, M)
    thr = torch.rand(1, K, M) if pool == "lts_min" else None
    opool = O.POOL_LTS_MIN if pool == "lts_min" else O.POOL_RBF_MAX
    dW_ref, _, dx_ref = O.shapelet_backward_autograd(xn.double(), W.double(), g.double(), stride, 0.9, mode, opool,
                                                     None if thr is None else thr.double(), need_dx=True)
    xd = xn.to(DEV).requires_grad_(True)
    Wd = W.to(DEV).requires_grad_(True)
    thd = None if thr is None else thr.to(DEV).requires_grad_(True)
    p, dmin, idx = shapelet_transform(SeriesPack.from_channel_major(xd), Wd, stride, 0.9, dist, pool, thd)
    (p * g.to(DEV)).sum().backward()
    torch.cuda.synchronize()
    assert_close(xd.grad, dx_ref, 2e-4, 2e-4 * float(dx_ref.abs().max()), f"{flag}/{pool} {shape} dx")
    assert_close(Wd.grad, dW_ref, 1e-4, 1e-4 * float(dW_ref.abs().max()), f"{flag}/{pool} {shape} dW (with dx requested)")
    # the input gradient alone (weights frozen): same values, the contraction is skipped
    xd2 = xn.to(DEV).requires_grad_(True)
    p2, _, _ = shapelet_transform(SeriesPack.from_channel_major(xd2), W.to(DEV), stride, 0.9, dist, pool,
                                  None if thr is None else thr.to(DEV))
    (p2 * g.to(DEV)).sum().backward()
    assert torch.equal(xd2.grad, xd.grad)


def test_input_gradient_of_the_squared_l2_function_is_zero_as_in_the_reference():
    from layers.shapelet_ops import SeriesPack, shapelet_transform
    torch.manual_seed(1)
    xd = torch.randn(2, 3, 80, device=DEV, requires_grad=True)
    Wd = torch.randn(4, 3, 11, device=DEV, requires_grad=True)
    p, _, _ = shapelet_transform(SeriesPack.from_channel_major(xd), Wd, 1, 1.0, "sql2")
    p.sum().backward()
    assert float(xd.grad.abs().sum()) == 0.0 and float(Wd.grad.abs().sum()) > 0.0      # Shapelet.py:40


# Series with more than 2048 windows: a sample spans several 128-row tiles of the tcgen05 forward and its arg-min is
# merged across them (64-bit atomicMin on (ordered distance | window index), then tc_finish_kernel).
LONG_ROWS = [
    # B, M, T,    K, L
    (3, 2, 2999, 5, 300),      # config-4 geometry T = 2999, L = .1 T: 2700 windows, two tiles per sample
    (2, 2, 5000, 3, 100),      # 4901 windows: three tiles, the last one short
    (5, 3, 2200, 10, 120),     # 2081 windows: the second tile holds three window groups; two shapelet blocks
]


@pytest.mark.parametrize("flag", ["cosine", "sql2", "pearson"])
@pytest.mark.parametrize("shape", LONG_ROWS)
def test_tcgen05_more_than_2048_windows_vs_oracle(flag, shape):
    from ctypes import byref
    from layers import ign_cabi as C
    B, M, T, K, L = shape
    mode, dist = MODES[flag]
    torch.manual_seed(9 + T + L)
    xn, W, g = torch.randn(B, M, T), torch.randn(K, M, L), torch.randn(B, K, M)
    desc = C.ShapeletDesc(B, M, T, C.padded_len(T), K, L, 1, 0.8, C.DIST[dist], 0, C.PRECISION["3xtf32"])
    assert C.ENGINE[C.lib.ign_shapelet_engine(byref(desc), 0)] == "tcgen05"
    ref = O.shapelet_forward(xn, W, 1, 0.8, mode)
    p, dmin, idx, dW, _ = run_layer(xn, W, 1, 0.8, dist, g=g, precision="3xtf32")
    assert_close(dmin.reshape(B, -1), ref.dmin, RTOL, ATOL, f"{flag} {shape} dmin")
    assert_close(p.reshape(B, -1), ref.p, RTOL, ATOL, f"{flag} {shape} p")
    index_parity(idx, ref.argmin_d, ref.d, False, L, f"{flag} {shape} argmin")
    dW_ref, _ = O.shapelet_backward_formula(xn.double(), W.double(), g.double(), 1, 0.8, mode)
    assert_close(dW, dW_ref, 1e-4, 1e-4 * float(dW_ref.abs().max()), f"{flag} {shape} dW")
    p2, d2, i2, _, _ = run_layer(xn, W, 1, 0.8, dist, precision="3xtf32")           # inference path, bit-deterministic
    assert torch.equal(p, p2) and torch.equal(dmin, d2) and torch.equal(idx, i2)
