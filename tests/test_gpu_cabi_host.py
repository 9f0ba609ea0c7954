"""GPU: the C ABI driven with plain host buffers (numpy + ctypes only — no torch types cross the
boundary), checked against the oracle."""
import ctypes

import numpy as np
import pytest
import torch

import ign_oracle as O

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("flag,dist", [("euclidean", 0), ("cosine", 2), ("pearson", 3)])
def test_sbm_transform_host(flag, dist):
    from layers import ign_cabi as C
    rng = np.random.default_rng(7)
    B, T, M = 5, 120, 7
    Ks, Ls, strides = [5, 5, 3], [12, 24, 60], [1, 1, 1]
    x = rng.standard_normal((B, T, M)).astype(np.float32)
    Ws = [rng.standard_normal((k, M, l)).astype(np.float32) for k, l in zip(Ks, Ls)]
    F = sum(k * M for k in Ks)
    probs = np.zeros((B, F), np.float32)
    dists = np.zeros((B, F), np.float32)
    ptrs = (ctypes.c_void_p * len(Ws))(*[w.ctypes.data for w in Ws])
    i32 = lambda a: (ctypes.c_int32 * len(a))(*a)
    rc = C.lib.ign_sbm_transform_host(x.ctypes.data, B, T, M, len(Ws), ptrs, i32(Ks), i32(Ls), i32(strides),
                                      1.0, dist, 0, probs.ctypes.data, dists.ctypes.data)
    assert rc == 0, C.last_error()
    mode = {"euclidean": O.DIST_L1, "cosine": O.DIST_COS, "pearson": O.DIST_PEARSON}[flag]
    xn = O.instance_norm(torch.from_numpy(x))
    ps, ds = [], []
    for W, s in zip(Ws, strides):
        o = O.shapelet_forward(xn, torch.from_numpy(W), s, 1.0, mode)
        ps.append(o.p); ds.append(o.dmin)
    np.testing.assert_allclose(probs, torch.cat(ps, -1).numpy(), rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(dists, torch.cat(ds, -1).numpy(), rtol=2e-5, atol=2e-6)


def test_instnorm_cluster_kernel_geometries():
    """instnorm_cluster_kernel (channel counts with gcd(M, 32) <= 2, 16-byte aligned sample slabs): cluster sizes 1..8, a last rank with
    fewer rows, ranks with no rows at all, large offsets (one-pass shifted variance) and a constant channel."""
    from layers.shapelet_ops import instance_norm
    torch.manual_seed(11)
    for (B, T, M) in [(1, 8, 3), (3, 20, 7), (2, 996, 125), (2, 1000, 125), (2, 100, 501), (2, 4100, 5), (3, 1651, 61),
                      (2, 100, 6), (2, 1000, 122)]:
        assert (T * M) % 4 == 0 or T == 1651
        x = torch.randn(B, T, M) * 2.5 + 40.0          # mean >> std: the two-pass reference must still be matched
        x[:, :, 0] = 3.25                               # a constant channel: std = 0 -> (x - mean) / 1e-8 = 0
        pack = instance_norm(x.cuda())
        ref = O.instance_norm(x)
        torch.testing.assert_close(pack.xn[:, :, :T].cpu(), ref, rtol=2e-5, atol=2e-5)
        assert float(pack.xn[:, :, T:].abs().sum()) == 0.0
        assert float(pack.xn[:, 0, :].abs().max()) == 0.0


def test_instnorm_and_window_stats_kernels():
    from layers.shapelet_ops import instance_norm
    torch.manual_seed(3)
    for (B, T, M) in [(3, 29, 12), (2, 1000, 125), (4, 130, 33), (2, 4100, 5), (1, 257, 16)]:
        x = torch.randn(B, T, M) * 3 + 1.5
        pack = instance_norm(x.cuda())
        ref = O.instance_norm(x)
        torch.testing.assert_close(pack.xn[:, :, :T].cpu(), ref, rtol=2e-5, atol=2e-6)
        assert float(pack.xn[:, :, T:].abs().sum()) == 0.0
        own = pack.xn[:, :, :T].double().cpu()       # window statistics are defined on the kernel's own xn
        r1 = torch.cumsum(own, -1)
        r2 = torch.cumsum(own ** 2, -1)
        # fused per-group window statistics against fp64 prefix sums
        L, s = max(3, T // 5), 1 if T < 3000 else 7
        Tw = (T - L) // s + 1
        j0 = torch.arange(Tw) * s
        sxx = (torch.cat([torch.zeros(B, M, 1, dtype=torch.double), r2], -1)[:, :, j0 + L] -
               torch.cat([torch.zeros(B, M, 1, dtype=torch.double), r2], -1)[:, :, j0])
        sx = (torch.cat([torch.zeros(B, M, 1, dtype=torch.double), r1], -1)[:, :, j0 + L] -
              torch.cat([torch.zeros(B, M, 1, dtype=torch.double), r1], -1)[:, :, j0])
        a0, _ = pack.window_stats("sql2", L, s)
        torch.testing.assert_close(a0[:, :, :Tw].double().cpu(), sxx, rtol=2e-7, atol=1e-6)
        assert a0.shape[-1] % 16 == 0
        if a0.shape[-1] > Tw:     # pad slots hold the ignore marker: +inf (sql2), NaN (cosine / pearson)
            assert bool(torch.isinf(a0[:, :, Tw:]).all())
        c0, _ = pack.window_stats("cosine", L, s)
        torch.testing.assert_close(c0[:, :, :Tw].double().cpu(), 1.0 / sxx.sqrt().clamp_min(1e-8), rtol=1e-6, atol=1e-7)
        if c0.shape[-1] > Tw:
            assert bool(torch.isnan(c0[:, :, Tw:]).all())
        q0, q1 = pack.window_stats("pearson", L, s)
        torch.testing.assert_close(q1[:, :, :Tw].double().cpu(), sx / L, rtol=1e-6, atol=1e-6)
        torch.testing.assert_close(q0[:, :, :Tw].double().cpu(), (sxx - sx * sx / L).clamp_min(0).sqrt(), rtol=1e-5, atol=1e-4)


def test_bad_arguments_return_status_not_crash():
    from ctypes import byref
    from layers import ign_cabi as C
    d = C.ShapeletDesc(2, 3, 10, 12, 4, 11, 1, 1.0, 0, 0, 0)
    rc = C.lib.ign_shapelet_forward(byref(d), *([None] * 9), 0, None)
    assert rc == 1 and "T < L" in C.last_error()
    d = C.ShapeletDesc(2, 3, 16, 16, 4, 5, 1, 1.0, 2, 0, 0)
    x = torch.zeros(2, 3, 16, device="cuda")
    rc = C.lib.ign_shapelet_forward(byref(d), x.data_ptr(), None, x.data_ptr(), None, x.data_ptr(),
                                    x.data_ptr(), None, None, None, 0, None)
    assert rc == 1 and "window statistics" in C.last_error()
