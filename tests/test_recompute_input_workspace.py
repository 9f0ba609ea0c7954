"""CPU: workspace planning of the recompute backward with input gradients (ign_shapelet_backward_recompute_input_workspace).
Host-side only, no GPU needed.  Config-4 corner K = 1000, B = 256, M = 125, T = 1000, L = 100, where the stored mode
would keep 2 x 116 GB."""
from ctypes import byref

import pytest


def desc(dist, K=1000):
    from layers import ign_cabi as C
    return C.ShapeletDesc(256, 125, 1000, 1000, K, 100, 1, 1.0, C.DIST[dist], C.POOL["rbf_max"], C.PRECISION["fp32"])


@pytest.mark.parametrize("dist", ["l1", "sql2", "cosine", "pearson"])
@pytest.mark.parametrize("budget_gb", [4, 12, 32])
def test_input_workspace_honours_the_budget_at_k1000(dist, budget_gb):
    from layers import ign_cabi as C
    d = desc(dist)
    assert 2 * C.lib.ign_shapelet_dstore_bytes(byref(d)) > 200 * 2 ** 30
    need = C.lib.ign_shapelet_backward_recompute_input_workspace(byref(d), budget_gb * 2 ** 30)
    assert 0 < need <= budget_gb * 2 ** 30, (dist, budget_gb, need)
    dw_only = C.lib.ign_shapelet_backward_recompute_workspace(byref(d), budget_gb * 2 ** 30)
    if dist in ("l1", "sql2"):          # in-place conversion, no distance buffer: the dW-only layout
        assert need == dw_only


@pytest.mark.parametrize("dist", ["cosine", "pearson"])
def test_input_workspace_adds_the_chunk_distances_for_cross_term_modes(dist):
    """At a budget that holds every shapelet in one chunk, both queries plan the same chunk; the input-gradient layout
    adds that chunk's window distances [B,M,K,Tw] (128-byte aligned)."""
    from layers import ign_cabi as C
    d = desc(dist, K=5)
    huge = 2 ** 40
    dist_bytes = 4 * 256 * 125 * 5 * C.padded_windows(1000, 100, 1)
    extra = (dist_bytes + 127) // 128 * 128
    assert dist_bytes == C.lib.ign_shapelet_dstore_bytes(byref(d))
    need = C.lib.ign_shapelet_backward_recompute_input_workspace(byref(d), huge)
    assert need == C.lib.ign_shapelet_backward_recompute_workspace(byref(d), huge) + extra


def test_input_workspace_rejects_a_bad_descriptor():
    from layers import ign_cabi as C
    bad = C.ShapeletDesc(2, 3, 10, 12, 4, 11, 1, 1.0, 0, 0, 0)     # T < L
    assert C.lib.ign_shapelet_backward_recompute_input_workspace(byref(bad), 2 ** 30) == 0
    assert "T < L" in C.last_error()
