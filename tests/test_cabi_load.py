"""CPU: the C-ABI library loads without a GPU and exports every symbol include/ign_b200.h declares
(no compute calls here)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "ign_b200.h")
LIB = os.path.join(ROOT, "speech-imagery-eeg_b200", "lib", "libign_b200.so")


def declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ign_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_abi3_surface():
    names = declared_functions()
    for n in ("ign_instnorm_forward", "ign_window_stats", "ign_shapelet_forward", "ign_shapelet_backward",
              "ign_gate_forward", "ign_gate_backward", "ign_sbm_transform_host", "ign_last_error"):
        assert n in names


def test_library_exports_every_declared_symbol():
    if not os.path.isfile(LIB):
        import __graft_entry__
        __graft_entry__.build()
    lib = ctypes.CDLL(LIB)
    for name in declared_functions():
        assert hasattr(lib, name), "libign_b200.so does not export %s" % name


def test_binding_covers_abi3_header_and_fails_loudly_without_gpu():
    import torch
    from layers import ign_cabi as C
    assert C.exported_symbols() == declared_functions()
    assert C.lib.ign_abi_version() == 3 == C.IGN_ABI_VERSION
    assert C.padded_len(1000) == 1000 and C.padded_len(29) == 32
    assert C.num_windows(1000, 100, 1) == 901 and C.num_windows(4000, 400, 8) == 451
    assert C.num_windows(5, 6, 1) == 0
    if not torch.cuda.is_available():
        assert C.lib.ign_device_check(-1) != 0
        assert "cuda" in C.last_error().lower()


def test_descriptor_validation_messages():
    from ctypes import byref
    from layers import ign_cabi as C
    bad = C.ShapeletDesc(2, 3, 10, 12, 4, 11, 1, 1.0, 0, 0, 0)     # T < L: the reference's unfold raises
    assert C.lib.ign_shapelet_backward_workspace(byref(bad)) == 0
    assert "T < L" in C.last_error()
    ok = C.ShapeletDesc(256, 125, 1000, 1000, 5, 100, 1, 1.0, 0, 0, 0)
    assert C.lib.ign_shapelet_backward_workspace(byref(ok)) > 0
    assert C.lib.ign_shapelet_dstore_bytes(byref(ok)) == 4 * 256 * 125 * 5 * 904


def test_engine_query_and_bounded_recompute_workspace():
    """Host-side planning only (no GPU needed): which engine a descriptor gets, and that the recompute backward's
    workspace honours its budget where the stored-distance mode would need hundreds of GB (config 4, K = 1000)."""
    from ctypes import byref
    from layers import ign_cabi as C
    L1, COS = C.DIST["l1"], C.DIST["cosine"]
    F32, X3 = C.PRECISION["fp32"], C.PRECISION["3xtf32"]
    eng = lambda d, bwd: C.ENGINE[C.lib.ign_shapelet_engine(byref(d), bwd)]
    assert eng(C.ShapeletDesc(256, 125, 1000, 1000, 5, 100, 1, 1.0, L1, 0, X3), 0) == "fp32"       # L1 has no cross term
    assert eng(C.ShapeletDesc(256, 125, 1000, 1000, 5, 100, 1, 1.0, COS, 0, F32), 0) == "fp32"
    assert eng(C.ShapeletDesc(256, 125, 1000, 1000, 5, 100, 1, 1.0, COS, 0, X3), 0) == "tcgen05"
    assert eng(C.ShapeletDesc(256, 125, 1000, 1000, 5, 100, 1, 1.0, COS, 0, X3), 1) == "tcgen05"
    assert "bf16" not in C.PRECISION
    big = C.ShapeletDesc(256, 125, 1000, 1000, 1000, 100, 1, 1.0, L1, 0, F32)
    stored = 2 * C.lib.ign_shapelet_dstore_bytes(byref(big))
    assert stored > 200 * 2 ** 30                                   # 116 GB + 116 GB: cannot run
    for budget_gb in (4, 12, 32):
        need = C.lib.ign_shapelet_backward_recompute_workspace(byref(big), budget_gb * 2 ** 30)
        assert 0 < need <= budget_gb * 2 ** 30, (budget_gb, need)
    # config 2 fits its budget in one chunk: the workspace is the stored-mode workspace plus the chunk's outputs
    small = C.ShapeletDesc(256, 125, 1000, 1000, 5, 100, 1, 1.0, L1, 0, F32)
    need = C.lib.ign_shapelet_backward_recompute_workspace(byref(small), 12 * 2 ** 30)
    assert C.lib.ign_shapelet_backward_workspace(byref(small)) <= need < 2 ** 30
