"""ctypes binding of libign_b200.so (include/ign_b200.h) — the only way Python reaches the kernels.

There is deliberately no fallback: if the shared library is missing this module raises at import
time, and every call raises RuntimeError with the library's message on a non-zero status.
"""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int32, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("IGN_B200_LIB", os.path.join(_HERE, "..", "lib", "libign_b200.so"))

IGN_ABI_VERSION = 3
DIST = {"l1": 0, "sql2": 1, "cosine": 2, "pearson": 3}
POOL = {"rbf_max": 0, "lts_min": 1}
PRECISION = {"fp32": 0, "3xtf32": 1, "tf32": 2}
ENGINE = {0: "fp32", 1: "tcgen05"}


class ShapeletDesc(Structure):
    _fields_ = [("B", c_int32), ("M", c_int32), ("T", c_int32), ("Tp", c_int32), ("K", c_int32),
                ("L", c_int32), ("stride", c_int32), ("eps", c_float), ("dist", c_int32),
                ("pool", c_int32), ("precision", c_int32)]


if not os.path.isfile(LIB_PATH):
    raise ImportError(
        "libign_b200.so not found at %s — build it with `python __graft_entry__.py` (or `make -C "
        "speech-imagery-eeg_b200/csrc`). This package has no CPU or PyTorch fallback." % LIB_PATH)

lib = ctypes.CDLL(LIB_PATH)

_P = c_void_p
_SIGNATURES = {
    "ign_abi_version": (c_int32, []),
    "ign_last_error": (c_char_p, []),
    "ign_device_check": (c_int32, [c_int32]),
    "ign_debug_bwd_phase_timing": (c_int32, [c_int32]),
    "ign_debug_bwd_phase_read": (c_int32, [_P, _P]),
    "ign_debug_tc_profile": (c_int32, [_P, c_int32]),
    "ign_debug_tc_trace": (c_int32, [_P, c_int32]),
    "ign_padded_len": (c_int32, [c_int32]),
    "ign_num_windows": (c_int32, [c_int32, c_int32, c_int32]),
    "ign_padded_windows": (c_int32, [c_int32, c_int32, c_int32]),
    "ign_instnorm_forward": (c_int32, [_P, _P, _P, _P, c_int32, c_int32, c_int32, _P]),
    "ign_stats_pitch": (c_int32, [c_int32, c_int32, c_int32]),
    "ign_window_stats": (c_int32, [_P, c_int32, c_int32, c_int32, c_int32, POINTER(c_int32), POINTER(c_int32), c_int32,
                                   POINTER(_P), POINTER(_P), _P]),
    "ign_shapelet_forward_workspace": (c_size_t, [POINTER(ShapeletDesc)]),
    "ign_shapelet_forward": (c_int32, [POINTER(ShapeletDesc)] + [_P] * 9 + [c_size_t, _P]),
    "ign_shapelet_engine": (c_int32, [POINTER(ShapeletDesc), c_int32]),
    "ign_shapelet_backward_workspace": (c_size_t, [POINTER(ShapeletDesc)]),
    "ign_shapelet_dstore_bytes": (c_size_t, [POINTER(ShapeletDesc)]),
    "ign_shapelet_backward_recompute_workspace": (c_size_t, [POINTER(ShapeletDesc), c_size_t]),
    "ign_shapelet_backward": (c_int32, [POINTER(ShapeletDesc)] + [_P] * 11 + [c_size_t, _P]),
    "ign_shapelet_backward_dmin": (c_int32, [POINTER(ShapeletDesc)] + [_P] * 12 + [c_size_t, _P]),
    "ign_shapelet_backward_input": (c_int32, [POINTER(ShapeletDesc)] + [_P] * 7 + [c_size_t, _P]),
    "ign_shapelet_backward_recompute_input_workspace": (c_size_t, [POINTER(ShapeletDesc), c_size_t]),
    "ign_shapelet_backward_recompute_input": (c_int32, [POINTER(ShapeletDesc)] + [_P] * 10 + [c_size_t, _P]),
    "ign_diversity_partials": (c_int32, [c_int32]),
    "ign_diversity_forward": (c_int32, [_P, _P, _P, c_int32, c_int32, c_int32, _P]),
    "ign_diversity_backward": (c_int32, [_P, _P, _P, _P, c_int32, c_int32, c_int32, _P]),
    "ign_gate_forward": (c_int32, [_P, _P, _P, _P, c_int32, c_int32, c_int32, c_float, _P]),
    "ign_gate_backward": (c_int32, [_P, _P, _P, _P, _P, _P, c_int32, c_int32, c_int32, c_float, _P]),
    "ign_sbm_transform_host": (c_int32, [_P, c_int32, c_int32, c_int32, c_int32, POINTER(_P),
                                         POINTER(c_int32), POINTER(c_int32), POINTER(c_int32), c_float,
                                         c_int32, c_int32, _P, _P]),
}
for _name, (_res, _args) in _SIGNATURES.items():
    _fn = getattr(lib, _name)   # AttributeError here = header/library mismatch: fail loudly
    _fn.restype = _res
    _fn.argtypes = _args

if lib.ign_abi_version() != IGN_ABI_VERSION:
    raise ImportError("libign_b200.so ABI %d != binding ABI %d" % (lib.ign_abi_version(), IGN_ABI_VERSION))


def exported_symbols():
    return sorted(_SIGNATURES)


def last_error() -> str:
    msg = lib.ign_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(status: int, what: str):
    if status != 0:
        raise RuntimeError("%s failed (ign status %d): %s" % (what, status, last_error()))


def padded_len(T: int) -> int:
    return lib.ign_padded_len(T)


def num_windows(T: int, L: int, stride: int) -> int:
    return lib.ign_num_windows(T, L, stride)


def padded_windows(T: int, L: int, stride: int) -> int:
    return lib.ign_padded_windows(T, L, stride)
