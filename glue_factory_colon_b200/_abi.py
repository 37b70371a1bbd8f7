"""ctypes binding of include/lightglue_b200.h.

There is no fallback: if the shared library is missing or the device is not a
B200-class GPU the import of the product path raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

LIB_PATH = Path(__file__).resolve().parent / "lib" / "liblightglue_b200.so"

F32, BF16, F32X3 = 0, 1, 2
EPI_ROWMAJOR, EPI_HEADS, EPI_LN_GELU = 0, 1, 2
ABI_VERSION = 8

_p, _i, _f = C.c_void_p, C.c_int, C.c_float


class MatchConfig(C.Structure):
    """lgb200_match_config (the whole-matcher entry points)."""
    _fields_ = [("precision", C.c_int), ("n_layers", C.c_int), ("input_dim", C.c_int), ("kdim", C.c_int),
                ("filter_threshold", C.c_float)]


class AdaptiveConfig(C.Structure):
    """lgb200_adaptive_config (lgb200_match_adaptive): a confidence <= 0 turns its mode off."""
    _fields_ = [("depth_confidence", C.c_float), ("width_confidence", C.c_float)]


_cfg = C.POINTER(MatchConfig)
_acfg = C.POINTER(AdaptiveConfig)

# name -> argtypes, exactly as declared in include/lightglue_b200.h
SIGNATURES = {
    "lgb200_abi_version": [],
    "lgb200_device_ok": [],
    "lgb200_pack_rows": [_p, _i, _i, _i, _i, _i, _p, _p, _p],
    "lgb200_posenc": [_p, _i, _i, _i, _p, _p, _p, _i, _i, _p, _p, _p],
    "lgb200_linear": [_i, _i, _p, _p, _i, _p, _p, _i, _i, _i, _p, _i, _f, _f, _f, _p, _p, _p, _p, _p, _p, _i,
                      _p, _p, _p, _p, _p, _p],
    "lgb200_attention": [_i, _p, _p, _p, _i, _i, _p, _i, _p, _p],
    "lgb200_attention_ordered": [_i, _p, _p, _p, _i, _i, _p, _p, _i, _p, _p],
    "lgb200_rowdot": [_i, _p, _p, _p, _i, _i, _p, _i, _p, _p],
    "lgb200_assign_lse": [_i, _p, _i, _i, _p, _p, _p],
    "lgb200_assign_scores": [_i, _p, _p, _p, _i, _i, _p, _i, _i, _p, _p, _p],
    "lgb200_filter_matches": [_p, _i, _i, _i, _p, _f, _p, _p, _i, _i, _i, _p, _p, _p, _p, _p, _i, _p],
    "lgb200_nn_scores": [_p, _p, _i, _i, _p, _i, _i, _p, _p, _p],
    "lgb200_nn_match": [_p, _i, _i, _i, _p, _f, _f, _i, _p, _p, _p, _p, _p, _p],
    "lgb200_npair_loss": [_p, _p, _i, _i, _i, _f, _p, _p, _p, _p],
    "lgb200_npair_loss_bwd": [_p, _p, _i, _i, _i, _f, _p, _p, _p, _p, _p, _p, _p],
    "lgb200_loss_reduce": [_p, _i, _i, _i, _p, _p, _p, _p, _p, _p, _p],
    "lgb200_loss_reduce_ragged": [_p, _i, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p],
    "lgb200_assign_loss": [_i, _p, _p, _p, _i, _i, _p, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p],
    "lgb200_exit_check": [_p, _i, _i, _p, _p, _f, _f, _i, _p, _p, _p],
    "lgb200_split_rows": [_p, C.c_longlong, _p, _p],
    "lgb200_split_dynamic": [_p, C.c_longlong, _p, _p, _i, _p, _i, _p],
    "lgb200_merge_rows": [_p, C.c_longlong, _f, _p, _p],
    "lgb200_x3_similarity": [_p, _i, _i, _p, _p, _p],
    "lgb200_x3_assign_lse": [_p, _i, _i, _p, _i, _i, _p, _p],
    "lgb200_x3_assign_scores": [_p, _p, _p, _i, _i, _p, _i, _i, _p, _p],
    "lgb200_attention_bwd": [_p, _p, _p, _p, _p, _i, _i, _p, _i, _p, _p, _p, _p, _p],
    "lgb200_attention_bwd_workspace": [_i, _i, _p],
    "lgb200_attention_bwd_bf16": [_p, _p, _p, _p, _p, _i, _i, _p, _i, _p, _p, _p, _p, _p],
    "lgb200_attention_bwd_bf16_workspace": [_i, _i, _p],
    "lgb200_heads_bwd": [_p, _p, _p, _p, _p, _p, _i, _i, _p, _i, _f, _f, _f, _p, _p, _p],
    "lgb200_ln_gelu_bwd": [_p, _p, _p, _p, _i, _i, _p, _p, _p, _p, _i, _p],
    "lgb200_assign_dsim": [_p, _i, _i, _i, _p, _i, _p, _p, _p, _p, _p],
    "lgb200_assign_dsim_ragged": [_p, _i, _i, _i, _p, _i, _p, _p, _p, _p, _p, _p],
    "lgb200_assign_bwd": [_p, _p, _i, _i, _i, _p, _i, _p, _p, _p, _p, _p, _p],
    "lgb200_assign_bwd_workspace": [_i, _i, _i, _p],
    "lgb200_posenc_bwd": [_p, _i, _i, _i, _p, _p, _p, _i, _i, _p, _p, _p],
    "lgb200_weight_table_size": [_cfg, _p, _p],
    "lgb200_pack_weights": [_cfg, _i, _p, _p, _p, C.c_longlong, _p, _p],
    "lgb200_match_workspace": [_cfg, _i, _i, _i, _p],
    "lgb200_match": [_cfg, _p, _i, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p,
                     C.c_longlong, _p],
    "lgb200_adaptive_table_size": [_cfg, _p, _p],
    "lgb200_pack_weights_adaptive": [_cfg, _i, _p, _p, _p, C.c_longlong, _p, _p],
    "lgb200_match_adaptive_workspace": [_cfg, _i, _i, _i, _p],
    "lgb200_match_adaptive": [_cfg, _acfg, _p, _i, _i, _i] + [_p] * 19 + [_p, C.c_longlong, _p],
    "lgb200_prune_compact": [_p, _p, _f, _f, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p],
}


class LightGlueB200Error(RuntimeError):
    pass


_lib = None


def load(path: Path = LIB_PATH):
    """Loads the library once and attaches prototypes.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if path == LIB_PATH and os.environ.get("LGB200_LIB"):  # development switch: A/B a variant build of the library
        path = Path(os.environ["LGB200_LIB"]).resolve()
    if not Path(path).exists():
        raise LightGlueB200Error(
            f"{path} is missing: build it with `python -m glue_factory_colon_b200.build` "
            "(there is no CPU or PyTorch fallback for the LightGlue hot path)"
        )
    lib = C.CDLL(str(path))
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.argtypes = argtypes
        fn.restype = C.c_int
    lib.lgb200_launch_count.argtypes = []
    lib.lgb200_launch_count.restype = C.c_ulonglong
    lib.lgb200_error_string.argtypes = [C.c_int]
    lib.lgb200_error_string.restype = C.c_char_p
    if lib.lgb200_abi_version() != ABI_VERSION:
        raise LightGlueB200Error("liblightglue_b200.so ABI version mismatch; rebuild the library")
    _lib = lib
    return lib


def check(code: int, what: str) -> None:
    if code != 0:
        msg = load().lgb200_error_string(code).decode()
        raise LightGlueB200Error(f"{what} failed with code {code}: {msg}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()
