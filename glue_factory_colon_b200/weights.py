"""Weight wire format of the LightGlue matcher (SURVEY.md 8(f) rank 4).

The state-dict keys of the reference class are the wire format: glue-factory checkpoints store them under
`matcher.<key>` inside a `{"model": ...}` dict (utils/experiments.py:141-148; tools/convert_weights/
convert_pth_to_tar.py:25-42), DDP adds `module.`, and the fork's C++ / LibTorch consumer loads a PLAIN dict of
CPU tensors written with the zipfile serializer (tools/convert_weights/official_save_tar_to_pth.py:17-30).
`glue_factory_colon_b200.LightGlue` has the same 252 keys, so these helpers only move prefixes and containers.
"""
from __future__ import annotations

from pathlib import Path
from typing import Dict, List, Mapping, Tuple, Union

import torch

_PREFIXES = ("module.", "matcher.")


def strip_prefixes(state: Mapping[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """`module.matcher.transformers.0...` / `matcher.transformers.0...` -> `transformers.0...`.
    Keys of other pipeline members (`extractor.*`, `solver.*`, ...) are dropped when a `matcher.` key is present."""
    def strip(k: str) -> str:
        changed = True
        while changed:
            changed = False
            for p in _PREFIXES:
                if k.startswith(p):
                    k, changed = k[len(p):], True
        return k

    keys = list(state.keys())
    has_matcher = any("matcher." in k[: len("module.matcher.")] for k in keys)
    out = {}
    for k, v in state.items():
        base = k[len("module."):] if k.startswith("module.") else k
        if has_matcher and not base.startswith("matcher."):
            continue
        out[strip(k)] = v
    return out


def unwrap_checkpoint(obj) -> Mapping[str, torch.Tensor]:
    """Accepts a raw state dict, a plain dict of tensors, or a glue-factory checkpoint `{"model": state, ...}`."""
    if isinstance(obj, Mapping) and "model" in obj and isinstance(obj["model"], Mapping):
        obj = obj["model"]
    if not isinstance(obj, Mapping) or not all(isinstance(v, torch.Tensor) for v in obj.values()):
        raise ValueError("not a state dict: expected a mapping of tensors (optionally under the key 'model')")
    return obj


def load_matcher_weights(model: torch.nn.Module, src: Union[str, Path, Mapping], strict: bool = True):
    """Loads LightGlue weights from any of the containers above into `model` (this repo's or the reference's)."""
    if isinstance(src, (str, Path)):
        src = torch.load(str(src), map_location="cpu", weights_only=True)
    state = strip_prefixes(unwrap_checkpoint(src))
    return model.load_state_dict(state, strict=strict)


def export_plain_state_dict(model: torch.nn.Module, path: Union[str, Path]) -> Dict[str, torch.Tensor]:
    """Writes the LibTorch-loadable file of official_save_tar_to_pth.py: a plain `dict` (no OrderedDict), every
    tensor on the CPU, zipfile serialization.  Returns the dict that was written."""
    plain = {k: v.detach().cpu().contiguous() for k, v in model.state_dict().items()}
    torch.save(plain, str(path), _use_new_zipfile_serialization=True)
    return plain


def to_pipeline_state_dict(state: Mapping[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """`transformers.0...` -> `matcher.transformers.0...` (what `TwoViewPipeline.load_state_dict` expects)."""
    return {f"matcher.{k}": v for k, v in strip_prefixes(state).items()}


# entry order of the packed-weight table of lgb200_match (include/lightglue_b200.h, "whole matcher")
NATIVE_LAYER_ENTRIES = ("qkv_w", "qkv_b", "sf0_w", "sf0_b", "sln_g", "sln_b", "sf3_w", "sf3_b",
                        "cqv_w", "cqv_b", "cf0_w", "cf0_b", "cln_g", "cln_b", "cf3_w", "cf3_b")


def native_table(model: torch.nn.Module, prec: int, adaptive: bool = False) -> Tuple[object, List[torch.Tensor]]:
    """The packed-weight table of lgb200_match built from `model._pack(prec)` on the model's device (prec = _abi.BF16
    or _abi.F32X3): (ctypes array of device pointers, the tensors they point into).  The tensors must outlive every
    call that uses the table.  adaptive=True: the table of lgb200_match_adaptive, with the MatchAssignment and the
    token-confidence head of every layer but the last appended (fp_w, fp_b, m_w, m_b, tk_w, tk_b per layer)."""
    import ctypes

    packed = model._pack(prec, next(model.parameters()).device)
    tensors = [lyr[k] for lyr in packed["layers"] for k in NATIVE_LAYER_ENTRIES]
    a = packed["assign"][-1]  # only the last layer's MatchAssignment runs in the forward
    tensors += [packed["wr"], a["fp_w"], a["fp_b"], a["m_w"], a["m_b"]]
    if "in_w" in packed:
        tensors += [packed["in_w"], packed["in_b"]]
    if adaptive:
        for a, t in zip(packed["assign"][:-1], packed["token"]):
            tensors += [a["fp_w"], a["fp_b"], a["m_w"], a["m_b"], t["w"], t["b"]]
    return (ctypes.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors]), tensors
