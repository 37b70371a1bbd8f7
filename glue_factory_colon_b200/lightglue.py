"""B200-native drop-in for `gluefactory.models.matchers.lightglue.LightGlue`.

Host side of the hot path.  Mirrors the reference's plugin contract
(reference: gluefactory/models/matchers/lightglue.py, cited as lightglue.py:LINE):

  * discovery: this module exposes `__main_model__` (reference
    models/__init__.py:20-25), so `model.matcher.name=glue_factory_colon_b200.lightglue`
    selects it through the reference's own `get_model` with no reference edits;
  * construction: `LightGlue(conf)` with the conf keys of lightglue.py:323-343,
    unknown keys accepted (the reference merge is non-struct, lightglue.py:351);
  * parameters: identical names and shapes (252 state-dict entries), so
    `matcher.*` checkpoints load unchanged;
  * call: `forward(data) -> dict` with the keys of lightglue.py:541-553.

All arithmetic runs in the hand-written sm_100a kernels of
`lib/liblightglue_b200.so` (C ABI: include/lightglue_b200.h).  PyTorch is used
for parameter storage, device memory and the stream only.  There is no CPU or
PyTorch fallback: CPU inputs raise.
"""
from __future__ import annotations

import ctypes
import gc
import math
import numbers
import os
from typing import Dict, Optional

import numpy as np
import torch
from torch import nn

from . import _abi
from ._abi import BF16, EPI_HEADS, EPI_LN_GELU, EPI_ROWMAJOR, F32, F32X3, MatchConfig, check, ptr
from .driver import crop_log_assignment
from .weights import native_table

LOG2E = 1.4426950408889634


def weight_planes(t: torch.Tensor) -> torch.Tensor:
    """Split-fp16 planes [2][N][K] of a weight matrix, the W operand of the F32X3 kernels: 256 w = hi + lo (LG_X3_EW in
    csrc/lg_internal.cuh: the power of two keeps the low plane a normal fp16 number; undone in the epilogues)."""
    t = t.detach().to(torch.float32) * 256.0
    hi = t.to(torch.float16)
    return torch.stack([hi, (t - hi.to(torch.float32)).to(torch.float16)]).contiguous()


def _capture(graph: "torch.cuda.CUDAGraph", fn):
    """fn() captured into `graph` -> what fn returns.  The cyclic garbage collector is off during the capture: a
    collection there can destroy another module's graphs (an adaptive entry's tail closure refers back to its module,
    so a dropped module is cyclic garbage, and torch.cuda.graph no longer collects before capturing), and destroying a
    graph during a capture invalidates the capture."""
    enabled = gc.isenabled()
    gc.disable()
    try:
        with torch.cuda.graph(graph):
            return fn()
    finally:
        if enabled:
            gc.enable()


class _Conf(dict):
    """Minimal attribute dict (the reference uses OmegaConf; not a dependency here)."""

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as exc:
            raise AttributeError(k) from exc

    def __setattr__(self, k, v):
        self[k] = v


def _merge_conf(default: dict, conf) -> _Conf:
    out = _Conf()
    for k, v in default.items():
        out[k] = _merge_conf(v, {}) if isinstance(v, dict) else v
    if conf is None:
        return out
    try:  # OmegaConf objects, when the caller has omegaconf
        from omegaconf import OmegaConf  # type: ignore

        if OmegaConf.is_config(conf):
            conf = OmegaConf.to_container(conf, resolve=True)
    except Exception:
        pass
    for k, v in dict(conf).items():
        if isinstance(v, dict) and isinstance(out.get(k), dict):
            out[k] = _merge_conf(out[k], v)
        else:
            out[k] = v
    return out


# ----- parameter holders: same module tree / names as the reference -----------------


def _ffn(d: int) -> nn.Sequential:
    # indices 0,1,3 carry parameters (lightglue.py:144-149); index 2 is the GELU slot
    return nn.Sequential(nn.Linear(2 * d, 2 * d), nn.LayerNorm(2 * d), nn.Identity(), nn.Linear(2 * d, d))


class _SelfBlockParams(nn.Module):  # lightglue.py:132-149
    def __init__(self, d: int):
        super().__init__()
        self.Wqkv = nn.Linear(d, 3 * d)
        self.out_proj = nn.Linear(d, d)
        self.ffn = _ffn(d)


class _CrossBlockParams(nn.Module):  # lightglue.py:167-184
    def __init__(self, d: int):
        super().__init__()
        self.to_qk = nn.Linear(d, d)
        self.to_v = nn.Linear(d, d)
        self.to_out = nn.Linear(d, d)
        self.ffn = _ffn(d)


class _LayerParams(nn.Module):  # lightglue.py:225-229
    def __init__(self, d: int):
        super().__init__()
        self.self_attn = _SelfBlockParams(d)
        self.cross_attn = _CrossBlockParams(d)


class _AssignParams(nn.Module):  # lightglue.py:272-277
    def __init__(self, d: int):
        super().__init__()
        self.matchability = nn.Linear(d, 1)
        self.final_proj = nn.Linear(d, d)


class _TokenParams(nn.Module):  # lightglue.py:69-72
    def __init__(self, d: int):
        super().__init__()
        self.token = nn.Sequential(nn.Linear(d, 1), nn.Identity())


class _PosEncParams(nn.Module):  # lightglue.py:53-59
    def __init__(self, m: int, f_dim: int):
        super().__init__()
        self.Wr = nn.Linear(m, f_dim // 2, bias=False)
        nn.init.normal_(self.Wr.weight.data, mean=0, std=1.0)


class LightGlue(nn.Module):
    default_conf = {
        "name": "lightglue",
        "input_dim": 256,
        "add_scale_ori": False,
        "descriptor_dim": 256,
        "n_layers": 9,
        "num_heads": 4,
        "flash": False,  # accepted for compatibility; attention is always the fused flash kernel
        "mp": False,  # True -> bf16 tcgen05 kernels (see `precision`)
        "depth_confidence": -1,
        "width_confidence": -1,
        "filter_threshold": 0.0,
        "checkpointed": False,
        "weights": None,
        "weights_from_version": "v0.1_arxiv",
        "loss": {"gamma": 1.0, "fn": "nll", "nll_balancing": 0.5},
        # B200 extension: "fp32" = fp32-accurate mode on the tensor cores (split-fp16 operands, three tcgen05 MMAs per
        # product, fp32 softmax / LayerNorm / GELU / residuals: 1e-3 parity on log_assignment), "bf16" = bf16 tcgen05
        # kernels (throughput mode), "fp32_simt" = the CUDA-core fp32 kernels (debug / cross-check),
        # "auto" = bf16 when conf.mp or torch autocast is active, else fp32.
        "precision": "auto",
        # B200 extension: capture the whole forward of a fixed input signature in a CUDA graph and replay it (eval
        # mode, no adaptive depth / width, no per-pair counts).  One pair at 2048 keypoints is ~90 launches of 5-20 us
        # each: issued from Python the forward is host-bound, replayed from a graph it is not.
        "cuda_graph": False,
        # with cuda_graph: return the graph's own output buffers (valid until the next call) instead of copies --
        # saves the 16.8 MB-per-pair copy of log_assignment at 2048 keypoints
        "graph_static_outputs": False,
        # B200 extension: with cuda_graph, an int K captures the forward once at K keypoints per image (lgb200_match at
        # B x K x K) and replays that graph for every input with max(m, n) <= K, zero-padded, with the counts
        # (num_keypoints0/1 or m / n) on the device: one capture serves a stream of varying keypoint counts.  bf16 / fp32
        # without adaptive depth / width; anything else takes the path it takes without this key.  A replay at K costs
        # a little more than one at the exact size, so streams of one fixed size are better served without it
        "graph_capacity": None,
        # B200 extension: arithmetic of a training step (module in training mode, autograd on; the no-grad forward
        # follows `precision`).  "fp32" = the fp32-accurate tensor-core mode; "bf16" = mixed precision: the bf16
        # inference kernels forward (outputs bit-equal to the no-grad forward with precision="bf16"), bf16 tensor-core
        # products with fp32 accumulation backward (train.py)
        "train_precision": "fp32",
    }

    required_data_keys = ["keypoints0", "keypoints1", "descriptors0", "descriptors1"]

    def __init__(self, conf=None) -> None:
        super().__init__()
        self.conf = conf = _merge_conf(self.default_conf, conf)
        self._train_bf16()  # (validates conf.train_precision)
        cap = conf.graph_capacity
        if cap is not None and (isinstance(cap, bool) or not isinstance(cap, numbers.Integral) or cap <= 0):
            raise ValueError(f"graph_capacity must be None or a positive int, got {cap!r}")
        d = conf.descriptor_dim
        if d != 256 or conf.num_heads != 4:
            raise NotImplementedError("the B200 kernels are specialised for descriptor_dim=256, num_heads=4")
        if conf.input_dim != d:
            self.input_proj = nn.Linear(conf.input_dim, d, bias=True)
        else:
            self.input_proj = nn.Identity()
        self.posenc = _PosEncParams(2 + 2 * bool(conf.add_scale_ori), d // conf.num_heads)
        n = conf.n_layers
        self.transformers = nn.ModuleList([_LayerParams(d) for _ in range(n)])
        self.log_assignment = nn.ModuleList([_AssignParams(d) for _ in range(n)])
        self.token_confidence = nn.ModuleList([_TokenParams(d) for _ in range(n - 1)])
        if conf.weights is not None:
            self._load_weights(conf.weights)
        self.register_buffer(
            "confidence_thresholds",
            torch.Tensor([self.confidence_threshold(i) for i in range(n)]),
        )
        self._packed: Dict = {}
        self._packs: Dict = {}
        self._pack_key = None
        self._graphs: Dict = {}
        # measurement hook (bench.py): a list to which the forward appends (start, end) CUDA events around every
        # self-attention launch, i.e. the dominant kernel timed inside the running step
        self._attn_events = None

    # ---- reference-compatible helpers ------------------------------------------------

    def confidence_threshold(self, layer_index: int) -> float:  # lightglue.py:555-558
        t = 0.8 + 0.1 * np.exp(-4.0 * layer_index / self.conf.n_layers)
        return float(np.clip(t, 0, 1))

    def _load_weights(self, weights) -> None:
        """lightglue.py:375-401: a path, or a file under DATA_PATH (gluefactory.settings.DATA_PATH when the reference
        is importable, else $GLUEFACTORY_DATA_PATH / $DATA_PATH); the release-URL branch needs a network and raises."""
        from pathlib import Path

        cands = [Path(weights)]
        try:
            from gluefactory.settings import DATA_PATH  # type: ignore

            cands.append(Path(DATA_PATH) / str(weights))
        except Exception:
            pass
        for var in ("GLUEFACTORY_DATA_PATH", "DATA_PATH"):
            if os.environ.get(var):
                cands.append(Path(os.environ[var]) / str(weights))
        path = next((c for c in cands if c.exists()), None)
        if path is None:
            raise FileNotFoundError(
                f"weights '{weights}' not found (tried {', '.join(map(str, cands))}); this build has no download path "
                f"for the official release files (lightglue.py:386-392)")
        from .weights import strip_prefixes, unwrap_checkpoint

        sd = dict(strip_prefixes(unwrap_checkpoint(torch.load(str(path), map_location="cpu", weights_only=True))))
        for i in range(self.conf.n_layers):  # rename old state dict entries (lightglue.py:395-400)
            sd = {k.replace(f"self_attn.{i}", f"transformers.{i}.self_attn"): v for k, v in sd.items()}
            sd = {k.replace(f"cross_attn.{i}", f"transformers.{i}.cross_attn"): v for k, v in sd.items()}
        self.load_state_dict(sd, strict=False)

    def compile(self, mode="reduce-overhead"):  # lightglue.py:410-420: nothing to compile
        return self

    # ---- loss (forward values; SURVEY.md 8(f) rank 2) ------------------------------------------

    def _log_assignment_of(self, lib, prec, d0, d1, layer: int, gt, token_layer: Optional[int] = None,
                           keep: Optional[dict] = None, counts: Optional[torch.Tensor] = None):
        """MatchAssignment `layer` applied to descriptors d0 [B,m,256] / d1 [B,n,256] (lightglue.py:279-288 as called
        from loss_params, :589-595) and the loss reductions on its output.  fp32 (CUDA cores) / fp32-accurate tensor-core
        mode (F32X3: split-fp16 final_proj and similarity GEMM): the forward's assignment kernels write scores
        [B,m+1,n+1], lgb200_loss_reduce reads them.  bf16: lgb200_assign_loss, the tcgen05 pass 2 with the
        reductions in its epilogue -- the matrix is never written.  Returns (pos_sum, pos_cnt, row_exp, row_arg,
        col_arg, dustbin column la[:, :m, n], dustbin row la[:, m, :n], token logits of `token_layer` or None).
        counts (device int32 [2B] or None): per-pair valid counts of a padded batch; the staged rows past them are
        zeroed, log_assignment takes the inference layout of such a batch and every reduction covers each pair's valid
        block only (lgb200_loss_reduce_ragged)."""
        bf = prec == BF16
        x3 = prec == F32X3  # fp32-accurate tensor-core mode: split-fp16 final_proj + similarity GEMM, fp32 normalisers
        hprec = F32 if x3 else prec  # the per-token heads read the fp32 rows in x3 mode
        dev = d0.device
        B, m, _ = d0.shape
        n = d1.shape[1]
        W = self._pack(prec, dev)
        st = torch.cuda.current_stream(dev).cuda_stream
        S = 2 * B
        pad = 256 if x3 else 128  # (the x3 similarity GEMM works on 256-column blocks)
        Lp = max(pad, ((max(m, n) + pad - 1) // pad) * pad)
        T = S * Lp
        f32 = dict(device=dev, dtype=torch.float32)
        adt = dict(device=dev, dtype=torch.bfloat16 if bf else torch.float32)
        lens = counts
        if counts is None and (m != Lp or n != Lp):
            lens = torch.tensor([m, n] * B, device=dev, dtype=torch.int32)
        x = torch.zeros(T, 256, **adt)
        for img, dsc, cnt in ((0, d0, m), (1, d1, n)):
            dsc = dsc.to(torch.float32).contiguous()
            x32_, x16_ = (None, x) if bf else (x, None)
            check(lib.lgb200_pack_rows(ptr(dsc), B, cnt, 256, img, Lp, ptr(x32_), ptr(x16_), st), "pack_rows")
        if counts is not None:
            x.masked_fill_((torch.arange(Lp, device=dev)[None] >= counts[:, None]).reshape(-1, 1), 0)
        a = W["assign"][layer]
        if x3:
            xs = torch.empty(2, T, 256, device=dev, dtype=torch.float16)
            check(lib.lgb200_split_rows(ptr(x), x.numel(), ptr(xs), st), "split_rows")
            md = torch.zeros(2, T, 256, device=dev, dtype=torch.float16)
            a_in, o32, o16 = xs, None, md
        else:
            md = torch.zeros(T, 256, **adt)
            a_in = x
            o32, o16 = (None, md) if bf else (md, None)
        check(
            lib.lgb200_linear(
                prec, EPI_ROWMAJOR, ptr(a_in), None, 256, ptr(a["fp_w"]), ptr(a["fp_b"]), T, 256, 256, ptr(lens), Lp,
                0.25, 1.0, 1.0, None, None, ptr(o32), ptr(o16), None, None, 0, None, None, None, None, None, st,
            ),
            "lgb200_linear",
        )
        z = torch.zeros(T, **f32)
        lse = torch.zeros(T, **f32)
        check(lib.lgb200_rowdot(hprec, ptr(x), ptr(a["m_w"]), ptr(a["m_b"]), S, Lp, ptr(lens), 0, ptr(z), st), "rowdot")
        sim = None
        if x3:
            sim = torch.empty(B, Lp, Lp, **f32)
            check(lib.lgb200_x3_similarity(ptr(md), B, Lp, ptr(lens), ptr(sim), st), "x3_similarity")
            check(lib.lgb200_x3_assign_lse(ptr(sim), B, Lp, ptr(lens), m, n, ptr(lse), st), "x3_assign_lse")
        else:
            check(lib.lgb200_assign_lse(prec, ptr(md), S, Lp, ptr(lens), ptr(lse), st), "assign_lse")
        R, C = m + 1, n + 1
        if keep is not None:  # what the backward pass (train.AssignFn) and the training forward need
            keep.update(z=z, lse=lse, Lp=Lp, lens=lens, md_planes=md if x3 else None, md16=md if bf else None)
        if bf:
            rows = torch.empty(3, B, m, **f32)
            row_arg = torch.empty(B, m, device=dev, dtype=torch.int32)
            col_arg = torch.empty(B, n, device=dev, dtype=torch.int32)
            ws = torch.empty(B * (R + C), device=dev, dtype=torch.int64)
            check(lib.lgb200_assign_loss(prec, ptr(md), ptr(z), ptr(lse), B, Lp, ptr(lens), R, C, ptr(gt), ptr(rows[0]),
                                         ptr(rows[1]), ptr(rows[2]), ptr(row_arg), ptr(col_arg), ptr(ws), st), "assign_loss")
            pos_sum, pos_cnt, row_exp = rows[0].sum(1), rows[1].sum(1), rows[2]
            zv = z.view(B, 2, Lp)
            ls = torch.nn.functional.logsigmoid
            dust0, dust1 = ls(-zv[:, 0, :m]), ls(-zv[:, 1, :n])  # lightglue.py:266-267
        else:
            scores = torch.empty(B, R, C, **f32)
            if x3:
                check(lib.lgb200_x3_assign_scores(ptr(sim), ptr(z), ptr(lse), B, Lp, ptr(lens), R, C, ptr(scores), st),
                      "x3_assign_scores")
            else:
                check(lib.lgb200_assign_scores(prec, ptr(md), ptr(z), ptr(lse), B, Lp, ptr(lens), R, C, ptr(scores), None,
                                               st), "assign_scores")
            pos_sum, pos_cnt, row_exp, row_arg, col_arg = self._reduce(lib, scores, gt, st, counts)
            dust0, dust1 = scores[:, :m, n], scores[:, m, :n]
            if keep is not None:
                keep["scores"] = scores
        logits = None
        if token_layer is not None:
            tk = W["token"][token_layer]
            lg_ = torch.zeros(T, **f32)
            check(lib.lgb200_rowdot(hprec, ptr(x), ptr(tk["w"]), ptr(tk["b"]), S, Lp, ptr(lens), 0, ptr(lg_), st), "rowdot")
            lv = lg_.view(B, 2, Lp)
            logits = (lv[:, 0, :m], lv[:, 1, :n])
        return pos_sum, pos_cnt, row_exp, row_arg, col_arg, dust0, dust1, logits

    def _assign_match_bf16(self, lib, d0, d1, layer: int, counts: Optional[torch.Tensor] = None,
                           keep: Optional[Dict] = None):
        """MatchAssignment `layer` and filter_matches on bf16 descriptors d0 [B,m,256] / d1 [B,n,256], with the kernels
        and arguments of the no-grad bf16 forward's tail (_forward_impl) -> (log_assignment [B,m+1,n+1], m0, m1, ms0,
        ms1).  The bf16 training forward's outputs are therefore the no-grad forward's, bit for bit.  counts: per-pair
        valid counts (device int32 [2B]) or None.  keep (dict): receives what the backward pass (train.LogAssignFn)
        needs, as for _log_assignment_of, plus the filter workspace fm_ws."""
        dev = d0.device
        B, m, _ = d0.shape
        n = d1.shape[1]
        W = self._pack(BF16, dev)
        st = torch.cuda.current_stream(dev).cuda_stream
        S = 2 * B
        Lp = max(128, ((max(m, n) + 127) // 128) * 128)
        T = S * Lp
        f32, b16 = dict(device=dev, dtype=torch.float32), dict(device=dev, dtype=torch.bfloat16)
        lens = counts
        if counts is None and (m != Lp or n != Lp):
            lens = torch.tensor([m, n] * B, device=dev, dtype=torch.int32)
        x = torch.zeros(T, 256, **b16)
        for img, dsc, cnt in ((0, d0, m), (1, d1, n)):
            check(lib.lgb200_pack_rows(ptr(dsc.to(torch.float32).contiguous()), B, cnt, 256, img, Lp, None, ptr(x), st),
                  "pack_rows")
        a = W["assign"][layer]
        md = torch.zeros(T, 256, **b16)
        check(lib.lgb200_linear(BF16, EPI_ROWMAJOR, ptr(x), None, 256, ptr(a["fp_w"]), ptr(a["fp_b"]), T, 256, 256,
                                ptr(lens), Lp, 0.25, 1.0, 1.0, None, None, None, ptr(md), None, None, 0, None, None,
                                None, None, None, st), "lgb200_linear")
        z, lse = torch.zeros(T, **f32), torch.zeros(T, **f32)
        check(lib.lgb200_rowdot(BF16, ptr(x), ptr(a["m_w"]), ptr(a["m_b"]), S, Lp, ptr(lens), 0, ptr(z), st), "rowdot")
        check(lib.lgb200_assign_lse(BF16, ptr(md), S, Lp, ptr(lens), ptr(lse), st), "assign_lse")
        R, C = m + 1, n + 1
        scores = torch.empty(B, R, C, **f32)
        fm_ws = torch.empty(B * (R + C), device=dev, dtype=torch.int64)
        check(lib.lgb200_assign_scores(BF16, ptr(md), ptr(z), ptr(lse), B, Lp, ptr(lens), R, C, ptr(scores), ptr(fm_ws),
                                       st), "assign_scores")
        m0 = torch.empty(B, m, device=dev, dtype=torch.int64)
        m1 = torch.empty(B, n, device=dev, dtype=torch.int64)
        ms0, ms1 = torch.empty(B, m, **f32), torch.empty(B, n, **f32)
        check(lib.lgb200_filter_matches(ptr(scores), B, R, C, ptr(lens), float(self.conf.filter_threshold), None, None,
                                        2 * Lp, m, n, ptr(m0), ptr(m1), ptr(ms0), ptr(ms1), ptr(fm_ws), 1, st),
              "filter_matches")
        if keep is not None:
            keep.update(z=z, lse=lse, Lp=Lp, lens=lens, md_planes=None, md16=md, fm_ws=fm_ws)
        return scores, m0, m1, ms0, ms1

    @staticmethod
    def _reduce(lib, la, gt, st, counts=None):
        """lgb200_loss_reduce on one log-assignment matrix: per-row positive sums / counts / exp sums and the
        row / column arg-maxima including the dustbins.  counts (device int32 [2B]): lgb200_loss_reduce_ragged, each
        pair over its valid block."""
        B, R, C = la.shape
        dev = la.device
        rows = torch.zeros(3, B, R - 1, device=dev, dtype=torch.float32)
        row_arg = torch.zeros(B, R - 1, device=dev, dtype=torch.int32)
        col_arg = torch.zeros(B, C - 1, device=dev, dtype=torch.int32)
        if counts is None:
            check(lib.lgb200_loss_reduce(ptr(la), B, R, C, ptr(gt), ptr(rows[0]), ptr(rows[1]), ptr(rows[2]),
                                         ptr(row_arg), ptr(col_arg), st), "loss_reduce")
        else:
            check(lib.lgb200_loss_reduce_ragged(ptr(la), B, R, C, ptr(counts), ptr(gt), ptr(rows[0]), ptr(rows[1]),
                                                ptr(rows[2]), ptr(row_arg), ptr(col_arg), st), "loss_reduce_ragged")
        return rows[0].sum(1), rows[1].sum(1), rows[2], row_arg, col_arg

    @staticmethod
    def _counts_of(data: dict, B: int, m: int, n: int) -> Optional[np.ndarray]:
        """Per-pair valid counts [B, 2] (host int32) from data["num_keypoints0/1"] (the B200 extension for padded
        batches, SURVEY.md 8(c)), or None without them -- and when every count equals the padded size, so that such a
        batch takes exactly the path of a batch without counts."""
        lens_host = np.empty((B, 2), dtype=np.int32)
        lens_host[:, 0], lens_host[:, 1] = m, n
        variable = False
        for idx in (0, 1):
            cnt = data.get(f"num_keypoints{idx}")
            if cnt is not None:
                lens_host[:, idx] = torch.as_tensor(cnt).to("cpu", torch.int32).numpy().reshape(-1)
                variable = True
        assert (lens_host[:, 0] <= m).all() and (lens_host[:, 1] <= n).all() and (lens_host >= 0).all()
        if not variable or ((lens_host[:, 0] == m).all() and (lens_host[:, 1] == n).all()):
            return None
        return lens_host

    def loss(self, pred, data):
        from . import train as _train

        r0 = pred["ref_descriptors0"]
        if torch.is_grad_enabled() and (r0.requires_grad or _train.wants_grad(self)):
            return self._loss_impl(pred, data, True)  # training step: the result carries an autograd graph
        with torch.no_grad():
            return self._loss_impl(pred, data, False)

    def _loss_impl(self, pred, data, with_grad: bool):
        """LightGlue.loss (lightglue.py:588-637) -> (losses, metrics) with the reference's keys.
        The dense [B,M+1,N+1] work -- MatchAssignment of every collected layer, the NLL sums of weight_loss
        (models/utils/losses.py:6-26), row_norm and the arg-maxima of TokenConfidence.loss (:82-95) -- runs in the
        library's kernels; what is left here is arithmetic on [B] and [B,N] vectors.  with_grad: every layer's
        MatchAssignment goes through train.AssignFn (in conf.train_precision; backward = lgb200_assign_dsim + cuBLAS
        GEMMs), the vector arithmetic below is tracked by autograd, and the token-confidence logits are a torch
        matrix-vector product on the detached descriptors (lightglue.py:83-84), so `losses["total"].mean().backward()`
        reaches every parameter the reference's does.
        With data["num_keypoints0/1"] every entry of `losses` and `metrics` is, per pair, that of the pair un-padded:
        ground truth outside the valid block is ignored (padded rows of gt_matches count as -2), means over an empty
        side are 0 (row_norm, the token-confidence BCE)."""
        lib = _abi.load()
        conf = self.conf
        r0, r1 = pred["ref_descriptors0"], pred["ref_descriptors1"]
        if not r0.is_cuda:
            raise _abi.LightGlueB200Error("glue_factory_colon_b200.LightGlue.loss runs on CUDA tensors only")
        dev = r0.device
        B, N, m, _ = r0.shape
        n = r1.shape[2]
        prec = self._precision()
        st = torch.cuda.current_stream(dev).cuda_stream
        L = conf.n_layers
        gt = data["gt_assignment"].to(dev).to(torch.bool).contiguous()
        assert gt.shape == (B, m, n), "gt_assignment must be [B, M, N]"
        gm0, gm1 = data["gt_matches0"].to(dev), data["gt_matches1"].to(dev)
        counts_h = self._counts_of(data, B, m, n)
        counts = valid0 = valid1 = None
        if counts_h is not None:  # padded batch: everything outside a pair's valid block is ignored
            counts = torch.from_numpy(counts_h.reshape(-1)).to(dev)
            valid0 = torch.arange(m, device=dev)[None] < counts[0::2, None]
            valid1 = torch.arange(n, device=dev)[None] < counts[1::2, None]
            gt = (gt & valid0[:, :, None] & valid1[:, None, :]).contiguous()
            gm0, gm1 = torch.where(valid0, gm0, -2), torch.where(valid1, gm1, -2)
        neg0, neg1 = (gm0 == -1).float(), (gm1 == -1).float()
        num_neg0, num_neg1 = neg0.sum(-1).clamp(min=1.0), neg1.sum(-1).clamp(min=1.0)
        bal = float(conf.loss.nll_balancing)

        def nll_of(layer_idx, mod, token_layer=None):  # weight_loss + NLLLoss.forward (losses.py:6-26, :44-60)
            if with_grad:
                from .train import AssignFn

                a = self.log_assignment[mod]
                d0_, d1_ = r0[:, layer_idx], r1[:, layer_idx]
                pos_sum, dust0, dust1, pos_cnt, _, row_arg, col_arg = AssignFn.apply(
                    self, mod, gt, counts, d0_, d1_, a.final_proj.weight, a.final_proj.bias, a.matchability.weight,
                    a.matchability.bias)
                logits = None
                if token_layer is not None:  # TokenConfidence.loss reads detached descriptors (lightglue.py:83-84)
                    tk = self.token_confidence[token_layer].token[0]
                    lin = torch.nn.functional.linear
                    logits = (lin(d0_.detach().float(), tk.weight, tk.bias).squeeze(-1),
                              lin(d1_.detach().float(), tk.weight, tk.bias).squeeze(-1))
            else:
                pos_sum, pos_cnt, _, row_arg, col_arg, dust0, dust1, logits = self._log_assignment_of(
                    lib, prec, r0[:, layer_idx], r1[:, layer_idx], mod, gt, token_layer, counts=counts)
            num_pos = pos_cnt.clamp(min=1.0)
            nll_pos = -pos_sum / num_pos
            nll_neg = (-(dust0 * neg0).sum(-1) - (dust1 * neg1).sum(-1)) / (num_neg0 + num_neg1)
            nll = bal * nll_pos + (1 - bal) * nll_neg
            return nll, nll_pos, nll_neg, num_pos, row_arg, col_arg, logits

        nll, nll_pos, nll_neg, num_pos, _, _, _ = nll_of(-1, L - 1)
        losses = {
            "total": nll, "last": nll.clone().detach(), "assignment_nll": nll, "nll_pos": nll_pos, "nll_neg": nll_neg,
            "num_matchable": num_pos, "num_unmatchable": (num_neg0 + num_neg1) / 2.0,
        }
        if self.training:
            losses["confidence"] = torch.zeros_like(nll)
        la_pred = pred["log_assignment"].detach().to(torch.float32).contiguous()
        _, _, row_exp_f, row_arg_f, col_arg_f = self._reduce(lib, la_pred, None, st, counts)
        if counts is None:
            losses["row_norm"] = row_exp_f.mean(1)  # lightglue.py:606
        else:  # (rows past the count hold 0; the mean over an empty side is 0)
            losses["row_norm"] = row_exp_f.sum(1) / valid0.sum(1).clamp(min=1)
        bce = torch.nn.functional.binary_cross_entropy_with_logits

        def bce_mean(lg, target, valid):
            e = bce(lg, target, reduction="none")
            if valid is None:
                return e.mean(-1)
            return torch.where(valid, e, 0.0).sum(-1) / valid.sum(-1).clamp(min=1)

        sum_w = 1.0
        for i in range(N - 1):
            nll_i, _, _, _, row_arg_i, col_arg_i, (lg0, lg1) = nll_of(i, i, token_layer=i)
            g = float(conf.loss.gamma)
            w = g ** (N - i - 1) if g > 0.0 else i + 1
            sum_w += w
            losses["total"] = losses["total"] + nll_i * w
            c0, c1 = (row_arg_f == row_arg_i).float(), (col_arg_f == col_arg_i).float()
            conf_i = (bce_mean(lg0, c0, valid0) + bce_mean(lg1, c1, valid1)) / 2.0
            losses["confidence"] = losses["confidence"] + conf_i / (N - 1)
        losses["total"] = losses["total"] / sum_w
        if self.training:
            losses["total"] = losses["total"] + losses["confidence"]
        metrics = {} if self.training else self._matcher_metrics(pred, {"gt_matches0": gm0})
        return losses, metrics

    @staticmethod
    def _matcher_metrics(pred, data):
        """Recall / precision / accuracy / ranking AP of matches0 against gt_matches0, same definitions as the
        reference's matcher_metrics (gluefactory/models/utils/metrics.py:5-57); [B,N] vector arithmetic."""
        mt, gt, sc = pred["matches0"], data["gt_matches0"], pred["matching_scores0"]
        same = (mt == gt).float()
        in_recall, in_acc = (gt > -1).float(), (gt >= -1).float()
        in_prec = ((mt > -1) & (gt >= -1)).float()
        eps = 1e-8
        order = torch.argsort(-sc, stable=True)  # ties: lowest index first (deterministic)
        tp, pm, rm = same.gather(-1, order), in_prec.gather(-1, order), in_recall.gather(-1, order)
        prec_curve = torch.cumsum(tp * pm, -1) / (eps + torch.cumsum(pm, -1))
        rec_curve = torch.cumsum(tp * rm, -1) / (eps + rm.sum(-1, keepdim=True))
        ap = ((rec_curve[..., 1:] - rec_curve[..., :-1]) * prec_curve[:, None, -1]).sum(-1)
        return {
            "match_recall": (same * in_recall).sum(1) / (eps + in_recall.sum(1)),
            "match_precision": (same * in_prec).sum(1) / (eps + in_prec.sum(1)),
            "accuracy": (same * in_acc).sum(1) / (eps + in_acc.sum(1)),
            "average_precision": ap,
        }

    # ---- weight packing ------------------------------------------------------------------

    def _precision(self) -> int:
        p = self.conf.precision
        if p == "auto":
            p = "bf16" if (self.conf.mp or torch.is_autocast_enabled()) else "fp32"
        if p not in ("fp32", "bf16", "fp32_simt"):
            raise ValueError(f"precision must be fp32, fp32_simt, bf16 or auto, got {p}")
        return {"bf16": BF16, "fp32": F32X3, "fp32_simt": F32}[p]

    def _train_bf16(self) -> bool:
        p = self.conf.get("train_precision", "fp32")
        if p not in ("fp32", "bf16"):
            raise ValueError(f"train_precision must be fp32 or bf16, got {p}")
        return p == "bf16"

    def _apply(self, fn, *args, **kwargs):  # .to() / .cuda() / .half(): parameters may be replaced
        self._plist = None
        return super()._apply(fn, *args, **kwargs)

    def _pack(self, prec: int, device) -> Dict:
        # identity + version of every parameter; walking the module tree costs 0.3 ms per call (a third of a one-pair
        # forward), the cached flat list 0.03 ms
        plist = getattr(self, "_plist", None)
        if plist is None:
            plist = self._plist = list(self.parameters())
        key = (prec, str(device), tuple((p.data_ptr(), p._version) for p in plist))
        hit = self._packs.get(prec)
        if hit is not None and hit[0] == key:
            self._packed, self._pack_key = hit[1], key
            return hit[1]
        # one pack per precision is kept (forward in the fp32 tensor-core mode, loss in the CUDA-core fp32 kernels);
        # captured CUDA graphs hold their own reference (see forward), so replacing one is safe
        wdt = torch.bfloat16 if prec == BF16 else torch.float32

        def W(t):
            t = t.detach().to(device=device, dtype=torch.float32)
            return weight_planes(t) if prec == F32X3 else t.to(wdt).contiguous()

        def Fp(t):
            return t.detach().to(device=device, dtype=torch.float32).contiguous()

        # Wqkv rows: reference row = head*192 + d*3 + part (lightglue.py:158) -> part*256 + head*64 + d
        perm = torch.arange(768).view(4, 64, 3).permute(2, 0, 1).reshape(-1)
        def fold_out_proj(ffn0, out_proj):
            """bf16 mode: x + ffn(cat[x, out_proj(ctx)]) (lightglue.py:163, :221-222) with the out_proj GEMM folded
            into the first FFN matrix -- W1.cat[x, Wo.ctx + bo] = [W1x | W1m.Wo].cat[x, ctx] + (b1 + W1m.bo) -- so the
            [T,256]x[256,256] launch and the `msg` round trip through HBM disappear (exact in real arithmetic; the
            product is formed in fp32 and rounded to bf16 once, like every other weight)."""
            w1 = ffn0.weight.detach().double()
            wo, bo = out_proj.weight.detach().double(), out_proj.bias.detach().double()
            d = wo.shape[0]
            return (torch.cat([w1[:, :d], w1[:, d:] @ wo], 1).float(),
                    (ffn0.bias.detach().double() + w1[:, d:] @ bo).float())

        fold = prec in (BF16, F32X3)
        layers = []
        for lyr in self.transformers:
            sa, ca = lyr.self_attn, lyr.cross_attn
            sf0 = fold_out_proj(sa.ffn[0], sa.out_proj) if fold else (sa.ffn[0].weight, sa.ffn[0].bias)
            cf0 = fold_out_proj(ca.ffn[0], ca.to_out) if fold else (ca.ffn[0].weight, ca.ffn[0].bias)
            layers.append(
                dict(
                    qkv_w=W(sa.Wqkv.weight[perm]), qkv_b=Fp(sa.Wqkv.bias[perm]),
                    so_w=W(sa.out_proj.weight), so_b=Fp(sa.out_proj.bias),
                    sf0_w=W(sf0[0]), sf0_b=Fp(sf0[1]),
                    sln_g=Fp(sa.ffn[1].weight), sln_b=Fp(sa.ffn[1].bias),
                    sf3_w=W(sa.ffn[3].weight), sf3_b=Fp(sa.ffn[3].bias),
                    cqv_w=W(torch.cat([ca.to_qk.weight, ca.to_v.weight], 0)),
                    cqv_b=Fp(torch.cat([ca.to_qk.bias, ca.to_v.bias], 0)),
                    co_w=W(ca.to_out.weight), co_b=Fp(ca.to_out.bias),
                    cf0_w=W(cf0[0]), cf0_b=Fp(cf0[1]),
                    cln_g=Fp(ca.ffn[1].weight), cln_b=Fp(ca.ffn[1].bias),
                    cf3_w=W(ca.ffn[3].weight), cf3_b=Fp(ca.ffn[3].bias),
                )
            )
        assign = [
            dict(fp_w=W(a.final_proj.weight), fp_b=Fp(a.final_proj.bias),
                 m_w=Fp(a.matchability.weight.view(-1)), m_b=Fp(a.matchability.bias))
            for a in self.log_assignment
        ]
        token = [dict(w=Fp(t.token[0].weight.view(-1)), b=Fp(t.token[0].bias)) for t in self.token_confidence]
        packed = dict(layers=layers, assign=assign, token=token, wr=Fp(self.posenc.Wr.weight))
        if isinstance(self.input_proj, nn.Linear):
            packed["in_w"], packed["in_b"] = W(self.input_proj.weight), Fp(self.input_proj.bias)
        self._packed, self._pack_key = packed, key
        self._packs[prec] = (key, packed)
        return packed

    # ---- forward ---------------------------------------------------------------------------

    _GRAPH_INPUTS = ("keypoints0", "keypoints1", "descriptors0", "descriptors1", "scales0", "scales1", "oris0", "oris1")

    def _pinned_snapshots(self, rows: int, cols: int) -> torch.Tensor:
        """Pinned int32 scratch for the adaptive path's device -> host reads (allocated once per shape: a
        cudaHostAlloc per forward would cost more than the forward)."""
        buf = getattr(self, "_snap_buf", None)
        if buf is None or buf.shape[0] < rows or buf.shape[1] < cols:
            buf = self._snap_buf = torch.zeros(max(rows, 16), max(cols, 64), dtype=torch.int32).pin_memory()
        return buf[:rows, :cols]

    def forward(self, data: dict) -> dict:
        from . import train as _train

        if _train.wants_grad(self, data):
            return self._forward_train(data)
        with torch.no_grad():
            return self._forward_nograd(data)

    def _forward_train(self, data: dict) -> dict:
        """Training step (module in training mode, autograd on): the transformer stack runs through
        train.TransformerFn -- the library's kernels forward, hand-written backward kernels + cuBLAS GEMMs backward, in
        conf.train_precision ("fp32": the fp32-accurate tensor-core mode; "bf16": the bf16 inference kernels and bf16
        products) -- so that `ref_descriptors0/1` carry an autograd graph to the descriptors and to every parameter
        (lightglue.py:484-498, :546-547).  conf.checkpointed (:485-494) selects recomputation of the attention
        operands in the backward pass instead of keeping them.  The last layer's MatchAssignment and filter_matches run
        through train.LogAssignFn, so that `log_assignment` and `matching_scores0/1` carry a graph too (as in the
        reference: a loss may read them; LightGlue.loss reads log_assignment detached, :606, :625-630).  The staged
        keypoints (with scales / orientations when add_scale_ori) are inputs of the transformer Function: keypoints0/1,
        scales0/1 and oris0/1 that require grad receive their gradient through the positional encoding.
        data["num_keypoints0/1"] (padded batches): every kernel reads the per-pair counts, the padding's descriptors and
        keypoints are replaced by zeros, and the outputs take the layout of the no-grad forward with the same counts."""
        from . import train as _train

        for key in self.required_data_keys:
            assert key in data, f"Missing key {key} in data"
        conf = self.conf
        kpts0, kpts1 = data["keypoints0"], data["keypoints1"]
        if not kpts0.is_cuda:
            raise _abi.LightGlueB200Error(
                "glue_factory_colon_b200.LightGlue runs on CUDA (sm_100a) tensors only; there is no CPU path")
        dev = kpts0.device
        B, m, _ = kpts0.shape
        n = kpts1.shape[1]
        counts_h = self._counts_of(data, B, m, n)  # None: no counts, or all full (exactly the path without counts)
        counts = None if counts_h is None else torch.from_numpy(counts_h.reshape(-1)).to(dev)

        def size_of(v):
            sz = data[v].get("image_size") if v in data else None
            if sz is None:
                return None
            if not isinstance(sz, torch.Tensor):
                sz = torch.tensor(sz)
            return sz.to(device=dev, dtype=torch.float32).reshape(-1, 2).expand(B, 2).contiguous()

        def kpts_of(idx, k):
            k = k.to(torch.float32)
            if conf.add_scale_ori:  # lightglue.py:436-454
                sc, ori = data[f"scales{idx}"], data[f"oris{idx}"]
                sc = sc if sc.dim() == 3 else sc[..., None]
                ori = ori if ori.dim() == 3 else ori[..., None]
                k = torch.cat([k, sc.to(k), ori.to(k)], -1)
            return k.contiguous()

        k0, k1 = kpts_of(0, kpts0), kpts_of(1, kpts1)
        geom = {"size0": size_of("view0"), "size1": size_of("view1"), "counts": counts_h}
        desc0 = data["descriptors0"].to(torch.float32)
        desc1 = data["descriptors1"].to(torch.float32)
        assert desc0.shape[-1] == conf.input_dim and desc1.shape[-1] == conf.input_dim
        params = [p for _, p in _train.transformer_params(self)]
        L = conf.n_layers
        r0, r1 = _train.TransformerFn.apply(self, geom, desc0, desc1, k0, k1, *params)
        a = self.log_assignment[L - 1]
        scores, m0, m1, ms0, ms1 = _train.LogAssignFn.apply(
            self, L - 1, counts, r0[:, -1], r1[:, -1], a.final_proj.weight, a.final_proj.bias, a.matchability.weight,
            a.matchability.bias)
        return {
            "matches0": m0, "matches1": m1, "matching_scores0": ms0, "matching_scores1": ms1,
            "ref_descriptors0": r0, "ref_descriptors1": r1, "log_assignment": scores,
            "prune0": torch.full((B, m), float(L), device=dev), "prune1": torch.full((B, n), float(L), device=dev),
        }

    def _forward_nograd(self, data: dict) -> dict:
        for key in self.required_data_keys:
            assert key in data, f"Missing key {key} in data"
        conf = self.conf
        if not (conf.cuda_graph and not self.training and data["keypoints0"].is_cuda):
            return self._forward_impl(data)
        # adaptive depth / width: the transformer stack (all layers; the kernels skip finished pairs and pruned rows
        # from device-side counts) is captured, the data-dependent tail -- one host read of the exit layers and the
        # pruned counts, MatchAssignment of the exit layer at the pruned shape, filter_matches -- runs eagerly behind
        # every replay (lightglue.py:501-536)
        adaptive = conf.depth_confidence > 0 or conf.width_confidence > 0
        cap = conf.get("graph_capacity")
        if (cap is not None and not adaptive and self._precision() in (BF16, F32X3)
                and max(data["keypoints0"].shape[1], data["keypoints1"].shape[1]) <= cap):
            return self._forward_capacity(data, int(cap))
        if "num_keypoints0" in data or "num_keypoints1" in data:
            return self._forward_impl(data)
        # ---- CUDA-graph path: static copies of the inputs, one captured forward per input signature ----
        ins = {k: data[k] for k in self._GRAPH_INPUTS if isinstance(data.get(k), torch.Tensor)}
        for v in ("view0", "view1"):
            sz = data.get(v, {}).get("image_size") if v in data else None
            if sz is not None:
                ins[v] = sz if isinstance(sz, torch.Tensor) else torch.tensor(sz)
        dev = data["keypoints0"].device
        prec = self._precision()
        self._pack(prec, dev)
        sig = (prec, self._pack_key, float(conf.depth_confidence), float(conf.width_confidence)) + tuple(
            (k, tuple(t.shape), t.dtype) for k, t in sorted(ins.items()))
        entry = self._graphs.get(sig)
        if entry is None:
            static = {k: t.to(dev).clone() for k, t in ins.items()}

            def as_data():
                d = {k: t for k, t in static.items() if not k.startswith("view")}
                d["view0"] = {"image_size": static["view0"]} if "view0" in static else {}
                d["view1"] = {"image_size": static["view1"]} if "view1" in static else {}
                return d

            warm = self._forward_impl(as_data(), static=adaptive)  # outside the capture: lazy initialisation, pools
            if adaptive:
                warm()
            torch.cuda.synchronize(dev)
            graph = torch.cuda.CUDAGraph()
            out = _capture(graph, lambda: self._forward_impl(as_data(), static=adaptive))  # adaptive: the tail closure
            if len(self._graphs) >= 8:  # a handful of signatures at most; drop the oldest
                self._graphs.pop(next(iter(self._graphs)))
            # the captured launches carry raw device pointers (and TMA tensor maps) into the weight pack: the entry
            # keeps the pack alive for as long as the graph can be replayed (a precision switch replaces self._packed)
            entry = self._graphs[sig] = (graph, static, out, self._packed)
        graph, static, out, _ = entry
        for k, t in ins.items():
            static[k].copy_(t, non_blocking=True)
        graph.replay()
        if adaptive:
            return out()  # fresh output tensors
        if conf.get("graph_static_outputs", False):  # caller consumes the results before the next call: no copies
            return dict(out)
        return {k: v.clone() for k, v in out.items()}  # the graph's output buffers are overwritten by the next replay

    def _forward_capacity(self, data: dict, cap: int) -> dict:
        """conf.graph_capacity: one CUDA graph of lgb200_match at B x cap x cap per (precision, weights, B, which image
        sizes are given) serves every input with max(m, n) <= cap.  The outputs are bit-equal to the eager forward of
        the input zero-padded to cap with the same counts, cropped to this input's shapes.  A call reads nothing back
        and makes no library call: it copies the pair in, replays and crops."""
        dev = data["keypoints0"].device
        B = data["keypoints0"].shape[0]
        prec = self._precision()
        self._pack(prec, dev)
        sizes = [data[v].get("image_size") if v in data else None for v in ("view0", "view1")]
        key = (prec, self._pack_key, B, cap, sizes[0] is not None, sizes[1] is not None)
        entry = self._graphs.get(key)
        if entry is None:
            entry = _CapacityGraph(self, prec, B, cap, data, sizes)
            if len(self._graphs) >= 8:  # shares the per-signature captures' limit: drop the oldest
                self._graphs.pop(next(iter(self._graphs)))
            self._graphs[key] = entry
        return entry(data, sizes, self.conf.get("graph_static_outputs", False))

    def _forward_impl(self, data: dict, static: bool = False):
        lib = _abi.load()
        conf = self.conf
        kpts0, kpts1 = data["keypoints0"], data["keypoints1"]
        if not kpts0.is_cuda:
            raise _abi.LightGlueB200Error(
                "glue_factory_colon_b200.LightGlue runs on CUDA (sm_100a) tensors only; there is no CPU path"
            )
        check(lib.lgb200_device_ok(), "device check")
        dev = kpts0.device
        B, m, _ = kpts0.shape
        _, n, _ = kpts1.shape
        # lightglue.py:430-432 -- unlike the reference (F6: UnboundLocalError) a missing view is size=None
        size0 = data["view0"].get("image_size") if "view0" in data else None
        size1 = data["view1"].get("image_size") if "view1" in data else None
        f32 = dict(device=dev, dtype=torch.float32)
        i32 = dict(device=dev, dtype=torch.int32)

        def prep_size(sz):
            if sz is None:
                return None
            if not isinstance(sz, torch.Tensor):
                sz = torch.tensor(sz)
            return sz.to(**f32).reshape(-1, 2).expand(B, 2).contiguous()

        size0, size1 = prep_size(size0), prep_size(size1)

        def prep_kpts(idx, k):
            k = k.to(torch.float32)
            if conf.add_scale_ori:  # lightglue.py:436-454
                sc, ori = data[f"scales{idx}"], data[f"oris{idx}"]
                sc = sc if sc.dim() == 3 else sc[..., None]
                ori = ori if ori.dim() == 3 else ori[..., None]
                k = torch.cat([k, sc.to(k), ori.to(k)], -1)
            return k.contiguous()

        k0, k1 = prep_kpts(0, kpts0), prep_kpts(1, kpts1)
        kdim = k0.shape[-1]
        desc0 = data["descriptors0"].to(torch.float32).contiguous()
        desc1 = data["descriptors1"].to(torch.float32).contiguous()
        assert desc0.shape[-1] == conf.input_dim
        assert desc1.shape[-1] == conf.input_dim

        prec = self._precision()
        bf = prec == BF16
        x3 = prec == F32X3   # fp32-accurate tensor-core mode: MMA operands are split-fp16 planes [2][rows][K]
        fold = bf or x3      # out_proj / to_out folded into the first FFN matrix (see _pack)
        W = self._pack(prec, dev)
        st = torch.cuda.current_stream(dev).cuda_stream
        L = conf.n_layers
        S = 2 * B
        gran = 256 if x3 else 128  # (the x3 similarity GEMM tiles the keys by 256)
        Lp = max(gran, ((max(m, n) + gran - 1) // gran) * gran)
        T = S * Lp

        # per-sequence valid counts (B200 extension for padded batches, SURVEY.md 8(c))
        lens_host = np.empty((B, 2), dtype=np.int32)
        lens_host[:, 0], lens_host[:, 1] = m, n
        variable = False
        for idx in (0, 1):
            cnt = data.get(f"num_keypoints{idx}")
            if cnt is not None:
                lens_host[:, idx] = torch.as_tensor(cnt).to("cpu", torch.int32).numpy().reshape(-1)
                variable = True
        assert (lens_host[:, 0] <= m).all() and (lens_host[:, 1] <= n).all() and (lens_host >= 0).all()
        do_early = conf.depth_confidence > 0 and not self.training
        do_prune = conf.width_confidence > 0 and not self.training
        adaptive = do_early or do_prune
        use_lens = variable or adaptive or m != Lp or n != Lp
        order_self = order_cross = None
        if not use_lens:
            lens = None
        elif variable:
            # one upload: lens | launch order of the self attention | of the cross attention (sequences sorted by key
            # count, longest first: a ragged batch's attention kernels then end on their shortest work items)
            flat = lens_host.reshape(-1)
            o_self = np.argsort(-flat, kind="stable").astype(np.int32)
            o_cross = np.argsort(-flat[np.arange(S) ^ 1], kind="stable").astype(np.int32)
            up = torch.from_numpy(np.concatenate([flat, o_self, o_cross])).to(dev)
            lens, order_self, order_cross = up[:S], up[S:2 * S], up[2 * S:]
            if os.environ.get("LGB200_ATTN_ORDER", "1") == "0":  # A/B switch
                order_self = order_cross = None
        else:  # all pairs (m, n): filled on the device (no host copy, so the forward can be captured in a CUDA graph)
            lens = torch.empty(S, **i32)
            lens[0::2] = m
            lens[1::2] = n
        lens_act = lens.clone() if adaptive else lens

        act = torch.bfloat16 if bf else torch.float32
        adt = dict(device=dev, dtype=act)
        # Residual stream x [T,256] in the activation dtype (bf16 mode keeps it in bf16 only: measured
        # against the fp32 oracle this is still 2x closer than the reference's own autocast run).
        # x3 mode: x stays the fp32 master (exact residual adds, token heads, returned descriptors) and xs holds its
        # split planes, the A operand of the projections.
        x = torch.empty(T, 256, **adt)
        rot = None if bf else torch.empty(T, 64, **f32)           # (cos, sin) fp32 pairs
        rot16 = torch.empty(T, 32, **i32) if bf else None          # packed fp16 (cos, sin)
        # padded rows must hold finite values (masked keys multiply V rows by exactly 0); without
        # padding every row is written before it is read, so the fills are skipped
        alloc = torch.zeros if use_lens else torch.empty
        if x3:
            h16 = dict(device=dev, dtype=torch.float16)
            xs = alloc(2, T, 256, **h16)
            q, k, v = alloc(2, T * 256, **h16), alloc(2, T * 256, **h16), alloc(2, T * 256, **h16)
            ctx, msg, hid = alloc(2, T, 256, **h16), alloc(2, T, 256, **h16), alloc(2, T, 512, **h16)
        else:
            xs = None
            q = alloc(T * 256, **adt)
            k = alloc(T * 256, **adt)
            v = alloc(T * 256, **adt)
            ctx = alloc(T, 256, **adt)
            msg = alloc(T, 256, **adt)
            hid = alloc(T, 512, **adt)

        def linear(epi, A0, Wt, bias, N, K, A1=None, K0=None, scale=(1.0, 1.0, 1.0), resid=None,
                   out=None, n_rot=0, outp=(None, None, None), gamma=None, beta=None, lens_=None, out32=None):
            """x3: A0 / A1 / out / outp are split planes, resid / out32 fp32."""
            if x3:
                r32, r16, o32, o16 = resid, None, out32, out
            else:
                r32, r16 = (None, resid) if bf else (resid, None)
                o32, o16 = (None, out) if bf else (out, None)
            check(
                lib.lgb200_linear(
                    prec, epi, ptr(A0), ptr(A1), K if K0 is None else K0, ptr(Wt), ptr(bias), T, N, K,
                    ptr(lens_), Lp, scale[0], scale[1], scale[2], ptr(r32), ptr(r16), ptr(o32), ptr(o16),
                    ptr(rot), ptr(rot16), n_rot, ptr(outp[0]), ptr(outp[1]), ptr(outp[2]), ptr(gamma),
                    ptr(beta), st,
                ),
                "lgb200_linear",
            )

        def split(src32, dst16):  # fp32 rows -> split planes
            check(lib.lgb200_split_rows(ptr(src32), src32.numel(), ptr(dst16), st), "split_rows")

        def pack(dsc, cnt, dim, img, dst):
            x32_, x16_ = (None, dst) if bf else (dst, None)
            check(lib.lgb200_pack_rows(ptr(dsc), B, cnt, dim, img, Lp, ptr(x32_), ptr(x16_), st), "pack_rows")

        hprec = F32 if x3 else prec  # the token / matchability heads read the fp32 master in x3 mode

        def rowdot(xt, wb, lens_, sigmoid, out):
            check(lib.lgb200_rowdot(hprec, ptr(xt), ptr(wb[0]), ptr(wb[1]), S, Lp, ptr(lens_), sigmoid, ptr(out), st),
                  "lgb200_rowdot")

        # ---- staging: descriptors (+ input_proj) and positional encoding ----
        if isinstance(self.input_proj, nn.Linear):
            din = conf.input_dim
            xin = torch.empty(T, din, **adt)
            for img, dsc, cnt in ((0, desc0, m), (1, desc1, n)):
                pack(dsc, cnt, din, img, xin)
            if x3:
                xin_s = torch.empty(2, T, din, **h16)
                split(xin, xin_s)
                linear(EPI_ROWMAJOR, xin_s, W["in_w"], W["in_b"], 256, din, out=xs, out32=x)
            else:
                linear(EPI_ROWMAJOR, xin, W["in_w"], W["in_b"], 256, din, out=x)
        else:
            for img, dsc, cnt in ((0, desc0, m), (1, desc1, n)):
                pack(dsc, cnt, 256, img, x)
            if x3:
                split(x, xs)
        for img, kk, cnt, sz in ((0, k0, m, size0), (1, k1, n, size1)):
            check(lib.lgb200_posenc(ptr(kk), B, cnt, kdim, ptr(sz), ptr(W["wr"]), ptr(lens), img, Lp, ptr(rot),
                                    ptr(rot16), st), "lgb200_posenc")

        # ---- adaptive state (device resident) ----
        if adaptive:
            conf_buf = torch.zeros(T, **f32)
            msig = torch.zeros(T, **f32)
            # device state read by the host: [done (B) | lens (S)], snapshotted into pinned memory without blocking
            state = torch.zeros(B + S, **i32)
            done = state[:B]
            if lens.data_ptr() != state[B:].data_ptr():
                state[B:].copy_(lens)
                lens = state[B:]
                lens_act = lens.clone()
            if variable:
                total = torch.from_numpy(lens_host.sum(1).astype(np.int32)).to(dev)
            else:  # filled on the device: no host copy inside a graph capture
                total = torch.full((B,), m + n, **i32)
            snaps = self._pinned_snapshots(L + 1, B + S)
            snap_ev = []
            polled = 0
        if do_prune:
            ind = torch.arange(Lp, **i32).repeat(S, 1).contiguous()
            prune_cnt = torch.ones(S, Lp, **i32)
            x_b, ind_b = torch.zeros_like(x), torch.zeros_like(ind)
            rot_b = None if bf else torch.zeros_like(rot)
            rot16_b = torch.zeros_like(rot16) if bf else None
        exit_layer = np.full(B, L - 1, dtype=np.int64)
        thresholds = [self.confidence_threshold(i) for i in range(L)]

        q_scale = LOG2E / math.sqrt(64.0)
        c_scale = math.sqrt(q_scale)
        collected0, collected1 = [], []  # training mode: every layer's descriptors (lightglue.py:495-497)
        for i in range(L):
            w = W["layers"][i]
            la = lens_act
            # self block (lightglue.py:151-164)
            xa = xs if x3 else x  # A operand of the projections
            linear(EPI_HEADS, xa, w["qkv_w"], w["qkv_b"], 768, 256, scale=(q_scale, 1.0, 1.0), n_rot=2,
                   outp=(q, k, v), lens_=la)
            if self._attn_events is not None:
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev0.record()
            check(lib.lgb200_attention_ordered(prec, ptr(q), ptr(k), ptr(v), S, Lp, ptr(la), ptr(order_self), 0, ptr(ctx),
                                               st), "attention")
            if self._attn_events is not None:
                ev1.record()
                self._attn_events.append((ev0, ev1))
            if not fold:  # (bf16 / x3: out_proj is folded into sf0_w, see _pack)
                linear(EPI_ROWMAJOR, ctx, w["so_w"], w["so_b"], 256, 256, out=msg, lens_=la)
            linear(EPI_LN_GELU, xa, w["sf0_w"], w["sf0_b"], 512, 512, A1=ctx if fold else msg, K0=256, gamma=w["sln_g"],
                   beta=w["sln_b"], out=hid, lens_=la)
            if x3:
                linear(EPI_ROWMAJOR, hid, w["sf3_w"], w["sf3_b"], 256, 512, resid=x, out=xs, out32=x, lens_=la)
            else:
                linear(EPI_ROWMAJOR, hid, w["sf3_w"], w["sf3_b"], 256, 512, resid=x, out=x, lens_=la)
            # cross block (lightglue.py:193-222)
            linear(EPI_HEADS, xa, w["cqv_w"], w["cqv_b"], 512, 256, scale=(c_scale, 1.0, 1.0), n_rot=0,
                   outp=(q, v, None), lens_=la)
            check(lib.lgb200_attention_ordered(prec, ptr(q), ptr(q), ptr(v), S, Lp, ptr(la), ptr(order_cross), 1, ptr(ctx),
                                               st), "attention")
            if not fold:
                linear(EPI_ROWMAJOR, ctx, w["co_w"], w["co_b"], 256, 256, out=msg, lens_=la)
            linear(EPI_LN_GELU, xa, w["cf0_w"], w["cf0_b"], 512, 512, A1=ctx if fold else msg, K0=256, gamma=w["cln_g"],
                   beta=w["cln_b"], out=hid, lens_=la)
            if x3:
                linear(EPI_ROWMAJOR, hid, w["cf3_w"], w["cf3_b"], 256, 512, resid=x, out=xs, out32=x, lens_=la)
            else:
                linear(EPI_ROWMAJOR, hid, w["cf3_w"], w["cf3_b"], 256, 512, resid=x, out=x, lens_=la)
            if self.training:
                xl = x.view(B, 2, Lp, 256)
                collected0.append(xl[:, 0, :m].clone())
                collected1.append(xl[:, 1, :n].clone())
            if i == L - 1 or not adaptive:
                continue
            thr = thresholds[i]
            if do_early:  # lightglue.py:501-505
                tk = W["token"][i]
                rowdot(x, (tk["w"], tk["b"]), la, 1, conf_buf)
                check(lib.lgb200_exit_check(ptr(conf_buf), B, Lp, ptr(lens), ptr(total), thr,
                                            float(conf.depth_confidence), i, ptr(done), ptr(lens_act), st), "exit_check")
                # No host round trip here (the reference syncs 2-3 times per layer, lightglue.py:501-521): the kernels
                # of later layers skip finished pairs by themselves (lens_active == 0), so the host only needs to
                # learn about the exit EVENTUALLY, to stop launching.  The flags are copied to pinned memory behind
                # the check and older snapshots are polled without blocking.
                # (static: the whole stack is being captured into a CUDA graph -- all layers are launched, finished
                # pairs cost empty kernels)
                if not static:
                    snaps[i, :B].copy_(done, non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record()
                    snap_ev.append(ev)
                    stop = False
                    while polled < len(snap_ev) and snap_ev[polled].query():
                        stop = stop or bool((snaps[polled, :B] != 0).all())
                        polled += 1
                    if stop:
                        break
            if do_prune:  # lightglue.py:506-521
                ma = W["assign"][i]
                rowdot(x, (ma["m_w"], ma["m_b"]), la, 1, msig)
                x32s, x16s = (None, x) if bf else (x, None)
                x32d, x16d = (None, x_b) if bf else (x_b, None)
                check(lib.lgb200_prune_compact(ptr(msig), ptr(conf_buf) if do_early else None, thr,
                                               float(conf.width_confidence), S, Lp, ptr(lens), ptr(lens_act),
                                               ptr(x32s), ptr(x32d), ptr(x16s), ptr(x16d), ptr(rot), ptr(rot_b),
                                               ptr(rot16), ptr(rot16_b), ptr(ind), ptr(ind_b), ptr(prune_cnt), st),
                      "prune_compact")
                x, x_b = x_b, x
                if x3:  # the split planes follow the compacted fp32 master
                    split(x, xs)
                rot, rot_b = rot_b, rot
                rot16, rot16_b = rot16_b, rot16
                ind, ind_b = ind_b, ind

        def tail():
            """Everything behind the transformer stack: the one host read of an adaptive forward, MatchAssignment of
            the exit layer(s), filter_matches, the output dict.  With static=True (CUDA-graph capture of an adaptive
            forward) it is returned instead of run: the graph holds the stack, the tail runs eagerly after a replay."""
            nonlocal exit_layer, st
            st = torch.cuda.current_stream(dev).cuda_stream  # (a captured stack was recorded on the capture stream)
            if adaptive:
                # the one blocking read of an adaptive forward: exit flags and (pruned) counts together
                snaps[L].copy_(state, non_blocking=True)
                torch.cuda.current_stream(dev).synchronize()
                st_h = snaps[L].numpy()
                done_h = st_h[:B]
                exit_layer = np.where(done_h != 0, done_h - 1, L - 1).astype(np.int64)
                lens_final = st_h[B:].reshape(B, 2).copy()
            # ---- log assignment (lightglue.py:523-524) ----
            md = msg  # reuse: [T,256] in the activation dtype (x3: split planes)
            sim = None
            z = torch.zeros(T, **f32)
            lse = torch.zeros(T, **f32)
            for e in np.unique(exit_layer):
                if adaptive and lens is not None and len(np.unique(exit_layer)) > 1:
                    sel = torch.from_numpy(np.repeat(exit_layer == e, 2)).to(dev)
                    lens_g = torch.where(sel, lens, torch.zeros_like(lens))
                else:
                    lens_g = lens
                a = W["assign"][int(e)]
                linear(EPI_ROWMAJOR, xs if x3 else x, a["fp_w"], a["fp_b"], 256, 256, scale=(0.25, 1.0, 1.0), out=md,
                       lens_=lens_g)
                rowdot(x, (a["m_w"], a["m_b"]), lens_g, 0, z)
                if x3:
                    if sim is None:
                        sim = torch.empty(B, Lp, Lp, **f32)
                    check(lib.lgb200_x3_similarity(ptr(md), B, Lp, ptr(lens_g), ptr(sim), st), "x3_similarity")
                    check(lib.lgb200_x3_assign_lse(ptr(sim), B, Lp, ptr(lens_g), m, n, ptr(lse), st), "x3_assign_lse")
                else:
                    check(lib.lgb200_assign_lse(prec, ptr(md), S, Lp, ptr(lens_g), ptr(lse), st), "assign_lse")
            if do_prune:  # pruned shape is data dependent (lightglue.py:285 note)
                R, C = int(lens_final[:, 0].max()) + 1, int(lens_final[:, 1].max()) + 1
            else:
                R, C = m + 1, n + 1
            scores = torch.empty(B, R, C, **f32)
            fm_ws = torch.empty(B * (R + C), device=dev, dtype=torch.int64)
            # bf16: the assignment epilogue also emits the row/column arg-maxima, so filter_matches never
            # re-reads the 1 GB score matrix
            if x3:
                check(lib.lgb200_x3_assign_scores(ptr(sim), ptr(z), ptr(lse), B, Lp, ptr(lens), R, C, ptr(scores), st),
                      "x3_assign_scores")
            else:
                check(lib.lgb200_assign_scores(prec, ptr(md), ptr(z), ptr(lse), B, Lp, ptr(lens), R, C, ptr(scores),
                                               ptr(fm_ws) if bf else None, st), "assign_scores")

            # ---- filter_matches (lightglue.py:525-536) ----
            m0 = torch.empty(B, m, device=dev, dtype=torch.int64)
            m1 = torch.empty(B, n, device=dev, dtype=torch.int64)
            ms0 = torch.empty(B, m, **f32)
            ms1 = torch.empty(B, n, **f32)
            check(
                lib.lgb200_filter_matches(
                    ptr(scores), B, R, C, ptr(lens), float(conf.filter_threshold),
                    ptr(ind) if do_prune else None, ptr(ind[1:]) if do_prune else None, 2 * Lp,
                    m, n, ptr(m0), ptr(m1), ptr(ms0), ptr(ms1), ptr(fm_ws), 1 if bf else 0, st,
                ),
                "filter_matches",
            )

            xv = x.view(B, 2, Lp, 256)
            if do_prune:
                pc = prune_cnt.view(B, 2, Lp)
                prune0, prune1 = pc[:, 0, :m].to(torch.int64), pc[:, 1, :n].to(torch.int64)
                k0f, k1f = R - 1, C - 1
                ref0, ref1 = xv[:, 0:1, :k0f], xv[:, 1:2, :k1f]
            else:  # lightglue.py:538-539
                prune0 = torch.full((B, m), float(L), **f32)
                prune1 = torch.full((B, n), float(L), **f32)
                ref0, ref1 = xv[:, 0:1, :m], xv[:, 1:2, :n]
            if self.training:  # [B, n_layers, N, 256] (lightglue.py:546-547)
                ref0, ref1 = torch.stack(collected0, 1), torch.stack(collected1, 1)
            return {
                "matches0": m0,
                "matches1": m1,
                "matching_scores0": ms0,
                "matching_scores1": ms1,
                # activation dtype, like the reference: fp32 by default, half precision under mp / autocast
                # (lightglue.py:466-468 casts desc to half; :541-553 returns the stacked layer outputs as they are).
                # Zero-copy views of the residual stream; the two fp32 copies cost 0.2 ms per 64-pair batch.
                "ref_descriptors0": ref0,
                "ref_descriptors1": ref1,
                "log_assignment": scores,
                "prune0": prune0,
                "prune1": prune1,
            }


        return tail if static else tail()


class _CapacityGraph:
    """The forward captured at a keypoint capacity K (conf.graph_capacity): one lgb200_match call at B x K x K on static
    inputs, device counts, a workspace and output buffers.  lgb200_match allocates nothing, synchronises nothing and
    reads no count on the host, so the graph serves any input of at most K keypoints per image.  The entry owns the
    packed weights its launches point into: a precision switch replaces the module's pack but cannot free them."""

    def __init__(self, model: LightGlue, prec: int, B: int, K: int, data: dict, sizes: list):
        conf = model.conf
        dev = data["keypoints0"].device
        self.B, self.K, self.n_layers = B, K, conf.n_layers
        kdim = 4 if conf.add_scale_ori else 2
        self.cfg = MatchConfig(prec, conf.n_layers, conf.input_dim, kdim, float(conf.filter_threshold))
        self.table, self.weights = native_table(model, prec)
        f32, i64 = dict(device=dev, dtype=torch.float32), dict(device=dev, dtype=torch.int64)
        self.kpts = [torch.zeros(B, K, kdim, **f32) for _ in range(2)]
        self.desc = [torch.zeros(B, K, conf.input_dim, **f32) for _ in range(2)]
        self.rows = [0, 0]  # rows of kpts / desc that may hold something other than zeros
        self.size = [None if s is None else torch.empty(B, 2, **f32) for s in sizes]
        self.counts = torch.empty(2, B, device=dev, dtype=torch.int32)
        lib = _abi.load()
        nb = ctypes.c_longlong(0)
        check(lib.lgb200_match_workspace(ctypes.byref(self.cfg), B, K, K, ctypes.byref(nb)), "match_workspace")
        self.ws = torch.empty(nb.value, device=dev, dtype=torch.uint8)
        act = torch.bfloat16 if prec == BF16 else torch.float32
        self.out = {
            "matches0": torch.empty(B, K, **i64), "matches1": torch.empty(B, K, **i64),
            "matching_scores0": torch.empty(B, K, **f32), "matching_scores1": torch.empty(B, K, **f32),
            "ref_descriptors0": torch.empty(B, K, 256, device=dev, dtype=act),
            "ref_descriptors1": torch.empty(B, K, 256, device=dev, dtype=act),
            "log_assignment": torch.empty(B, K + 1, K + 1, **f32),
        }
        self._load(data, sizes)
        self._launch(lib)  # outside the capture: lazy initialisation
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        _capture(self.graph, lambda: self._launch(lib))

    def _launch(self, lib) -> None:
        o = self.out
        check(lib.lgb200_match(
            ctypes.byref(self.cfg), self.table, self.B, self.K, self.K, ptr(self.kpts[0]), ptr(self.kpts[1]),
            ptr(self.desc[0]), ptr(self.desc[1]), ptr(self.size[0]), ptr(self.size[1]), ptr(self.counts[0]),
            ptr(self.counts[1]), ptr(o["matches0"]), ptr(o["matches1"]), ptr(o["matching_scores0"]),
            ptr(o["matching_scores1"]), ptr(o["log_assignment"]), ptr(o["ref_descriptors0"]),
            ptr(o["ref_descriptors1"]), ptr(self.ws), self.ws.numel(),
            torch.cuda.current_stream(self.ws.device).cuda_stream), "lgb200_match")

    def _load(self, data: dict, sizes: list) -> None:
        """The pair into the static inputs: its rows, zeros over the rows a larger earlier input left (so every row past
        m / n is zero and the result cannot depend on an earlier call), the counts min(num_keypoints, m) or m, the image
        sizes.  Copies only: nothing is read back."""
        B = self.B
        for i in (0, 1):
            kp, dsc, k, d = data[f"keypoints{i}"], data[f"descriptors{i}"], self.kpts[i], self.desc[i]
            c = kp.shape[1]
            assert dsc.shape[-1] == d.shape[-1]
            k[:, :c, :2].copy_(kp, non_blocking=True)
            if k.shape[2] == 4:  # add_scale_ori (lightglue.py:436-454)
                k[:, :c, 2].copy_(data[f"scales{i}"].reshape(B, c), non_blocking=True)
                k[:, :c, 3].copy_(data[f"oris{i}"].reshape(B, c), non_blocking=True)
            d[:, :c].copy_(dsc, non_blocking=True)
            if self.rows[i] > c:
                k[:, c:self.rows[i]].zero_()
                d[:, c:self.rows[i]].zero_()
            self.rows[i] = c
            cnt = data.get(f"num_keypoints{i}")
            if cnt is None:
                self.counts[i].fill_(c)
            else:
                self.counts[i].copy_(torch.as_tensor(cnt).reshape(-1).clamp(max=c), non_blocking=True)
            if sizes[i] is not None:
                self.size[i].copy_(torch.as_tensor(sizes[i]).reshape(-1, 2), non_blocking=True)

    def __call__(self, data: dict, sizes: list, static_outputs: bool) -> dict:
        """Load, replay, and fresh outputs in the shapes of the eager forward for this input: log_assignment cropped
        to [B, m+1, n+1] with the dustbins moved to row m and column n.  static_outputs: the graph's own buffers (valid
        until the next call) when they already have those shapes: m == n == K and no counts given."""
        B, K = self.B, self.K
        m, n = data["keypoints0"].shape[1], data["keypoints1"].shape[1]
        self._load(data, sizes)
        self.graph.replay()
        o = self.out
        dev = self.ws.device
        prune0 = torch.full((B, m), float(self.n_layers), device=dev, dtype=torch.float32)
        prune1 = torch.full((B, n), float(self.n_layers), device=dev, dtype=torch.float32)
        if static_outputs and m == n == K and "num_keypoints0" not in data and "num_keypoints1" not in data:
            return {
                "matches0": o["matches0"], "matches1": o["matches1"],
                "matching_scores0": o["matching_scores0"], "matching_scores1": o["matching_scores1"],
                "ref_descriptors0": o["ref_descriptors0"][:, None], "ref_descriptors1": o["ref_descriptors1"][:, None],
                "log_assignment": o["log_assignment"], "prune0": prune0, "prune1": prune1,
            }
        return {
            "matches0": o["matches0"][:, :m].clone(), "matches1": o["matches1"][:, :n].clone(),
            "matching_scores0": o["matching_scores0"][:, :m].clone(),
            "matching_scores1": o["matching_scores1"][:, :n].clone(),
            "ref_descriptors0": o["ref_descriptors0"][:, None, :m].clone(),
            "ref_descriptors1": o["ref_descriptors1"][:, None, :n].clone(),
            "log_assignment": crop_log_assignment(o["log_assignment"], m, n),
            "prune0": prune0, "prune1": prune1,
        }


__main_model__ = LightGlue
