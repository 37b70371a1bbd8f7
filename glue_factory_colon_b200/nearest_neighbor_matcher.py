"""B200 drop-in for `gluefactory.models.matchers.nearest_neighbor_matcher.NearestNeighborMatcher`
(SURVEY.md 8(f) rank 3): same conf keys, same input / output dict, fp32.

Compute runs in the C-ABI library: the similarity and the dual log-softmax reuse the fp32 similarity kernels of
MatchAssignment (`lgb200_assign_lse`, `lgb200_nn_scores`), `find_nn` + `mutual_check` are `lgb200_nn_match`.
There is no CPU path.  Select it in glue-factory with `model.matcher.name=glue_factory_colon_b200.nearest_neighbor_matcher`.

Training (`loss: "N_pair"`) works as in the reference: with autograd on, `similarity` carries a graph to
`descriptors0/1` when they require grad, and `loss` returns `n_pair_nll` / `total` with a graph to `similarity` and the
learnable `temperature`, so `losses["total"].mean().backward()` trains both the descriptors and the temperature.  The
forward values are those of the no-grad path bit for bit; `log_assignment` (which no loss reads) is returned without a
graph.  Backward: `lgb200_npair_loss_bwd` (one streaming pass over similarity and ground truth) gives d similarity and
d temperature; d descriptors = dSim . d1 and dSim^T . d0 as three fp16 tensor-core products on split planes with fp32
output (`train.bmm3`), exactly zero on rows past `num_keypoints0/1`.
"""
from __future__ import annotations

from types import SimpleNamespace

import torch
import torch.nn.functional as F
from torch import nn

from . import _abi
from ._abi import F32, check, ptr
from .train import bmm3

_OUT_KEYS = ("matches0", "matches1", "matching_scores0", "matching_scores1", "similarity", "log_assignment")


class NearestNeighborMatcher(nn.Module):
    # nearest_neighbor_matcher.py:47-53
    default_conf = {"ratio_thresh": None, "distance_thresh": None, "mutual_check": True, "loss": None}
    required_data_keys = ["descriptors0", "descriptors1"]

    def __init__(self, conf=None):
        super().__init__()
        merged = dict(self.default_conf)
        merged.update(dict(conf or {}))  # unknown keys (name, trainable, ...) are accepted like BaseModel does
        self.conf = SimpleNamespace(**merged)
        if self.conf.loss == "N_pair":  # :55-58
            self.register_parameter("temperature", nn.Parameter(torch.tensor(1.0)))

    def forward(self, data: dict) -> dict:
        for key in self.required_data_keys:
            assert key in data, f"Missing key {key} in data"
        d0, d1 = data["descriptors0"], data["descriptors1"]
        if not d0.is_cuda:
            raise _abi.LightGlueB200Error("glue_factory_colon_b200.NearestNeighborMatcher runs on CUDA tensors only")
        if torch.is_grad_enabled() and (d0.requires_grad or d1.requires_grad):
            return dict(zip(_OUT_KEYS, _SimilarityFn.apply(self, data, d0, d1)))
        with torch.no_grad():
            return self._match(data, d0, d1)[0]

    def _match(self, data: dict, d0, d1):
        """-> (outputs, per-pair counts [B, 2] int32 on the host; None when a side is empty)."""
        lib = _abi.load()
        check(lib.lgb200_device_ok(), "device check")
        B, N, D = d0.shape
        M = d1.shape[1]
        assert d1.shape[0] == B and d1.shape[2] == D
        if D > 256:
            raise ValueError("descriptor dimension above 256 is not supported by the similarity kernel")
        dev = d0.device
        f32 = dict(device=dev, dtype=torch.float32)
        i64 = dict(device=dev, dtype=torch.int64)
        if N == 0 or M == 0:  # find_nn with no candidates (:17-18): nothing to compute
            return {
                "matches0": torch.full((B, N), -1, **i64), "matches1": torch.full((B, M), -1, **i64),
                "matching_scores0": torch.zeros(B, N, **f32), "matching_scores1": torch.zeros(B, M, **f32),
                "similarity": torch.zeros(B, N, M, **f32), "log_assignment": torch.zeros(B, N + 1, M + 1, **f32),
            }, None
        Lp = (max(N, M) + 127) // 128 * 128
        S = 2 * B
        # staging: [S, Lp, 256] fp32, sequence s = 2b + image, rows >= count and columns >= D zero
        md = torch.zeros(B, 2, Lp, 256, **f32)
        md[:, 0, :N, :D] = d0
        md[:, 1, :M, :D] = d1
        counts = torch.empty(B, 2, dtype=torch.int32)
        counts[:, 0], counts[:, 1] = N, M
        for idx in (0, 1):  # B200 extension, as in the LightGlue drop-in: per-pair valid counts of a padded batch
            cnt = data.get(f"num_keypoints{idx}")
            if cnt is not None:
                counts[:, idx] = torch.as_tensor(cnt).to("cpu", torch.int32).reshape(-1)
        lens = counts.reshape(-1).to(dev)
        st = torch.cuda.current_stream(dev).cuda_stream
        lse = torch.empty(S * Lp, **f32)
        check(lib.lgb200_assign_lse(F32, ptr(md), S, Lp, ptr(lens), ptr(lse), st), "assign_lse")
        sim = torch.empty(B, N, M, **f32)
        la = torch.empty(B, N + 1, M + 1, **f32)
        check(lib.lgb200_nn_scores(ptr(md), ptr(lse), B, Lp, ptr(lens), N + 1, M + 1, ptr(sim), ptr(la), st), "nn_scores")
        ws = torch.empty(B * (N + M), **i64)
        m0, m1 = torch.empty(B, N, **i64), torch.empty(B, M, **i64)
        ms0, ms1 = torch.empty(B, N, **f32), torch.empty(B, M, **f32)
        check(
            lib.lgb200_nn_match(ptr(sim), B, N, M, ptr(lens), float(self.conf.ratio_thresh or 0.0),
                                float(self.conf.distance_thresh or 0.0), int(bool(self.conf.mutual_check)),
                                ptr(ws), ptr(m0), ptr(m1), ptr(ms0), ptr(ms1), st),
            "nn_match",
        )
        return {"matches0": m0, "matches1": m1, "matching_scores0": ms0, "matching_scores1": ms1,
                "similarity": sim, "log_assignment": la}, counts

    def loss(self, pred, data):
        """nearest_neighbor_matcher.py:85-109.  `N_pair`: three streaming passes over the similarity matrix in
        `lgb200_npair_loss`; with autograd on and `similarity` or `temperature` requiring grad, `n_pair_nll` / `total`
        carry a graph to both (backward: `lgb200_npair_loss_bwd`) and `n_pair_temperature` is the parameter itself, as
        in the reference.  Metrics as the reference's matcher_metrics in eval mode.  Any other conf.loss raises
        NotImplementedError, which TwoViewPipeline.loss treats as "skip" (two_view_pipeline.py:417-429)."""
        if self.conf.loss != "N_pair":
            raise NotImplementedError
        sim = pred["similarity"]
        if not sim.is_cuda:
            raise _abi.LightGlueB200Error("glue_factory_colon_b200.NearestNeighborMatcher.loss runs on CUDA tensors only")
        dev = sim.device
        gt = data["gt_assignment"].to(dev).to(torch.bool).contiguous()
        assert gt.shape == sim.shape, "gt_assignment must be [B, N, M]"
        if torch.is_grad_enabled() and (sim.requires_grad or self.temperature.requires_grad):
            nll, num = _NPairLossFn.apply(sim.to(torch.float32).contiguous(), self.temperature, gt)
            temperature = self.temperature[None]
        else:
            with torch.no_grad():
                nll, num, _, _ = _npair_loss(sim.to(torch.float32).contiguous(), float(self.temperature), gt)
            temperature = self.temperature.detach()[None]
        losses = {"n_pair_nll": nll, "total": nll, "num_matchable": num, "n_pair_temperature": temperature}
        if self.training:
            return losses, {}
        from .lightglue import LightGlue

        with torch.no_grad():
            return losses, LightGlue._matcher_metrics(pred, {"gt_matches0": data["gt_matches0"].to(dev)})


def _npair_loss(sim, temperature: float, gt):
    """lgb200_npair_loss -> (nll [B], num [B], workspace LR | LC, row counts [B, N])."""
    lib = _abi.load()
    B, N, M = sim.shape
    f32 = dict(device=sim.device, dtype=torch.float32)
    rows = torch.empty(2, B, N, **f32)
    ws = torch.empty(B * (N + M), **f32)
    check(lib.lgb200_npair_loss(ptr(sim), ptr(gt), B, N, M, temperature, ptr(ws), ptr(rows[0]), ptr(rows[1]),
                                torch.cuda.current_stream(sim.device).cuda_stream), "npair_loss")
    num = rows[1].sum(1).clamp(min=1.0)
    nll = -(rows[0].sum(1) / num) / 2
    return nll, num, ws, rows[1]


class _NPairLossFn(torch.autograd.Function):
    """(similarity fp32 [B, N, M], temperature) -> (nll [B], num_matchable [B], not differentiable)."""

    @staticmethod
    def forward(ctx, sim, temperature, gt):
        T = float(temperature)
        nll, num, ws, row_cnt = _npair_loss(sim, T, gt)
        ctx.save_for_backward(sim, gt, ws, row_cnt, num)
        ctx.T = T
        ctx.mark_non_differentiable(num)
        return nll, num

    @staticmethod
    def backward(ctx, g_nll, _):
        sim, gt, ws, row_cnt, num = ctx.saved_tensors
        lib = _abi.load()
        B, N, M = sim.shape
        f32 = dict(device=sim.device, dtype=torch.float32)
        coef = (-g_nll.to(torch.float32) / (2 * num)).contiguous()
        col_cnt, dtemp_rows = torch.empty(B, M, **f32), torch.empty(B, N, **f32)
        dsim = torch.empty(B, N, M, **f32) if ctx.needs_input_grad[0] else None
        check(lib.lgb200_npair_loss_bwd(ptr(sim), ptr(gt), B, N, M, ctx.T, ptr(ws), ptr(row_cnt), ptr(coef),
                                        ptr(col_cnt), ptr(dsim), ptr(dtemp_rows),
                                        torch.cuda.current_stream(sim.device).cuda_stream), "npair_loss_bwd")
        dtemp = dtemp_rows.sum().reshape(()) if ctx.needs_input_grad[1] else None
        return dsim, dtemp, None


def _planes(lib, t):
    """fp32 contiguous t -> (split-fp16 planes [2, *t.shape] of g t, 1 / g on the device), g from lgb200_split_dynamic."""
    p = torch.empty(2, *t.shape, device=t.device, dtype=torch.float16)
    inv = torch.empty(2, device=t.device, dtype=torch.float32)
    check(lib.lgb200_split_dynamic(ptr(t), t.numel(), ptr(p), ptr(inv), 0, None, 0,
                                   torch.cuda.current_stream(t.device).cuda_stream), "lgb200_split_dynamic")
    return p, inv[0]


def _pad8(x, rows: int):
    """fp32 x [B, r, c] zero-padded to [B, rows, c rounded up to 8] (element counts and fp16 leading dimensions that
    the split and the tensor-core products accept)."""
    x = x.to(torch.float32)
    cols = (x.shape[2] + 7) // 8 * 8
    if (rows, cols) == tuple(x.shape[1:]):
        return x.contiguous()
    return F.pad(x, (0, cols - x.shape[2], 0, rows - x.shape[1]))


class _SimilarityFn(torch.autograd.Function):
    """(descriptors0, descriptors1) -> the matcher's outputs in _OUT_KEYS order; only `similarity` = d0 . d1^T is
    differentiable.  Forward: the no-grad path's kernels, so every output is bit-equal to it."""

    @staticmethod
    def forward(ctx, matcher, data, d0, d1):
        out, counts = matcher._match(data, d0, d1)
        ctx.save_for_backward(d0, d1)
        ctx.counts = counts
        ctx.mark_non_differentiable(*(out[k] for k in _OUT_KEYS if k != "similarity"))
        return tuple(out[k] for k in _OUT_KEYS)

    @staticmethod
    def backward(ctx, *grads):
        d0, d1 = ctx.saved_tensors
        need0, need1 = ctx.needs_input_grad[2], ctx.needs_input_grad[3]
        B, N, D = d0.shape
        M = d1.shape[1]
        if N == 0 or M == 0:
            return None, None, torch.zeros_like(d0) if need0 else None, torch.zeros_like(d1) if need1 else None
        lib = _abi.load()
        dsim = grads[_OUT_KEYS.index("similarity")]
        x0, x1 = d0.detach(), d1.detach()
        counts = ctx.counts
        if (counts < torch.tensor([N, M], dtype=counts.dtype)).any():
            # similarity entries outside a pair's valid block are constants (0), and padded rows must not reach a product
            cnt = counts.to(d0.device)
            v0 = torch.arange(N, device=d0.device)[None] < cnt[:, :1]
            v1 = torch.arange(M, device=d0.device)[None] < cnt[:, 1:]
            dsim = torch.where(v0[:, :, None] & v1[:, None, :], dsim, 0.0)
            x0, x1 = torch.where(v0[..., None], x0, 0.0), torch.where(v1[..., None], x1, 0.0)
        Mp = (M + 7) // 8 * 8
        sp, si = _planes(lib, _pad8(dsim, N))
        g0 = g1 = None
        if need0:  # dSim . d1
            p1, i1 = _planes(lib, _pad8(x1, Mp))
            g0 = bmm3(sp, p1, si * i1)[:, :, :D].to(d0.dtype).contiguous()
        if need1:  # dSim^T . d0
            p0, i0 = _planes(lib, _pad8(x0, N))
            g1 = bmm3(sp.transpose(2, 3), p0, si * i0)[:, :M, :D].to(d1.dtype).contiguous()
        return None, None, g0, g1


__main_model__ = NearestNeighborMatcher
