"""Training path of the B200 LightGlue drop-in: forward that keeps what the backward needs, and the backward pass.

The reference trains through `LightGlue.forward` / `LightGlue.loss` with autograd (lightglue.py:484-498 collects every
layer's descriptors in training mode, :588-637 turns them into the deep-supervision NLL; train.py calls
`loss.backward()`).  Here the same contract is met by `torch.autograd.Function`s whose backward is written by hand:

  * `TransformerFn`  descriptors (+ every transformer / posenc / input_proj parameter) -> ref_descriptors0/1
    [B, n_layers, N, 256].  It keeps the two block inputs of every layer plus -- unless conf.checkpointed
    (lightglue.py:485-494) -- q / k / v / context (/ message); with conf.checkpointed those are recomputed in the
    backward pass with the same kernels.  The pre-LayerNorm activations are always recomputed (one GEMM).  Backward =
    the hand-written kernels of csrc/lg_bwd.cu: flash-attention backward (lgb200_attention_bwd /
    lgb200_attention_bwd_bf16), rotary / head-split backward incl. the gradient of the rotary angles
    (lgb200_heads_bwd), GELU . LayerNorm backward (lgb200_ln_gelu_bwd).  The layer loop, the keep / recompute policy
    and the posenc / input_proj tail are shared; the kernels and GEMMs of each block come from `_F32Blocks` or
    `_Bf16Blocks` (conf.train_precision).
  * `AssignFn`       MatchAssignment of one layer (lightglue.py:272-288) reduced to what NLLLoss reads
    (losses.py:6-26: the sum of log_assignment over the ground-truth matches and the two dustbin vectors).  Forward =
    the library's assignment + reduction kernels; backward = lgb200_assign_dsim (d similarity of the double softmax).
  * `LogAssignFn`    the training forward's log_assignment / matches / matching_scores of the last layer (lightglue.py:
    272-288, 294-319) with a graph for losses that read them; backward = lgb200_assign_bwd (any upstream gradient).
The staged keypoints are inputs of TransformerFn: with keypoints (scales, orientations) that require grad,
lgb200_posenc_bwd turns the rotary-angle gradient into their gradient (lightglue.py:28-40, 61-66).

conf.train_precision = "fp32" (the default): fp32-accurate whatever conf.precision says.  Forward = the library's
tensor-core kernels in the split-fp16 / three-MMA mode (lg_x3.cu / lg_x3_attn.cu).  Plain GEMMs of the backward pass
(dX = dY.W, dW = dY^T.X) go to cuBLAS -- they are library GEMMs with nothing to fuse -- as three fp16 tensor-core GEMMs
on split planes with fp32 accumulation (_Kern.mm3).  Gradients span a range (1e-8 ... 1e-2) that a fixed plane scaling
does not cover, so lgb200_split_dynamic scales every gradient tensor by its own power of two first.

conf.train_precision = "bf16" (mixed precision, the counterpart of the reference under torch.autocast(bfloat16)): the
forward runs the bf16 inference kernels exactly as the no-grad forward with precision="bf16" does (bf16 weight pack with
out_proj / to_out folded into the first FFN matrix, bf16 residual stream, rot16), so the training forward's outputs are
bit-equal to it; the backward recomputes the pre-LayerNorm activations in fp32 from the bf16 operands, runs the bf16
attention backward (one bf16 tcgen05 MMA per product) and does every plain GEMM as ONE bf16 cuBLAS product with fp32
output.  Gradients of the folded weights follow by the chain rule (see _Bf16Blocks.ffn_bwd).  `AssignFn` uses the bf16
assignment kernels.

Padded batches (data["num_keypoints0/1"], the counts padding.py produces): every kernel of the stack reads the
per-pair counts from the device `lens`, the staged descriptor and keypoint rows past the counts are zeroed (so the
padding's values cannot reach an output or a gradient), and AssignFn reduces each pair over its valid block only.  A
padded batch with counts trains like the same pairs run one at a time, un-padded (DESIGN.md 3.9).

CPU tensors raise as everywhere else in this package.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, List, Tuple

import numpy as np
import torch
from torch import nn

from . import _abi
from ._abi import BF16, EPI_HEADS, EPI_LN_GELU, EPI_ROWMAJOR, F32, F32X3, check, ptr
from .lightglue import weight_planes

LOG2E = 1.4426950408889634
Q_SCALE = LOG2E / math.sqrt(64.0)   # folded into q: the attention kernels work in the log2 domain
C_SCALE = math.sqrt(Q_SCALE)        # cross block: to_qk feeds both sides (lightglue.py:208)
AI, WI = 1.0 / 64.0, 1.0 / 256.0       # inverse plane scalings of activations / weights (LG_X3_EA, LG_X3_EW)
N_PARTIALS = 296                    # CTAs of lgb200_ln_gelu_bwd (2 per SM)
_X3_WEIGHTS = ("qkv_w", "so_w", "sf0_w", "sf3_w", "cqv_w", "co_w", "cf0_w", "cf3_w")
# packed Wqkv row r holds reference row _PERM[r] (lightglue.py:158: head*192 + d*3 + part -> part*256 + head*64 + d)
_PERM = torch.arange(768).view(4, 64, 3).permute(2, 0, 1).reshape(-1)


class _Kern:
    """Launch helpers for one (B, m, n) problem: S = 2B sequences padded to Lp rows, lens on the device.
    counts (host int array [B, 2], or None): per-pair valid counts of a padded batch; m / n stay the padded sizes."""

    def __init__(self, dev, B: int, m: int, n: int, counts=None):
        self.lib = _abi.load()
        check(self.lib.lgb200_device_ok(), "device check")
        self.dev, self.B, self.m, self.n = dev, B, m, n
        self.S = 2 * B
        self.Lp = max(128, ((max(m, n) + 127) // 128) * 128)
        self.T = self.S * self.Lp
        self.counts = counts
        self.lens = self.valid = None
        if counts is not None:  # one host -> device upload
            self.lens = torch.from_numpy(np.ascontiguousarray(counts, dtype=np.int32).reshape(-1)).to(dev)
            self.valid = (torch.arange(self.Lp, device=dev)[None] < self.lens[:, None]).reshape(-1)  # [T] bool
        elif m != self.Lp or n != self.Lp:
            self.lens = torch.tensor([m, n] * B, device=dev, dtype=torch.int32)

    def mask_rows(self, x):
        """Zeroes the rows of x [T, ...] past the per-pair counts, in place (nothing without counts)."""
        if self.valid is not None:
            x.view(self.T, -1).masked_fill_(~self.valid[:, None], 0)
        return x

    @property
    def st(self):
        return torch.cuda.current_stream(self.dev).cuda_stream

    def zeros(self, *shape):
        return torch.zeros(*shape, device=self.dev, dtype=torch.float32)

    def empty(self, *shape):
        return torch.empty(*shape, device=self.dev, dtype=torch.float32)

    def linear(self, epi, A0, W, b, N, K, A1=None, K0=None, scale=(1.0, 1.0, 1.0), resid=None, out=None, rot=None,
               n_rot=0, outp=(None, None, None), gamma=None, beta=None):
        check(self.lib.lgb200_linear(F32, epi, ptr(A0), ptr(A1), K if K0 is None else K0, ptr(W), ptr(b), self.T, N, K,
                                     ptr(self.lens), self.Lp, scale[0], scale[1], scale[2], ptr(resid), None, ptr(out),
                                     None, ptr(rot), None, n_rot, ptr(outp[0]), ptr(outp[1]), ptr(outp[2]), ptr(gamma),
                                     ptr(beta), self.st), "lgb200_linear")

    def linear3(self, epi, A0, W, b, N, K, A1=None, K0=None, scale=(1.0, 1.0, 1.0), resid=None, out=None, out32=None,
                rot=None, n_rot=0, outp=(None, None, None), gamma=None, beta=None):
        """The same layer in the fp32-accurate tensor-core mode (lg_x3.cu): A0 / A1 / W / out / outp are split-fp16
        planes, resid / out32 / rot fp32."""
        check(self.lib.lgb200_linear(F32X3, epi, ptr(A0), ptr(A1), K if K0 is None else K0, ptr(W), ptr(b), self.T, N, K,
                                     ptr(self.lens), self.Lp, scale[0], scale[1], scale[2], ptr(resid), None, ptr(out32),
                                     ptr(out), ptr(rot), None, n_rot, ptr(outp[0]), ptr(outp[1]), ptr(outp[2]), ptr(gamma),
                                     ptr(beta), self.st), "lgb200_linear (x3)")

    def planes(self, *shape):
        return torch.zeros(2, *shape, device=self.dev, dtype=torch.float16)

    def unsplit(self, p, *shape, out=None):
        """split planes (x * 64 = hi + lo) -> fp32"""
        n = p.numel() // 2
        out = torch.empty(n, device=self.dev, dtype=torch.float32) if out is None else out
        check(self.lib.lgb200_merge_rows(ptr(p), n, AI, ptr(out), self.st), "lgb200_merge_rows")
        return out.view(*shape) if shape else out

    def split(self, t):
        """fp32 -> split-fp16 planes [2][n] (x * 64 = hi + lo), the operand format of the LGB200_F32X3 kernels."""
        out = torch.empty(2, t.numel(), device=self.dev, dtype=torch.float16)
        check(self.lib.lgb200_split_rows(ptr(t), t.numel(), ptr(out), self.st), "lgb200_split_rows")
        return out

    def asplit(self, t):
        """activation [M, N] fp32 -> planes [2, M, N] (scale 64)"""
        return self.split(t).view(2, *t.shape)

    def gsplit(self, t, colsum: bool = False):
        """gradient [M, N] fp32 -> (planes [2, M, N] of g t, 1 / g on the device): lgb200_split_dynamic picks the power of
        two g per tensor (gradients have no fixed range).  colsum: also t.sum(0) (the bias gradient), from per-CTA
        partials of the same pass over t."""
        t = t.contiguous()
        out = torch.empty(2, *t.shape, device=self.dev, dtype=torch.float16)
        inv = torch.empty(2, device=self.dev, dtype=torch.float32)
        part = torch.empty(N_PARTIALS, t.shape[-1], device=self.dev, dtype=torch.float32) if colsum else None
        check(self.lib.lgb200_split_dynamic(ptr(t), t.numel(), ptr(out), ptr(inv), t.shape[-1] if colsum else 0, ptr(part),
                                            N_PARTIALS if colsum else 0, self.st), "lgb200_split_dynamic")
        return (out, inv[0], part.sum(0)) if colsum else (out, inv[0])

    @staticmethod
    def mm3(A, B, scale):
        """fp32-accurate A.B from plane pairs A [2, M, K], B [2, K, N] (views may be transposed): lo.hi + hi.lo + hi.hi as
        three fp16 tensor-core GEMMs with fp32 accumulation and fp32 output (cuBLAS: plain library GEMMs), times `scale`
        (the product of the inverse plane scalings; float or 0-dim device tensor)."""
        f32 = torch.float32
        r = torch.mm(A[1], B[0], out_dtype=f32)
        # beta = 1: accumulated in the GEMM epilogue; out = r: in place (without it ATen copies r into a new output first)
        torch.addmm(r, A[0], B[1], out_dtype=f32, out=r)
        torch.addmm(r, A[0], B[0], out_dtype=f32, out=r)
        return r.mul_(scale)

    def attention(self, qp, kp, vp, kv_xor, ctx):
        """Forward attention on the tensor cores in the fp32-accurate mode (lg_x3_attn.cu: split-fp16 operands, three
        tcgen05 MMAs per product, fp32 softmax) on the planes of the x3 projections -> the context's planes; ctx
        [T,256] receives it in fp32."""
        cp = torch.zeros(2, self.T, 256, device=self.dev, dtype=torch.float16)
        check(self.lib.lgb200_attention(F32X3, ptr(qp), ptr(kp), ptr(vp), self.S, self.Lp, ptr(self.lens), kv_xor, ptr(cp),
                                        self.st), "lgb200_attention")
        self.unsplit(cp, out=ctx)
        return cp

    def attention_bwd(self, q, k, v, ctx, dctx, kv_xor):
        """Flash-attention backward, fp32 dctx -> fp32 dq, dk, dv: lgb200_attention_bwd on fp32 q / k / v / ctx, or
        lgb200_attention_bwd_bf16 on the bf16 ones the bf16 forward kept."""
        name = "lgb200_attention_bwd_bf16" if q.dtype == torch.bfloat16 else "lgb200_attention_bwd"
        dq, dk, dv = self.empty(self.T * 256), self.empty(self.T * 256), self.empty(self.T * 256)
        n_ws = C.c_longlong(0)
        check(getattr(self.lib, name + "_workspace")(self.S, self.Lp, C.byref(n_ws)), name + "_workspace")
        ws = self.empty(n_ws.value)
        check(getattr(self.lib, name)(ptr(q), ptr(k), ptr(v), ptr(ctx), ptr(dctx), self.S, self.Lp, ptr(self.lens),
                                      kv_xor, ptr(dq), ptr(dk), ptr(dv), ptr(ws), self.st), name)
        return dq, dk, dv

    # ---- bf16 mixed-precision training (conf.train_precision = "bf16") ----

    def zeros16(self, *shape):
        return torch.zeros(*shape, device=self.dev, dtype=torch.bfloat16)

    def linear16(self, epi, A0, W, b, N, K, A1=None, K0=None, scale=(1.0, 1.0, 1.0), resid=None, out=None, out32=None,
                 rot16=None, n_rot=0, outp=(None, None, None), gamma=None, beta=None, lens=True):
        """lgb200_linear(LGB200_BF16): bf16 A0 / A1 / W / resid / out / outp, fp32 out32; lens=False: no counts."""
        check(self.lib.lgb200_linear(BF16, epi, ptr(A0), ptr(A1), K if K0 is None else K0, ptr(W), ptr(b), self.T, N, K,
                                     ptr(self.lens) if lens else None, self.Lp, scale[0], scale[1], scale[2], None,
                                     ptr(resid), ptr(out32), ptr(out), None, ptr(rot16), n_rot, ptr(outp[0]),
                                     ptr(outp[1]), ptr(outp[2]), ptr(gamma), ptr(beta), self.st), "lgb200_linear (bf16)")

    def attention16(self, q, k, v, kv_xor):
        ctx = self.zeros16(self.T, 256)
        check(self.lib.lgb200_attention(BF16, ptr(q), ptr(k), ptr(v), self.S, self.Lp, ptr(self.lens), kv_xor, ptr(ctx),
                                        self.st), "lgb200_attention (bf16)")
        return ctx

    def heads_bwd(self, dq, dk, dv, q, k, rot, n_parts, scales, dtheta):
        out = self.empty(self.T, 256 * n_parts)
        check(self.lib.lgb200_heads_bwd(ptr(dq), ptr(dk), ptr(dv), ptr(q), ptr(k), ptr(rot), self.S, self.Lp,
                                        ptr(self.lens), n_parts, scales[0], scales[1], scales[2], ptr(out), ptr(dtheta),
                                        self.st), "lgb200_heads_bwd")
        return out

    def ln_gelu_bwd(self, h, gamma, beta, da):
        dh, act, part = self.empty(self.T, 512), self.empty(self.T, 512), self.empty(N_PARTIALS, 1024)
        check(self.lib.lgb200_ln_gelu_bwd(ptr(h), ptr(gamma), ptr(beta), ptr(da), self.T, self.Lp, ptr(self.lens), ptr(dh),
                                          ptr(act), ptr(part), N_PARTIALS, self.st), "lgb200_ln_gelu_bwd")
        return dh, act, part.sum(0)

    def pack2(self, a0, a1, dtype=torch.float32):
        """[B, m, dim] / [B, n, dim] -> [T, dim] fp32 or bf16 (image img of pair b in the rows of sequence 2b + img),
        rows past the padded sizes and the per-pair counts zero."""
        dst = torch.zeros(self.T, a0.shape[-1], device=self.dev, dtype=dtype)
        f32 = dtype == torch.float32
        for img, src in ((0, a0), (1, a1)):
            src = src.to(torch.float32).contiguous()
            check(self.lib.lgb200_pack_rows(ptr(src), self.B, src.shape[1], src.shape[2], img, self.Lp,
                                            ptr(dst) if f32 else None, None if f32 else ptr(dst), self.st),
                  "lgb200_pack_rows")
        return self.mask_rows(dst)

    def unpack(self, x):
        xv = x.view(self.B, 2, self.Lp, x.shape[-1])
        return xv[:, 0, : self.m], xv[:, 1, : self.n]

    def posenc(self, geom, Wr, rot, rot16=None):
        """lgb200_posenc for both images: rot [T,64] fp32 (+ rot16 [T,32] packed fp16) from the staged keypoints."""
        for img, kk, cnt, sz in ((0, geom["k0"], self.m, geom["size0"]), (1, geom["k1"], self.n, geom["size1"])):
            check(self.lib.lgb200_posenc(ptr(kk), self.B, cnt, kk.shape[-1], ptr(sz), ptr(Wr), ptr(self.lens), img,
                                         self.Lp, ptr(rot), ptr(rot16), self.st), "lgb200_posenc")

    def posenc_bwd(self, geom, Wr, dtheta, need):
        """d staged keypoints [B, cnt, kdim] of image 0 / 1 from the rotary-angle gradient dtheta [T,32]
        (lgb200_posenc_bwd); None, and nothing launched, where need[img] is False."""
        out = []
        for img, kk, cnt, sz in ((0, geom["k0"], self.m, geom["size0"]), (1, geom["k1"], self.n, geom["size1"])):
            dk = None
            if need[img]:
                dk = torch.empty_like(kk)
                check(self.lib.lgb200_posenc_bwd(ptr(kk), self.B, cnt, kk.shape[-1], ptr(sz), ptr(Wr), ptr(self.lens),
                                                 img, self.Lp, ptr(dtheta), ptr(dk), self.st), "lgb200_posenc_bwd")
            out.append(dk)
        return out


def bmm3(A, B, scale):
    """Batched _Kern.mm3: fp32-accurate A.B from plane pairs A [2, b, M, K], B [2, b, K, N] (views may be transposed)
    as three fp16 tensor-core bmms with fp32 accumulation and fp32 output, times `scale` (float or 0-dim device
    tensor)."""
    f32 = torch.float32
    o = torch.bmm(A[1], B[0], out_dtype=f32)
    torch.baddbmm(o, A[0], B[1], out_dtype=f32, out=o)
    torch.baddbmm(o, A[0], B[0], out_dtype=f32, out=o)
    return o.mul_(scale)


def normalize_keypoints(kpts: torch.Tensor, size) -> torch.Tensor:
    """lightglue.py:28-40 (only needed for the gradient of posenc.Wr; the forward's posenc kernel has it fused)."""
    if size is None:
        size = 1 + kpts.max(-2).values - kpts.min(-2).values
    size = size.to(kpts)
    shift = size / 2
    scale = size.max(-1).values / 2
    return (kpts - shift[..., None, :]) / scale[..., None, None]


def _posenc_rows(k: _Kern, geom: Dict) -> torch.Tensor:
    """[T, kdim]: the rows posenc.Wr multiplies (lightglue.py:61-66) -- keypoints normalised as the posenc kernel does
    (over each pair's valid points when size is None), scale / orientation un-normalised (lightglue.py:436-454);
    rows past the per-pair counts zero."""
    kdim = geom["k0"].shape[-1]
    kn = k.zeros(k.T, kdim)
    knv = kn.view(k.B, 2, k.Lp, kdim)
    for img, kk, sz, cnt in ((0, geom["k0"], geom["size0"], k.m), (1, geom["k1"], geom["size1"], k.n)):
        if k.counts is None:
            knv[:, img, :cnt, :2] = normalize_keypoints(kk[..., :2], sz)
            knv[:, img, :cnt, 2:] = kk[..., 2:]
            continue
        valid = k.valid.view(k.B, 2, k.Lp)[:, img, :cnt, None]
        xy = kk[..., :2]
        if sz is None:  # extent of the valid points only (an empty side gives non-finite values, all masked)
            sz = 1 + torch.where(valid, xy, -math.inf).max(-2).values - torch.where(valid, xy, math.inf).min(-2).values
        knv[:, img, :cnt, :2] = torch.where(valid, normalize_keypoints(xy, sz), 0.0)
        knv[:, img, :cnt, 2:] = torch.where(valid, kk[..., 2:], 0.0)
    return kn


def transformer_params(model) -> List[Tuple[object, nn.Parameter]]:
    """(key, parameter) of everything TransformerFn differentiates, in a fixed order."""
    out: List[Tuple[object, nn.Parameter]] = []
    if isinstance(model.input_proj, nn.Linear):
        out += [("in_w", model.input_proj.weight), ("in_b", model.input_proj.bias)]
    out.append(("wr", model.posenc.Wr.weight))
    for i, lyr in enumerate(model.transformers):
        sa, ca = lyr.self_attn, lyr.cross_attn
        out += [
            ((i, "qkv_w"), sa.Wqkv.weight), ((i, "qkv_b"), sa.Wqkv.bias),
            ((i, "so_w"), sa.out_proj.weight), ((i, "so_b"), sa.out_proj.bias),
            ((i, "sf0_w"), sa.ffn[0].weight), ((i, "sf0_b"), sa.ffn[0].bias),
            ((i, "sln_g"), sa.ffn[1].weight), ((i, "sln_b"), sa.ffn[1].bias),
            ((i, "sf3_w"), sa.ffn[3].weight), ((i, "sf3_b"), sa.ffn[3].bias),
            ((i, "cqk_w"), ca.to_qk.weight), ((i, "cqk_b"), ca.to_qk.bias),
            ((i, "cv_w"), ca.to_v.weight), ((i, "cv_b"), ca.to_v.bias),
            ((i, "co_w"), ca.to_out.weight), ((i, "co_b"), ca.to_out.bias),
            ((i, "cf0_w"), ca.ffn[0].weight), ((i, "cf0_b"), ca.ffn[0].bias),
            ((i, "cln_g"), ca.ffn[1].weight), ((i, "cln_b"), ca.ffn[1].bias),
            ((i, "cf3_w"), ca.ffn[3].weight), ((i, "cf3_b"), ca.ffn[3].bias),
        ]
    return out


# ---- the transformer stack (lightglue.py:151-164, 193-222, 456-498) ------------------------------------------------
# _F32Blocks / _Bf16Blocks hold what depends on conf.train_precision -- the weight pack, the staging, the positional
# encoding and the kernels and GEMMs of one block forward and backward -- behind the same methods; TransformerFn owns
# the layer loop, the keep / recompute policy of conf.checkpointed and the posenc / input_proj tail.  A block's saved
# tuple starts with the attention operands (q, k, v, ctx) of the self block, (qk, v, ctx) of the cross block.


class _F32Blocks:
    """conf.train_precision = "fp32": the fp32-accurate tensor-core kernels on split-fp16 planes forward (lg_x3.cu /
    lg_x3_attn.cu), three fp16 tensor-core GEMMs on split planes for every plain GEMM of the backward (_Kern.mm3);
    fp32 residual stream.  Saved tuples end with the message: (q, k, v, ctx, msg) / (qk, v, ctx, msg), q / k / v fp32
    or None (not kept)."""

    def __init__(self, k: _Kern, model):
        self.k, self.model = k, model
        self.W = model._pack(F32, k.dev)
        for w in self.W["layers"]:  # split-fp16 planes of the weight matrices, cached with the pack (rebuilt with it)
            if "x3" not in w:
                w["x3"] = {name: weight_planes(w[name]) for name in _X3_WEIGHTS}

    def stage(self, desc0, desc1):
        """-> (x [T,256]: the first block input, the staged input of input_proj or None)"""
        k = self.k
        x = k.pack2(desc0, desc1)
        if not isinstance(self.model.input_proj, nn.Linear):
            return x, None
        out = k.zeros(k.T, 256)
        k.linear(EPI_ROWMAJOR, x, self.W["in_w"], self.W["in_b"], 256, x.shape[1], out=out)
        return out, x

    def posenc(self, geom):
        """self.rot: rotary angles [T,64] fp32 from the staged keypoints."""
        self.rot = self.k.zeros(self.k.T, 64)
        self.k.posenc(geom, self.W["wr"], self.rot)

    def self_attend(self, w, x, heads: bool = True):
        """-> (q, k, v, ctx, msg); q / k / v None unless `heads` (the backward kernels read them in fp32)."""
        k, T, wx = self.k, self.k.T, w["x3"]
        qp, kp, vp = k.planes(T * 256), k.planes(T * 256), k.planes(T * 256)
        k.linear3(EPI_HEADS, k.split(x), wx["qkv_w"], w["qkv_b"], 768, 256, scale=(Q_SCALE, 1.0, 1.0), rot=self.rot,
                  n_rot=2, outp=(qp, kp, vp))
        ctx = k.zeros(T, 256)
        cp = k.attention(qp, kp, vp, 0, ctx)
        msg = k.zeros(T, 256)
        k.linear3(EPI_ROWMAJOR, cp, wx["so_w"], w["so_b"], 256, 256, out32=msg)
        if not heads:
            return None, None, None, ctx, msg
        return k.unsplit(qp, T * 256), k.unsplit(kp, T * 256), k.unsplit(vp, T * 256), ctx, msg

    def cross_attend(self, w, x, heads: bool = True):
        k, T, wx = self.k, self.k.T, w["x3"]
        qp, vp = k.planes(T * 256), k.planes(T * 256)
        k.linear3(EPI_HEADS, k.split(x), wx["cqv_w"], w["cqv_b"], 512, 256, scale=(C_SCALE, 1.0, 1.0), n_rot=0,
                  outp=(qp, vp, None))
        ctx = k.zeros(T, 256)
        cp = k.attention(qp, qp, vp, 1, ctx)
        msg = k.zeros(T, 256)
        k.linear3(EPI_ROWMAJOR, cp, wx["co_w"], w["co_b"], 256, 256, out32=msg)
        if not heads:
            return None, None, ctx, msg
        return k.unsplit(qp, T * 256), k.unsplit(vp, T * 256), ctx, msg

    def ffn(self, w, pre: str, x, s):
        """x + ffn(cat[x, msg]) (lightglue.py:164, 220-221), msg = s[-1]."""
        k, wx = self.k, w["x3"]
        out = k.zeros(k.T, 256)
        hp = k.planes(k.T, 512)
        k.linear3(EPI_LN_GELU, k.split(x), wx[pre + "f0_w"], w[pre + "f0_b"], 512, 512, A1=k.split(s[-1]), K0=256,
                  gamma=w[pre + "ln_g"], beta=w[pre + "ln_b"], out=hp)
        k.linear3(EPI_ROWMAJOR, hp, wx[pre + "f3_w"], w[pre + "f3_b"], 256, 512, resid=x, out32=out)
        return out

    def ffn_bwd(self, i: int, w, pre: str, x, s, dy):
        """Backward of y = ffn(cat[x, out_proj(ctx)]) given dy [T,256] and the block's saved tuple s: (d x through the
        ffn, d ctx, parameter gradients incl. those of out_proj / to_out)."""
        k, wx = self.k, w["x3"]
        c, msg = s[-2:]
        h = k.zeros(k.T, 512)  # pre-LayerNorm activations, recomputed
        k.linear3(EPI_ROWMAJOR, k.split(x), wx[pre + "f0_w"], w[pre + "f0_b"], 512, 512, A1=k.split(msg), K0=256,
                  out32=h)
        dyp, dyi, b3 = k.gsplit(dy, colsum=True)
        da = k.mm3(dyp, wx[pre + "f3_w"], dyi * WI)
        dh, act, gsum = k.ln_gelu_bwd(h, w[pre + "ln_g"], w[pre + "ln_b"], da)
        g3 = k.mm3(dyp.transpose(1, 2), k.asplit(act), dyi * AI)
        dhp, dhi, b0 = k.gsplit(dh, colsum=True)
        dht = dhp.transpose(1, 2)
        g0 = torch.cat([k.mm3(dht, k.asplit(x), dhi * AI), k.mm3(dht, k.asplit(msg), dhi * AI)], 1)
        dcat = k.mm3(dhp, wx[pre + "f0_w"], dhi * WI)
        del h, dyp, dyi, da, dh, act, dhp, dhi, dht  # not held across the out_proj backward: keeps the peak memory down
        po = "so" if pre == "s" else "co"
        gw, gb, dc = self.proj_bwd(w, po + "_w", dcat[:, 256:].contiguous(), c)
        g = {
            pre + "f3_w": g3, pre + "f3_b": b3,
            pre + "ln_g": gsum[:512], pre + "ln_b": gsum[512:],
            pre + "f0_w": g0, pre + "f0_b": b0,
            po + "_w": gw, po + "_b": gb,
        }
        return dcat[:, :256], dc, g

    def proj_bwd(self, w, name: str, dy, x):
        """Backward of y = x W^T + b for the weight `name` ([N, K], planes in w["x3"]): (dy^T x, dy^T 1, dy W)."""
        k = self.k
        dyp, dyi, db = k.gsplit(dy, colsum=True)
        return k.mm3(dyp.transpose(1, 2), k.asplit(x), dyi * AI), db, k.mm3(dyp, w["x3"][name], dyi * WI)

    def input_proj_bwd(self, dx, xin):
        """(d input_proj.weight, d input_proj.bias, d its input) from dx [T,256] (lightglue.py:464-465)."""
        return dx.t() @ xin, dx.sum(0), dx @ self.W["in_w"]


def _mm16(a, b):
    """a . b as one bf16 tensor-core GEMM with fp32 accumulation and fp32 output (cuBLAS)."""
    return torch.mm(a.to(torch.bfloat16), b.to(torch.bfloat16), out_dtype=torch.float32)


class _Bf16Blocks:
    """conf.train_precision = "bf16": the bf16 inference kernels forward, with the arguments of the no-grad forward with
    precision="bf16" (bf16 pack with out_proj / to_out folded into the first FFN matrix, bf16 residual stream, rot16),
    one bf16 tensor-core GEMM with fp32 output for every plain GEMM of the backward.  Saved tuples: (q, k, v, ctx) /
    (qk, v, ctx), bf16."""

    def __init__(self, k: _Kern, model):
        self.k, self.model = k, model
        self.W = model._pack(BF16, k.dev)

    def stage(self, desc0, desc1):
        """-> (x [T,256] bf16: the first block input, the staged input of input_proj or None)"""
        k = self.k
        x = k.pack2(desc0, desc1, torch.bfloat16)
        if not isinstance(self.model.input_proj, nn.Linear):
            return x, None
        out = k.zeros16(k.T, 256)
        k.linear16(EPI_ROWMAJOR, x, self.W["in_w"], self.W["in_b"], 256, x.shape[1], out=out, lens=False)
        return out, x

    def posenc(self, geom):
        """self.rot: fp32 angles [T,64] for lgb200_heads_bwd; self.rot16 [T,32]: packed fp16 cos / sin for the
        forward's QKV epilogue (one call)."""
        k = self.k
        self.rot = k.zeros(k.T, 64)
        self.rot16 = torch.zeros(k.T, 32, device=k.dev, dtype=torch.int32)
        k.posenc(geom, self.W["wr"], self.rot, self.rot16)

    def self_attend(self, w, x, heads: bool = True):
        """Self block up to the context, as the no-grad bf16 forward runs it: (q, k, v, ctx), kept whatever `heads`."""
        k = self.k
        q, kk, v = k.zeros16(k.T * 256), k.zeros16(k.T * 256), k.zeros16(k.T * 256)
        k.linear16(EPI_HEADS, x, w["qkv_w"], w["qkv_b"], 768, 256, scale=(Q_SCALE, 1.0, 1.0), rot16=self.rot16, n_rot=2,
                   outp=(q, kk, v))
        return q, kk, v, k.attention16(q, kk, v, 0)

    def cross_attend(self, w, x, heads: bool = True):
        k = self.k
        qk, v = k.zeros16(k.T * 256), k.zeros16(k.T * 256)
        k.linear16(EPI_HEADS, x, w["cqv_w"], w["cqv_b"], 512, 256, scale=(C_SCALE, 1.0, 1.0), rot16=self.rot16, n_rot=0,
                   outp=(qk, v, None))
        return qk, v, k.attention16(qk, qk, v, 1)

    def ffn(self, w, pre: str, x, s):
        """x + ffn(cat[x, out_proj(ctx)]) with out_proj folded into the first FFN matrix, ctx = s[-1]: a new bf16
        tensor."""
        k = self.k
        hid = k.zeros16(k.T, 512)
        k.linear16(EPI_LN_GELU, x, w[pre + "f0_w"], w[pre + "f0_b"], 512, 512, A1=s[-1], K0=256, gamma=w[pre + "ln_g"],
                   beta=w[pre + "ln_b"], out=hid)
        out = x.clone()  # (the no-grad forward updates its residual stream in place; the block input is kept here)
        k.linear16(EPI_ROWMAJOR, hid, w[pre + "f3_w"], w[pre + "f3_b"], 256, 512, resid=out, out=out)
        return out

    def ffn_bwd(self, i: int, w, pre: str, x, s, dy):
        """Backward of y = ffn(cat[x, proj(c)]) in the folded form h = [W1x | W1m.Wo].cat[x, c] + (b1 + W1m.bo), given
        dy [T,256] and the saved tuple s (c = s[-1]): (d x through the ffn, d c, parameter gradients incl. those of
        proj).  With G = dh^T c (the [512,256] block of d W1') and gb = sum dh: dW1m = G Wo^T + gb bo^T (W1m enters the
        folded bias too), dWo = W1m^T G, dbo = W1m^T gb, db1 = gb."""
        k, c = self.k, s[-1]
        blk = self.model.transformers[i]
        ffn0, proj = (blk.self_attn.ffn[0], blk.self_attn.out_proj) if pre == "s" else \
            (blk.cross_attn.ffn[0], blk.cross_attn.to_out)
        h = k.empty(k.T, 512)  # pre-LayerNorm activations, recomputed in fp32 from the same bf16 operands
        k.linear16(EPI_ROWMAJOR, x, w[pre + "f0_w"], w[pre + "f0_b"], 512, 512, A1=c, K0=256, out32=h)
        dy16 = dy.to(torch.bfloat16)
        da = _mm16(dy16, w[pre + "f3_w"])
        dh, act, gsum = k.ln_gelu_bwd(h, w[pre + "ln_g"], w[pre + "ln_b"], da)
        dh16 = dh.to(torch.bfloat16)
        g3 = _mm16(dy16.t(), act)
        gx, G = _mm16(dh16.t(), x), _mm16(dh16.t(), c)
        dcat = _mm16(dh16, w[pre + "f0_w"])
        gb = dh.sum(0)
        d = proj.weight.shape[0]
        w1m, wo, bo = ffn0.weight.detach()[:, d:], proj.weight.detach(), proj.bias.detach()
        po = "so" if pre == "s" else "co"
        g = {
            pre + "f3_w": g3, pre + "f3_b": dy.sum(0),
            pre + "ln_g": gsum[:512], pre + "ln_b": gsum[512:],
            pre + "f0_w": torch.cat([gx, G @ wo.t() + torch.outer(gb, bo)], 1), pre + "f0_b": gb,
            po + "_w": w1m.t() @ G, po + "_b": w1m.t() @ gb,
        }
        return dcat[:, :256], dcat[:, 256:].contiguous(), g

    def proj_bwd(self, w, name: str, dy, x):
        """Backward of y = x W^T + b with bf16 x / W = w[name]: (dy^T x, dy^T 1, dy W)."""
        dy16 = dy.to(torch.bfloat16)
        return _mm16(dy16.t(), x), dy.sum(0), _mm16(dy16, w[name])

    def input_proj_bwd(self, dx, xin):
        """(d input_proj.weight, d input_proj.bias, d its input) from dx [T,256] (lightglue.py:464-465)."""
        return dx.t() @ xin.float(), dx.sum(0), dx @ self.model.input_proj.weight.detach()


class TransformerFn(torch.autograd.Function):
    """ref_descriptors0/1 = all layers' outputs of the transformer stack (lightglue.py:456-498) in conf.train_precision:
    fp32, or bf16 as the no-grad bf16 forward returns them."""

    @staticmethod
    def forward(ctx, model, geom: Dict, desc0, desc1, k0, k1, *params):
        """k0 / k1 [B, m / n, kdim]: the staged keypoint rows (coordinates, plus scale and orientation with
        add_scale_ori) -- inputs, so that their gradient reaches whatever the caller built them from."""
        B, m, _ = desc0.shape
        n = desc1.shape[1]
        geom = dict(geom, k0=k0, k1=k1)
        k = _Kern(desc0.device, B, m, n, geom.get("counts"))
        P = (_Bf16Blocks if model._train_bf16() else _F32Blocks)(k, model)
        x, xin = P.stage(desc0, desc1)
        P.posenc(geom)
        # conf.checkpointed (lightglue.py:485-494): keep only the block inputs and recompute q / k / v / context /
        # message in the backward pass (26 x T KB per layer less in fp32); otherwise they are kept, as autograd would
        keep = not bool(model.conf.checkpointed)
        xs_in, xs_mid, outs, kept = [], [], [], []
        for w in P.W["layers"]:
            xs_in.append(x)
            sa = P.self_attend(w, x, heads=keep)
            x = P.ffn(w, "s", x, sa)
            xs_mid.append(x)
            ca = P.cross_attend(w, x, heads=keep)
            x = P.ffn(w, "c", x, ca)
            outs.append(x)
            kept.append((sa, ca) if keep else None)
        ctx.P, ctx.geom = P, geom
        ctx.xs_in, ctx.xs_mid, ctx.xin, ctx.kept = xs_in, xs_mid, xin, kept
        ctx.keys = [key for key, _ in transformer_params(model)]
        r0 = torch.stack([k.unpack(o)[0] for o in outs], 1)
        r1 = torch.stack([k.unpack(o)[1] for o in outs], 1)
        return r0, r1

    @staticmethod
    def backward(ctx, g0, g1):
        P, geom = ctx.P, ctx.geom
        k, rot = P.k, P.rot
        dx = k.zeros(k.T, 256)
        dtheta = k.zeros(k.T, 32)
        grads: Dict[object, torch.Tensor] = {}
        perm = _PERM.to(dx.device)
        for i in reversed(range(len(ctx.xs_in))):
            w = P.W["layers"][i]
            dx = dx + k.pack2(g0[:, i], g1[:, i])
            x_in, x_mid = ctx.xs_in[i], ctx.xs_mid[i]
            # ---- cross block (lightglue.py:193-222) ----
            s = ctx.kept[i][1] if ctx.kept[i] is not None else P.cross_attend(w, x_mid)
            qk, v, c = s[:3]  # (unpacked here: releases the previous block's v / c before the FFN backward)
            dxa, dc, g = P.ffn_bwd(i, w, "c", x_mid, s, dx)
            for name, val in g.items():
                grads[(i, name)] = val
            dq, dk, dv = k.attention_bwd(qk, qk, v, c, dc, 1)
            dqv = k.heads_bwd(dq, dk, dv, None, None, None, 2, (C_SCALE, 1.0, 1.0), None)
            gw, gb, dxp = P.proj_bwd(w, "cqv_w", dqv, x_mid)
            grads[(i, "cqk_w")], grads[(i, "cv_w")] = gw[:256], gw[256:]
            grads[(i, "cqk_b")], grads[(i, "cv_b")] = gb[:256], gb[256:]
            dxm = dx + dxa + dxp
            # ---- self block (lightglue.py:151-164) ----
            s = ctx.kept[i][0] if ctx.kept[i] is not None else P.self_attend(w, x_in)
            ctx.kept[i] = None
            q, kk, v, c = s[:4]
            dxa, dc, g = P.ffn_bwd(i, w, "s", x_in, s, dxm)
            for name, val in g.items():
                grads[(i, name)] = val
            dq, dk, dv = k.attention_bwd(q, kk, v, c, dc, 0)
            dqkv = k.heads_bwd(dq, dk, dv, q.float(), kk.float(), rot, 3, (Q_SCALE, 1.0, 1.0), dtheta)
            gw = torch.empty(768, 256, device=dqkv.device, dtype=torch.float32)
            gb = torch.empty(768, device=dqkv.device, dtype=torch.float32)
            gw[perm], gb[perm], dxp = P.proj_bwd(w, "qkv_w", dqkv, x_in)
            grads[(i, "qkv_w")], grads[(i, "qkv_b")] = gw, gb
            dx = dxm + dxa + dxp
        # positional encoding: theta = Wr . normalised keypoints (lightglue.py:61-66)
        grads["wr"] = dtheta.t() @ _posenc_rows(k, geom)
        need = ctx.needs_input_grad
        gk0, gk1 = k.posenc_bwd(geom, P.W["wr"], dtheta, need[4:6])
        if ctx.xin is not None:  # input_proj (lightglue.py:464-465)
            grads["in_w"], grads["in_b"], dx = P.input_proj_bwd(dx, ctx.xin)
        gd0, gd1 = k.unpack(k.mask_rows(dx))
        return (None, None, gd0.contiguous() if need[2] else None, gd1.contiguous() if need[3] else None, gk0, gk1,
                *[grads[key] if need[6 + j] else None for j, key in enumerate(ctx.keys)])


class AssignFn(torch.autograd.Function):
    """MatchAssignment `layer` on (d0, d1) reduced to the inputs of NLLLoss: pos_sum [B] = sum of log_assignment over
    the ground-truth matches, dust0 [B,m] / dust1 [B,n] = the dustbin column / row (differentiable); pos_cnt, row_exp,
    row_arg, col_arg as in lgb200_loss_reduce (not differentiable).  counts (device int32 [2B] or None): per-pair valid
    counts of a padded batch -- every pair is then reduced over its valid block (lgb200_loss_reduce_ragged semantics)
    and the gradients are exactly 0 outside it; gt must be False outside it."""

    @staticmethod
    def forward(ctx, model, layer: int, gt, counts, d0, d1, fp_w, fp_b, m_w, m_b):
        lib = _abi.load()
        keep: Dict = {}
        pos_sum, pos_cnt, row_exp, row_arg, col_arg, dust0, dust1, _ = model._log_assignment_of(
            lib, BF16 if model._train_bf16() else F32X3, d0, d1, layer, gt, keep=keep, counts=counts)
        ctx.save_for_backward(d0, d1, fp_w, m_w, gt, keep["z"], keep["lse"])
        ctx.counts = counts
        ctx.Lp = keep["Lp"]
        # what the backward recomputes the similarity from: x3 mode, the split planes of final_proj(desc) / 4 (33 MB at
        # 8 x 2048, recomputed on tcgen05); bf16, final_proj(desc) / 4 as the forward's kernels computed it
        ctx.md_planes, ctx.md16, ctx.lens = keep["md_planes"], keep["md16"], keep["lens"]
        ctx.mark_non_differentiable(pos_cnt, row_exp, row_arg, col_arg)
        return pos_sum, dust0.contiguous(), dust1.contiguous(), pos_cnt, row_exp, row_arg, col_arg

    @staticmethod
    def backward(ctx, g_pos, g_d0, g_d1, *_):
        d0, d1, fp_w, m_w, gt, z, lse = ctx.saved_tensors
        lib = _abi.load()
        B, m, _ = d0.shape
        n = d1.shape[1]
        Lp = ctx.Lp
        dev = d0.device
        x0, x1 = d0.to(torch.float32), d1.to(torch.float32)
        st = torch.cuda.current_stream(dev).cuda_stream
        sim, md = _assign_similarity(lib, st, x0, x1, ctx.md_planes, ctx.md16, ctx.lens, Lp)
        g = (g_pos if g_pos is not None else torch.zeros(B, device=dev)).to(torch.float32).contiguous()
        r = (g[:, None] * gt.sum(2)).contiguous()
        c = (g[:, None] * gt.sum(1)).contiguous()
        counts = ctx.counts
        if counts is None:
            check(lib.lgb200_assign_dsim(ptr(sim), B, m, n, ptr(lse), Lp, ptr(gt), ptr(g), ptr(r), ptr(c), st),
                  "assign_dsim")
        else:  # exact zeros outside every pair's valid block
            check(lib.lgb200_assign_dsim_ragged(ptr(sim), B, m, n, ptr(lse), Lp, ptr(counts), ptr(gt), ptr(g), ptr(r),
                                                ptr(c), st), "assign_dsim_ragged")
        zv = z.view(B, 2, Lp)
        z0, z1 = zv[:, 0, :m], zv[:, 1, :n]
        gd0 = g_d0 if g_d0 is not None else torch.zeros_like(z0)
        gd1 = g_d1 if g_d1 is not None else torch.zeros_like(z1)
        # la = ... + logsigmoid(z0_i) + logsigmoid(z1_j) inside, logsigmoid(-z) in the dustbins (lightglue.py:262-267)
        dz0 = r * torch.sigmoid(-z0) - gd0 * torch.sigmoid(z0)
        dz1 = c * torch.sigmoid(-z1) - gd1 * torch.sigmoid(z1)
        return (None, None, None, None,
                *_assign_input_grads(lib, st, sim, dz0, dz1, x0, x1, fp_w, m_w, md, ctx.md_planes, Lp, counts))


def _assign_similarity(lib, st, x0, x1, mdp, md16, lens, Lp):
    """The similarity [B,m,n] fp32 of MatchAssignment (lightglue.py:281-284) recomputed for a backward pass from what
    the forward kept -- the split planes mdp of final_proj(desc) / 4 in the x3 mode, or md16 = final_proj(desc) / 4 of the
    bf16 forward -> (sim, md); md = (md0, md1) of the bf16 forward for the d md products, None in the x3 mode."""
    B, m, _ = x0.shape
    n = x1.shape[1]
    f32 = torch.float32
    if md16 is not None:  # bf16: the similarity as one bf16 bmm with fp32 output (bf16 output: ~0.1 at |sim| ~ 30)
        mv = md16.view(B, 2, Lp, 256)
        md0, md1 = mv[:, 0, :m], mv[:, 1, :n]
        return torch.bmm(md0, md1.transpose(1, 2), out_dtype=f32).contiguous(), (md0, md1)
    sim = torch.empty(B, Lp, Lp, device=x0.device, dtype=f32)
    check(lib.lgb200_x3_similarity(ptr(mdp), B, Lp, ptr(lens), ptr(sim), st), "x3_similarity")
    return sim[:, :m, :n].contiguous(), None


def _assign_input_grads(lib, st, sim, dz0, dz1, x0, x1, fp_w, m_w, md, mdp, Lp, counts):
    """Backward of MatchAssignment (lightglue.py:272-288) from d sim [B,m,n] (in sim) and the matchability logits'
    gradients dz0 [B,m] / dz1 [B,n] to (d desc0, d desc1, d final_proj.weight, d final_proj.bias, d matchability.weight,
    d matchability.bias).  md / mdp as returned by / given to _assign_similarity; counts: rows past them get 0."""
    B, m, n = sim.shape
    dev = sim.device
    f32 = torch.float32
    if md is not None:  # bf16
        md0, md1 = md
        s16 = sim.to(torch.bfloat16)
        dmd0 = torch.bmm(s16, md1, out_dtype=f32)
        dmd1 = torch.bmm(s16.transpose(1, 2), md0, out_dtype=f32)
    else:  # three fp16 tensor-core products per GEMM, as _Kern.mm3
        sp = torch.empty(2, B, m, n, device=dev, dtype=torch.float16)
        inv = torch.empty(2, device=dev, dtype=torch.float32)
        check(lib.lgb200_split_dynamic(ptr(sim), sim.numel(), ptr(sp), ptr(inv), 0, None, 0, st), "lgb200_split_dynamic")
        mv = mdp.view(2, B, 2, Lp, 256)
        mp0, mp1 = mv[:, :, 0, :m], mv[:, :, 1, :n]
        dmd0 = bmm3(sp, mp1, inv[0] * AI)
        dmd1 = bmm3(sp.transpose(2, 3), mp0, inv[0] * AI)
    if counts is not None:  # rows past the counts: no matchability gradient (their z is not a keypoint's)
        v0 = torch.arange(m, device=dev)[None] < counts[0::2, None]
        v1 = torch.arange(n, device=dev)[None] < counts[1::2, None]
        dz0, dz1 = torch.where(v0, dz0, 0.0), torch.where(v1, dz1, 0.0)
    mw = m_w.reshape(1, 1, 256)
    gx0 = 0.25 * (dmd0 @ fp_w) + dz0[..., None] * mw
    gx1 = 0.25 * (dmd1 @ fp_w) + dz1[..., None] * mw
    if counts is not None:
        gx0, gx1 = torch.where(v0[..., None], gx0, 0.0), torch.where(v1[..., None], gx1, 0.0)
    g_fp_w = 0.25 * (dmd0.reshape(-1, 256).t() @ x0.reshape(-1, 256) + dmd1.reshape(-1, 256).t() @ x1.reshape(-1, 256))
    g_fp_b = 0.25 * (dmd0.sum((0, 1)) + dmd1.sum((0, 1)))
    g_m_w = ((dz0[..., None] * x0).sum((0, 1)) + (dz1[..., None] * x1).sum((0, 1))).reshape(m_w.shape)
    g_m_b = (dz0.sum() + dz1.sum()).reshape(1)
    return gx0, gx1, g_fp_w, g_fp_b, g_m_w, g_m_b


class LogAssignFn(torch.autograd.Function):
    """The training forward's tail: MatchAssignment `layer` (lightglue.py:272-288) and filter_matches (:294-319) on the
    last layer's descriptors d0 / d1 -> (log_assignment [B,m+1,n+1], matches0, matches1, matching_scores0,
    matching_scores1), with the kernels and arguments the step used before it had a graph, so the values are the same
    bits.  log_assignment and the matching scores are differentiable w.r.t. d0, d1 and the final_proj / matchability
    parameters; the matches are not.  counts (device int32 [2B] or None): per-pair valid counts of a padded batch.

    Backward: G = d loss / d log_assignment, plus the matching-score terms as autograd differentiates the reference's
    filter_matches -- ms0_i = exp(la[i, m0_i]) on mutual rows, ms1_j = exp(la[m1_j, j]) on mutual columns (below the
    threshold too), 0 elsewhere -- then lgb200_assign_bwd on the recomputed similarity, then AssignFn's tail.  The
    forward keeps z, lse, the filter workspace (the packed row / column maxima) and what the similarity is recomputed
    from (AssignFn's choice); nothing runs unless the loss reads these outputs."""

    @staticmethod
    def forward(ctx, model, layer: int, counts, d0, d1, fp_w, fp_b, m_w, m_b):
        lib = _abi.load()
        keep: Dict = {}
        if model._train_bf16():
            scores, m0, m1, ms0, ms1 = model._assign_match_bf16(lib, d0, d1, layer, counts, keep=keep)
        else:  # (the fp32-accurate tensor-core kernels, as the rest of the training forward)
            dev = d0.device
            B, m, _ = d0.shape
            n = d1.shape[1]
            model._log_assignment_of(lib, F32X3, d0, d1, layer, None, keep=keep, counts=counts)
            scores = keep["scores"]
            m0 = torch.empty(B, m, device=dev, dtype=torch.int64)
            m1 = torch.empty(B, n, device=dev, dtype=torch.int64)
            ms0 = torch.empty(B, m, device=dev, dtype=torch.float32)
            ms1 = torch.empty(B, n, device=dev, dtype=torch.float32)
            keep["fm_ws"] = torch.empty(B * (m + n + 2), device=dev, dtype=torch.int64)
            st = torch.cuda.current_stream(dev).cuda_stream
            check(lib.lgb200_filter_matches(ptr(scores), B, m + 1, n + 1, ptr(keep["lens"]),
                                            float(model.conf.filter_threshold), None, None, 0, m, n, ptr(m0), ptr(m1),
                                            ptr(ms0), ptr(ms1), ptr(keep["fm_ws"]), 0, st), "filter_matches")
        ctx.save_for_backward(d0, d1, fp_w, m_w, keep["z"], keep["lse"], keep["fm_ws"])
        ctx.counts, ctx.Lp = counts, keep["Lp"]
        ctx.md_planes, ctx.md16, ctx.lens = keep["md_planes"], keep["md16"], keep["lens"]
        ctx.mark_non_differentiable(m0, m1)
        return scores, m0, m1, ms0, ms1

    @staticmethod
    def backward(ctx, g_la, _g_m0, _g_m1, g_ms0, g_ms1):
        d0, d1, fp_w, m_w, z, lse, fm_ws = ctx.saved_tensors
        lib = _abi.load()
        B, m, _ = d0.shape
        n = d1.shape[1]
        Lp, counts = ctx.Lp, ctx.counts
        dev = d0.device
        st = torch.cuda.current_stream(dev).cuda_stream
        G = torch.zeros(B, m + 1, n + 1, device=dev, dtype=torch.float32)
        if g_la is not None:
            G.copy_(g_la)
        if g_ms0 is not None or g_ms1 is not None:
            # the raw mutual pairs: lgb200_filter_matches again on the packed maxima the forward left in fm_ws, with a
            # threshold below every score (scores are >= 0), so every mutual pair is a match
            mm0 = torch.empty(B, m, device=dev, dtype=torch.int64)
            mm1 = torch.empty(B, n, device=dev, dtype=torch.int64)
            ms0 = torch.empty(B, m, device=dev, dtype=torch.float32)
            ms1 = torch.empty(B, n, device=dev, dtype=torch.float32)
            check(lib.lgb200_filter_matches(None, B, m + 1, n + 1, ptr(ctx.lens), -1.0, None, None, 0, m, n, ptr(mm0),
                                            ptr(mm1), ptr(ms0), ptr(ms1), ptr(fm_ws), 1, st), "filter_matches")
            bi = torch.arange(B, device=dev)[:, None]
            # rows, then columns: two index_put_ calls, each with distinct indices, so sums into one entry of G have a
            # fixed order (a row / column without a mutual pair adds an exact 0)
            if g_ms0 is not None:
                ii = torch.arange(m, device=dev)[None].expand(B, m)
                G.index_put_((bi.expand(B, m), ii, mm0.clamp(min=0)), torch.where(mm0 >= 0, g_ms0 * ms0, 0.0),
                             accumulate=True)
            if g_ms1 is not None:
                jj = torch.arange(n, device=dev)[None].expand(B, n)
                G.index_put_((bi.expand(B, n), mm1.clamp(min=0), jj), torch.where(mm1 >= 0, g_ms1 * ms1, 0.0),
                             accumulate=True)
        x0, x1 = d0.to(torch.float32), d1.to(torch.float32)
        sim, md = _assign_similarity(lib, st, x0, x1, ctx.md_planes, ctx.md16, ctx.lens, Lp)
        dz0 = torch.empty(B, m, device=dev, dtype=torch.float32)
        dz1 = torch.empty(B, n, device=dev, dtype=torch.float32)
        n_ws = C.c_longlong(0)
        check(lib.lgb200_assign_bwd_workspace(B, m, n, C.byref(n_ws)), "lgb200_assign_bwd_workspace")
        ws = torch.empty(n_ws.value, device=dev, dtype=torch.float32)
        check(lib.lgb200_assign_bwd(ptr(G), ptr(sim), B, m, n, ptr(lse), Lp, ptr(counts), ptr(z), ptr(dz0), ptr(dz1),
                                    ptr(ws), st), "lgb200_assign_bwd")
        return (None, None, None,
                *_assign_input_grads(lib, st, sim, dz0, dz1, x0, x1, fp_w, m_w, md, ctx.md_planes, Lp, counts))


def wants_grad(model, data=None) -> bool:
    """Training step: module in training mode, autograd on, something to differentiate."""
    if not (model.training and torch.is_grad_enabled()):
        return False
    if any(p.requires_grad for p in model.parameters()):
        return True
    return data is not None and any(
        isinstance(data.get(kk), torch.Tensor) and data[kk].requires_grad
        for kk in ("descriptors0", "descriptors1", "keypoints0", "keypoints1", "scales0", "scales1", "oris0", "oris1"))
