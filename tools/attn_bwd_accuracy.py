"""Attention backward (lgb200_attention_bwd) against float64 autograd at long sequences: relative error (norm-wise and
largest entry) of dQ / dK / dV.  usage: attn_bwd_accuracy.py [S] [Lp]"""
import ctypes
import math
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from glue_factory_colon_b200 import _abi  # noqa: E402
from glue_factory_colon_b200._abi import ptr  # noqa: E402

S = int(sys.argv[1]) if len(sys.argv) > 1 else 2
Lp = int(sys.argv[2]) if len(sys.argv) > 2 else 2048
dev = torch.device("cuda:0")
lib = _abi.load()
g = torch.Generator().manual_seed(1)
q = (torch.randn(S, 4, Lp, 64, generator=g) * 0.6).to(dev)
k = (torch.randn(S, 4, Lp, 64, generator=g) * 0.6).to(dev)
v = (torch.randn(S, 4, Lp, 64, generator=g) + 0.5).to(dev)   # non-zero mean: same-sign sums show accumulator rounding
dctx = (torch.randn(S, Lp, 256, generator=g) * 1e-3 + 5e-4).to(dev)
qd, kd, vd = (t.double().requires_grad_(True) for t in (q, k, v))   # float64 on the GPU
a = torch.softmax(qd @ kd.transpose(-1, -2) * math.log(2.0), -1)
ctx_ref = (a @ vd).permute(0, 2, 1, 3).reshape(S, Lp, 256)
(ctx_ref * dctx.double()).sum().backward()
st = torch.cuda.current_stream(dev).cuda_stream
ctx = torch.zeros(S, Lp, 256, device=dev)
assert lib.lgb200_attention(_abi.F32, ptr(q), ptr(k), ptr(v), S, Lp, None, 0, ptr(ctx), st) == 0
dq, dk, dv = (torch.empty(S, 4, Lp, 64, device=dev) for _ in range(3))
n_ws = ctypes.c_longlong(0)
assert lib.lgb200_attention_bwd_workspace(S, Lp, ctypes.byref(n_ws)) == 0
ws = torch.empty(n_ws.value, device=dev)
assert lib.lgb200_attention_bwd(ptr(q), ptr(k), ptr(v), ptr(ctx), ptr(dctx), S, Lp, None, 0, ptr(dq), ptr(dk), ptr(dv),
                                ptr(ws), st) == 0
for name, got, ref in (("dq", dq, qd.grad), ("dk", dk, kd.grad), ("dv", dv, vd.grad)):
    d = got.double() - ref
    print(f"S={S} Lp={Lp} {name}: norm-wise {float(d.norm() / ref.norm()):.2e}  max |d| / max |ref| {float(d.abs().max() / ref.abs().max()):.2e}"
          f"  mean signed d / mean |ref| {float(d.mean() / ref.abs().mean()):+.2e}")
