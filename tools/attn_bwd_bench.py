"""Attention backward kernels alone: S sequences x 4 heads x Lp keypoints.  Two arms, timed alternately on the same
inputs: the fp32 entry lgb200_attention_bwd (csrc/lg_bwd.cu -> the x3 tcgen05 kernel) and the bf16 entry
lgb200_attention_bwd_bf16 (the same kernel template on bf16 operands, fed by the bf16 forward).  Prints ms per call and
the useful TFLOP/s on one product count for both (8 tile products of 2.Lp^2.64 per head: 1 statistics + 3 dQ +
4 dK/dV), and the card's name and power limit.  Usage: python tools/attn_bwd_bench.py [S] [Lp] [reps]"""
import ctypes
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from glue_factory_colon_b200 import _abi  # noqa: E402
from glue_factory_colon_b200._abi import ptr  # noqa: E402

S = int(sys.argv[1]) if len(sys.argv) > 1 else 16
Lp = int(sys.argv[2]) if len(sys.argv) > 2 else 2048
REPS = int(sys.argv[3]) if len(sys.argv) > 3 else 10
dev = torch.device("cuda:0")
lib = _abi.load()
g = torch.Generator().manual_seed(0)
q, k = ((torch.randn(S, 4, Lp, 64, generator=g) * 0.6).to(dev) for _ in range(2))
v = torch.randn(S, 4, Lp, 64, generator=g).to(dev)
dctx = torch.randn(S, Lp, 256, generator=g).to(dev)
ctx = torch.zeros(S, Lp, 256, device=dev)
st = torch.cuda.current_stream(dev).cuda_stream
assert lib.lgb200_attention(_abi.F32, ptr(q), ptr(k), ptr(v), S, Lp, None, 0, ptr(ctx), st) == 0
dq, dk, dv = (torch.empty(S, 4, Lp, 64, device=dev) for _ in range(3))
n_ws = ctypes.c_longlong(0)
assert lib.lgb200_attention_bwd_workspace(S, Lp, ctypes.byref(n_ws)) == 0
ws = torch.empty(n_ws.value, device=dev)


q16, k16, v16 = (t.to(torch.bfloat16) for t in (q, k, v))
ctx16 = torch.zeros(S, Lp, 256, device=dev, dtype=torch.bfloat16)
assert lib.lgb200_attention(_abi.BF16, ptr(q16), ptr(k16), ptr(v16), S, Lp, None, 0, ptr(ctx16), st) == 0
assert lib.lgb200_attention_bwd_bf16_workspace(S, Lp, ctypes.byref(n_ws)) == 0
ws16 = torch.empty(n_ws.value, device=dev)
dq16, dk16, dv16 = (torch.empty(S, 4, Lp, 64, device=dev) for _ in range(3))


def call_x3():
    rc = lib.lgb200_attention_bwd(ptr(q), ptr(k), ptr(v), ptr(ctx), ptr(dctx), S, Lp, None, 0, ptr(dq), ptr(dk), ptr(dv),
                                  ptr(ws), st)
    assert rc == 0


def call_bf16():
    rc = lib.lgb200_attention_bwd_bf16(ptr(q16), ptr(k16), ptr(v16), ptr(ctx16), ptr(dctx), S, Lp, None, 0, ptr(dq16),
                                       ptr(dk16), ptr(dv16), ptr(ws16), st)
    assert rc == 0


def timed(call):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(REPS):
        call()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / REPS


arms = {"x3 (fp32-accurate, three fp16 MMAs per product)": call_x3, "bf16 (one bf16 MMA per product)": call_bf16}
for call in arms.values():
    for _ in range(2):
        call()
torch.cuda.synchronize()
times = {name: [] for name in arms}
for _ in range(3):  # alternating rounds
    for name, call in arms.items():
        times[name].append(timed(call))
flop = 8 * 2.0 * Lp * Lp * 64 * 4 * S
card = torch.cuda.get_device_name(dev)
try:
    import subprocess

    plim = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
except OSError:
    plim = "unknown"
for name, ts in times.items():
    ms = min(ts)
    print(f"attention backward {name} S={S} Lp={Lp}: {ms:.3f} ms per call (rounds {', '.join(f'{t:.3f}' for t in ts)}), "
          f"{flop / ms / 1e9:.1f} TFLOP/s useful; {card}, power limit {plim}")
rel = lambda a, b: float((a - b).norm() / b.norm())  # noqa: E731
print(f"bf16 vs x3 arm, norm-wise: dq {rel(dq16, dq):.2e} dk {rel(dk16, dk):.2e} dv {rel(dv16, dv):.2e}")
