"""Training step (forward in training mode + LightGlue.loss + backward) through the drop-in's hand-written backward
pass, and through the UNMODIFIED reference module (baseline/_ref, PyTorch autograd over cuBLAS / SDPA kernels) on the
same GPU and the same batch.  Arms: conf.train_precision "fp32" (fp32-accurate) and "bf16" (mixed precision), each kept
and checkpointed, timed in alternating rounds; the reference in fp32 and under torch.autocast("cuda", bfloat16) (what a
glue-factory user training with mixed precision runs) if baseline/_ref is present.  One JSON line per arm and round with
ms per step and peak memory, plus the card's name and power limit.  Usage: python tools/train_bench.py [B] [kpts] [reps]
[rounds]"""
import json
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402
from glue_factory_colon_b200 import LightGlue  # noqa: E402
from glue_factory_colon_b200.synthetic import make_pairs  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 32
N = int(sys.argv[2]) if len(sys.argv) > 2 else 512
REPS = int(sys.argv[3]) if len(sys.argv) > 3 else 5
ROUNDS = int(sys.argv[4]) if len(sys.argv) > 4 else 2
dev = torch.device("cuda:0")
conf = {"filter_threshold": 0.1}
data = make_pairs(B, N, N, seed=3, device=dev, with_gt=True)


def step(model, autocast=False):
    model.zero_grad(set_to_none=True)
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
        pred = model(data)
        losses, _ = model.loss(pred, data)
    losses["total"].mean().backward()
    return float(losses["total"].mean().detach())


def timed(model, label, extra=None, autocast=False, warm=2):
    for _ in range(warm):
        val = step(model, autocast)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(REPS):
        val = step(model, autocast)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / REPS
    rec = {"impl": label, "pairs": B, "kpts": N, "ms_per_step": round(ms, 2), "pairs_per_s": round(B / ms * 1e3, 1),
           "loss": round(val, 5), "peak_mem_gb": round(torch.cuda.max_memory_allocated() / 2**30, 2)}
    rec.update(extra or {})
    print(json.dumps(rec), flush=True)
    return rec


def card():
    import subprocess

    try:
        plim = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True).stdout.strip()
    except OSError:
        plim = "unknown"
    return {"gpu": torch.cuda.get_device_name(dev), "power_limit": plim}


print(json.dumps(card()), flush=True)
arms = []  # (label, model, autocast)
for tp in ("fp32", "bf16"):
    for ckpt in (False, True):
        torch.manual_seed(0)
        ours = LightGlue({**conf, "checkpointed": ckpt, "train_precision": tp}).to(dev).train()
        arms.append((f"glue_factory_colon_b200 train_precision={tp}, checkpointed={ckpt}", ours, False))
for ckpt in (False, True):
    ref = bench.load_reference_module({**conf, "checkpointed": ckpt})
    if ref is None:
        print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref missing"}))
        break
    ref = ref.to(dev).train()
    arms.append((f"unmodified reference module, fp32 autograd, checkpointed={ckpt}", ref, False))
    arms.append((f"unmodified reference module, torch.autocast(bfloat16), checkpointed={ckpt}", ref, True))
for r in range(ROUNDS):
    for label, model, ac in arms:
        try:
            timed(model, label, {"round": r}, autocast=ac, warm=2 if r == 0 else 1)
        except Exception as exc:  # noqa: BLE001
            print(json.dumps({"impl": label, "error": repr(exc)[:200]}), flush=True)
        torch.cuda.empty_cache()
print(json.dumps(card()), flush=True)
