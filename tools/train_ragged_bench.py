"""Training step on a ragged batch: per-pair keypoint counts drawn from U[N/4, N], every pair padded to N.  For each
conf.train_precision the step is timed with the counts (num_keypoints0/1: padded tiles skipped, padding ignored) and
on the same tensors without them (the padding treated as real keypoints, the only option before counts were accepted
in training), in alternating rounds.  One JSON line per arm and round with ms per step and peak memory, plus the card's
name and power limit.  Usage: python tools/train_ragged_bench.py [B] [N] [reps] [rounds]"""
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from glue_factory_colon_b200 import LightGlue  # noqa: E402
from glue_factory_colon_b200.padding import pad_and_stack, pad_to_length  # noqa: E402
from glue_factory_colon_b200.synthetic import make_pairs, to_device  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 32
N = int(sys.argv[2]) if len(sys.argv) > 2 else 512
REPS = int(sys.argv[3]) if len(sys.argv) > 3 else 5
ROUNDS = int(sys.argv[4]) if len(sys.argv) > 4 else 2
dev = torch.device("cuda:0")
conf = {"filter_threshold": 0.1}


def ragged_batch():
    g = torch.Generator().manual_seed(3)
    counts = torch.randint(N // 4, N + 1, (2, B), generator=g)
    pairs = [make_pairs(1, int(counts[0, b]), int(counts[1, b]), seed=100 + b, with_gt=True) for b in range(B)]
    torch.manual_seed(0)
    data = {}
    for i in (0, 1):
        data[f"keypoints{i}"] = pad_and_stack([p[f"keypoints{i}"][0] for p in pairs], N, -2, mode="random_c")
        data[f"descriptors{i}"] = pad_and_stack([p[f"descriptors{i}"][0] for p in pairs], N, -2, mode="random")
        data[f"view{i}"] = {"image_size": torch.cat([p[f"view{i}"]["image_size"] for p in pairs])}
        data[f"gt_matches{i}"] = pad_and_stack([p[f"gt_matches{i}"][0] for p in pairs], N, -1, mode="minus_one")
    data["gt_assignment"] = torch.stack([pad_to_length(pad_to_length(p["gt_assignment"][0], N, -1), N, -2)
                                         for p in pairs])
    with_counts = dict(data, num_keypoints0=counts[0].to(torch.int32), num_keypoints1=counts[1].to(torch.int32))
    return to_device(with_counts, dev), to_device(data, dev), float(counts.float().mean())


def step(model, data):
    model.zero_grad(set_to_none=True)
    losses, _ = model.loss(model(data), data)
    losses["total"].mean().backward()
    return float(losses["total"].mean().detach())


def timed(model, data, label, extra, warm):
    for _ in range(warm):
        val = step(model, data)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(REPS):
        val = step(model, data)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / REPS
    rec = {"impl": label, "pairs": B, "padded_kpts": N, "ms_per_step": round(ms, 2), "loss": round(val, 5),
           "peak_mem_gb": round(torch.cuda.max_memory_allocated() / 2**30, 2), **extra}
    print(json.dumps(rec), flush=True)


def card():
    try:
        plim = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True).stdout.strip()
    except OSError:
        plim = "unknown"
    return {"gpu": torch.cuda.get_device_name(dev), "power_limit": plim}


print(json.dumps(card()), flush=True)
ragged, padded, mean_count = ragged_batch()
print(json.dumps({"pairs": B, "padded_kpts": N, "mean_count": round(mean_count, 1)}), flush=True)
arms = []
for tp in ("fp32", "bf16"):
    torch.manual_seed(0)
    model = LightGlue({**conf, "train_precision": tp}).to(dev).train()
    arms.append((f"train_precision={tp}, with counts", model, ragged))
    arms.append((f"train_precision={tp}, without counts (padding as keypoints)", model, padded))
for r in range(ROUNDS):
    for label, model, data in arms:
        timed(model, data, label, {"round": r}, warm=2 if r == 0 else 1)
        torch.cuda.empty_cache()
print(json.dumps(card()), flush=True)
