"""Training step of the nearest-neighbour matcher with the N_pair loss: forward, `loss` and `total.mean().backward()` of
the drop-in against the same algorithm in fp32 torch autograd (the reference's ops -- einsum, find_nn, mutual_check,
dual log-softmax, N_pair loss -- from oracle/nn_oracle.py, on the same GPU), in alternating rounds, with ms per step and
peak memory (inputs included).  Then lgb200_npair_loss_bwd alone, with the L2 overwritten before every launch, and its
bytes (similarity and ground truth read, d similarity written) over the 7.7 TB/s HBM bound of the data sheet.  One JSON
line per measurement, plus the card's name and power limit.  Usage: python tools/nn_train_bench.py [reps] [rounds]"""
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from glue_factory_colon_b200 import _abi  # noqa: E402
from glue_factory_colon_b200._abi import check, ptr  # noqa: E402
from glue_factory_colon_b200.nearest_neighbor_matcher import NearestNeighborMatcher, _npair_loss  # noqa: E402
from glue_factory_colon_b200.synthetic import make_pairs, to_device  # noqa: E402
from oracle import nn_oracle  # noqa: E402

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 10
ROUNDS = int(sys.argv[2]) if len(sys.argv) > 2 else 2
SIZES = ((16, 1024), (16, 2048))  # pairs x keypoints per image, D = 256
HBM_BYTES_PER_S = 7.7e12
dev = torch.device("cuda:0")


def card():
    try:
        plim = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True).stdout.strip()
    except OSError:
        plim = "unknown"
    return {"gpu": torch.cuda.get_device_name(dev), "power_limit": plim}


def dropin_arm(data):
    model = NearestNeighborMatcher({"loss": "N_pair"}).to(dev).train()
    d0, d1 = data["descriptors0"].clone().requires_grad_(), data["descriptors1"].clone().requires_grad_()
    batch = dict(data, descriptors0=d0, descriptors1=d1)

    def step():
        d0.grad = d1.grad = model.temperature.grad = None
        losses, _ = model.loss(model(batch), batch)
        losses["total"].mean().backward()
        return losses["total"].mean().detach()

    return step, (d0, d1, model.temperature)


def torch_arm(data):
    d0, d1 = data["descriptors0"].clone().requires_grad_(), data["descriptors1"].clone().requires_grad_()
    temperature = torch.tensor(1.0, device=dev, requires_grad=True)

    def step():
        d0.grad = d1.grad = temperature.grad = None
        with torch.device(dev):  # the reference's index tensors are created without a device
            pred = nn_oracle.forward({"mutual_check": True}, None, sim=torch.einsum("bnd,bmd->bnm", d0, d1))
        losses = nn_oracle.npair_loss(pred["similarity"], data["gt_assignment"], temperature)
        losses["total"].mean().backward()
        return losses["total"].mean().detach()

    return step, (d0, d1, temperature)


def timed(step, reps):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        val = step()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, torch.cuda.max_memory_allocated() / 2**30, float(val)


def kernel_alone(data, reps):
    """lgb200_npair_loss_bwd on the drop-in's similarity, per-launch events, 512 MB written between launches."""
    lib = _abi.load()
    with torch.no_grad():
        sim = NearestNeighborMatcher({})(data)["similarity"]
    gt = data["gt_assignment"].contiguous()
    B, N, M = sim.shape
    _, num, ws, row_cnt = _npair_loss(sim, 1.0, gt)
    coef = (-1.0 / (2 * num)).contiguous()
    col_cnt, dtemp_rows, dsim = torch.empty(B, M, device=dev), torch.empty(B, N, device=dev), torch.empty_like(sim)
    flush = torch.empty(2**27, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    times = []
    for i in range(reps + 3):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        check(lib.lgb200_npair_loss_bwd(ptr(sim), ptr(gt), B, N, M, 1.0, ptr(ws), ptr(row_cnt), ptr(coef), ptr(col_cnt),
                                        ptr(dsim), ptr(dtemp_rows), st), "npair_loss_bwd")
        e1.record()
        if i >= 3:
            times.append((e0, e1))
    torch.cuda.synchronize()
    ms = sorted(a.elapsed_time(b) for a, b in times)
    med = ms[len(ms) // 2]
    nbytes = B * N * M * (4 + 1 + 4)
    return {"kernel": "lgb200_npair_loss_bwd", "pairs": B, "kpts": N, "ms_median": round(med, 4),
            "ms_min": round(ms[0], 4), "bytes": nbytes, "TB_per_s": round(nbytes / med / 1e9, 2),
            "share_of_7.7TBps": round(nbytes / med / 1e9 / (HBM_BYTES_PER_S / 1e12), 3)}


print(json.dumps(card()), flush=True)
for B, N in SIZES:
    data = to_device(make_pairs(B, N, N, seed=5, with_gt=True), dev)
    arms = [("drop-in (lgb200 kernels)", *dropin_arm(data)), ("fp32 torch autograd (reference ops)", *torch_arm(data))]
    for _, step, _ in arms:  # warm-up
        step()
        step()
    for r in range(ROUNDS):
        for label, step, _ in arms:
            ms, mem, val = timed(step, REPS)
            print(json.dumps({"impl": label, "pairs": B, "kpts": N, "dim": 256, "round": r, "ms_per_step": round(ms, 2),
                              "peak_mem_gb": round(mem, 2), "loss": round(val, 6)}), flush=True)
            torch.cuda.empty_cache()
    # same inputs, same step: how far apart the two arms' gradients are (max |d| over max |g| of the torch arm)
    (_, _, ga), (_, _, gb) = arms
    print(json.dumps({"pairs": B, "kpts": N, "grad_rel_diff": [
        float((a.grad - b.grad).abs().max() / b.grad.abs().max()) for a, b in zip(ga, gb)]}), flush=True)
    del arms, ga, gb
    torch.cuda.empty_cache()
    print(json.dumps(kernel_alone(data, 50)), flush=True)
    del data
    torch.cuda.empty_cache()
print(json.dumps(card()), flush=True)
