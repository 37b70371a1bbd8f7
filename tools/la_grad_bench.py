"""Cost of training through `log_assignment`, `matching_scores0/1` and the keypoints, and proof that today's loss is
untouched.  One JSON line per measurement, plus the card's name and power limit.

1. lgb200_assign_bwd alone at 8 x 2048^2 and 16 x 2048^2, L2 overwritten (a 256 MB write) before every launch: time
   per call (CUDA events), bytes from the shapes -- G read twice, the similarity read and written, plus the
   partials, sums and dz -- and that over the 7.7 TB/s HBM bound of the data sheet.
2. Training steps at 32 x 512 and 8 x 2048 keypoints, train_precision fp32 and bf16, each version of the package in its
   own process, the two alternating (--parent DIR: a copy of the parent commit's package, e.g. exported with
   `git archive HEAD~1 glue_factory_colon_b200 | tar -x -C DIR`, built with its own build.py):
     "today"  LightGlue.loss's total, descriptors requiring grad (the step both versions run): ms per step, peak
              memory, launches per step;
     "extra"  the same plus sum W.log_assignment + sum v.matching_scores0 + sum u.matching_scores1 (this version only),
              with and without keypoints that require grad.
   Both versions also run one seeded step of every case in DUMP_CASES and dump a digest of its losses, forward outputs,
   parameter gradients and input gradients; the digests are compared per case (bit_equal_to_parent).
The dumps go to a temporary directory.  Usage: python tools/la_grad_bench.py [--parent DIR] [--steps K] [--rounds R]"""
import argparse
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
HBM_BYTES_PER_S = 7.7e12
CONFIGS = ((32, 512), (8, 2048))
# name -> (conf over the timed model's, make_pairs arguments, counts, inputs that require grad, loss mode).  counts:
# num_keypoints0/1 below the padded size, and an empty side in the last pair.
KPTS = ("keypoints0", "keypoints1", "scales0", "scales1", "oris0", "oris1")
DUMP_CASES = {
    "today": ({}, {}, False, (), "today"),
    "checkpointed": ({"checkpointed": True}, {}, False, (), "today"),
    "padded_counts": ({}, {}, True, (), "extra"),
    "dim128_scale_ori": ({"input_dim": 128, "add_scale_ori": True}, {"dim": 128, "scale_ori": True}, False, KPTS,
                         "extra"),
    "extra": ({}, {}, False, (), "extra"),
}
OUTPUTS = ("ref_descriptors0", "ref_descriptors1", "log_assignment", "matches0", "matches1", "matching_scores0",
           "matching_scores1")


def digest(t):
    """dtype, shape and SHA-256 of the bytes of t: equal digests are equal bits."""
    import torch

    t = t.detach().contiguous()
    h = hashlib.sha256(t.reshape(-1).view(torch.uint8).cpu().numpy().tobytes()).hexdigest()
    return f"{t.dtype} {tuple(t.shape)} {h}"


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True).stdout.strip()
    except OSError:
        out = "unknown"
    return {"card": out}


def kernel_bench(reps=20):
    import ctypes

    import torch

    sys.path.insert(0, str(ROOT))
    from glue_factory_colon_b200 import _abi
    from glue_factory_colon_b200._abi import check, ptr

    lib = _abi.load()
    dev = torch.device("cuda:0")
    st = torch.cuda.current_stream(dev).cuda_stream
    flush = torch.empty(64 * 2**20, device=dev)  # 256 MB: twice the L2
    for B in (8, 16):
        m = n = Lp = 2048
        g = torch.Generator(device=dev).manual_seed(B)
        G = torch.randn(B, m + 1, n + 1, device=dev, generator=g)
        sim0 = torch.randn(B, m, n, device=dev, generator=g) * 2
        sim = sim0.clone()
        lse = torch.zeros(2 * B, Lp, device=dev)
        lse.view(B, 2, Lp)[:, 0] = torch.logsumexp(sim0, 2)
        lse.view(B, 2, Lp)[:, 1] = torch.logsumexp(sim0, 1)
        z = torch.randn(2 * B * Lp, device=dev, generator=g)
        dz0, dz1 = torch.empty(B, m, device=dev), torch.empty(B, n, device=dev)
        n_ws = ctypes.c_longlong(0)
        check(lib.lgb200_assign_bwd_workspace(B, m, n, ctypes.byref(n_ws)), "workspace")
        ws = torch.empty(n_ws.value, device=dev)
        ts = []
        for i in range(reps + 3):
            sim.copy_(sim0)
            flush.fill_(float(i))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            check(lib.lgb200_assign_bwd(ptr(G), ptr(sim), B, m, n, ptr(lse), Lp, None, ptr(z), ptr(dz0), ptr(dz1),
                                        ptr(ws), st), "assign_bwd")
            e1.record()
            torch.cuda.synchronize()
            if i >= 3:
                ts.append(e0.elapsed_time(e1))
        ts.sort()
        P = (m + 31) // 32
        nbytes = 4 * (2 * B * (m + 1) * (n + 1) + 2 * B * m * n + 2 * B * P * n + 3 * B * (m + n))
        med = ts[len(ts) // 2]
        print(json.dumps({"kernel": "lgb200_assign_bwd", "shape": f"{B}x{m}x{n}", "ms_median": round(med, 4),
                          "ms_min": round(ts[0], 4), "ms_max": round(ts[-1], 4), "bytes": nbytes,
                          "TB_per_s": round(nbytes / med / 1e9, 3),
                          "share_of_7.7TBps": round(nbytes / med / 1e9 / (HBM_BYTES_PER_S / 1e12), 3)}), flush=True)


def worker(args):
    """One version of the package (args.pkg) in this process: one dump step, then timed steps."""
    sys.path.insert(0, args.pkg)
    sys.path.insert(1, str(ROOT))
    import torch

    from glue_factory_colon_b200 import LightGlue, _abi
    from glue_factory_colon_b200.synthetic import make_pairs, to_device

    assert Path(_abi.__file__).resolve().is_relative_to(Path(args.pkg).resolve()), _abi.__file__
    lib = _abi.load()
    dev = torch.device("cuda:0")
    B, N = args.B, args.N
    torch.manual_seed(0)
    model = LightGlue({"n_layers": 9, "filter_threshold": 0.1, "train_precision": args.prec}).to(dev).train()
    data = to_device(make_pairs(B=B, n0=N, n1=N, seed=3, with_gt=True), dev)
    g = torch.Generator(device=dev).manual_seed(1)
    W = torch.randn(B, N + 1, N + 1, device=dev, generator=g) * 1e-3
    v, u = torch.randn(B, N, device=dev, generator=g) * 0.1, torch.randn(B, N, device=dev, generator=g) * 0.1

    def step(mode, model=model, data=data, leaves=()):
        d = dict(data)
        leaves = ("descriptors0", "descriptors1") + leaves + (("keypoints0", "keypoints1") if mode == "extra_kpts" else ())
        for k in leaves:
            d[k] = data[k].clone().requires_grad_(True)
        model.zero_grad(set_to_none=True)
        pred = model(d)
        losses, _ = model.loss(pred, d)
        loss = losses["total"].mean()
        if mode != "today":
            loss = loss + (W * pred["log_assignment"]).sum() + (v * pred["matching_scores0"]).sum() + \
                (u * pred["matching_scores1"]).sum()
        loss.backward()
        return losses, d, pred, leaves

    if args.dump:
        out = {}
        for case, (conf, kw, counts, leaves, mode) in DUMP_CASES.items():
            torch.manual_seed(0)
            m_ = LightGlue({"n_layers": 9, "filter_threshold": 0.1, "train_precision": args.prec, **conf}).to(dev).train()
            d_ = to_device(make_pairs(B=B, n0=N, n1=N, seed=3, with_gt=True, **kw), dev)
            if counts:
                c0, c1 = [N - (61 * b) % N for b in range(B)], [N - (97 * b) % N for b in range(B)]
                c1[-1] = 0
                d_["num_keypoints0"], d_["num_keypoints1"] = torch.tensor(c0), torch.tensor(c1)
            losses, d, pred, leaves = step(mode, m_, d_, leaves)
            ts = {"loss." + k: t for k, t in losses.items()}
            ts.update({"out." + k: pred[k] for k in OUTPUTS})
            ts.update({"grad." + k: p.grad for k, p in m_.named_parameters() if p.grad is not None})
            ts.update({"grad." + k: d[k].grad for k in leaves})
            out.update({f"{case}/{k}": digest(t) for k, t in ts.items()})
            del m_, d_, losses, d, pred, ts
        torch.save(out, args.dump)
    for mode in args.modes.split(","):
        for _ in range(2):
            step(mode)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        c0 = lib.lgb200_launch_count()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step(mode)
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3 / args.steps
        print(json.dumps({"version": args.name, "B": B, "N": N, "train_precision": args.prec, "loss": mode,
                          "ms_per_step": round(ms, 2), "peak_GB": round(torch.cuda.max_memory_allocated(dev) / 1e9, 3),
                          "launches_per_step": (lib.lgb200_launch_count() - c0) // args.steps}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent")
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--pkg")
    ap.add_argument("--name")
    ap.add_argument("--B", type=int)
    ap.add_argument("--N", type=int)
    ap.add_argument("--prec")
    ap.add_argument("--modes")
    ap.add_argument("--dump")
    args = ap.parse_args()
    if args.worker:
        return worker(args)
    print(json.dumps(card()), flush=True)
    kernel_bench()
    out = Path(tempfile.mkdtemp(prefix="la_grad_bench_"))
    versions = [("branch", str(ROOT))] + ([("parent", str(Path(args.parent).resolve()))] if args.parent else [])
    for B, N in CONFIGS:
        for prec in ("fp32", "bf16"):
            for r in range(args.rounds):
                for name, pkg in (versions if r % 2 == 0 else versions[::-1]):
                    modes = "today,extra,extra_kpts" if name == "branch" else "today"
                    cmd = [sys.executable, __file__, "--worker", "--pkg", pkg, "--name", name, "--B", str(B),
                           "--N", str(N), "--prec", prec, "--modes", modes, "--steps", str(args.steps)]
                    if r == 0:
                        cmd += ["--dump", str(out / f"{name}_{B}x{N}_{prec}.pt")]
                    subprocess.run(cmd, check=True, env=dict(os.environ, PYTHONDONTWRITEBYTECODE="1"))
            if args.parent:
                import torch

                a = torch.load(out / f"branch_{B}x{N}_{prec}.pt")
                b = torch.load(out / f"parent_{B}x{N}_{prec}.pt")
                for case in DUMP_CASES:
                    keys = {k for k in set(a) | set(b) if k.startswith(case + "/")}
                    diff = sorted(k for k in keys if a.get(k) != b.get(k))
                    print(json.dumps({"B": B, "N": N, "train_precision": prec, "case": case,
                                      "tensors_compared": len(keys), "bit_equal_to_parent": not diff,
                                      "differing": diff[:10]}), flush=True)
    shutil.rmtree(out)


if __name__ == "__main__":
    main()
