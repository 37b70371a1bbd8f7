"""lgb200_match (the whole matcher behind the C ABI) against LightGlue.forward, bf16.

Batch-1 latency at 512 / 1024 / 2048 keypoints, five arms: Python eager, Python `cuda_graph`, native eager (the ctypes
call included), native graph captured at the exact size, native graph captured at a 2048 x 2048 capacity and replayed
with the pair's counts.  Then 64 x 2048 throughput, native against LightGlue.forward, the two arms alternating.
CUDA events around back-to-back calls after warm-ups; every figure is the median of 7 windows, with min-max.

    python tools/native_match_bench.py [--out FILE]
"""
import argparse
import ctypes
import json
import statistics
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from glue_factory_colon_b200 import LightGlue, _abi  # noqa: E402
from glue_factory_colon_b200._abi import BF16, MatchConfig, check, ptr  # noqa: E402
from glue_factory_colon_b200.synthetic import make_pairs  # noqa: E402
from glue_factory_colon_b200.weights import native_table  # noqa: E402

DEV = torch.device("cuda:0")


class Native:
    """lgb200_match at a fixed capacity B x m x n: table, workspace, output buffers."""

    def __init__(self, model, B, m, n):
        self.lib = _abi.load()
        c = model.conf
        self.cfg = MatchConfig(BF16, c.n_layers, c.input_dim, 2, float(c.filter_threshold))
        self.table, self.keep = native_table(model, BF16)
        self.B, self.m, self.n = B, m, n
        nb = ctypes.c_longlong(0)
        check(self.lib.lgb200_match_workspace(ctypes.byref(self.cfg), B, m, n, ctypes.byref(nb)), "match_workspace")
        self.ws = torch.empty(nb.value, dtype=torch.uint8, device=DEV)
        i64, f32 = dict(device=DEV, dtype=torch.int64), dict(device=DEV, dtype=torch.float32)
        self.out = dict(m0=torch.empty(B, m, **i64), m1=torch.empty(B, n, **i64), s0=torch.empty(B, m, **f32),
                        s1=torch.empty(B, n, **f32), la=torch.empty(B, m + 1, n + 1, **f32))

    def __call__(self, ins):
        o = self.out
        check(self.lib.lgb200_match(
            ctypes.byref(self.cfg), self.table, self.B, self.m, self.n, ptr(ins["k0"]), ptr(ins["k1"]), ptr(ins["d0"]),
            ptr(ins["d1"]), ptr(ins["s0"]), ptr(ins["s1"]), ptr(ins.get("c0")), ptr(ins.get("c1")), ptr(o["m0"]),
            ptr(o["m1"]), ptr(o["s0"]), ptr(o["s1"]), ptr(o["la"]), None, None, ptr(self.ws), self.ws.numel(),
            torch.cuda.current_stream(DEV).cuda_stream), "lgb200_match")
        return o


def inputs(data, cap=None):
    """Device inputs; with cap: zero-padded to cap keypoints with the true counts in c0 / c1."""
    B, m, _ = data["keypoints0"].shape
    n = data["keypoints1"].shape[1]
    ins = {}
    for i, cnt in ((0, m), (1, n)):
        k, d = data[f"keypoints{i}"].float(), data[f"descriptors{i}"].float()
        if cap is not None:
            k = torch.cat([k, k.new_zeros(B, cap - cnt, 2)], 1)
            d = torch.cat([d, d.new_zeros(B, cap - cnt, 256)], 1)
            ins[f"c{i}"] = torch.full((B,), cnt, dtype=torch.int32, device=DEV)
        ins[f"k{i}"], ins[f"d{i}"] = k.to(DEV).contiguous(), d.to(DEV).contiguous()
        ins[f"s{i}"] = data[f"view{i}"]["image_size"].to(DEV).float().contiguous()
    return ins


def timed(fn, calls, windows=7, warm=5):
    """ms per call: median, min, max over `windows` windows of `calls` back-to-back calls (CUDA events)."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    res = []
    for _ in range(windows):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(calls):
            fn()
        e1.record()
        e1.synchronize()
        res.append(e0.elapsed_time(e1) / calls)
    return statistics.median(res), min(res), max(res)


def graph_of(fn):
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    args = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()[0]
    lines = [{"card": card, "torch": torch.__version__}]
    print(f"card: {card}")
    torch.manual_seed(0)
    model = LightGlue({"precision": "bf16", "filter_threshold": 0.1}).eval().to(DEV)
    model_g = LightGlue({"precision": "bf16", "filter_threshold": 0.1, "cuda_graph": True}).eval().to(DEV)
    model_g.load_state_dict(model.state_dict())
    cap = 2048
    nat_cap = Native(model, 1, cap, cap)
    for kp in (512, 1024, 2048):
        data = make_pairs(1, kp, kp, seed=7)
        ddev = {k: (v.to(DEV) if torch.is_tensor(v) else {kk: vv.to(DEV) for kk, vv in v.items()})
                for k, v in data.items()}
        nat = Native(model, 1, kp, kp)
        ins, ins_cap = inputs(data), inputs(data, cap)
        g_exact = graph_of(lambda: nat(ins))
        g_cap = graph_of(lambda: nat_cap(ins_cap))
        with torch.no_grad():
            ref = model(ddev)
        nat(ins)
        torch.cuda.synchronize()
        same = torch.equal(nat.out["la"], ref["log_assignment"]) and torch.equal(nat.out["m0"], ref["matches0"])
        arms = {}
        with torch.no_grad():
            arms["python_eager"] = timed(lambda: model(ddev), 50)
            arms["python_cuda_graph"] = timed(lambda: model_g(ddev), 50)
        arms["native_eager"] = timed(lambda: nat(ins), 50)
        arms["native_graph_exact"] = timed(g_exact.replay, 50)
        arms["native_graph_cap2048"] = timed(g_cap.replay, 50)
        for arm, (med, lo, hi) in arms.items():
            print(f"B=1 {kp:5d} kpts  {arm:22s} {med:.3f} ms per pair  (min {lo:.3f}, max {hi:.3f})")
            lines.append({"B": 1, "kpts": kp, "arm": arm, "ms_median": round(med, 4), "ms_min": round(lo, 4),
                          "ms_max": round(hi, 4)})
        print(f"B=1 {kp:5d} kpts  native eager bit-equal to LightGlue.forward: {same}")
        lines.append({"B": 1, "kpts": kp, "native_bit_equal": same})
        del g_exact, g_cap

    B, kp = 64, 2048
    data = make_pairs(B, kp, kp, seed=9)
    ddev = {k: (v.to(DEV) if torch.is_tensor(v) else {kk: vv.to(DEV) for kk, vv in v.items()}) for k, v in data.items()}
    nat = Native(model, B, kp, kp)
    ins = inputs(data)
    with torch.no_grad():
        ref = model(ddev)
        nat(ins)
        torch.cuda.synchronize()
        same = torch.equal(nat.out["la"], ref["log_assignment"]) and torch.equal(nat.out["m0"], ref["matches0"])
        del ref
        py, na = [], []
        for _ in range(2):  # warm-up of both arms
            model(ddev), nat(ins)
        torch.cuda.synchronize()
        for _ in range(7):  # alternating windows of 5 batches each
            py.append(timed(lambda: model(ddev), 5, windows=1, warm=0)[0])
            na.append(timed(lambda: nat(ins), 5, windows=1, warm=0)[0])
    for arm, ts in (("python_forward", py), ("native", na)):
        med = statistics.median(ts)
        print(f"B={B} {kp} kpts  {arm:15s} {med:.2f} ms per batch = {B / med * 1e3:.0f} pairs/s  "
              f"(min {min(ts):.2f}, max {max(ts):.2f} ms)")
        lines.append({"B": B, "kpts": kp, "arm": arm, "ms_median": round(med, 3), "ms_min": round(min(ts), 3),
                      "ms_max": round(max(ts), 3), "pairs_per_s": round(B / med * 1e3, 1)})
    print(f"B={B} {kp} kpts  native bit-equal to LightGlue.forward: {same}")
    lines.append({"B": B, "kpts": kp, "native_bit_equal": same})
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
