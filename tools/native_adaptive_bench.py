"""Adaptive depth and width from Python and from C (lgb200_match_adaptive), batch 1, bf16 and fp32.

The heads are biased as in tools/adaptive_bench.py (depth_confidence 0.95, width_confidence 0.99; token confidence high
from layer 4 on, so pairs exit there; matchability low on even layers, so those layers prune).  Two workloads:
  * fixed 2048 x 2048: Python eager; Python `cuda_graph` (the captured stack plus the eager host tail); lgb200_match_
    adaptive called eagerly; the same call captured in a CUDA graph at the exact size.  Also the cost of the L-1
    MatchAssignment groups that early exit adds to the native tail when no pair exits at their layer: the same calls
    (lgb200_linear, lgb200_rowdot, the normalisers) with all counts 0, captured and replayed on their own;
  * a seeded stream of pairs (default 200) with m, n ~ U[512, 2048]: Python eager; Python `cuda_graph` (one capture per
    input shape, counted); lgb200_match_adaptive captured once at capacity 2048 and replayed with the counts, each pair
    copied into the static inputs (zeros past its rows).  Peak memory of one pass above what was allocated before it.
Times: CUDA events around back-to-back calls, the arms alternating window by window (order rotating); median and
min-max over the windows.  Every output of every arm is checked bit-equal to Python eager's (log_assignment cropped to
the pruned counts, ref_descriptors on each pair's rows < its count).

    python tools/native_adaptive_bench.py [--pairs 200] [--windows 5] [--out FILE]
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
from glue_factory_colon_b200._abi import BF16, F32, F32X3, AdaptiveConfig, MatchConfig, check, ptr  # noqa: E402
from glue_factory_colon_b200.driver import crop_log_assignment  # noqa: E402
from glue_factory_colon_b200.synthetic import make_pairs  # noqa: E402
from glue_factory_colon_b200.weights import native_table  # noqa: E402

DEV = torch.device("cuda:0")
CAP = 2048
CONF = {"filter_threshold": 0.1, "depth_confidence": 0.95, "width_confidence": 0.99}


def make_model(prec, **extra):
    torch.manual_seed(0)
    m = LightGlue({"precision": prec, **CONF, **extra}).eval()
    sd = m.state_dict()
    for i in range(m.conf.n_layers - 1):
        sd[f"token_confidence.{i}.token.0.bias"].fill_(3.0 if i >= 4 else -3.0)
        sd[f"log_assignment.{i}.matchability.bias"].fill_(-4.5 if i % 2 == 0 else 0.0)
    return m.to(DEV)


class Native:
    """lgb200_match_adaptive at B = 1 and capacity m x n: static inputs (with counts), workspace, outputs."""

    def __init__(self, model, m, n, counts):
        self.lib = _abi.load()
        c = model.conf
        prec = {"bf16": BF16, "fp32": F32X3}[c.precision]
        self.cfg = MatchConfig(prec, c.n_layers, c.input_dim, 2, float(c.filter_threshold))
        self.acfg = AdaptiveConfig(float(c.depth_confidence), float(c.width_confidence))
        self.table, self.keep = native_table(model, prec, adaptive=True)
        self.m, self.n = m, n
        nb = ctypes.c_longlong(0)
        check(self.lib.lgb200_match_adaptive_workspace(ctypes.byref(self.cfg), 1, m, n, ctypes.byref(nb)), "ws")
        self.ws = torch.empty(nb.value, dtype=torch.uint8, device=DEV)
        f32, i32, i64 = (dict(device=DEV, dtype=d) for d in (torch.float32, torch.int32, torch.int64))
        act = torch.bfloat16 if prec == BF16 else torch.float32
        self.ins = {"kpts0": torch.zeros(1, m, 2, **f32), "kpts1": torch.zeros(1, n, 2, **f32),
                    "desc0": torch.zeros(1, m, 256, **f32), "desc1": torch.zeros(1, n, 256, **f32),
                    "size0": torch.zeros(1, 2, **f32), "size1": torch.zeros(1, 2, **f32),
                    "counts0": torch.full((1,), m, **i32) if counts else None,
                    "counts1": torch.full((1,), n, **i32) if counts else None}
        self.out = {"matches0": torch.empty(1, m, **i64), "matches1": torch.empty(1, n, **i64),
                    "matching_scores0": torch.empty(1, m, **f32), "matching_scores1": torch.empty(1, n, **f32),
                    "log_assignment": torch.empty(1, m + 1, n + 1, **f32),
                    "ref_descriptors0": torch.empty(1, m, 256, device=DEV, dtype=act),
                    "ref_descriptors1": torch.empty(1, n, 256, device=DEV, dtype=act),
                    "prune0": torch.empty(1, m, **i32), "prune1": torch.empty(1, n, **i32),
                    "exit_layer": torch.empty(1, **i32), "final_counts": torch.empty(1, 2, **i32)}
        self.graph = None

    def load(self, d):
        """The pair into the static inputs: its rows, zeros past them, its counts."""
        for i in (0, 1):
            k = d[f"keypoints{i}"].shape[1]
            self.ins[f"kpts{i}"][:, :k].copy_(d[f"keypoints{i}"])
            self.ins[f"kpts{i}"][:, k:].zero_()
            self.ins[f"desc{i}"][:, :k].copy_(d[f"descriptors{i}"])
            self.ins[f"desc{i}"][:, k:].zero_()
            self.ins[f"size{i}"].copy_(d[f"view{i}"]["image_size"].reshape(1, 2))
            if self.ins[f"counts{i}"] is not None:
                self.ins[f"counts{i}"].fill_(k)

    def call(self):
        i, o = self.ins, self.out
        check(self.lib.lgb200_match_adaptive(
            ctypes.byref(self.cfg), ctypes.byref(self.acfg), self.table, 1, self.m, self.n, ptr(i["kpts0"]),
            ptr(i["kpts1"]), ptr(i["desc0"]), ptr(i["desc1"]), ptr(i["size0"]), ptr(i["size1"]), ptr(i["counts0"]),
            ptr(i["counts1"]), ptr(o["matches0"]), ptr(o["matches1"]), ptr(o["matching_scores0"]),
            ptr(o["matching_scores1"]), ptr(o["log_assignment"]), ptr(o["ref_descriptors0"]),
            ptr(o["ref_descriptors1"]), ptr(o["prune0"]), ptr(o["prune1"]), ptr(o["exit_layer"]),
            ptr(o["final_counts"]), ptr(self.ws), self.ws.numel(), torch.cuda.current_stream(DEV).cuda_stream),
            "lgb200_match_adaptive")

    def capture(self):
        self.call()
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.call()

    def __call__(self, d):
        self.load(d)
        self.graph.replay() if self.graph is not None else self.call()
        return self.out


def bit_equal(nat, ref, m, n):
    """nat (capacity layout) against Python eager's outputs for a pair with m x n keypoints."""
    k0, k1 = (int(v) for v in nat["final_counts"][0])
    if not torch.equal(crop_log_assignment(nat["log_assignment"], k0, k1), ref["log_assignment"]):
        return False
    for key, cnt in (("matches0", m), ("matches1", n), ("matching_scores0", m), ("matching_scores1", n)):
        if not torch.equal(nat[key][:, :cnt], ref[key]):
            return False
    for i, cnt, k in ((0, m, k0), (1, n, k1)):
        if not torch.equal(nat[f"prune{i}"][:, :cnt].to(ref[f"prune{i}"].dtype), ref[f"prune{i}"]):
            return False
        if not torch.equal(nat[f"ref_descriptors{i}"][0, :k], ref[f"ref_descriptors{i}"][0, -1, :k]):
            return False
    return True


def timed(fn, items):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for d in items:
        fn(d)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / len(items)


def alternate(arms, items, windows):
    times = {name: [] for name in arms}
    names = list(arms)
    for w in range(windows):
        for j in range(len(names)):
            name = names[(w + j) % len(names)]
            times[name].append(timed(arms[name], items))
    return {name: dict(ms_median=round(statistics.median(t), 4), ms_min=round(min(t), 4), ms_max=round(max(t), 4))
            for name, t in times.items()}


def empty_groups_ms(prec, L, reps=200):
    """The L-1 MatchAssignment groups early exit adds to the tail, when no pair exits at their layer: final_proj,
    matchability and the normalisers at B = 1, Lp = 2048 with every count 0, captured and replayed alone."""
    lib = _abi.load()
    x3 = prec == "fp32"
    S, Lp, T = 2, CAP, 2 * CAP
    lens = torch.zeros(S, device=DEV, dtype=torch.int32)
    f32 = dict(device=DEV, dtype=torch.float32)
    if x3:
        xs, md = torch.zeros(2, T, 256, device=DEV, dtype=torch.float16), torch.zeros(2, T, 256, device=DEV, dtype=torch.float16)
        x, w = torch.zeros(T, 256, **f32), torch.zeros(2, 256, 256, device=DEV, dtype=torch.float16)
        sim = torch.zeros(1, Lp, Lp, **f32)
    else:
        x = xs = torch.zeros(T, 256, device=DEV, dtype=torch.bfloat16)
        md, w = torch.zeros(T, 256, device=DEV, dtype=torch.bfloat16), torch.zeros(256, 256, device=DEV, dtype=torch.bfloat16)
    b, mw, mb = torch.zeros(256, **f32), torch.zeros(256, **f32), torch.zeros(1, **f32)
    z, lse = torch.zeros(T, **f32), torch.zeros(T, **f32)
    st = lambda: torch.cuda.current_stream(DEV).cuda_stream  # noqa: E731
    pr = F32X3 if x3 else BF16

    def groups():
        for _ in range(L - 1):
            check(lib.lgb200_linear(pr, 0, ptr(xs), None, 256, ptr(w), ptr(b), T, 256, 256, ptr(lens), Lp, 0.25, 1.0,
                                    1.0, None, None, None, ptr(md), None, None, 0, None, None, None, None, None, st()),
                  "linear")
            check(lib.lgb200_rowdot(F32 if x3 else BF16, ptr(x), ptr(mw), ptr(mb), S, Lp, ptr(lens), 0, ptr(z), st()),
                  "rowdot")
            if x3:
                check(lib.lgb200_x3_similarity(ptr(md), 1, Lp, ptr(lens), ptr(sim), st()), "sim")
                check(lib.lgb200_x3_assign_lse(ptr(sim), 1, Lp, ptr(lens), CAP, CAP, ptr(lse), st()), "lse")
            else:
                check(lib.lgb200_assign_lse(BF16, ptr(md), S, Lp, ptr(lens), ptr(lse), st()), "lse")

    groups()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        groups()
    for _ in range(10):
        g.replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def peak_pass(fn, items):
    torch.cuda.synchronize()
    start = torch.cuda.memory_allocated(DEV)
    torch.cuda.reset_peak_memory_stats(DEV)
    for d in items:
        fn(d)
    torch.cuda.synchronize()
    return round((torch.cuda.max_memory_allocated(DEV) - start) / 2**20, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=200)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    args = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()[0]
    lines = [{"card": card, "torch": torch.__version__, "pairs": args.pairs, "windows": args.windows, **CONF}]
    print(f"card: {card}", flush=True)
    g = torch.Generator().manual_seed(0)
    sizes = torch.randint(512, CAP + 1, (args.pairs, 2), generator=g).tolist()
    stream = [make_pairs(1, m, n, seed=i, device=DEV) for i, (m, n) in enumerate(sizes)]
    fixed = [make_pairs(1, CAP, CAP, seed=400, device=DEV)] * 20
    for prec in ("bf16", "fp32"):
        with torch.no_grad():
            eager = make_model(prec)
            graphed = make_model(prec, cuda_graph=True)
            L = eager.conf.n_layers
            # ---- fixed 2048 x 2048 ----
            nat_e = Native(eager, CAP, CAP, counts=False)
            nat_g = Native(eager, CAP, CAP, counts=False)
            nat_g.load(fixed[0])
            nat_g.capture()
            ref = eager(fixed[0])
            lib = _abi.load()
            c0 = lib.lgb200_launch_count()
            nat_e(fixed[0])
            launches = lib.lgb200_launch_count() - c0
            ok = {"python_cuda_graph": all(torch.equal(graphed(fixed[0])[k], ref[k]) for k in ref),
                  "native_eager": bit_equal(nat_e(fixed[0]), ref, CAP, CAP),
                  "native_graph_exact": bit_equal(nat_g(fixed[0]), ref, CAP, CAP)}
            arms = {"python_eager": eager, "python_cuda_graph": graphed, "native_eager": nat_e,
                    "native_graph_exact": nat_g}
            res = alternate(arms, fixed, args.windows)
            k = nat_g.out["final_counts"][0].tolist()
            meta = {"exit_layer": int(nat_g.out["exit_layer"][0]), "final_counts": k,
                    "native_launches_per_call": launches,
                    "empty_groups_ms": round(empty_groups_ms(prec, L), 4)}
            print(f"{prec} fixed {CAP}^2: exit layer {meta['exit_layer']}, pruned counts {k}, "
                  f"{launches} native launches, {L - 1} empty tail groups {meta['empty_groups_ms']:.4f} ms", flush=True)
            lines.append({"precision": prec, "workload": f"fixed {CAP}x{CAP}", **meta})
            for name, r in res.items():
                r["bit_equal_to_eager"] = ok.get(name, True)
                print(f"{prec} fixed  {name:22s} {r['ms_median']:.3f} ms (min {r['ms_min']:.3f}, max {r['ms_max']:.3f})"
                      f"  bit-equal {r['bit_equal_to_eager']}", flush=True)
                lines.append({"precision": prec, "workload": f"fixed {CAP}x{CAP}", "arm": name, **r})
            del nat_e, nat_g
            # ---- stream of varying sizes ----
            nat_c = Native(eager, CAP, CAP, counts=True)
            nat_c.load(stream[0])
            nat_c.capture()
            stats = {}
            for name, fn in (("python_eager", eager), ("native_graph_capacity", nat_c)):
                stats[name] = {"peak_mb": peak_pass(fn, stream)}
            graphed._graphs.clear()
            caps = 0
            torch.cuda.synchronize()
            start = torch.cuda.memory_allocated(DEV)
            torch.cuda.reset_peak_memory_stats(DEV)
            for d in stream:
                keys = set(graphed._graphs)
                graphed(d)
                caps += len(set(graphed._graphs) - keys)
            torch.cuda.synchronize()
            stats["python_cuda_graph"] = {"peak_mb": round((torch.cuda.max_memory_allocated(DEV) - start) / 2**20, 1),
                                          "captures_per_pass": caps}
            same = {"python_cuda_graph": True, "native_graph_capacity": True}
            for (m, n), d in zip(sizes, stream):
                want = eager(d)
                same["python_cuda_graph"] &= all(torch.equal(graphed(d)[k], want[k]) for k in want)
                same["native_graph_capacity"] &= bit_equal(nat_c(d), want, m, n)
            arms = {"python_eager": eager, "python_cuda_graph": graphed, "native_graph_capacity": nat_c}
            res = alternate(arms, stream, args.windows)
            for name, r in res.items():
                r.update(stats[name])
                r["bit_equal_to_eager"] = same.get(name, True)
                print(f"{prec} stream {name:22s} {r['ms_median']:.3f} ms per pair (min {r['ms_min']:.3f}, max "
                      f"{r['ms_max']:.3f})  peak {r['peak_mb']} MB"
                      + (f"  captures per pass {r['captures_per_pass']}" if "captures_per_pass" in r else "")
                      + f"  bit-equal {r['bit_equal_to_eager']}", flush=True)
                lines.append({"precision": prec, "workload": f"stream of {args.pairs}, m, n ~ U[512, {CAP}]",
                              "arm": name, **r})
            del nat_c, eager, graphed
            torch.cuda.empty_cache()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
