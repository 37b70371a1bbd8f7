"""`cuda_graph` with and without `graph_capacity` on a stream of pairs whose keypoint counts change with every call, as
a detector-thresholded extractor gives them to the batch-1 eval flow (eval/hpatches.py:46).

Batch 1, a seeded stream of pairs (default 200) with m and n drawn independently from U[512, 2048], image sizes given,
in bf16 and fp32.  Three arms on the same weights: eager, `cuda_graph` alone (one capture per input signature, at most 8
kept), and `cuda_graph` with `graph_capacity=2048`.  Per arm and precision:
  * ms per pair: CUDA events around the whole stream run back to back; the arms alternate window by window (the order
    rotates), median and min-max over the windows;
  * captures during one pass of the stream (new entries of `model._graphs`) and the peak memory allocated during that
    pass above what was allocated before it (the first pass of each arm, run alone: it includes the capture);
  * whether every output of the graph arms is bit-equal to eager's, else the largest |d log_assignment| and the share
    of equal `matches0`.

    python tools/graph_capacity_bench.py [--pairs 200] [--windows 5] [--out FILE]
"""
import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from glue_factory_colon_b200 import LightGlue  # noqa: E402
from glue_factory_colon_b200.synthetic import make_pairs  # noqa: E402

DEV = torch.device("cuda:0")
CAP = 2048


def stream(n_pairs, seed=0):
    g = torch.Generator().manual_seed(seed)
    sizes = torch.randint(512, CAP + 1, (n_pairs, 2), generator=g).tolist()
    return sizes, [make_pairs(1, m, n, seed=seed * 1000 + i, device=DEV) for i, (m, n) in enumerate(sizes)]


def one_pass(model, pairs):
    """Captures and peak memory of one pass over the stream."""
    torch.cuda.synchronize()
    start = torch.cuda.memory_allocated(DEV)
    torch.cuda.reset_peak_memory_stats(DEV)
    captures = 0
    for d in pairs:
        before = set(model._graphs)
        model(d)
        captures += len(set(model._graphs) - before)
    torch.cuda.synchronize()
    return captures, (torch.cuda.max_memory_allocated(DEV) - start) / 2**20


def compare(eager, model, pairs):
    """(every output bit-equal to eager's, max |d log_assignment|, share of equal matches0) over the stream."""
    same, dmax, agree, total = True, 0.0, 0, 0
    for d in pairs:
        want, got = eager(d), model(d)
        same = same and all(torch.equal(got[k], want[k]) for k in want)
        g, w = got["log_assignment"], want["log_assignment"]
        dmax = max(dmax, float(torch.where(g == w, 0.0, (g - w).abs()).max()))
        agree += int((got["matches0"] == want["matches0"]).sum())
        total += want["matches0"].numel()
    return same, dmax, agree / max(total, 1)


def timed_pass(model, pairs):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for d in pairs:
        model(d)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / len(pairs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=200)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    args = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()[0]
    lines = [{"card": card, "torch": torch.__version__, "pairs": args.pairs, "windows": args.windows}]
    print(f"card: {card}")
    sizes, pairs = stream(args.pairs)
    print(f"stream: {len(pairs)} pairs, m and n in [{min(min(s) for s in sizes)}, {max(max(s) for s in sizes)}]")
    torch.manual_seed(0)
    for prec in ("bf16", "fp32"):
        base = {"precision": prec, "filter_threshold": 0.1}
        arms = {"eager": LightGlue(base).eval().to(DEV)}
        arms["cuda_graph"] = LightGlue({**base, "cuda_graph": True}).eval().to(DEV)
        arms[f"cuda_graph+capacity{CAP}"] = LightGlue({**base, "cuda_graph": True, "graph_capacity": CAP}).eval().to(DEV)
        for mdl in arms.values():
            mdl.load_state_dict(arms["eager"].state_dict())
        res = {}
        with torch.no_grad():
            for name, mdl in arms.items():  # alone, first pass: captures and peak memory (and the warm-up)
                res[name] = dict(zip(("captures", "peak_mb"), one_pass(mdl, pairs)))
            for name, mdl in arms.items():
                if name != "eager":
                    res[name].update(zip(("bit_equal_to_eager", "max_abs_d_log_assignment", "matches0_agree"),
                                         compare(arms["eager"], mdl, pairs)))
            names = list(arms)
            times = {name: [] for name in names}
            for w in range(args.windows):
                for j in range(len(names)):
                    name = names[(w + j) % len(names)]
                    times[name].append(timed_pass(arms[name], pairs))
        for name in names:
            ts = times[name]
            r = res[name]
            r.update(ms_median=round(statistics.median(ts), 4), ms_min=round(min(ts), 4), ms_max=round(max(ts), 4))
            print(f"{prec:4s} {name:22s} {r['ms_median']:.3f} ms per pair (min {r['ms_min']:.3f}, max {r['ms_max']:.3f})"
                  f"  captures per pass {r['captures']:3d}  peak {r['peak_mb']:8.1f} MB"
                  + (f"  bit-equal to eager: {r['bit_equal_to_eager']}"
                     + ("" if r["bit_equal_to_eager"] else
                        f" (max |d la| {r['max_abs_d_log_assignment']:.3g}, matches0 agree {r['matches0_agree']:.5f})")
                     if "bit_equal_to_eager" in r else ""))
            lines.append({"precision": prec, "arm": name, **{k: (round(v, 6) if isinstance(v, float) else v)
                                                             for k, v in r.items()}})
        del arms
        torch.cuda.empty_cache()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
