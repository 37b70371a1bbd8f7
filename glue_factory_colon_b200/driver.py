"""Batched, streamed pair driver for the B200 LightGlue (SURVEY.md 8(f) rank 1).

The reference calls the matcher once per dataloader batch from `TwoViewPipeline._forward`
(models/two_view_pipeline.py:326-335) between two `torch.cuda.synchronize()` calls (`_profile_call`, :78-102),
and its eval loops run at batch 1 (utils/export_predictions.py:36-90; eval/hpatches.py:46).  The kernels here
want tens of pairs per launch, and the model already takes per-pair keypoint counts (`num_keypoints0/1`), so
this driver does the part the call site cannot: it takes a stream of independent pairs with arbitrary keypoint
counts, groups them into padded batches under a pair and token budget, uploads batch i+1 from pinned host
memory on a copy stream while batch i runs, reads the matches back asynchronously, and yields one result dict
per pair, in input order, trimmed to the pair's own counts -- without a device-wide synchronize.

Host logic only: all compute is `LightGlue.forward` (C-ABI kernels).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, Iterable, Iterator, List, Optional, Sequence, Tuple

import torch


def _round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


def plan_batches(
    counts: Sequence[Tuple[int, int]],
    max_pairs: int = 64,
    max_tokens: int = 64 * 2 * 2048,
    bucket: int = 128,
    by_size: bool = False,
) -> List[List[int]]:
    """Greedy batching.  `counts[i] = (n0, n1)`.  A batch is closed when adding the next pair
    would exceed `max_pairs` or make the PADDED token count B * (N0p + N1p) exceed `max_tokens`
    (N0p / N1p = the batch maxima rounded up to `bucket`).  Every pair lands in exactly one batch; a single pair
    larger than the token budget gets a batch of its own.  Order-preserving by default; `by_size` visits the pairs
    largest first, so that a batch holds pairs of similar size: every kernel pads a batch to its largest pair, and
    the attention cost of the padding grows with its square."""
    if max_pairs < 1 or bucket < 1:
        raise ValueError("max_pairs and bucket must be positive")
    batches: List[List[int]] = []
    cur: List[int] = []
    m0 = m1 = 0
    visit = range(len(counts))
    if by_size:
        visit = sorted(visit, key=lambda i: (-max(counts[i]), -min(counts[i]), i))
    for i in visit:
        n0, n1 = counts[i]
        if n0 < 0 or n1 < 0:
            raise ValueError("negative keypoint count")
        c0, c1 = max(m0, _round_up(max(n0, 1), bucket)), max(m1, _round_up(max(n1, 1), bucket))
        if cur and (len(cur) + 1 > max_pairs or (len(cur) + 1) * (c0 + c1) > max_tokens):
            batches.append(cur)
            cur, c0, c1 = [], _round_up(max(n0, 1), bucket), _round_up(max(n1, 1), bucket)
        cur.append(i)
        m0, m1 = c0, c1
    if cur:
        batches.append(cur)
    return batches


def collate_pairs(pairs: Sequence[dict], bucket: int = 128, pin: bool = False) -> dict:
    """Zero-pads a list of single-pair dicts into one model input dict with `num_keypoints0/1`.

    A pair dict holds `keypoints0/1` [n,2], `descriptors0/1` [n,D] and optionally `image_size0/1` [2] (W,H),
    `scales0/1`, `oris0/1` [n].  Pairs without an image size cannot be mixed with pairs that have one."""
    B = len(pairs)
    n0 = [int(p["keypoints0"].shape[0]) for p in pairs]
    n1 = [int(p["keypoints1"].shape[0]) for p in pairs]
    N0, N1 = _round_up(max(max(n0), 1), bucket), _round_up(max(max(n1), 1), bucket)
    D = int(pairs[0]["descriptors0"].shape[-1])

    def buf(*shape, dtype=torch.float32):
        t = torch.zeros(*shape, dtype=dtype)
        return t.pin_memory() if pin else t

    out = {
        "keypoints0": buf(B, N0, 2), "keypoints1": buf(B, N1, 2),
        "descriptors0": buf(B, N0, D), "descriptors1": buf(B, N1, D),
        "num_keypoints0": torch.tensor(n0, dtype=torch.int32), "num_keypoints1": torch.tensor(n1, dtype=torch.int32),
        "view0": {}, "view1": {},
    }
    have_size = ["image_size0" in p for p in pairs]
    if any(have_size) and not all(have_size):
        raise ValueError("either every pair of a batch carries image_size0/1 or none does")
    if all(have_size):
        out["view0"]["image_size"] = buf(B, 2)
        out["view1"]["image_size"] = buf(B, 2)
    extra = [k for k in ("scales0", "scales1", "oris0", "oris1") if k in pairs[0]]
    for k in extra:
        out[k] = buf(B, N0 if k.endswith("0") else N1)
    for b, p in enumerate(pairs):
        out["keypoints0"][b, : n0[b]] = p["keypoints0"]
        out["keypoints1"][b, : n1[b]] = p["keypoints1"]
        out["descriptors0"][b, : n0[b]] = p["descriptors0"]
        out["descriptors1"][b, : n1[b]] = p["descriptors1"]
        if all(have_size):
            out["view0"]["image_size"][b] = torch.as_tensor(p["image_size0"], dtype=torch.float32)
            out["view1"]["image_size"][b] = torch.as_tensor(p["image_size1"], dtype=torch.float32)
        for k in extra:
            n = n0[b] if k.endswith("0") else n1[b]
            out[k][b, :n] = p[k].reshape(-1)
    return out


def crop_log_assignment(scores: torch.Tensor, n0: int, n1: int) -> torch.Tensor:
    """[..., R, C] padded score matrices (valid block, dustbin column C-1, dustbin row R-1; leading dimensions, such as
    a batch, are kept) -> the [..., n0+1, n1+1] matrices the reference would have produced for the un-padded pairs."""
    R, C = scores.shape[-2:]
    out = scores.new_empty(*scores.shape[:-2], n0 + 1, n1 + 1)
    out[..., :n0, :n1] = scores[..., :n0, :n1]
    out[..., :n0, n1] = scores[..., :n0, C - 1]
    out[..., n0, :n1] = scores[..., R - 1, :n1]
    out[..., n0, n1] = scores[..., R - 1, C - 1]
    return out


@dataclass
class _InFlight:
    idx: List[int]
    counts: List[Tuple[int, int]]
    host: Dict[str, torch.Tensor]
    done: torch.cuda.Event
    scores: Optional[torch.Tensor]


class BatchedPairMatcher:
    """Streams independent pairs through a `LightGlue` module in padded batches.

    >>> drv = BatchedPairMatcher(model, max_pairs=64)
    >>> for res in drv.match(pairs):          # pairs: iterable of per-pair dicts (CPU tensors)
    ...     res["matches0"], res["matching_scores0"]   # CPU tensors trimmed to the pair's n0 / n1
    """

    D2H_KEYS = ("matches0", "matches1", "matching_scores0", "matching_scores1")

    def __init__(self, matcher, max_pairs: int = 64, max_tokens: int = 64 * 2 * 2048, bucket: int = 128,
                 device: Optional[torch.device] = None, return_log_assignment: bool = False, window: int = 256,
                 sort_by_size: bool = True):
        self.matcher = matcher
        self.max_pairs, self.max_tokens, self.bucket = max_pairs, max_tokens, bucket
        self.device = torch.device(device) if device is not None else next(matcher.parameters()).device
        if self.device.type != "cuda":
            raise RuntimeError("BatchedPairMatcher needs the matcher on a CUDA device (there is no CPU path)")
        self.return_log_assignment = return_log_assignment
        self.window = max(window, max_pairs)  # pairs pulled from the iterator before batches are planned
        self.sort_by_size = sort_by_size      # batches of similar-sized pairs within a window (results stay in input order)

    # ------------------------------------------------------------------------------------------
    def _upload(self, host: dict, stream: torch.cuda.Stream):
        from .synthetic import to_device

        counts = {k: host[k] for k in ("num_keypoints0", "num_keypoints1")}
        with torch.cuda.stream(stream):
            dev = to_device({k: v for k, v in host.items() if k not in counts}, self.device, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(stream)
        dev.update(counts)  # the model reads the per-pair counts on the host: keep them there (no device round trip)
        return dev, ev

    def _launch(self, dev: dict, ready: torch.cuda.Event, idx, counts, compute: torch.cuda.Stream) -> _InFlight:
        compute.wait_event(ready)
        out = self.matcher(dev)
        host = {}
        for k in self.D2H_KEYS:
            h = torch.empty(out[k].shape, dtype=out[k].dtype).pin_memory()
            h.copy_(out[k], non_blocking=True)
            host[k] = h
        # every uploaded tensor (nested view dicts included: image_size, scales, oris are read by the compute-stream
        # kernels without a copy) was allocated on the copy stream and is consumed on `compute`
        def mark(obj):
            if isinstance(obj, torch.Tensor):
                if obj.is_cuda:
                    obj.record_stream(compute)
            elif isinstance(obj, dict):
                for v in obj.values():
                    mark(v)

        mark(dev)
        done = torch.cuda.Event()
        done.record(compute)
        return _InFlight(list(idx), list(counts), host, done, out["log_assignment"] if self.return_log_assignment else None)

    def _emit(self, fl: _InFlight) -> Iterator[Tuple[int, dict]]:
        fl.done.synchronize()  # this batch only; later batches keep running
        for b, (i, (n0, n1)) in enumerate(zip(fl.idx, fl.counts)):
            res = {
                "matches0": fl.host["matches0"][b, :n0].clone(),
                "matches1": fl.host["matches1"][b, :n1].clone(),
                "matching_scores0": fl.host["matching_scores0"][b, :n0].clone(),
                "matching_scores1": fl.host["matching_scores1"][b, :n1].clone(),
            }
            if fl.scores is not None:
                res["log_assignment"] = crop_log_assignment(fl.scores[b], n0, n1)
            yield i, res

    # ------------------------------------------------------------------------------------------
    @torch.no_grad()
    def match(self, pairs: Iterable[dict]) -> Iterator[dict]:
        """Yields one result dict per input pair, in input order."""
        copy_stream = torch.cuda.Stream(device=self.device)
        compute = torch.cuda.current_stream(self.device)
        it = iter(pairs)
        base = 0
        pending: Dict[int, dict] = {}
        next_out = 0
        in_flight: List[_InFlight] = []

        def drain(keep: int):
            nonlocal next_out
            while len(in_flight) > keep:
                for i, res in self._emit(in_flight.pop(0)):
                    pending[i] = res
                while next_out in pending:
                    yield pending.pop(next_out)
                    next_out += 1

        while True:
            chunk = []
            for p in it:
                chunk.append(p)
                if len(chunk) >= self.window:
                    break
            if not chunk:
                break
            counts = [(int(p["keypoints0"].shape[0]), int(p["keypoints1"].shape[0])) for p in chunk]
            plan = plan_batches(counts, self.max_pairs, self.max_tokens, self.bucket, by_size=self.sort_by_size)
            staged = None
            for bi, idx in enumerate(plan):
                if staged is None:
                    host = collate_pairs([chunk[i] for i in idx], self.bucket, pin=True)
                    staged = self._upload(host, copy_stream)
                dev, ready = staged
                # stage the next batch while this one is queued behind the previous launches
                staged = None
                if bi + 1 < len(plan):
                    nhost = collate_pairs([chunk[i] for i in plan[bi + 1]], self.bucket, pin=True)
                    staged = self._upload(nhost, copy_stream)
                in_flight.append(self._launch(dev, ready, [base + i for i in idx], [counts[i] for i in idx], compute))
                yield from drain(keep=2)  # at most two batches of results outstanding
            base += len(chunk)
        yield from drain(keep=0)
