"""conf.graph_capacity (a B200 extension of conf.cuda_graph): one CUDA graph of lgb200_match captured at B x K x K serves
every input with max(m, n) <= K, with or without num_keypoints0/1.  Its outputs are bit-equal to the eager forward of
the input zero-padded to K with the counts set, cropped to the input's shapes."""
import pytest
import torch

from glue_factory_colon_b200 import LightGlue, _abi
from glue_factory_colon_b200.driver import crop_log_assignment
from glue_factory_colon_b200.lightglue import _CapacityGraph
from glue_factory_colon_b200.synthetic import make_pairs

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
K = 1024
KEYS = ("matches0", "matches1", "matching_scores0", "matching_scores1", "ref_descriptors0", "ref_descriptors1",
        "log_assignment", "prune0", "prune1")


def _models(precision, seed=5, capacity=K, **conf):
    """(eager, cuda_graph + graph_capacity, cuda_graph alone), same weights."""
    torch.manual_seed(seed)
    base = {"filter_threshold": 0.1, "precision": precision, **conf}
    eager = LightGlue(base).eval().to(DEV)
    cap = LightGlue({**base, "cuda_graph": True, "graph_capacity": capacity}).eval().to(DEV)
    graph = LightGlue({**base, "cuda_graph": True}).eval().to(DEV)
    cap.load_state_dict(eager.state_dict())
    graph.load_state_dict(eager.state_dict())
    return eager, cap, graph


def _capacity_entries(model):
    return [e for e in model._graphs.values() if isinstance(e, _CapacityGraph)]


def _pair(B, m, n, seed, with_size=True, counts=None, **kw):
    d = make_pairs(B, m, n, seed=seed, with_size=with_size, device=DEV, **kw)
    if counts is not None:
        d["num_keypoints0"], d["num_keypoints1"] = torch.tensor(counts[0]), torch.tensor(counts[1])
    return d


def _padded(data, cap):
    """The input zero-padded to `cap` keypoints per image, with num_keypoints0/1 = min(given, m) or m."""
    out = dict(data)
    B = data["keypoints0"].shape[0]
    for i in (0, 1):
        c = data[f"keypoints{i}"].shape[1]
        for k in (f"keypoints{i}", f"descriptors{i}", f"scales{i}", f"oris{i}"):
            if k in data:
                t = data[k]
                out[k] = torch.cat([t, t.new_zeros(B, cap - c, *t.shape[2:])], 1)
        cnt = data.get(f"num_keypoints{i}")
        out[f"num_keypoints{i}"] = torch.full((B,), c) if cnt is None else torch.as_tensor(cnt).clamp(max=c)
    return out


def _crop(out, m, n):
    """Outputs of a forward at capacity cropped to an m x n input (dustbins moved to row m / column n)."""
    return {
        "matches0": out["matches0"][:, :m], "matches1": out["matches1"][:, :n],
        "matching_scores0": out["matching_scores0"][:, :m], "matching_scores1": out["matching_scores1"][:, :n],
        "ref_descriptors0": out["ref_descriptors0"][:, :, :m], "ref_descriptors1": out["ref_descriptors1"][:, :, :n],
        "log_assignment": crop_log_assignment(out["log_assignment"], m, n),
        "prune0": out["prune0"][:, :m], "prune1": out["prune1"][:, :n],
    }


def _reference_at_capacity(eager, data, cap=K):
    m, n = data["keypoints0"].shape[1], data["keypoints1"].shape[1]
    return _crop(eager(_padded(data, cap)), m, n)


def _differences(got, want):
    """Keys whose shape, dtype or bits differ -> description (max |difference| for float outputs)."""
    bad = {}
    assert set(got) == set(want), (sorted(got), sorted(want))
    for k in want:
        g, w = got[k], want[k]
        if g.shape != w.shape or g.dtype != w.dtype:
            bad[k] = f"shape / dtype {tuple(g.shape)} {g.dtype} vs {tuple(w.shape)} {w.dtype}"
        elif not torch.equal(g, w):
            if g.is_floating_point():
                fin = torch.isfinite(w) & torch.isfinite(g)
                dif = (g.double() - w.double())[fin].abs()
                bad[k] = (f"max |d| {float(dif.max()) if dif.numel() else 0.0:.3g}, "
                          f"{int((g != w).sum())} of {w.numel()} differ, non-finite mismatch "
                          f"{int((torch.isfinite(w) != torch.isfinite(g)).sum())}")
            else:
                bad[k] = f"{int((g != w).sum())} of {w.numel()} differ"
    return bad


def _assert_same(got, want, what):
    bad = _differences(got, want)
    assert not bad, f"{what}: {bad}"


CASES = {
    "700x311": (dict(), dict(B=1, m=700, n=311)),
    "1024x1024": (dict(), dict(B=1, m=1024, n=1024)),
    "5x0": (dict(), dict(B=1, m=5, n=0)),
    "1x1": (dict(), dict(B=1, m=1, n=1)),
    "dim128_scale_ori": (dict(input_dim=128, add_scale_ori=True), dict(B=1, m=700, n=311, dim=128, scale_ori=True)),
    "B3_counts": (dict(), dict(B=3, m=600, n=900, counts=([600, 129, 1], [77, 900, 260]))),
}
CASE_IDS = [f"{c}-{'size' if s else 'nosize'}" for c in CASES for s in (True, False)
            if s or c in ("700x311", "1024x1024", "5x0", "1x1")]


def _case(cid, seed=21):
    name, size = cid.rsplit("-", 1)
    conf, kw = CASES[name]
    kw = dict(kw)
    return conf, _pair(kw.pop("B"), kw.pop("m"), kw.pop("n"), seed, with_size=size == "size", **kw)


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("cid", CASE_IDS)
def test_bit_equal_to_the_forward_at_capacity(precision, cid):
    conf, data = _case(cid)
    eager, cap, _ = _models(precision, **conf)
    got = cap(data)
    assert len(cap._graphs) == 1 and len(_capacity_entries(cap)) == 1
    _assert_same(got, _reference_at_capacity(eager, data), f"{precision} {cid}")
    got = cap(data)  # a replay of the kept graph
    _assert_same(got, _reference_at_capacity(eager, data), f"{precision} {cid}, second call")


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("cid", CASE_IDS)
def test_against_the_exact_shape_forward(precision, cid):
    """Does turning graph_capacity on change the results of the eager forward at the input's own shape?  No: bit-equal
    in both precisions.  An image without keypoints is the exception: the eager forward at that shape raises (a tensor
    with no rows has no data pointer, and the library refuses NULL inputs), the capacity graph returns what the
    eager forward gives for the padded input with the counts (test_bit_equal_to_the_forward_at_capacity)."""
    conf, data = _case(cid)
    eager, cap, _ = _models(precision, **conf)
    got = cap(data)
    B, m, n = data["keypoints0"].shape[0], data["keypoints0"].shape[1], data["keypoints1"].shape[1]
    if min(m, n) == 0:
        with pytest.raises(_abi.LightGlueB200Error, match="NULL"):
            eager(data)
        assert got["log_assignment"].shape == (B, m + 1, n + 1)
        assert bool((got["matches0"] == -1).all()) and bool((got["matching_scores0"] == 0).all())
        return
    want = eager(data)
    bad = _differences(got, want)
    print(f"[capacity vs exact] {precision} {cid}: {bad or 'bit-equal'}")
    assert not bad, f"{precision} {cid}: {bad}"


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_one_graph_serves_a_stream(precision):
    eager, cap, _ = _models(precision)
    g = torch.Generator().manual_seed(31)
    sizes = torch.randint(1, K + 1, (30, 2), generator=g).tolist()
    sizes[7], sizes[8] = [K, K], [3, 1]  # full capacity, then a tiny pair right after it
    for i, (m, n) in enumerate(sizes):
        counts = None
        if i % 3 == 2:  # a third of the calls carry counts (some past m / n: clamped)
            counts = ([max(m - 17 * i, 0)], [n + 5])
        data = _pair(1, m, n, 100 + i, counts=counts)
        got = cap(data)
        _assert_same(got, _reference_at_capacity(eager, data), f"{precision} call {i} ({m} x {n}, counts {counts})")
        del got, data
        if i == 1:
            torch.cuda.synchronize()
            mem = torch.cuda.memory_allocated(DEV)
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated(DEV) == mem
    assert len(cap._graphs) == 1 and len(_capacity_entries(cap)) == 1


def test_returned_tensors_are_fresh():
    eager, cap, _ = _models("bf16")
    d1, d2 = _pair(1, 700, 311, 41), _pair(1, 300, 900, 42)
    o1 = cap(d1)
    keep = {k: v.clone() for k, v in o1.items()}
    cap(d2)
    _assert_same(o1, keep, "after a later replay")
    # graph_static_outputs: the graph's own buffers only when they have the output shapes (m == n == K, no counts)
    cap.conf.graph_static_outputs = True
    entry = _capacity_entries(cap)[0]
    full = _pair(1, K, K, 43)
    o = cap(full)
    assert o["log_assignment"].data_ptr() == entry.out["log_assignment"].data_ptr()
    _assert_same(o, _reference_at_capacity(eager, full), "static outputs")
    o = cap(dict(full, num_keypoints0=torch.tensor([K]), num_keypoints1=torch.tensor([K])))
    assert o["log_assignment"].data_ptr() != entry.out["log_assignment"].data_ptr()
    o = cap(d1)
    assert o["matches0"].data_ptr() != entry.out["matches0"].data_ptr()
    _assert_same(o, _reference_at_capacity(eager, d1), "static outputs, smaller input")


def test_recapture_after_a_weight_change_and_precision_switches():
    eager, cap, _ = _models("fp32")
    data = _pair(1, 700, 311, 51)
    _assert_same(cap(data), _reference_at_capacity(eager, data), "first capture")
    with torch.no_grad():
        cap.log_assignment[-1].matchability.bias.add_(0.5)
        eager.log_assignment[-1].matchability.bias.add_(0.5)
    _assert_same(cap(data), _reference_at_capacity(eager, data), "after the weight change")
    assert len(_capacity_entries(cap)) == 2
    cap._graphs.clear()
    want = {}
    for prec in ("fp32", "bf16"):
        eager.conf.precision = prec
        want[prec] = _reference_at_capacity(eager, data)
    for rnd, prec in enumerate(["fp32", "bf16", "fp32", "bf16", "fp32"]):
        cap.conf.precision = prec
        junk = [torch.randn(1 << 20, device=DEV) for _ in range(8)]  # a freed pack would be reused
        _assert_same(cap(data), want[prec], f"round {rnd} ({prec})")
        del junk
    assert len(_capacity_entries(cap)) == 2  # one capture per precision, replayed after the switches


def _fallback_equal(cap, graph, data):
    got, want = cap(data), graph(data)
    _assert_same({k: v.detach() for k, v in got.items()}, {k: v.detach() for k, v in want.items()}, "fallback")
    assert not _capacity_entries(cap)


def test_fallbacks_take_the_existing_paths():
    # larger than the capacity: the per-signature capture, or eager with counts
    _, cap, graph = _models("bf16", capacity=256)
    _fallback_equal(cap, graph, _pair(1, 300, 200, 61))
    assert len(cap._graphs) == 1
    _fallback_equal(cap, graph, _pair(1, 300, 200, 62, counts=([250], [200])))
    assert len(cap._graphs) == 1
    # fp32_simt
    _, cap, graph = _models("fp32_simt", capacity=512)
    _fallback_equal(cap, graph, _pair(1, 300, 200, 63))
    # adaptive depth / width: the per-signature capture of the transformer stack
    _, cap, graph = _models("bf16", capacity=512, depth_confidence=0.95, width_confidence=0.99)
    _fallback_equal(cap, graph, _pair(1, 300, 200, 64))
    assert len(cap._graphs) == 1
    # a training step (module in training mode, autograd on)
    _, cap, graph = _models("fp32", capacity=512, n_layers=3)
    cap.train(), graph.train()
    _fallback_equal(cap, graph, _pair(1, 300, 200, 65))
    assert not cap._graphs


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_a_replay_makes_no_library_call(precision):
    lib = _abi.load()
    eager, cap, _ = _models(precision)
    cap(_pair(1, 700, 311, 71))  # the capture
    data = _pair(1, 512, 1000, 72, counts=([400], [1000]))
    torch.cuda.synchronize()
    n0 = lib.lgb200_launch_count()
    got = cap(data)
    torch.cuda.synchronize()
    assert lib.lgb200_launch_count() == n0
    ref = _reference_at_capacity(eager, data)
    assert lib.lgb200_launch_count() > n0  # (the counter does count the eager forward's launches)
    _assert_same(got, ref, precision)
