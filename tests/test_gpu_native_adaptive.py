"""GPU tests of adaptive depth and width behind the C ABI (lgb200_pack_weights_adaptive, lgb200_match_adaptive):
bit-equal to LightGlue.forward with the same conf in both precisions (in its shapes: log_assignment cropped to the
largest pruned counts, ref_descriptors on each pair's own rows), a batch whose pairs exit at different layers, the
everything-pruned corner, the path without adaptive modes against lgb200_match, native packing, and one CUDA graph
captured at a capacity replayed with other inputs and counts."""
import ctypes

import pytest
import torch

from test_gpu_native_match import Native, _bits, _cfg, _inputs, _model, _native_pack, _python, _ulp_close
from test_gpu_native_match import FOLDED
from test_gpu_train_ragged import _padded, _pairs
from glue_factory_colon_b200 import _abi
from glue_factory_colon_b200._abi import BF16, AdaptiveConfig, check, ptr
from glue_factory_colon_b200.driver import crop_log_assignment
from glue_factory_colon_b200.synthetic import make_pairs
from glue_factory_colon_b200.weights import NATIVE_LAYER_ENTRIES, native_table

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
MODES = {"depth+width": (0.95, 0.99), "width": (-1.0, 0.99), "depth": (0.95, -1.0)}


class NativeAdaptive:
    """Output buffers, workspace and adaptive table of lgb200_match_adaptive at a fixed capacity B x m x n."""

    def __init__(self, model, B, m, n, table=None):
        self.lib = _abi.load()
        self.cfg = _cfg(model)
        c = model.conf
        self.acfg = AdaptiveConfig(float(c.depth_confidence), float(c.width_confidence))
        self.table, self.keep = native_table(model, self.cfg.precision, adaptive=True) if table is None else (table, None)
        self.B, self.m, self.n = B, m, n
        nb = ctypes.c_longlong(0)
        check(self.lib.lgb200_match_adaptive_workspace(ctypes.byref(self.cfg), B, m, n, ctypes.byref(nb)), "workspace")
        self.ws = torch.empty(nb.value, dtype=torch.uint8, device=DEV)
        act = torch.bfloat16 if self.cfg.precision == BF16 else torch.float32
        i64, f32, i32 = (dict(device=DEV, dtype=d) for d in (torch.int64, torch.float32, torch.int32))
        self.out = {
            "matches0": torch.empty(B, m, **i64), "matches1": torch.empty(B, n, **i64),
            "matching_scores0": torch.empty(B, m, **f32), "matching_scores1": torch.empty(B, n, **f32),
            "log_assignment": torch.empty(B, m + 1, n + 1, **f32),
            "ref_descriptors0": torch.empty(B, m, 256, device=DEV, dtype=act),
            "ref_descriptors1": torch.empty(B, n, 256, device=DEV, dtype=act),
            "prune0": torch.empty(B, m, **i32), "prune1": torch.empty(B, n, **i32),
            "exit_layer": torch.empty(B, **i32), "final_counts": torch.empty(B, 2, **i32),
        }

    def __call__(self, ins, stream=None):
        o = self.out
        st = (stream or torch.cuda.current_stream(DEV)).cuda_stream
        check(self.lib.lgb200_match_adaptive(
            ctypes.byref(self.cfg), ctypes.byref(self.acfg), self.table, self.B, self.m, self.n, ptr(ins["kpts0"]),
            ptr(ins["kpts1"]), ptr(ins["desc0"]), ptr(ins["desc1"]), ptr(ins["size0"]), ptr(ins["size1"]),
            ptr(ins["counts0"]), ptr(ins["counts1"]), ptr(o["matches0"]), ptr(o["matches1"]),
            ptr(o["matching_scores0"]), ptr(o["matching_scores1"]), ptr(o["log_assignment"]),
            ptr(o["ref_descriptors0"]), ptr(o["ref_descriptors1"]), ptr(o["prune0"]), ptr(o["prune1"]),
            ptr(o["exit_layer"]), ptr(o["final_counts"]), ptr(self.ws), self.ws.numel(), st), "lgb200_match_adaptive")
        return o


def _adaptive_model(precision, mode, seed=6, token_bias=3.0, match_bias=-4.5, **conf):
    """Heads that prune and (depth) exit, as in tools/adaptive_bench.py: token confidence high from layer 4 (or the
    last layer that has a head), matchability low on even layers."""
    depth, width = MODES[mode]
    model = _model(precision, seed=seed, depth_confidence=depth, width_confidence=width, filter_threshold=0.1, **conf)
    L = model.conf.n_layers
    with torch.no_grad():
        for i in range(L - 1):
            model.token_confidence[i].token[0].bias.fill_(token_bias if i >= min(4, L - 2) else -token_bias)
            model.log_assignment[i].matchability.bias.fill_(match_bias if i % 2 == 0 else 0.0)
    return model


def _run(model, data):
    B, m, _ = data["keypoints0"].shape
    nat = NativeAdaptive(model, B, m, data["keypoints1"].shape[1])
    out = nat(_inputs(model, data))
    torch.cuda.synchronize()
    return out


def _assert_equal_to_eager(nat, ref, pruned, what):
    """nat (capacity layout) against LightGlue.forward's outputs, bit for bit, in the eager shapes."""
    k = nat["final_counts"].cpu()
    la = nat["log_assignment"]
    if pruned:
        la = crop_log_assignment(la, int(k[:, 0].max()), int(k[:, 1].max()))
    assert la.shape == ref["log_assignment"].shape, (what, la.shape, ref["log_assignment"].shape)
    assert torch.equal(_bits(la), _bits(ref["log_assignment"])), f"{what}: log_assignment differs"
    for key in ("matches0", "matches1", "matching_scores0", "matching_scores1"):
        assert torch.equal(_bits(nat[key]), _bits(ref[key])), f"{what}: {key} differs"
    for i in (0, 1):
        p = nat[f"prune{i}"].to(ref[f"prune{i}"].dtype)
        assert torch.equal(p, ref[f"prune{i}"]), f"{what}: prune{i} differs"
        d, r = nat[f"ref_descriptors{i}"], ref[f"ref_descriptors{i}"][:, -1]
        for b in range(d.shape[0]):
            kb = int(k[b, i])
            assert torch.equal(_bits(d[b, :kb]), _bits(r[b, :kb])), f"{what}: ref_descriptors{i} pair {b} differs"
            assert not d[b, kb:].any(), f"{what}: ref_descriptors{i} pair {b} not zero past its count"


def _drop_sizes(data):
    data["view0"], data["view1"] = {}, {}
    return data


CASES = {
    "1x512x480": (dict(), lambda: make_pairs(B=1, n0=512, n1=480, seed=51)),
    "1x512x480_nosize": (dict(), lambda: _drop_sizes(make_pairs(B=1, n0=512, n1=480, seed=52))),
    "3x384x384": (dict(), lambda: make_pairs(B=3, n0=384, n1=384, seed=53)),
    "padded_counts": (dict(), lambda: _padded(_pairs([600, 129, 1], [77, 900, 260]), 600, 900)),
    "dim128_scale_ori": (dict(input_dim=128, add_scale_ori=True, n_layers=3),
                         lambda: make_pairs(B=2, n0=200, n1=333, seed=3, dim=128, scale_ori=True)),
    "3_layers": (dict(n_layers=3), lambda: make_pairs(B=2, n0=512, n1=256, seed=4)),
}


@pytest.mark.parametrize("mode", sorted(MODES))
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_bit_equal_to_the_python_forward(case, precision, mode):
    conf, make = CASES[case]
    model = _adaptive_model(precision, mode, **conf)
    data = make()
    nat, ref = _run(model, data), _python(model, data)
    _assert_equal_to_eager(nat, ref, "width" in mode, f"{precision} {mode} {case}")
    L = model.conf.n_layers
    ex = nat["exit_layer"].cpu()
    assert bool(((ex >= 0) & (ex <= L - 1)).all())
    if mode == "width":
        assert bool((ex == L - 1).all())
    if case == "1x512x480":  # the heads act: the pair exits at layer 4 / (width alone) even layers prune
        if "depth" in mode:
            assert int(ex.min()) == 4
        else:
            assert int(nat["final_counts"].sum()) < 512 + 480


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_pairs_exiting_at_different_layers(precision):
    """One batch, three pairs: one confident from the first layer on (exits at layer 0), one never confident (runs to
    the last layer), one with half of its points confident (pruned where matchability is low, no exit).  The token
    heads read one channel, which the descriptors bias per pair; the residual stream carries its sign."""
    model = _adaptive_model(precision, "depth+width", match_bias=-10.0)
    L, c = model.conf.n_layers, 17
    with torch.no_grad():
        for i in range(L - 1):
            model.token_confidence[i].token[0].weight.zero_()
            model.token_confidence[i].token[0].weight[0, c] = 10.0
            model.token_confidence[i].token[0].bias.zero_()
    data = make_pairs(B=3, n0=512, n1=480, seed=61)
    g = torch.Generator().manual_seed(0)
    for i in (0, 1):
        d = data[f"descriptors{i}"]
        d[0, :, c] += 5.0
        d[1, :, c] -= 5.0
        d[2, :, c] += 5.0 * (torch.randint(0, 2, (d.shape[1],), generator=g).float() * 2 - 1)
    nat, ref = _run(model, data), _python(model, data)
    _assert_equal_to_eager(nat, ref, True, f"{precision} ragged exit")
    ex, k = nat["exit_layer"].cpu(), nat["final_counts"].cpu()
    assert len(set(ex.tolist())) >= 2, ex
    assert len({tuple(r) for r in k.tolist()}) >= 2, k
    for b in range(3):  # each pair's block equals its own B = 1 forward
        one = {key: (v[b:b + 1] if isinstance(v, torch.Tensor) else {"image_size": v["image_size"][b:b + 1]})
               for key, v in data.items() if key.startswith(("keypoints", "descriptors", "view"))}
        r1 = _python(model, one)
        k0, k1 = int(k[b, 0]), int(k[b, 1])
        la = crop_log_assignment(nat["log_assignment"][b:b + 1], k0, k1)
        assert torch.equal(_bits(la), _bits(r1["log_assignment"])), f"{precision} pair {b}: log_assignment"
        for key in ("matches0", "matches1", "matching_scores0", "matching_scores1"):
            assert torch.equal(_bits(nat[key][b:b + 1]), _bits(r1[key])), f"{precision} pair {b}: {key}"
        for i, kk in ((0, k0), (1, k1)):
            assert torch.equal(_bits(nat[f"ref_descriptors{i}"][b, :kk]), _bits(r1[f"ref_descriptors{i}"][0, -1, :kk]))
            assert torch.equal(nat[f"prune{i}"][b:b + 1].long(), r1[f"prune{i}"])


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_everything_pruned(precision):
    model = _adaptive_model(precision, "width")
    with torch.no_grad():
        for i in range(model.conf.n_layers - 1):
            model.log_assignment[i].matchability.bias.fill_(-10.0)
    data = make_pairs(B=2, n0=300, n1=260, seed=62)
    nat, ref = _run(model, data), _python(model, data)
    assert not nat["final_counts"].any()
    assert ref["log_assignment"].shape == (2, 1, 1)
    _assert_equal_to_eager(nat, ref, True, f"{precision} everything pruned")
    assert bool((nat["matches0"] == -1).all()) and bool((nat["matches1"] == -1).all())


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_without_adaptive_modes_equals_lgb200_match(precision):
    model = _model(precision, n_layers=3, filter_threshold=0.1)
    data = _padded(_pairs([300, 129, 1], [260, 260, 77]), 320, 280)
    ins = _inputs(model, data)
    nat = NativeAdaptive(model, 3, 320, 280)
    plain = Native(model, 3, 320, 280)
    nat(ins)
    plain(ins)
    torch.cuda.synchronize()
    for key, v in plain.out.items():
        assert torch.equal(_bits(nat.out[key]), _bits(v)), f"{precision}: {key} differs from lgb200_match"
    assert bool((nat.out["prune0"] == 3).all()) and bool((nat.out["prune1"] == 3).all())
    assert bool((nat.out["exit_layer"] == 2).all())
    counts = torch.stack([data["num_keypoints0"], data["num_keypoints1"]], 1).to(DEV, torch.int32)
    assert torch.equal(nat.out["final_counts"], counts)


def _native_pack_adaptive(model, cfg):
    lib = _abi.load()
    sd = {k: v.detach().to(DEV, torch.float32).contiguous() for k, v in model.state_dict().items()}
    names = (ctypes.c_char_p * len(sd))(*[k.encode() for k in sd])
    ptrs = (ctypes.c_void_p * len(sd))(*[v.data_ptr() for v in sd.values()])
    e, nb = ctypes.c_int(0), ctypes.c_longlong(0)
    check(lib.lgb200_adaptive_table_size(ctypes.byref(cfg), ctypes.byref(e), ctypes.byref(nb)), "table_size")
    buf = torch.full((nb.value,), 0xFF, dtype=torch.uint8, device=DEV)
    table = (ctypes.c_void_p * e.value)()
    check(lib.lgb200_pack_weights_adaptive(ctypes.byref(cfg), len(sd), names, ptrs, ptr(buf), nb.value, table,
                                           torch.cuda.current_stream(DEV).cuda_stream), "pack_weights_adaptive")
    torch.cuda.synchronize()
    return table, buf


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("conf", [dict(), dict(input_dim=128, add_scale_ori=True, n_layers=3)], ids=["default", "dim128"])
def test_native_packing_against_pack(precision, conf):
    model = _adaptive_model(precision, "depth+width", **conf)
    cfg = _cfg(model)
    table, buf = _native_pack_adaptive(model, cfg)
    base_table, base_buf = _native_pack(model, cfg)
    ref_table, ref = native_table(model, cfg.precision, adaptive=True)
    assert len(table) == len(ref_table) == len(base_table) + 6 * (model.conf.n_layers - 1)
    assert torch.equal(buf[:base_buf.numel()], base_buf)  # the prefix is lgb200_pack_weights' pack, byte for byte
    assert all(table[i] - buf.data_ptr() == base_table[i] - base_buf.data_ptr() for i in range(len(base_table)))
    n_layer_entries = len(NATIVE_LAYER_ENTRIES) * model.conf.n_layers
    for idx, t in enumerate(ref):
        nbytes = t.numel() * t.element_size()
        off = table[idx] - buf.data_ptr()
        assert off % 256 == 0 and 0 <= off and off + nbytes <= buf.numel()
        nat = buf[off:off + nbytes].view(t.dtype).view(t.shape)
        if torch.equal(_bits(nat), _bits(t)):
            continue
        folded = idx < n_layer_entries and idx % len(NATIVE_LAYER_ENTRIES) in FOLDED
        assert folded, f"entry {idx} differs and is not a folded FFN1 entry"
        assert _ulp_close(nat, t, t.dtype == torch.float16), f"entry {idx}: more than 1 ulp from _pack"
    # a forward on the native pack exits where the forward on _pack's table does (the token heads are bit-equal)
    data = make_pairs(B=1, n0=512, n1=480, seed=63, dim=model.conf.input_dim, scale_ori=model.conf.add_scale_ori)
    a = NativeAdaptive(model, 1, 512, 480, table=table)(_inputs(model, data))
    torch.cuda.synchronize()
    assert torch.equal(a["exit_layer"], _run(model, data)["exit_layer"])


def _zero_padded(data, cap):
    """data (B = 1) written into capacity-sized inputs, zeros past its rows, with the counts."""
    out = {}
    for i in (0, 1):
        for key in (f"keypoints{i}", f"descriptors{i}"):
            t = data[key]
            z = t.new_zeros(t.shape[0], cap, t.shape[2])
            z[:, :t.shape[1]] = t
            out[key] = z
        out[f"view{i}"] = data[f"view{i}"]
        out[f"num_keypoints{i}"] = torch.tensor([data[f"keypoints{i}"].shape[1]])
    return out


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_graph_capture_at_capacity_replays_any_counts(precision):
    model = _adaptive_model(precision, "depth+width")
    lib = _abi.load()
    cap, L = 1024, model.conf.n_layers
    nat = NativeAdaptive(model, 1, cap, cap)
    eager = NativeAdaptive(model, 1, cap, cap)
    first = _zero_padded(make_pairs(B=1, n0=cap, n1=cap, seed=70), cap)
    static = _inputs(model, first)
    nat(static)  # outside the capture: lazy initialisation
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        nat(static)
    for seed, (c0, c1) in ((71, (1024, 1024)), (72, (700, 311)), (73, (5, 0))):
        if c1 > 0:
            small = make_pairs(B=1, n0=c0, n1=c1, seed=seed)
            padded = _zero_padded(small, cap)
        else:  # (an empty image has no exact-shape forward: its tensor has no data pointer)
            small = None
            padded = make_pairs(B=1, n0=cap, n1=cap, seed=seed)
            padded["num_keypoints0"], padded["num_keypoints1"] = torch.tensor([c0]), torch.tensor([c1])
        new = _inputs(model, padded)
        for k, t in new.items():
            static[k].copy_(t)
        graph.replay()
        torch.cuda.synchronize()
        assert int(nat.out["final_counts"][0, 0]) <= c0 and int(nat.out["final_counts"][0, 1]) <= c1
        ref = _python(model, padded)
        _assert_equal_to_eager(nat.out, ref, True, f"{precision} replay {c0}/{c1} vs padded forward")
        if small is not None:
            ref_s = _python(model, small)
            got = {k: v[:, :c0] if k.endswith("0") and k != "final_counts" else
                   v[:, :c1] if k.endswith("1") else v for k, v in nat.out.items()}
            _assert_equal_to_eager(got, ref_s, True, f"{precision} replay {c0}/{c1} vs exact-shape forward")
        eager(new)
        torch.cuda.synchronize()
        _assert_equal_to_eager(eager.out, ref, True, f"{precision} eager {c0}/{c1}")

    # no allocation, a non-default stream, the documented launch count
    ins = _inputs(model, padded)
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated(DEV)
    side = torch.cuda.Stream(DEV)
    side.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(side):
        eager(ins, stream=side)
    side.synchronize()
    assert torch.cuda.memory_allocated(DEV) == before
    _assert_equal_to_eager(eager.out, ref, True, f"{precision} side stream")
    plain = Native(model, 1, cap, cap)
    x3 = precision == "fp32"
    g = 3 + (2 if x3 else 0)  # final_proj, matchability, (x3_similarity, x3_assign_lse's two kernels | assign_lse)
    for mode in MODES:
        depth, width = MODES[mode]
        eager.acfg = AdaptiveConfig(depth, width)
        d, w = int(depth > 0), int(width > 0)
        n0 = lib.lgb200_launch_count()
        plain(ins)
        n1 = lib.lgb200_launch_count()
        eager(ins)
        n2 = lib.lgb200_launch_count()
        torch.cuda.synchronize()
        want = (n1 - n0) + 1 + (L - 1) * (2 * d + (2 + x3) * w) + d * (1 + (L - 1) * g) + 1
        assert n2 - n1 == want, (mode, n1 - n0, n2 - n1, want)
