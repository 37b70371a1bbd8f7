"""GPU tests of the whole matcher behind the C ABI (lgb200_pack_weights, lgb200_match): bit-equal to LightGlue.forward
in both precisions, native packing against LightGlue._pack, capture into a CUDA graph at a fixed capacity replayed with
other counts, and the C++ example built against the header alone."""
import ctypes
import subprocess

import pytest
import torch

from helpers import ROOT, oracle_batch
from test_gpu_parity import compare_to_oracle, fp32_la_tol
from test_gpu_train_ragged import LEN0, LEN1, N0S, N1S, _padded, _pairs
from glue_factory_colon_b200 import LightGlue, _abi, build
from glue_factory_colon_b200._abi import BF16, F32X3, MatchConfig, check, ptr
from glue_factory_colon_b200.synthetic import make_pairs, to_device
from glue_factory_colon_b200.weights import NATIVE_LAYER_ENTRIES, native_table

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
PREC = {"bf16": BF16, "fp32": F32X3}
KEYS = ("matches0", "matches1", "matching_scores0", "matching_scores1", "log_assignment")
FOLDED = {NATIVE_LAYER_ENTRIES.index(k) for k in ("sf0_w", "sf0_b", "cf0_w", "cf0_b")}


def _model(precision, seed=5, **conf):
    torch.manual_seed(seed)
    return LightGlue({"filter_threshold": 0.0, "precision": precision, **conf}).eval().to(DEV)


def _cfg(model):
    c = model.conf
    return MatchConfig(PREC[c.precision], c.n_layers, c.input_dim, 4 if c.add_scale_ori else 2,
                       float(c.filter_threshold))


def _inputs(model, data):
    """The fp32 device inputs of lgb200_match for a LightGlue data dict (keypoints with scale / orientation appended
    under add_scale_ori, image sizes [B,2] or None, counts int32 [B] or None)."""
    ins = {}
    for i in (0, 1):
        k = data[f"keypoints{i}"].to(DEV, torch.float32)
        B = k.shape[0]
        if model.conf.add_scale_ori:
            k = torch.cat([k, data[f"scales{i}"].to(k)[..., None], data[f"oris{i}"].to(k)[..., None]], -1)
        ins[f"kpts{i}"] = k.contiguous()
        ins[f"desc{i}"] = data[f"descriptors{i}"].to(DEV, torch.float32).contiguous()
        sz = data.get(f"view{i}", {}).get("image_size")
        ins[f"size{i}"] = None if sz is None else sz.to(DEV, torch.float32).reshape(-1, 2).expand(B, 2).contiguous()
        cnt = data.get(f"num_keypoints{i}")
        ins[f"counts{i}"] = None if cnt is None else cnt.to(DEV, torch.int32).contiguous()
    return ins


class Native:
    """Output buffers, workspace and table of lgb200_match at a fixed capacity B x m x n."""

    def __init__(self, model, B, m, n, table=None):
        self.lib = _abi.load()
        self.cfg = _cfg(model)
        self.table, self.keep = native_table(model, self.cfg.precision) if table is None else (table, None)
        self.B, self.m, self.n = B, m, n
        nb = ctypes.c_longlong(0)
        check(self.lib.lgb200_match_workspace(ctypes.byref(self.cfg), B, m, n, ctypes.byref(nb)), "match_workspace")
        self.ws = torch.empty(nb.value, dtype=torch.uint8, device=DEV)
        act = torch.bfloat16 if self.cfg.precision == BF16 else torch.float32
        i64, f32 = dict(device=DEV, dtype=torch.int64), dict(device=DEV, dtype=torch.float32)
        self.out = {
            "matches0": torch.empty(B, m, **i64), "matches1": torch.empty(B, n, **i64),
            "matching_scores0": torch.empty(B, m, **f32), "matching_scores1": torch.empty(B, n, **f32),
            "log_assignment": torch.empty(B, m + 1, n + 1, **f32),
            "ref_descriptors0": torch.empty(B, m, 256, device=DEV, dtype=act),
            "ref_descriptors1": torch.empty(B, n, 256, device=DEV, dtype=act),
        }

    def __call__(self, ins, stream=None):
        o = self.out
        st = (stream or torch.cuda.current_stream(DEV)).cuda_stream
        check(self.lib.lgb200_match(
            ctypes.byref(self.cfg), self.table, self.B, self.m, self.n, ptr(ins["kpts0"]), ptr(ins["kpts1"]),
            ptr(ins["desc0"]), ptr(ins["desc1"]), ptr(ins["size0"]), ptr(ins["size1"]), ptr(ins["counts0"]),
            ptr(ins["counts1"]), ptr(o["matches0"]), ptr(o["matches1"]), ptr(o["matching_scores0"]),
            ptr(o["matching_scores1"]), ptr(o["log_assignment"]), ptr(o["ref_descriptors0"]),
            ptr(o["ref_descriptors1"]), ptr(self.ws), self.ws.numel(), st), "lgb200_match")
        return o


def _bits(t):
    return t.contiguous().view(torch.uint8)


def _assert_bit_equal(nat, ref, what):
    for k in KEYS:
        assert torch.equal(_bits(nat[k]), _bits(ref[k])), f"{what}: {k} differs"
    for i in (0, 1):
        r = ref[f"ref_descriptors{i}"][:, -1]  # [B, 1, n, 256]: the last layer
        assert torch.equal(_bits(nat[f"ref_descriptors{i}"]), _bits(r)), f"{what}: ref_descriptors{i} differs"


def _python(model, data):
    with torch.no_grad():
        out = model(to_device(data, DEV))
    return out


def _native(model, data):
    B, m, _ = data["keypoints0"].shape
    nat = Native(model, B, m, data["keypoints1"].shape[1])
    out = nat(_inputs(model, data))
    torch.cuda.synchronize()
    return out


def _drop_sizes(data):
    data["view0"], data["view1"] = {}, {}
    return data


CASES = {
    "1x1024x1024": (dict(), lambda: make_pairs(B=1, n0=1024, n1=1024, seed=1)),
    "3x300x260_nosize": (dict(), lambda: _drop_sizes(make_pairs(B=3, n0=300, n1=260, seed=2))),
    "padded_counts": (dict(n_layers=3), lambda: _padded(_pairs(N0S, N1S), LEN0, LEN1)),
    "dim128_scale_ori": (dict(input_dim=128, add_scale_ori=True, n_layers=3),
                         lambda: make_pairs(B=2, n0=200, n1=333, seed=3, dim=128, scale_ori=True)),
    "3_layers": (dict(n_layers=3), lambda: make_pairs(B=2, n0=512, n1=256, seed=4)),
}


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_bit_equal_to_the_python_forward(precision, case):
    conf, make = CASES[case]
    model = _model(precision, **conf)
    data = make()
    _assert_bit_equal(_native(model, data), _python(model, data), f"{precision} {case}")


def test_bit_equal_at_production_size_bf16():
    """4 x 2048: multi-tile persistent CTAs and full key rings in every kernel."""
    model = _model("bf16")
    data = make_pairs(B=4, n0=2048, n1=2048, seed=6)
    _assert_bit_equal(_native(model, data), _python(model, data), "bf16 4x2048")


def _native_pack(model, cfg):
    """lgb200_pack_weights on the model's state dict -> (table, pack buffer)."""
    lib = _abi.load()
    sd = {k: v.detach().to(DEV, torch.float32).contiguous() for k, v in model.state_dict().items()}
    names = (ctypes.c_char_p * len(sd))(*[k.encode() for k in sd])
    ptrs = (ctypes.c_void_p * len(sd))(*[v.data_ptr() for v in sd.values()])
    e, nb = ctypes.c_int(0), ctypes.c_longlong(0)
    check(lib.lgb200_weight_table_size(ctypes.byref(cfg), ctypes.byref(e), ctypes.byref(nb)), "weight_table_size")
    buf = torch.full((nb.value,), 0xFF, dtype=torch.uint8, device=DEV)
    table = (ctypes.c_void_p * e.value)()
    check(lib.lgb200_pack_weights(ctypes.byref(cfg), len(sd), names, ptrs, ptr(buf), nb.value, table,
                                  torch.cuda.current_stream(DEV).cuda_stream), "pack_weights")
    torch.cuda.synchronize()
    return table, buf


def _ulp_close(nat, ref, planes):
    """Folded entries: within one unit in the last place of the stored format.  fp32 / bf16: the bit patterns differ by
    at most 1.  fp16 planes (256 w = hi + lo): hi + lo differ by at most one ulp of lo plus one fp32 ulp of 256 w."""
    if not planes:
        it = torch.int32 if ref.dtype == torch.float32 else torch.int16
        return bool(((nat.view(it).long() - ref.view(it).long()).abs() <= 1).all())
    vn = nat[0].double() + nat[1].double()
    vr = ref[0].double() + ref[1].double()
    ulp_lo = torch.exp2(torch.floor(torch.log2(ref[1].double().abs().clamp(min=2.0 ** -14))) - 10)
    ulp_t = torch.exp2(torch.floor(torch.log2(vr.abs().clamp(min=2.0 ** -100))) - 23)
    return bool(((vn - vr).abs() <= ulp_lo + ulp_t).all())


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("conf", [dict(), dict(input_dim=128, add_scale_ori=True, n_layers=3)], ids=["default", "dim128"])
def test_native_packing_against_pack(precision, conf):
    model = _model(precision, **conf)
    cfg = _cfg(model)
    table, buf = _native_pack(model, cfg)
    ref_table, ref = native_table(model, cfg.precision)
    assert len(table) == len(ref_table)
    base = buf.data_ptr()
    n_layer_entries = len(NATIVE_LAYER_ENTRIES) * model.conf.n_layers
    differ = []
    for idx, t in enumerate(ref):
        nbytes = t.numel() * t.element_size()
        off = table[idx] - base
        assert off % 256 == 0 and 0 <= off and off + nbytes <= buf.numel()
        nat = buf[off:off + nbytes].view(t.dtype).view(t.shape)
        if torch.equal(_bits(nat), _bits(t)):
            continue
        folded = idx < n_layer_entries and idx % len(NATIVE_LAYER_ENTRIES) in FOLDED
        assert folded, f"entry {idx} differs and is not a folded FFN1 entry"
        assert _ulp_close(nat, t, t.dtype == torch.float16), f"entry {idx}: more than 1 ulp from _pack"
        differ.append(idx)
    print(f"[native pack {precision}] {len(differ)} of {len(ref)} entries differ from _pack (folded FFN1, <= 1 ulp)")
    # a forward on the native pack stays within the oracle tolerances
    data = make_pairs(B=2, n0=300, n1=260, seed=8, dim=model.conf.input_dim, scale_ori=model.conf.add_scale_ori)
    out = Native(model, 2, 300, 260, table=table)(_inputs(model, data))
    torch.cuda.synchronize()
    res = oracle_batch(model.cpu(), model.conf, data)
    compare_to_oracle(out, res, 300, 260, fp32=precision == "fp32", la_tol=fp32_la_tol("fp32"))


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_graph_capture_at_capacity_replays_any_counts(precision):
    model = _model(precision)
    lib = _abi.load()
    cap = 1024
    nat = Native(model, 1, cap, cap)
    eager = Native(model, 1, cap, cap)
    first = make_pairs(B=1, n0=cap, n1=cap, seed=10)
    first["num_keypoints0"], first["num_keypoints1"] = torch.tensor([cap]), torch.tensor([cap])
    static = _inputs(model, first)
    nat(static)  # outside the capture: lazy initialisation
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        nat(static)
    for seed, (c0, c1) in ((11, (1024, 1024)), (12, (700, 311)), (13, (5, 0))):
        data = make_pairs(B=1, n0=cap, n1=cap, seed=seed)
        data["num_keypoints0"], data["num_keypoints1"] = torch.tensor([c0]), torch.tensor([c1])
        new = _inputs(model, data)
        for k, t in new.items():
            static[k].copy_(t)
        graph.replay()
        torch.cuda.synchronize()
        ref = _python(model, data)
        _assert_bit_equal(nat.out, ref, f"{precision} replay {c0}/{c1} vs LightGlue.forward")
        eager(new)
        torch.cuda.synchronize()
        _assert_bit_equal(eager.out, ref, f"{precision} eager {c0}/{c1}")

    # no allocation, a non-default stream, launches = the Python forward's + the lens / order kernel
    ins = _inputs(model, data)
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated(DEV)
    side = torch.cuda.Stream(DEV)
    side.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(side):
        eager(ins, stream=side)
    side.synchronize()
    assert torch.cuda.memory_allocated(DEV) == before
    _assert_bit_equal(eager.out, ref, f"{precision} side stream")
    for counts in (True, False):
        d = dict(data) if counts else {k: v for k, v in data.items() if not k.startswith("num_keypoints")}
        i_d = _inputs(model, d)
        n0 = lib.lgb200_launch_count()
        _python(model, d)
        n1 = lib.lgb200_launch_count()
        eager(i_d)
        n2 = lib.lgb200_launch_count()
        torch.cuda.synchronize()
        assert n2 - n1 == (n1 - n0) + (1 if counts else 0), (counts, n1 - n0, n2 - n1)


@pytest.fixture(scope="module")
def demo(tmp_path_factory):
    exe = tmp_path_factory.mktemp("demo") / "native_match_demo"
    lib_dir = build.LIB.parent
    subprocess.run([build._nvcc(), "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                    "-I", str(ROOT / "include"), str(ROOT / "tools" / "native_match_demo.cpp"),
                    "-L", str(lib_dir), "-llightglue_b200", "-Xlinker", f"-rpath={lib_dir}", "-o", str(exe)],
                   check=True)
    return exe


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_cpp_example(demo, tmp_path, precision):
    model = _model(precision, n_layers=3)
    B, m, n = 2, 300, 260
    data = make_pairs(B=B, n0=m, n1=n, seed=14)
    data["num_keypoints0"], data["num_keypoints1"] = torch.tensor([300, 129]), torch.tensor([77, 260])
    c = model.conf
    (tmp_path / "config.txt").write_text(f"{PREC[precision]} {c.n_layers} {c.input_dim} 2 {c.filter_threshold} {B} {m} {n}\n")
    (tmp_path / "weights").mkdir()
    for k, v in model.state_dict().items():
        (tmp_path / "weights" / f"{k}.bin").write_bytes(v.detach().float().cpu().contiguous().numpy().tobytes())
    for i in (0, 1):
        for name, t in ((f"kpts{i}", data[f"keypoints{i}"]), (f"desc{i}", data[f"descriptors{i}"]),
                        (f"size{i}", data[f"view{i}"]["image_size"])):
            (tmp_path / f"{name}.bin").write_bytes(t.float().contiguous().numpy().tobytes())
        (tmp_path / f"counts{i}.bin").write_bytes(data[f"num_keypoints{i}"].to(torch.int32).numpy().tobytes())
    subprocess.run([str(demo), str(tmp_path)], check=True)
    ref = _python(model, data)

    def load(name, dtype, shape):
        return torch.frombuffer(bytearray((tmp_path / f"{name}.bin").read_bytes()), dtype=dtype).view(shape).to(DEV)

    act = torch.bfloat16 if precision == "bf16" else torch.float32
    got = {"matches0": load("matches0", torch.int64, (B, m)), "matches1": load("matches1", torch.int64, (B, n)),
           "matching_scores0": load("scores0", torch.float32, (B, m)),
           "matching_scores1": load("scores1", torch.float32, (B, n)),
           "log_assignment": load("log_assignment", torch.float32, (B, m + 1, n + 1)),
           "ref_descriptors0": load("desc_out0", act, (B, m, 256)), "ref_descriptors1": load("desc_out1", act, (B, n, 256))}
    _assert_bit_equal(got, ref, f"C++ example {precision}")
