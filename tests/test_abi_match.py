"""CPU tests of the whole-matcher entry points (lgb200_weight_table_size, lgb200_pack_weights, lgb200_match_workspace,
lgb200_match): exported with the binding's argument counts, bad arguments rejected before any CUDA call, the documented
table and workspace sizes, and the header's list of required weights against the state dict."""
import ctypes
import re

import pytest

from helpers import ROOT

HEADER = ROOT / "include" / "lightglue_b200.h"
COUNTS = {"lgb200_weight_table_size": 3, "lgb200_pack_weights": 8, "lgb200_match_workspace": 5, "lgb200_match": 23}
P = 4096  # a non-NULL pointer that is never dereferenced: validation fails first


@pytest.fixture(scope="module")
def lib():
    from glue_factory_colon_b200 import _abi, build

    build.build()
    return _abi.load()


def _cfg(precision=1, n_layers=9, input_dim=256, kdim=2, thr=0.0):
    from glue_factory_colon_b200._abi import MatchConfig

    return MatchConfig(precision, n_layers, input_dim, kdim, thr)


def _align(b):
    return (b + 255) // 256 * 256


def _table_formula(precision, n_layers, input_dim, kdim):
    """(entries, pack bytes) from the entry list documented in the header."""
    w = 2 if precision == 1 else 4  # bf16 / fp16 plane pair per weight element
    layer = [("W", 768 * 256), ("F", 768), ("W", 512 * 512), ("F", 512), ("F", 512), ("F", 512), ("W", 256 * 512),
             ("F", 256), ("W", 512 * 256), ("F", 512), ("W", 512 * 512), ("F", 512), ("F", 512), ("F", 512),
             ("W", 256 * 512), ("F", 256)]
    tail = [("F", 32 * kdim), ("W", 256 * 256), ("F", 256), ("F", 256), ("F", 1)]
    if input_dim != 256:
        tail += [("W", 256 * input_dim), ("F", 256)]
    entries = layer * n_layers + tail
    return len(entries), sum(_align(k * (w if t == "W" else 4)) for t, k in entries)


def _workspace_formula(precision, input_dim, B, m, n):
    x3 = precision == 2
    gran = 256 if x3 else 128
    Lp = max(gran, -(-max(m, n) // gran) * gran)
    T = 2 * B * Lp
    act = op = 4 if x3 else 2
    parts = [T * 256 * act]                                   # x
    if input_dim != 256:
        parts.append(T * input_dim * act)                     # xin
        if x3:
            parts.append(T * input_dim * op)                  # its planes
    parts.append(T * 64 * 4 if x3 else T * 32 * 4)            # rot / rot16
    if x3:
        parts.append(T * 256 * op)                            # xs
    parts += [T * 256 * op] * 5 + [T * 512 * op]              # q, k, v, ctx, msg, hid
    parts += [T * 4, T * 4]                                   # z, lse
    if x3:
        parts.append(B * Lp * Lp * 4)                         # sim
    parts += [8 * B * (m + n + 2), 3 * 2 * B * 4]             # filter workspace, lens | orders
    return sum(_align(p) for p in parts)


@pytest.mark.parametrize("name", sorted(COUNTS))
def test_exported_with_the_header_argument_count(lib, name):
    from glue_factory_colon_b200 import _abi

    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    assert hasattr(ctypes.CDLL(str(_abi.LIB_PATH)), name)
    assert len(_abi.SIGNATURES[name]) == COUNTS[name]
    m = re.search(r"\b" + name + r"\s*\(([^;]*?)\)\s*;", text, flags=re.S)
    assert m and len([p for p in m.group(1).split(",") if p.strip()]) == COUNTS[name]
    assert _abi.ABI_VERSION == 8 and lib.lgb200_abi_version() == 8
    assert lib.lgb200_error_string(-6).decode() == "required weight missing"


@pytest.mark.parametrize("conf", [(1, 9, 256, 2), (2, 9, 256, 2), (1, 3, 128, 4), (2, 1, 128, 4), (2, 5, 512, 2)])
def test_weight_table_size(lib, conf):
    entries, nbytes = ctypes.c_int(0), ctypes.c_longlong(0)
    assert lib.lgb200_weight_table_size(ctypes.byref(_cfg(*conf)), ctypes.byref(entries), ctypes.byref(nbytes)) == 0
    assert (entries.value, nbytes.value) == _table_formula(*conf)


def test_weight_table_size_validation(lib):
    e, b = ctypes.c_int(0), ctypes.c_longlong(0)
    f = lib.lgb200_weight_table_size
    assert f(None, ctypes.byref(e), ctypes.byref(b)) == -2
    assert f(ctypes.byref(_cfg()), None, ctypes.byref(b)) == -2
    assert f(ctypes.byref(_cfg()), ctypes.byref(e), None) == -2
    for bad in (dict(n_layers=0), dict(kdim=3), dict(input_dim=100), dict(input_dim=0)):
        assert f(ctypes.byref(_cfg(**bad)), ctypes.byref(e), ctypes.byref(b)) == -1, bad
    for prec in (0, 3, -1):  # LGB200_F32 (the CUDA-core mode) and unknown values
        assert f(ctypes.byref(_cfg(precision=prec)), ctypes.byref(e), ctypes.byref(b)) == -3, prec


@pytest.mark.parametrize("prec", [1, 2])
@pytest.mark.parametrize("shape", [(1, 1024, 1024), (3, 300, 260), (3, 320, 280), (4, 2048, 2048), (2, 0, 77),
                                   (1, 129, 1)])
def test_match_workspace_size(lib, prec, shape):
    B, m, n = shape
    for din in (256, 128):
        nbytes = ctypes.c_longlong(0)
        assert lib.lgb200_match_workspace(ctypes.byref(_cfg(prec, input_dim=din)), B, m, n, ctypes.byref(nbytes)) == 0
        assert nbytes.value == _workspace_formula(prec, din, B, m, n), (prec, din, shape)


def test_match_workspace_validation(lib):
    nb = ctypes.c_longlong(0)
    f = lib.lgb200_match_workspace
    assert f(None, 1, 5, 5, ctypes.byref(nb)) == -2 and f(ctypes.byref(_cfg()), 1, 5, 5, None) == -2
    for B, m, n in ((0, 5, 5), (-1, 5, 5), (1, -1, 5), (1, 5, -1)):
        assert f(ctypes.byref(_cfg()), B, m, n, ctypes.byref(nb)) == -1, (B, m, n)
    assert f(ctypes.byref(_cfg(precision=0)), 1, 5, 5, ctypes.byref(nb)) == -3


def _match_args(cfg, ws_bytes=1 << 40):
    # (cfg, table, B, m, n, kpts0, kpts1, desc0, desc1, size0, size1, counts0, counts1, matches0, matches1, scores0,
    #  scores1, log_assignment, desc_out0, desc_out1, workspace, workspace_bytes, stream)
    table = (ctypes.c_void_p * 256)(*([P] * 256))
    return [ctypes.byref(cfg), table, 2, 300, 260, P, P, P, P, None, None, None, None, P, P, P, P, P, None, None, P,
            ws_bytes, None]


def test_match_argument_validation_without_gpu(lib):
    f = lib.lgb200_match
    cfg = _cfg()
    for i in (0, 1, 5, 6, 7, 8, 13, 14, 15, 16, 17, 20):
        args = _match_args(cfg)
        args[i] = None
        assert f(*args) == -2, i
    table = (ctypes.c_void_p * 256)(*([P] * 256))
    table[3] = None  # a NULL table entry
    args = _match_args(cfg)
    args[1] = table
    assert f(*args) == -2
    for B, m, n in ((0, 300, 260), (-1, 300, 260), (2, -1, 260), (2, 300, -5)):
        args = _match_args(cfg)
        args[2:5] = [B, m, n]
        assert f(*args) == -1, (B, m, n)
    for bad in (dict(n_layers=0), dict(kdim=3), dict(kdim=1), dict(input_dim=200)):
        assert f(*_match_args(_cfg(**bad))) == -1, bad
    for prec in (0, 3):
        assert f(*_match_args(_cfg(precision=prec))) == -3, prec
    nb = ctypes.c_longlong(0)
    assert lib.lgb200_match_workspace(ctypes.byref(cfg), 2, 300, 260, ctypes.byref(nb)) == 0
    assert f(*_match_args(cfg, ws_bytes=nb.value - 1)) == -1
    args = _match_args(cfg)
    args[20] = P + 16  # a workspace that is not 256-byte aligned
    assert f(*args) == -1


def _state_dict_names(conf):
    from glue_factory_colon_b200 import LightGlue

    return list(LightGlue(conf).state_dict().keys())


def _names_array(names):
    return (ctypes.c_char_p * len(names))(*[k.encode() for k in names])


def test_pack_weights_argument_validation_without_gpu(lib):
    f = lib.lgb200_pack_weights
    cfg = _cfg(n_layers=2)
    e, nb = ctypes.c_int(0), ctypes.c_longlong(0)
    assert lib.lgb200_weight_table_size(ctypes.byref(cfg), ctypes.byref(e), ctypes.byref(nb)) == 0
    names = _state_dict_names({"n_layers": 2})
    cn, ptrs, table = _names_array(names), (ctypes.c_void_p * len(names))(*([P] * len(names))), (ctypes.c_void_p * e.value)()
    # (cfg, n, names, tensors, pack_buf, pack_bytes, table, stream)
    for i in (0, 2, 3, 4, 6):
        args = [ctypes.byref(cfg), len(names), cn, ptrs, P, nb.value, table, None]
        args[i] = None
        assert f(*args) == -2, i
    assert f(ctypes.byref(cfg), -1, cn, ptrs, P, nb.value, table, None) == -1
    assert f(ctypes.byref(cfg), len(names), cn, ptrs, P, nb.value - 1, table, None) == -1
    assert f(ctypes.byref(cfg), len(names), cn, ptrs, P + 16, nb.value, table, None) == -1  # unaligned pack_buf
    assert f(ctypes.byref(_cfg(n_layers=0)), len(names), cn, ptrs, P, nb.value, table, None) == -1
    assert f(ctypes.byref(_cfg(kdim=5)), len(names), cn, ptrs, P, nb.value, table, None) == -1
    assert f(ctypes.byref(_cfg(precision=0)), len(names), cn, ptrs, P, nb.value, table, None) == -3
    # every required name missing in turn -> LGB200_ERR_WEIGHTS; a NULL tensor of a required name -> NULL
    required = _required_names(2, 256)
    for k in required:
        rest = [x for x in names if x != k]
        r = f(ctypes.byref(cfg), len(rest), _names_array(rest), (ctypes.c_void_p * len(rest))(*([P] * len(rest))), P,
              nb.value, table, None)
        assert r == -6, k
    i = names.index("posenc.Wr.weight")
    ptrs_null = (ctypes.c_void_p * len(names))(*[None if j == i else P for j in range(len(names))])
    assert f(ctypes.byref(cfg), len(names), cn, ptrs_null, P, nb.value, table, None) == -2
    # a cfg with 3 layers needs transformers.2.*: a 2-layer state dict lacks it
    cfg3 = _cfg(n_layers=3)
    assert lib.lgb200_weight_table_size(ctypes.byref(cfg3), ctypes.byref(e), ctypes.byref(nb)) == 0
    table3 = (ctypes.c_void_p * e.value)()
    assert f(ctypes.byref(cfg3), len(names), cn, ptrs, P, nb.value, table3, None) == -6
    # an input_proj is required exactly when input_dim != 256
    assert f(ctypes.byref(_cfg(n_layers=2, input_dim=128)), len(names), cn, ptrs, P, 1 << 40,
             (ctypes.c_void_p * 64)(), None) == -6


def _required_names(L, input_dim):
    """The header's BEGIN / END REQUIRED WEIGHTS block, expanded for n_layers = L."""
    text = HEADER.read_text()
    block = text[text.index("BEGIN REQUIRED WEIGHTS"):text.index("END REQUIRED WEIGHTS")]
    out = []
    for line in block.splitlines()[1:]:
        line = line.strip().lstrip("*")
        if "(input_dim != 256 only)" in line:
            if input_dim == 256:
                continue
            line = line.replace("(input_dim != 256 only)", "")
        for tok in line.split():
            if "{l}" in tok:
                out += [tok.replace("{l}", str(i)) for i in range(L)]
            else:
                out.append(tok.replace("{L-1}", str(L - 1)))
    return out


@pytest.mark.parametrize("conf", [{"n_layers": 9}, {"n_layers": 3, "input_dim": 128},
                                  {"n_layers": 9, "add_scale_ori": True},
                                  {"n_layers": 2, "input_dim": 128, "add_scale_ori": True}])
def test_header_lists_the_weights_the_forward_reads(conf):
    """The forward without adaptive depth / width reads every state-dict entry except the token-confidence heads
    (adaptive depth, lightglue.py:501-505), the MatchAssignment of every layer but the last (adaptive width and the
    loss, :506-521, :589-595) and the confidence_thresholds buffer."""
    L = conf["n_layers"]
    keys = _state_dict_names(conf)
    read = [k for k in keys
            if not k.startswith("token_confidence.") and k != "confidence_thresholds"
            and not (k.startswith("log_assignment.") and not k.startswith(f"log_assignment.{L - 1}."))]
    req = _required_names(L, conf.get("input_dim", 256))
    assert len(req) == len(set(req))
    assert sorted(req) == sorted(read)
