"""CPU tests of the adaptive whole-matcher entry points (lgb200_adaptive_table_size, lgb200_pack_weights_adaptive,
lgb200_match_adaptive_workspace, lgb200_match_adaptive): exported with the binding's argument counts, bad arguments
rejected before any CUDA call, the documented table and workspace sizes, and the header's lists of required weights
against the state dict."""
import ctypes
import re

import pytest

from helpers import ROOT
from test_abi_match import _align, _cfg, _names_array, _required_names, _state_dict_names, _table_formula
from test_abi_match import _workspace_formula

HEADER = ROOT / "include" / "lightglue_b200.h"
COUNTS = {"lgb200_adaptive_table_size": 3, "lgb200_pack_weights_adaptive": 8, "lgb200_match_adaptive_workspace": 5,
          "lgb200_match_adaptive": 28}
P = 4096  # a non-NULL pointer that is never dereferenced: validation fails first


@pytest.fixture(scope="module")
def lib():
    from glue_factory_colon_b200 import _abi, build

    build.build()
    return _abi.load()


def _acfg(depth=0.95, width=0.99):
    from glue_factory_colon_b200._abi import AdaptiveConfig

    return AdaptiveConfig(depth, width)


@pytest.mark.parametrize("name", sorted(COUNTS))
def test_exported_with_the_header_argument_count(lib, name):
    from glue_factory_colon_b200 import _abi

    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    assert hasattr(ctypes.CDLL(str(_abi.LIB_PATH)), name)
    assert len(_abi.SIGNATURES[name]) == COUNTS[name]
    m = re.search(r"\b" + name + r"\s*\(([^;]*?)\)\s*;", text, flags=re.S)
    assert m and len([p for p in m.group(1).split(",") if p.strip()]) == COUNTS[name]
    assert _abi.ABI_VERSION == 8 and lib.lgb200_abi_version() == 8


def test_new_names_do_not_shadow_lgb200_match():
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    assert len(re.findall(r"\blgb200_match\s*\(", text)) == 1
    for name in COUNTS:
        assert not re.search(r"\blgb200_match\s*\(", name + "(")


def _adaptive_table_formula(precision, n_layers, input_dim, kdim):
    entries, nbytes = _table_formula(precision, n_layers, input_dim, kdim)
    w = 2 if precision == 1 else 4
    per_layer = [256 * 256 * w, 256 * 4, 256 * 4, 4, 256 * 4, 4]  # fp_w, fp_b, m_w, m_b, tk_w, tk_b
    return entries + 6 * (n_layers - 1), nbytes + (n_layers - 1) * sum(_align(b) for b in per_layer)


@pytest.mark.parametrize("conf", [(1, 9, 256, 2), (2, 9, 256, 2), (1, 3, 128, 4), (2, 1, 128, 4), (2, 5, 512, 2)])
def test_adaptive_table_size(lib, conf):
    entries, nbytes = ctypes.c_int(0), ctypes.c_longlong(0)
    f = lib.lgb200_adaptive_table_size
    assert f(ctypes.byref(_cfg(*conf)), ctypes.byref(entries), ctypes.byref(nbytes)) == 0
    assert (entries.value, nbytes.value) == _adaptive_table_formula(*conf)
    e, b = ctypes.c_int(0), ctypes.c_longlong(0)
    assert f(None, ctypes.byref(e), ctypes.byref(b)) == -2
    assert f(ctypes.byref(_cfg()), None, ctypes.byref(b)) == -2 and f(ctypes.byref(_cfg()), ctypes.byref(e), None) == -2
    for bad in (dict(n_layers=0), dict(kdim=3), dict(input_dim=100)):
        assert f(ctypes.byref(_cfg(**bad)), ctypes.byref(e), ctypes.byref(b)) == -1, bad
    assert f(ctypes.byref(_cfg(precision=0)), ctypes.byref(e), ctypes.byref(b)) == -3


def _adaptive_workspace_formula(precision, input_dim, n_layers, B, m, n):
    x3 = precision == 2
    gran = 256 if x3 else 128
    Lp = max(gran, -(-max(m, n) // gran) * gran)
    T = 2 * B * Lp
    act = 4 if x3 else 2
    parts = [T * 4] * 5                                       # ind, prune_cnt, conf, msig, ind_b
    parts += [T * 256 * act, T * 64 * 4 if x3 else T * 32 * 4]  # x_b, rot_b
    parts += [(2 * B + 2 * B) * 4, n_layers * 2 * B * 4]        # done | lens_active | total, per-exit-layer counts
    return _workspace_formula(precision, input_dim, B, m, n) + sum(_align(p) for p in parts)


@pytest.mark.parametrize("prec", [1, 2])
@pytest.mark.parametrize("shape", [(1, 1024, 1024), (3, 300, 260), (4, 2048, 2048), (2, 0, 77), (1, 129, 1)])
def test_adaptive_workspace_size(lib, prec, shape):
    B, m, n = shape
    for din, L in ((256, 9), (128, 3)):
        nbytes = ctypes.c_longlong(0)
        cfg = _cfg(prec, n_layers=L, input_dim=din)
        assert lib.lgb200_match_adaptive_workspace(ctypes.byref(cfg), B, m, n, ctypes.byref(nbytes)) == 0
        assert nbytes.value == _adaptive_workspace_formula(prec, din, L, B, m, n), (prec, din, shape)


def test_adaptive_workspace_validation(lib):
    nb = ctypes.c_longlong(0)
    f = lib.lgb200_match_adaptive_workspace
    assert f(None, 1, 5, 5, ctypes.byref(nb)) == -2 and f(ctypes.byref(_cfg()), 1, 5, 5, None) == -2
    for B, m, n in ((0, 5, 5), (-1, 5, 5), (1, -1, 5), (1, 5, -1)):
        assert f(ctypes.byref(_cfg()), B, m, n, ctypes.byref(nb)) == -1, (B, m, n)
    assert f(ctypes.byref(_cfg(precision=0)), 1, 5, 5, ctypes.byref(nb)) == -3


def _args(cfg, acfg, B=2, m=300, n=260, ws_bytes=1 << 40):
    # (cfg, acfg, table, B, m, n, kpts0, kpts1, desc0, desc1, size0, size1, counts0, counts1, matches0, matches1,
    #  scores0, scores1, log_assignment, desc_out0, desc_out1, prune0, prune1, exit_layer, final_counts, workspace,
    #  workspace_bytes, stream)
    table = (ctypes.c_void_p * 512)(*([P] * 512))
    return [ctypes.byref(cfg), None if acfg is None else ctypes.byref(acfg), table, B, m, n, P, P, P, P, None, None,
            None, None, P, P, P, P, P, None, None, None, None, None, None, P, ws_bytes, None]


@pytest.mark.parametrize("modes", [(0.95, 0.99), (0.95, -1.0), (-1.0, 0.99), (-1.0, -1.0)])
def test_match_adaptive_argument_validation_without_gpu(lib, modes):
    f = lib.lgb200_match_adaptive
    cfg, acfg = _cfg(), _acfg(*modes)
    for i in (0, 1, 2, 6, 7, 8, 9, 14, 15, 16, 17, 18, 25):
        args = _args(cfg, acfg)
        args[i] = None
        assert f(*args) == -2, i
    for B, m, n in ((0, 300, 260), (-1, 300, 260), (2, -1, 260), (2, 300, -5)):
        assert f(*_args(cfg, acfg, B, m, n)) == -1, (B, m, n)
    for bad in (dict(n_layers=0), dict(kdim=3), dict(input_dim=200)):
        assert f(*_args(_cfg(**bad), acfg)) == -1, bad
    for prec in (0, 3):
        assert f(*_args(_cfg(precision=prec), acfg)) == -3, prec
    nb = ctypes.c_longlong(0)
    assert lib.lgb200_match_adaptive_workspace(ctypes.byref(cfg), 2, 300, 260, ctypes.byref(nb)) == 0
    assert f(*_args(cfg, acfg, ws_bytes=nb.value - 1)) == -1
    args = _args(cfg, acfg)
    args[25] = P + 16  # a workspace that is not 256-byte aligned
    assert f(*args) == -1
    # a NULL entry of the base table is refused always, one of the adaptive heads when a mode is on
    ne, ne_ad, nbt = ctypes.c_int(0), ctypes.c_int(0), ctypes.c_longlong(0)
    assert lib.lgb200_weight_table_size(ctypes.byref(cfg), ctypes.byref(ne), ctypes.byref(nbt)) == 0
    assert lib.lgb200_adaptive_table_size(ctypes.byref(cfg), ctypes.byref(ne_ad), ctypes.byref(nbt)) == 0
    for idx in (3, ne_ad.value - 1):
        args = _args(cfg, acfg)
        table = (ctypes.c_void_p * 512)(*([P] * 512))
        table[idx] = None
        args[2] = table
        on = modes[0] > 0 or modes[1] > 0
        if idx < ne.value or on:
            assert f(*args) == -2, idx
    # width pruning beyond lgb200_prune_compact's 8192 rows per sequence
    big = 8193
    nb = ctypes.c_longlong(0)
    assert lib.lgb200_match_adaptive_workspace(ctypes.byref(cfg), 1, big, 100, ctypes.byref(nb)) == 0
    if modes[1] > 0:
        assert f(*_args(cfg, acfg, 1, big, 100, ws_bytes=nb.value)) == -1


def test_match_adaptive_requires_acfg(lib):
    assert lib.lgb200_match_adaptive(*_args(_cfg(), None)) == -2


def _adaptive_names(L):
    """The header's BEGIN / END ADAPTIVE WEIGHTS block, expanded for n_layers = L."""
    text = HEADER.read_text()
    block = text[text.index("BEGIN ADAPTIVE WEIGHTS"):text.index("END ADAPTIVE WEIGHTS")]
    out = []
    for line in block.splitlines()[1:]:
        for tok in line.strip().lstrip("*").split():
            assert "{l}" in tok, tok
            out += [tok.replace("{l}", str(i)) for i in range(L - 1)]
    return out


@pytest.mark.parametrize("conf", [{"n_layers": 9}, {"n_layers": 3, "input_dim": 128},
                                  {"n_layers": 9, "add_scale_ori": True},
                                  {"n_layers": 2, "input_dim": 128, "add_scale_ori": True}])
def test_header_lists_every_weight_the_adaptive_forward_reads(conf):
    """The adaptive forward reads every state-dict entry except the confidence_thresholds buffer."""
    L = conf["n_layers"]
    keys = _state_dict_names(conf)
    req = _required_names(L, conf.get("input_dim", 256)) + _adaptive_names(L)
    assert len(req) == len(set(req))
    assert sorted(req) == sorted(k for k in keys if k != "confidence_thresholds")


def test_pack_weights_adaptive_argument_validation_without_gpu(lib):
    f = lib.lgb200_pack_weights_adaptive
    cfg = _cfg(n_layers=3)
    e, nb = ctypes.c_int(0), ctypes.c_longlong(0)
    assert lib.lgb200_adaptive_table_size(ctypes.byref(cfg), ctypes.byref(e), ctypes.byref(nb)) == 0
    names = _state_dict_names({"n_layers": 3})
    cn, ptrs, table = _names_array(names), (ctypes.c_void_p * len(names))(*([P] * len(names))), (ctypes.c_void_p * e.value)()
    for i in (0, 2, 3, 4, 6):
        args = [ctypes.byref(cfg), len(names), cn, ptrs, P, nb.value, table, None]
        args[i] = None
        assert f(*args) == -2, i
    assert f(ctypes.byref(cfg), -1, cn, ptrs, P, nb.value, table, None) == -1
    assert f(ctypes.byref(cfg), len(names), cn, ptrs, P, nb.value - 1, table, None) == -1
    assert f(ctypes.byref(cfg), len(names), cn, ptrs, P + 16, nb.value, table, None) == -1
    assert f(ctypes.byref(_cfg(n_layers=0)), len(names), cn, ptrs, P, nb.value, table, None) == -1
    assert f(ctypes.byref(_cfg(precision=0)), len(names), cn, ptrs, P, nb.value, table, None) == -3
    # every required name, base or adaptive, missing in turn -> LGB200_ERR_WEIGHTS before any launch
    for k in _required_names(3, 256) + _adaptive_names(3):
        rest = [x for x in names if x != k]
        r = f(ctypes.byref(cfg), len(rest), _names_array(rest), (ctypes.c_void_p * len(rest))(*([P] * len(rest))), P,
              nb.value, table, None)
        assert r == -6, k
    i = names.index("token_confidence.1.token.0.bias")
    ptrs_null = (ctypes.c_void_p * len(names))(*[None if j == i else P for j in range(len(names))])
    assert f(ctypes.byref(cfg), len(names), cn, ptrs_null, P, nb.value, table, None) == -2
