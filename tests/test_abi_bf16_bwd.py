"""CPU tests of the bf16 attention backward's C-ABI entry points (ABI v7): argument validation and workspace size,
checked before any CUDA call, and the train_precision conf key."""
import ctypes

import pytest


@pytest.fixture(scope="module")
def lib():
    from glue_factory_colon_b200 import _abi, build

    build.build()
    return _abi.load()


def test_bf16_attention_bwd_argument_validation_without_gpu(lib):
    n_ws = ctypes.c_longlong(0)
    assert lib.lgb200_attention_bwd_bf16_workspace(4, 256, ctypes.byref(n_ws)) == 0
    assert n_ws.value == 2 * 4 * 4 * 256 + 16 + 4 * 256 * 256 // 2  # statistics + pad + dO as bf16 (two per float)
    assert lib.lgb200_attention_bwd_bf16_workspace(4, 200, ctypes.byref(n_ws)) == -1
    assert lib.lgb200_attention_bwd_bf16_workspace(0, 256, ctypes.byref(n_ws)) == -1
    assert lib.lgb200_attention_bwd_bf16_workspace(4, 256, None) == -2
    assert lib.lgb200_attention_bwd_bf16(None, None, None, None, None, 4, 256, None, 0, None, None, None, None, None) == -2
    p = ctypes.c_void_p(16)  # never dereferenced: the shape checks fail first
    args = [p] * 5
    outs = [p] * 3
    assert lib.lgb200_attention_bwd_bf16(*args, 4, 200, None, 0, *outs, p, None) == -1   # Lp % 128
    assert lib.lgb200_attention_bwd_bf16(*args, 3, 256, None, 1, *outs, p, None) == -1   # cross needs pairs
    assert lib.lgb200_attention_bwd_bf16(*args, 4, 256, None, 2, *outs, p, None) == -1   # kv_xor
    assert lib.lgb200_attention_bwd_bf16(*args, 4, 256, None, 0, p, None, p, p, None) == -2


def test_train_precision_conf_key():
    from glue_factory_colon_b200 import LightGlue

    assert LightGlue.default_conf["train_precision"] == "fp32"
    assert LightGlue({"n_layers": 1, "train_precision": "bf16"}).conf.train_precision == "bf16"
    with pytest.raises(ValueError):
        LightGlue({"n_layers": 1, "train_precision": "bfloat16"})
