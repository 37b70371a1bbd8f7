"""CPU tests of the ragged loss-side entry points (ABI 8): lgb200_loss_reduce_ragged and lgb200_assign_dsim_ragged are
exported with the binding's argument counts and reject bad arguments before any CUDA call."""
import ctypes
import re

import pytest

from helpers import ROOT

HEADER = ROOT / "include" / "lightglue_b200.h"


@pytest.fixture(scope="module")
def lib():
    from glue_factory_colon_b200 import _abi, build

    build.build()
    return _abi.load()


def test_abi_version_is_8_and_the_ragged_entry_points_are_exported(lib):
    from glue_factory_colon_b200 import _abi

    assert _abi.ABI_VERSION == 8 and lib.lgb200_abi_version() == 8
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    raw = ctypes.CDLL(str(_abi.LIB_PATH))
    for name, n_args in (("lgb200_loss_reduce_ragged", 12), ("lgb200_assign_dsim_ragged", 12)):
        assert hasattr(raw, name), name
        assert len(_abi.SIGNATURES[name]) == n_args
        m = re.search(r"\b" + name + r"\s*\(([^;]*?)\)\s*;", text, flags=re.S)
        assert m and len([p for p in m.group(1).split(",") if p.strip()]) == n_args, name


def test_ragged_argument_validation_without_gpu(lib):
    """NULL matrices / counts and impossible shapes are refused (-2 = NULL, -1 = shape) before any CUDA call."""
    p = 4096  # a non-NULL pointer that is never dereferenced: validation fails first
    # lgb200_loss_reduce_ragged(la, B, R, C, lens, gt, row_pos, row_cnt, row_exp, row_arg, col_arg, stream)
    assert lib.lgb200_loss_reduce_ragged(None, 2, 5, 5, p, None, None, None, None, None, None, None) == -2
    assert lib.lgb200_loss_reduce_ragged(p, 2, 5, 5, None, None, None, None, None, None, None, None) == -2
    assert lib.lgb200_loss_reduce_ragged(p, -1, 5, 5, p, None, None, None, None, None, None, None) == -1
    assert lib.lgb200_loss_reduce_ragged(p, 2, 0, 5, p, None, None, None, None, None, None, None) == -1
    assert lib.lgb200_loss_reduce_ragged(p, 2, 5, 0, p, None, None, None, None, None, None, None) == -1
    assert lib.lgb200_loss_reduce_ragged(p, 0, 5, 5, p, None, None, None, None, None, None, None) == 0  # nothing to do
    # lgb200_assign_dsim_ragged(sim, B, m, n, lse, Lp, lens, gt, g_pos, r, c, stream)
    assert lib.lgb200_assign_dsim_ragged(p, 2, 100, 100, p, 128, None, p, p, p, p, None) == -2
    assert lib.lgb200_assign_dsim_ragged(None, 2, 100, 100, p, 128, p, p, p, p, p, None) == -2
    assert lib.lgb200_assign_dsim_ragged(p, 2, 100, 100, p, 128, p, None, p, p, p, None) == -2
    assert lib.lgb200_assign_dsim_ragged(p, 2, 200, 100, p, 128, p, p, p, p, p, None) == -1  # m > Lp
    assert lib.lgb200_assign_dsim_ragged(p, 0, 100, 100, p, 128, p, p, p, p, p, None) == -1
    assert lib.lgb200_assign_dsim_ragged(p, 2, 100, 0, p, 128, p, p, p, p, p, None) == -1
