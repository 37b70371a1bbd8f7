"""CPU tests of lgb200_npair_loss_bwd (the backward of the nearest-neighbour matcher's N_pair loss): exported with the
binding's argument count and rejecting bad arguments before any CUDA call."""
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


def test_npair_bwd_is_exported_with_the_header_argument_count(lib):
    from glue_factory_colon_b200 import _abi

    name = "lgb200_npair_loss_bwd"
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    assert hasattr(ctypes.CDLL(str(_abi.LIB_PATH)), name)
    assert len(_abi.SIGNATURES[name]) == 13
    m = re.search(r"\b" + name + r"\s*\(([^;]*?)\)\s*;", text, flags=re.S)
    assert m and len([p for p in m.group(1).split(",") if p.strip()]) == 13


def test_npair_bwd_argument_validation_without_gpu(lib):
    """NULL inputs / outputs and impossible shapes are refused (-2 = NULL, -1 = shape); dsim alone may be NULL."""
    p = 4096  # a non-NULL pointer that is never dereferenced: validation fails first
    f = lib.lgb200_npair_loss_bwd
    # (sim, gt, B, N, M, T, workspace, row_cnt, coef, col_cnt, dsim, dtemp_rows, stream)
    for i in (0, 1, 6, 7, 8, 9, 11):
        args = [p, p, 2, 5, 7, 1.0, p, p, p, p, p, p, None]
        args[i] = None
        assert f(*args) == -2, i
    for B, N, M in ((0, 5, 7), (-1, 5, 7), (2, 0, 7), (2, 5, 0), (2, -3, 7), (65536, 5, 7)):
        assert f(p, p, B, N, M, 1.0, p, p, p, p, None, p, None) == -1, (B, N, M)
