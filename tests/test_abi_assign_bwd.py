"""CPU tests of lgb200_assign_bwd (backward of the log-assignment for any upstream gradient), its workspace query and
lgb200_posenc_bwd (keypoint gradients through the positional encoding): exported with the binding's argument counts,
rejecting bad arguments before any CUDA call, and the documented workspace size."""
import ctypes
import math
import re

import pytest

from helpers import ROOT

HEADER = ROOT / "include" / "lightglue_b200.h"
COUNTS = {"lgb200_assign_bwd": 13, "lgb200_assign_bwd_workspace": 4, "lgb200_posenc_bwd": 12}


@pytest.fixture(scope="module")
def lib():
    from glue_factory_colon_b200 import _abi, build

    build.build()
    return _abi.load()


@pytest.mark.parametrize("name", sorted(COUNTS))
def test_exported_with_the_header_argument_count(lib, name):
    from glue_factory_colon_b200 import _abi

    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    assert hasattr(ctypes.CDLL(str(_abi.LIB_PATH)), name)
    assert len(_abi.SIGNATURES[name]) == COUNTS[name]
    m = re.search(r"\b" + name + r"\s*\(([^;]*?)\)\s*;", text, flags=re.S)
    assert m and len([p for p in m.group(1).split(",") if p.strip()]) == COUNTS[name]
    assert _abi.ABI_VERSION == 8 and lib.lgb200_abi_version() == 8


def test_assign_bwd_argument_validation_without_gpu(lib):
    """-2 = NULL, -1 = shape.  lens and z may be NULL; with z, dz0 and dz1 are required."""
    p = 4096  # a non-NULL pointer that is never dereferenced: validation fails first
    f = lib.lgb200_assign_bwd
    # (G, sim, B, m, n, lse, Lp, lens, z, dz0, dz1, workspace, stream)
    for i in (0, 1, 5, 11):
        args = [p, p, 2, 5, 7, p, 128, None, None, None, None, p, None]
        args[i] = None
        assert f(*args) == -2, i
    for i in (9, 10):
        args = [p, p, 2, 5, 7, p, 128, None, p, p, p, p, None]
        args[i] = None
        assert f(*args) == -2, i
    for B, m, n, Lp in ((0, 5, 7, 128), (-1, 5, 7, 128), (65536, 5, 7, 128), (2, 0, 7, 128), (2, 5, 0, 128),
                        (2, 129, 7, 128), (2, 5, 129, 128), (2, 5, 7, 100), (2, 5, 7, 0)):
        assert f(p, p, B, m, n, p, Lp, None, None, None, None, p, None) == -1, (B, m, n, Lp)


def test_assign_bwd_workspace_size(lib):
    n_floats = ctypes.c_longlong(0)
    for B, m, n in ((1, 1, 1), (2, 150, 131), (3, 320, 280), (16, 2048, 2048), (2, 33, 5)):
        assert lib.lgb200_assign_bwd_workspace(B, m, n, ctypes.byref(n_floats)) == 0
        assert n_floats.value == B * m + B * n + B * math.ceil(m / 32) * n, (B, m, n)
    assert lib.lgb200_assign_bwd_workspace(2, 5, 7, None) == -2
    for B, m, n in ((0, 5, 7), (2, 0, 7), (2, 5, 0), (-2, 5, 7)):
        assert lib.lgb200_assign_bwd_workspace(B, m, n, ctypes.byref(n_floats)) == -1, (B, m, n)


def test_posenc_bwd_argument_validation_without_gpu(lib):
    """size and lens may be NULL; kdim is 2 or 4."""
    p = 4096
    f = lib.lgb200_posenc_bwd
    # (kpts, B, n, kdim, size, Wr, lens, img, Lp, dtheta, dkpts, stream)
    for i in (0, 5, 9, 10):
        args = [p, 2, 100, 2, None, p, None, 0, 128, p, p, None]
        args[i] = None
        assert f(*args) == -2, i
    for B, n, kdim, img, Lp in ((0, 100, 2, 0, 128), (2, 100, 3, 0, 128), (2, 100, 2, 2, 128), (2, 129, 2, 0, 128),
                                (2, -1, 2, 0, 128), (2, 100, 4, 0, 96), (2, 100, 2, -1, 128)):
        assert f(p, B, n, kdim, None, p, None, img, Lp, p, p, None) == -1, (B, n, kdim, img, Lp)
