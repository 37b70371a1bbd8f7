"""Host side of the CUDA-graph options: conf.graph_capacity is checked when the module is built, and a capture runs with
the cyclic garbage collector off."""
import contextlib
import gc

import pytest
import torch

from glue_factory_colon_b200 import LightGlue
from glue_factory_colon_b200 import lightglue as lg


@pytest.mark.parametrize("cap", [None, 1, 2048])
def test_graph_capacity_accepted(cap):
    assert LightGlue({"cuda_graph": True, "graph_capacity": cap}).conf.graph_capacity == cap


@pytest.mark.parametrize("cap", [0, -512, 2048.0, 1.5, True, "2048"])
def test_graph_capacity_rejected(cap):
    with pytest.raises(ValueError, match="graph_capacity"):
        LightGlue({"cuda_graph": True, "graph_capacity": cap})


def test_capture_runs_without_the_garbage_collector(monkeypatch):
    seen = []

    @contextlib.contextmanager
    def fake_graph(graph):
        seen.append(("enter", graph, gc.isenabled()))
        yield
        seen.append(("exit", graph, gc.isenabled()))

    monkeypatch.setattr(torch.cuda, "graph", fake_graph)
    assert gc.isenabled()
    assert lg._capture("g", lambda: gc.isenabled()) is False
    assert seen == [("enter", "g", False), ("exit", "g", False)] and gc.isenabled()

    def fails():
        raise RuntimeError("capture failed")

    with pytest.raises(RuntimeError, match="capture failed"):
        lg._capture("g", fails)
    assert gc.isenabled()
    gc.disable()  # a caller that runs without the collector keeps it off
    try:
        lg._capture("g", lambda: None)
        assert not gc.isenabled()
    finally:
        gc.enable()
