"""The U-Net's CUDA-graph captures hold Python's cyclic garbage collector off: a collection inside a capture can destroy
the captured graphs of an unreachable model, which invalidates the open capture. Checked without a device by standing
in for torch.cuda.graph."""
import contextlib
import gc

import pytest
import torch

from diffusion_pruning_b200 import unet


@pytest.fixture
def recorded(monkeypatch):
    seen = []

    @contextlib.contextmanager
    def fake_graph(g):
        seen.append(("enter", g, gc.isenabled()))
        yield
        seen.append(("exit", g, gc.isenabled()))
    monkeypatch.setattr(torch.cuda, "graph", fake_graph)
    enabled = gc.isenabled()
    yield seen
    gc.enable() if enabled else gc.disable()


def test_gc_is_off_during_capture_and_restored(recorded):
    gc.enable()
    with unet._graph_capture("g"):
        inside = gc.isenabled()
    assert not inside
    assert recorded == [("enter", "g", False), ("exit", "g", False)]
    assert gc.isenabled()


def test_gc_restored_when_capture_raises(recorded):
    gc.enable()
    with pytest.raises(RuntimeError):
        with unet._graph_capture("g"):
            raise RuntimeError("capture failed")
    assert gc.isenabled()


def test_gc_left_off_when_it_was_off(recorded):
    gc.disable()
    with unet._graph_capture("g"):
        pass
    assert not gc.isenabled()
