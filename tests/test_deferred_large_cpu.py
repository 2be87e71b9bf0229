"""CPU: the int16 transfer form of a batch's edge list (preprocess.LocalEdges with dtype=torch.int16, graphs of up to 1024 nodes)
and the size envelope of the fused BFS + graph readout entry points, which refuse a max_n they cannot address before any CUDA
call (host buffers stand in for device pointers, so nothing is launched)."""
import ctypes
import os

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import importlib.util
    spec = importlib.util.spec_from_file_location("gnan_build", os.path.join(ROOT, "graph-neural-additive-networks---gnan_b200", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.build()
    from gnan_b200 import _lib
    return _lib.load()


def test_local_edges_int16_host_form():
    """int16 endpoints inside the graph, per-graph edge offsets, stable grouping by graph, 4 bytes per directed edge"""
    from gnan_b200.preprocess import LocalEdges
    node_off = np.array([0, 3, 3, 8, 1032])                                   # graph 3 has 1024 nodes
    ei = torch.tensor([[4, 0, 1031, 1, 7, 8, 600], [5, 2, 8, 0, 3, 1031, 9]])
    le = LocalEdges.from_edge_index(ei, node_off, dtype=torch.int16)
    assert le.src.dtype == le.dst.dtype == le.dtype == torch.int16 and le.edge_off.dtype == torch.int32
    assert le.nbytes() == 7 * 2 * 2 + 5 * 4
    assert le.edge_off.tolist() == [0, 2, 2, 4, 7]
    assert le.src.tolist() == [0, 1, 1, 4, 1023, 0, 592] and le.dst.tolist() == [2, 0, 2, 0, 0, 1023, 1]
    small = torch.tensor([[4, 0, 263, 1, 7, 8], [5, 2, 8, 0, 3, 263]])                 # the uint8 test's batch
    same = LocalEdges.from_edge_index(small, np.array([0, 3, 3, 8, 264]), dtype=torch.int16)
    narrow = LocalEdges.from_edge_index(small, np.array([0, 3, 3, 8, 264]))
    assert narrow.dtype == torch.uint8 and narrow.nbytes() == 12 + 20
    assert same.src.tolist() == narrow.src.tolist() and same.dst.tolist() == narrow.dst.tolist()
    assert same.edge_off.tolist() == narrow.edge_off.tolist()


def test_local_edges_width_limits():
    from gnan_b200 import _lib
    from gnan_b200.preprocess import LocalEdges
    with pytest.raises(ValueError, match=str(_lib.APSP_BATCHED_MAX_NODES)):
        LocalEdges.from_edge_index(torch.tensor([[0], [1]]), np.array([0, 1025]), dtype=torch.int16)
    with pytest.raises(ValueError, match="256"):
        LocalEdges.from_edge_index(torch.tensor([[0], [1]]), np.array([0, 257]))          # the default width stays uint8
    with pytest.raises(ValueError):
        LocalEdges.from_edge_index(torch.tensor([[0], [3]]), np.array([0, 3, 600]), dtype=torch.int16)   # leaves its graph
    with pytest.raises(TypeError):
        LocalEdges.from_edge_index(torch.tensor([[0], [1]]), np.array([0, 2]), dtype=torch.int32)
    le = LocalEdges.from_edge_index(torch.tensor([[0], [1]]), np.array([0, 1024]), dtype=torch.int16)
    assert le.src.tolist() == [0] and le.dst.tolist() == [1]


def test_local_edges_to_keeps_the_width():
    from gnan_b200.preprocess import LocalEdges
    le = LocalEdges.from_edge_index(torch.tensor([[0, 700], [700, 0]]), np.array([0, 900]), dtype=torch.int16)
    moved = le.to("cpu")
    assert moved.dtype == torch.int16 and torch.equal(moved.src, le.src) and moved.nbytes() == le.nbytes()


def _readout_call(lib, name, max_n, B=2):
    arr = (ctypes.c_int64 * 64)()
    buf = ctypes.addressof(arr)
    return getattr(lib, name)(buf, buf, buf, buf, B, max_n, 8, buf, 1, buf, 1, buf, buf, buf, buf, buf, buf, buf, None)


@pytest.mark.parametrize("name,cap", [("gnan_bfs_graph_readout_fwd", 256), ("gnan_bfs_graph_readout_fwd_i16", 1024)])
@pytest.mark.parametrize("over", [True, False])
def test_fused_readout_refuses_sizes_it_cannot_address(lib, name, cap, over):
    rc = _readout_call(lib, name, cap + 1 if over else 0)
    assert rc == 2
    msg = lib.gnan_last_error()
    assert str(cap).encode() in msg and name[len("gnan_"):].encode() in msg


def test_fused_readout_envelope_is_checked_first(lib):
    """nbins / C outside the one-pass envelope: refused the same way, whatever the endpoint width"""
    arr = (ctypes.c_int64 * 64)()
    buf = ctypes.addressof(arr)
    rc = lib.gnan_bfs_graph_readout_fwd_i16(buf, buf, buf, buf, 2, 300, 65, buf, 1, buf, 1, buf, buf, buf, buf, buf, buf, buf, None)
    assert rc == 2 and b"nbins" in lib.gnan_last_error()


def test_edges_from_local_i16_validates_without_gpu(lib):
    rc = lib.gnan_edges_from_local_i16(None, None, None, None, 1, 4, None, None)
    assert rc == 1 and b"edges_from_local_i16" in lib.gnan_last_error()
    assert lib.gnan_edges_from_local_i16(None, None, None, None, 0, 0, None, None) == 0
