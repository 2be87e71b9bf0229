"""CPU: the size envelope of the batched BFS (gnan_apsp_bfs_batched_ex) is refused before any CUDA call, naming the cap, and the
Python constant matches the header's."""
import ctypes
import os
import re

import pytest

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


def test_python_cap_equals_header_define():
    from gnan_b200 import _lib
    src = open(os.path.join(ROOT, "include", "gnan_b200.h")).read()
    m = re.search(r"#define\s+GNAN_APSP_BATCHED_MAX_NODES\s+(\d+)", src)
    assert m and int(m.group(1)) == _lib.APSP_BATCHED_MAX_NODES == 1024


@pytest.mark.parametrize("max_n", [1025, 0])
def test_batched_bfs_refuses_outside_its_envelope(lib, max_n):
    """Host buffers stand in for device pointers: a refusal must come before anything touches them."""
    from gnan_b200 import _lib
    arr = (ctypes.c_int64 * 16)()
    buf = ctypes.addressof(arr)
    rc = lib.gnan_apsp_bfs_batched_ex(buf, buf, buf, buf, 2, max_n, buf, buf, None, 48, buf, None, buf, None)
    assert rc == 2
    assert str(_lib.APSP_BATCHED_MAX_NODES).encode() in lib.gnan_last_error()
