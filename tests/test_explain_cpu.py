"""CPU: gnan_b200.interpret.explain through the real modules (each module's `_aggregation`, the compressed feature form, the graph /
node / NAM readout cases) on every golden case of the unmodified reference, with the CUDA ops replaced by dense torch definitions:
those of tests/test_dist_modules_cpu.py and tests/test_modules_composition_cpu.py, plus the explanation ops below, which restate
their C ABI semantics (include/gnan_b200.h) the dense way, without the baseline-plus-exceptions algebra the kernels use. The same
cases run on the kernels in tests/test_gpu_explain.py."""
import ctypes
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import gnan_lut
from tests import _explain_f64 as X
from tests import _golden as G
from tests._build import build_module
from tests.test_dist_modules_cpu import _install_torch_ops
from tests.test_cabi import lib_path  # noqa: F401  (fixture: builds the library)
from tests.test_modules_composition_cpu import _from_reference_format, _install_torch_entries_ops

TOL = 1e-5


def _install_torch_explain_ops(setter):
    from gnan_b200 import ops

    def explain_segments(grp_ptr, ent_row, node_off):
        K, B = grp_ptr.numel() - 1, node_off.numel() - 1
        seg = torch.empty(K, B + 1, dtype=torch.int64)
        for k in range(K):
            e0, e1 = int(grp_ptr[k]) + 1, int(grp_ptr[k + 1])
            seg[k] = e0 + torch.searchsorted(ent_row[e0:e1], node_off.long())
        return seg

    def entry_matrix(Y, grp_ptr, ent_row, n):
        """Yx[j,k,:] = f_k(x_jk): every row takes its feature's baseline unless it is listed as an exception"""
        K = grp_ptr.numel() - 1
        Yx = Y[grp_ptr[:-1]].unsqueeze(0).repeat(n, 1, 1)
        for k in range(K):
            e = torch.arange(int(grp_ptr[k]) + 1, int(grp_ptr[k + 1]))
            Yx[ent_row[e], k] = Y[e]
        return Yx

    def explain_graph_features(Y, grp_ptr, ent_row, seg, colw, colw_sum):
        K, B = grp_ptr.numel() - 1, seg.shape[1] - 1
        F = torch.empty(B, K, Y.shape[1])
        for k in range(K):
            yb = Y[grp_ptr[k]]
            for b in range(B):
                e = torch.arange(int(seg[k, b]), int(seg[k, b + 1]))
                F[b, k] = yb * colw_sum[b] + (colw[ent_row[e]] * (Y[e] - yb)).sum(0)
        return F

    def explain_rows_features(hop, hop_off, node_off, ncols, rows, n_rows, T, per_row, rscale, Y, grp_ptr, ent_row, seg):
        N = int(node_off[-1])
        Yx = entry_matrix(Y, grp_ptr, ent_row, N)
        ids = rows.tolist() if rows is not None else list(range(n_rows))
        nbins = T.shape[-2]
        out = []
        for i in ids:
            if hop_off is None:
                h, cols = hop[i, :N].long(), slice(0, N)
            else:
                b = int(torch.searchsorted(node_off.long(), torch.tensor(i), right=True)) - 1
                r0, r1 = int(node_off[b]), int(node_off[b + 1])
                n = r1 - r0
                h = hop[int(hop_off[b]) + (i - r0) * n:int(hop_off[b]) + (i - r0 + 1) * n].long()
                cols = slice(r0, r1)
            d = h.clamp(max=nbins - 1)
            w = (T[i] if per_row else T)[d]                                           # [n,Cr]
            if rscale is not None:
                w = w * rscale[i][d][:, None]
            out.append((w[:, None, :] * Yx[cols]).sum(0))
        return torch.stack(out) if out else Y.new_zeros(0, grp_ptr.numel() - 1, Y.shape[1])

    def gather_segment_sum(src, order, seg_ptr):
        return torch.stack([src[int(seg_ptr[s]):int(seg_ptr[s + 1])].sum(0) for s in range(seg_ptr.numel() - 1)])

    for name, fn in (("explain_segments", explain_segments), ("explain_graph_features", explain_graph_features),
                     ("explain_rows_features", explain_rows_features), ("gather_segment_sum", gather_segment_sum)):
        setter(ops, name, fn)


def _mode(z):
    if z["variant"] == "batched":
        return "raw"
    if not z["normalize_rho"]:
        return "none"
    return "input" if z["variant"] == "gnanpy_tensor" else "output"


def reference_explanation(z):
    """(features, A, nodes, A_nodes) in float64 from the golden weights; A None where the features are not a plain sum"""
    p_fs, p_rho = X.params(z["fs"]), X.params(z["rho"])
    x = torch.tensor(z["x"]).double()
    mode = _mode(z)
    if z["variant"] == "batched":
        hop = torch.tensor(z["dist_batch"]).round().long()
        bv = torch.tensor(z["batch_vector"]).long()
        F, A, terms, W = X.node_rows(p_fs, p_rho, x, hop, None, mode)
        if not z["is_graph_task"]:
            return F, A, None, None
        B = int(bv.max()) + 1
        Fg = torch.zeros(B, *F.shape[1:], dtype=F.dtype).index_add(0, bv, F)
        Ag = torch.zeros(B, *A.shape[1:], dtype=A.dtype).index_add(0, bv, A)
        return (Fg, Ag) + X.colw_nodes(W, terms)
    hop = gnan_lut.hops_from_reference(torch.tensor(z["node_distances"]))
    cnt = gnan_lut.counts_from_hops(hop)
    if not z["is_graph_task"]:
        if z["variant"] == "gnan_loop" and "node_ids" in z:
            ids = torch.tensor(z["node_ids"]).long()
            hop, cnt = hop[ids], cnt[ids]
        F, A, _, _ = X.node_rows(p_fs, p_rho, x, hop, cnt, mode)
        return F, A, None, None
    F, A, nodes, An = X.graph_row(p_fs, p_rho, x, hop, cnt, mode)
    if "readout" in z:
        return X.nam_features(X.params(z["readout"]), F[None, :, 0]), None, None, None
    return F[None], A[None], nodes, An


def _explain_golden(z, dedup):
    from gnan_b200 import interpret
    m = build_module(z).eval()
    m.dedup = dedup
    if z["variant"] == "batched":
        return interpret.explain(m, (torch.tensor(z["x"]), torch.tensor(z["dist_batch"]), torch.tensor(z["batch_vector"])))
    data = SimpleNamespace(x=torch.tensor(z["x"]), edge_index=torch.tensor(z["edge_index"]), node_distances=torch.tensor(z["node_distances"]),
                           normalization_matrix=torch.tensor(z["normalization_matrix"]))
    ids = z["node_ids"].tolist() if (z["variant"] == "gnan_loop" and "node_ids" in z) else None
    return interpret.explain(m, data, ids)


@pytest.mark.parametrize("dedup", [True, False], ids=["dedup", "no_dedup"])
@pytest.mark.parametrize("name", G.MODEL_CASES + G.BATCHED_CASES)
def test_explanations_decompose_the_golden_outputs(name, dedup, monkeypatch):
    from gnan_b200 import _inputs
    _install_torch_ops(monkeypatch.setattr)
    _install_torch_entries_ops(monkeypatch.setattr)
    _install_torch_explain_ops(monkeypatch.setattr)
    monkeypatch.setattr(_inputs, "from_reference_format", _from_reference_format)
    z = G.load(name)
    e = _explain_golden(z, dedup)
    want_out = z["out"].T if (z["is_graph_task"] and z["variant"] != "batched") else z["out"]
    assert tuple(e.out.shape) == want_out.shape and e.features.shape[:1] == e.out.shape[:1] and e.features.shape[2] == e.out.shape[1]
    assert G.rel_err(e.out.numpy(), want_out) < TOL
    assert G.rel_err(e.features.sum(dim=1).numpy(), want_out) < TOL
    F, A, nodes, An = reference_explanation(z)
    assert e.features.shape == F.shape
    if A is None:                                     # NAM readout: g_k of the per-feature graph value
        assert G.rel_err(e.features.numpy(), F.numpy()) < TOL
    else:
        assert bool(((e.features.double() - F).abs() <= TOL * A + 1e-12).all()), float(((e.features.double() - F).abs() / A.clamp(min=1e-30)).max())
    if nodes is None:
        assert e.nodes is None
    else:
        assert bool(((e.nodes.double() - nodes).abs() <= TOL * An + 1e-12).all())
        bv = torch.tensor(z["batch_vector"]).long() if z["variant"] == "batched" else torch.zeros(nodes.shape[0], dtype=torch.long)
        per_graph = torch.zeros_like(e.out).index_add(0, bv, e.nodes)
        assert G.rel_err(per_graph.numpy(), want_out) < TOL


def test_explain_entry_points_validate_their_arguments_without_gpu(lib_path):
    """NULL pointers and impossible sizes are refused before any CUDA call"""
    from gnan_b200 import _lib
    lib = _lib.load()
    arr = (ctypes.c_int64 * 8)()
    buf = ctypes.addressof(arr)
    assert lib.gnan_explain_segments(None, buf, 2, buf, 1, buf, None) == 1 and b"NULL" in lib.gnan_last_error()
    assert lib.gnan_explain_segments(buf, buf, 0, buf, 1, buf, None) == 1
    assert lib.gnan_explain_segments(buf, buf, 2, buf, -1, buf, None) == 1
    assert lib.gnan_explain_graph_features(buf, buf, buf, buf, 2, 3, 1, None, buf, buf, None) == 1 and b"NULL" in lib.gnan_last_error()
    assert lib.gnan_explain_graph_features(buf, buf, buf, buf, 2, 0, 1, None, None, None, None) == 0       # no graphs: nothing to do
    args = [buf, 16, None, buf, 1, 4, None, 4, buf, 0, 5, 1, None, buf, buf, buf, buf, 2, 1, buf, None]
    bad = list(args); bad[0] = None                                                                           # hop
    assert lib.gnan_explain_rows_features(*bad) == 1 and b"NULL" in lib.gnan_last_error()
    bad = list(args); bad[19] = None                                                                          # F
    assert lib.gnan_explain_rows_features(*bad) == 1
    bad = list(args); bad[11] = 3                                                                             # Cr neither 1 nor C
    assert lib.gnan_explain_rows_features(*bad) == 1
    bad = list(args); bad[1] = 2                                                                              # ld_hop < ncols
    assert lib.gnan_explain_rows_features(*bad) == 1
    bad = list(args); bad[1] = bad[5] = 1 << 20                                                               # a row larger than shared memory
    assert lib.gnan_explain_rows_features(*bad) == 2


@pytest.mark.parametrize("name,ids", [("gnan_loop_shared_rho", [0, -1]), ("gnanpy_tensor_node", [-3]), ("models_tensor_node_shared_rho", [0, 10 ** 6])])
def test_node_ids_outside_the_rows_are_refused(name, ids, monkeypatch):
    """node_ids index hop rows, tables and normalisers on the device: a negative or too large id is refused before any kernel"""
    from gnan_b200 import _inputs, interpret
    _install_torch_ops(monkeypatch.setattr)
    _install_torch_entries_ops(monkeypatch.setattr)
    _install_torch_explain_ops(monkeypatch.setattr)
    monkeypatch.setattr(_inputs, "from_reference_format", _from_reference_format)
    z = G.load(name)
    m = build_module(z).eval()
    data = SimpleNamespace(x=torch.tensor(z["x"]), node_distances=torch.tensor(z["node_distances"]),
                           normalization_matrix=torch.tensor(z["normalization_matrix"]))
    with pytest.raises(IndexError):
        interpret.explain(m, data, ids)
