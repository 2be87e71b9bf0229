"""GPU: gnan_b200.interpret.explain on the kernels of csrc/explain.cu against the float64 restatement of the reference's per-feature
terms (tests/_explain_f64.py): every contribution within |err| <= 1e-5 * A, A the sum of the absolute values of its terms (the
convention of tests/test_gpu_graph_readout_f64.py). Also: e.out is the eval-mode fp32 forward bit for bit, the node contributions
of a graph sum to its output, and two calls are bit-identical."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import apsp as oapsp
from oracle import gnan_lut
from tests import _explain_f64 as X
from tests import _golden as G
from tests._build import build_module
from tests.test_explain_cpu import reference_explanation
from tests.test_gpu_parity import random_graph

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5
NAMES = ("w1", "b1", "wh", "bh", "wo", "bo")


def f64(st):
    d = {n: getattr(st, n).detach().double().cpu() for n in NAMES}
    if st.n_layers == 1:
        d.update(w1=None, b1=None, wh=None, bh=None)
    return d


def forward_fp32(model, inputs, node_ids=None):
    from gnan_b200.GNAN import GNAN as RowGNAN
    model.eval()
    model.precision = "fp32"
    with torch.no_grad():
        if isinstance(inputs, tuple):
            return model(*inputs)
        return model(inputs, node_ids) if isinstance(model, RowGNAN) else model(inputs)


def explain_checked(model, inputs, node_ids=None):
    """explain twice (bit-identical), e.out == the fp32 eval forward, sum over features == out"""
    from gnan_b200 import interpret
    e = interpret.explain(model, inputs, node_ids)
    again = interpret.explain(model, inputs, node_ids)
    assert torch.equal(e.features, again.features) and torch.equal(e.out, again.out)
    assert (e.nodes is None) == (again.nodes is None) and (e.nodes is None or torch.equal(e.nodes, again.nodes))
    from gnan_b200.GNAN import GNAN as RowGNAN
    want = forward_fp32(model, inputs, node_ids)
    if node_ids is not None and not isinstance(model, RowGNAN):
        want = want[torch.as_tensor(node_ids, device=want.device, dtype=torch.long)]
    elif want.shape != e.out.shape:                    # [C,1] of a single graph
        want = want.T
    assert torch.equal(e.out, want)
    torch.cuda.synchronize()
    return e


def assert_close(got, want, A, tag=""):
    err = (got.double().cpu() - want).abs()
    worst = float((err / A.clamp(min=1e-30)).max()) if err.numel() else 0.0
    assert bool((err <= TOL * A + 1e-30).all()), (tag, worst)


def assert_sums(e, graph_of=None):
    """sum over features == out, and for graph rows the node contributions summed per graph == out (norm-wise)"""
    assert G.rel_err(e.features.sum(dim=1).cpu().numpy(), e.out.cpu().numpy()) < TOL
    if e.nodes is not None:
        per_graph = torch.zeros_like(e.out).index_add(0, graph_of, e.nodes)
        assert G.rel_err(per_graph.cpu().numpy(), e.out.cpu().numpy()) < TOL


# ---- golden cases --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", G.MODEL_CASES + G.BATCHED_CASES)
def test_golden_cases(name):
    z = G.load(name)
    m = build_module(z, device=DEV).eval()
    if z["variant"] == "batched":
        inputs = (torch.tensor(z["x"]), torch.tensor(z["dist_batch"]).to(DEV), torch.tensor(z["batch_vector"]).to(DEV))
    else:
        inputs = SimpleNamespace(x=torch.tensor(z["x"]), edge_index=torch.tensor(z["edge_index"]),
                                 node_distances=torch.tensor(z["node_distances"]), normalization_matrix=torch.tensor(z["normalization_matrix"]))
    ids = z["node_ids"].tolist() if (z["variant"] == "gnan_loop" and "node_ids" in z) else None
    e = explain_checked(m, inputs, ids)
    F, A, nodes, An = reference_explanation(z)
    if A is None:
        assert G.rel_err(e.features.cpu().numpy(), F.numpy()) < TOL
    else:
        assert_close(e.features, F, A, name)
    if nodes is not None:
        assert_close(e.nodes, nodes, An, name + " nodes")
        bv = torch.tensor(z["batch_vector"]).long().to(DEV) if z["variant"] == "batched" else torch.zeros(nodes.shape[0], dtype=torch.long, device=DEV)
        assert_sums(e, bv)


# ---- random single graphs: node tasks -------------------------------------------------------------------------------------
def features_of(rng, n, K):
    """normal columns, a sparse indicator column, the constant column (no exceptions); K = 1: one dense column"""
    x = rng.normal(size=(n, K)).astype(np.float32)
    if K >= 3:
        x[:, 1] = (rng.random(n) < 0.1).astype(np.float32)
        x[:, -1] = 1.0
    return torch.tensor(x)


def build(kind, K, C, L, H, rpf, norm, graph=False, readout=0):
    from gnan_b200 import GNAN as g, models as mo
    torch.manual_seed(0)
    if kind == "gnanpy":
        m = g.TensorGNAN(K, C, L, H, normalize_rho=norm, is_graph_task=graph)
    elif kind == "models":
        m = mo.TensorGNAN(K, C, L, H, normalize_rho=norm, is_graph_task=graph, rho_per_feature=rpf, readout_n_layers=readout)
    else:
        m = g.GNAN(K, C, L, H, normalize_rho=norm, rho_per_feature=rpf)
    m = m.to(DEV)
    m.fs.xavier_normal_(1.0); m.rho.xavier_normal_(1.0)
    with torch.no_grad():
        for p in m.parameters():
            if p.dim() <= 2 and p.numel() and float(p.abs().max()) == 0.0:
                p.normal_(0.0, 0.3)
    return m


def mode_of(kind, norm):
    return ("input" if kind == "gnanpy" else "output") if norm else "none"


NODE_CASES = [  # kind, K, C, L, H, rho_per_feature, normalize, directed
    ("gnanpy", 6, 1, 3, 64, True, True, False), ("gnanpy", 6, 3, 2, 8, True, False, True), ("gnanpy", 5, 7, 3, 64, True, True, True),
    ("gnanpy", 1, 2, 1, 8, True, True, False), ("gnanpy", 4, 40, 3, 8, True, True, False),
    ("models", 6, 3, 3, 64, False, True, False), ("models", 6, 3, 3, 64, True, True, True), ("models", 5, 2, 2, 8, True, False, False),
    ("models", 7, 40, 3, 64, False, True, True), ("models", 1, 7, 1, 8, True, True, True),
    ("gnan", 6, 3, 3, 64, False, True, False), ("gnan", 6, 7, 2, 8, True, True, True), ("gnan", 4, 1, 1, 8, False, False, False),
]


# GNAN.GNAN's own forward refuses an empty row list (the row aggregation of zero selected hop rows), so that pair is not a case here
@pytest.mark.parametrize("case,ids_kind", [(c, k) for c in NODE_CASES for k in ("all", "subset", "duplicates", "empty")
                                           if not (k == "empty" and c[0] == "gnan")],
                         ids=lambda v: "-".join(map(str, v)) if isinstance(v, tuple) else v)
def test_node_rows_vs_float64(case, ids_kind):
    from gnan_b200.preprocess import apsp
    kind, K, C, L, H, rpf, norm, directed = case
    rng = np.random.default_rng(K * 100 + C)
    n = 150
    ei = random_graph(rng, n, 2.0, directed, n_isolated=4)
    x = features_of(rng, n, K)
    hd = apsp(torch.tensor(ei), n, device=DEV)
    m = build(kind, K, C, L, H, rpf, norm)
    ids = {"all": None, "subset": [3, 140, 7, 77], "duplicates": [5, 5, 149, 0, 5], "empty": []}[ids_kind]
    e = explain_checked(m, SimpleNamespace(x=x, hop_data=hd), ids)
    hop = torch.tensor(oapsp.apsp(ei, n)).long()
    cnt = gnan_lut.counts_from_hops(hop)
    sel = torch.arange(n) if ids is None else torch.tensor(ids, dtype=torch.long)
    F, A, _, _ = X.node_rows(f64(m.fs), f64(m.rho), x, hop[sel], cnt[sel], mode_of(kind, norm))
    assert e.features.shape == F.shape and e.nodes is None
    assert_close(e.features, F, A, str(case))
    if e.features.shape[0]:
        assert_sums(e)


# ---- packed batches -------------------------------------------------------------------------------------------------------
SIZES = [1, 2, 9, 30, 64, 150, 17, 3]           # a 1-node graph, an edgeless 2-node graph, one larger than 128 nodes


def packed_batch(rng, directed, K, sizes=SIZES):
    from gnan_b200.preprocess import apsp_batched
    node_off = np.concatenate([[0], np.cumsum(sizes)])
    eis = [np.zeros((2, 0), np.int64) if n <= 2 else random_graph(rng, n, 2.2, directed, n_isolated=1 if n > 8 else 0) for n in sizes]
    ei = torch.tensor(np.concatenate([e + node_off[i] for i, e in enumerate(eis)], axis=1))
    x = features_of(rng, int(node_off[-1]), K)
    pk = apsp_batched(ei, node_off, device=DEV, x=x.to(DEV))
    return pk, eis, node_off, x


def packed_reference(m, eis, node_off, x, mode, graph):
    F, A, Nd, An = [], [], [], []
    for i, e in enumerate(eis):
        r0, r1 = int(node_off[i]), int(node_off[i + 1])
        hop = torch.tensor(oapsp.apsp(e, r1 - r0)).long()
        cnt = gnan_lut.counts_from_hops(hop) if mode != "raw" else None
        if graph:
            f, a, nd, an = X.graph_row(f64(m.fs), f64(m.rho), x[r0:r1], hop, cnt, mode)
            F.append(f[None]); A.append(a[None]); Nd.append(nd); An.append(an)
        else:
            f, a, _, _ = X.node_rows(f64(m.fs), f64(m.rho), x[r0:r1], hop, cnt, mode)
            F.append(f); A.append(a)
    return torch.cat(F), torch.cat(A), (torch.cat(Nd) if graph else None), (torch.cat(An) if graph else None)


@pytest.mark.parametrize("graph", [True, False], ids=["graph", "node"])
@pytest.mark.parametrize("kind,C,rpf,norm,directed", [("gnanpy", 3, True, True, False), ("gnanpy", 2, True, False, True),
                                                      ("models", 1, False, True, False), ("models", 3, True, True, True),
                                                      ("models", 7, True, False, False), ("batched", 2, True, True, False),
                                                      ("batched", 1, True, True, True)])
def test_packed_batches_vs_float64(kind, C, rpf, norm, directed, graph):
    rng = np.random.default_rng(C * 10 + directed)
    K = 5
    pk, eis, node_off, x = packed_batch(rng, directed, K)
    if kind == "batched":
        from gnan_b200 import batched
        torch.manual_seed(0)
        m = batched.TensorGNAN(K, C, 2, hidden_channels=16, is_graph_task=graph).to(DEV)
        mode = "raw"
    else:
        m = build(kind, K, C, 3, 64, rpf, norm, graph=graph)
        mode = mode_of(kind, norm)
    e = explain_checked(m, pk)
    F, A, nodes, An = packed_reference(m, eis, node_off, x, mode, graph)
    assert e.features.shape == F.shape
    assert_close(e.features, F, A, f"{kind} {C}")
    if graph:
        assert_close(e.nodes, nodes, An, "nodes")
        assert_sums(e, pk.batch_vector)
    else:
        assert e.nodes is None
        sub = explain_checked(m, pk, [0, 3, 3, int(node_off[-1]) - 1])       # a row list of a packed node-level output
        assert torch.equal(sub.features, e.features[[0, 3, 3, int(node_off[-1]) - 1]])


def test_deferred_molecule_batch_next_to_its_materialised_twin():
    """the fused BFS + readout path (distances never written) against the same batch after its distances were materialised"""
    from gnan_b200.preprocess import LocalEdges, apsp_batched
    rng = np.random.default_rng(7)
    sizes = [int(v) for v in rng.integers(1, 129, size=200)]
    node_off = np.concatenate([[0], np.cumsum(sizes)])
    eis = [random_graph(rng, n, 2.2, False) for n in sizes]
    ei = torch.tensor(np.concatenate([e + node_off[i] for i, e in enumerate(eis)], axis=1))
    x = features_of(rng, int(node_off[-1]), 5).to(DEV)
    le = LocalEdges.from_edge_index(ei, node_off)
    fused = apsp_batched(le, node_off, device=DEV, x=x, nbins=48, rscale=True)
    twin = apsp_batched(le, node_off, device=DEV, x=x, nbins=48, rscale=True)
    twin.hop                                                                     # materialise the twin's distances
    m = build("models", 5, 1, 3, 64, False, True, graph=True)
    e = explain_checked(m, fused)
    assert fused.deferred and not twin.deferred
    t = explain_checked(m, twin)
    F, A, nodes, An = packed_reference(m, eis, node_off, x.cpu(), "output", True)
    assert_close(e.features, F, A, "fused")
    assert_close(t.features, F, A, "materialised")
    assert_close(e.nodes, nodes, An, "fused nodes")
    assert_sums(e, fused.batch_vector)


@pytest.mark.parametrize("packed", [False, True])
def test_nam_readout(packed):
    rng = np.random.default_rng(11)
    K, C = 6, 3
    m = build("models", K, C, 3, 64, False, True, graph=True, readout=2)
    if packed:
        pk, eis, node_off, x = packed_batch(rng, False, K)
        e = explain_checked(m, pk)
    else:
        from gnan_b200.preprocess import apsp
        n = 60
        eis, node_off = [random_graph(rng, n, 2.0, False, n_isolated=2)], np.array([0, n])
        x = features_of(rng, n, K)
        e = explain_checked(m, SimpleNamespace(x=x, hop_data=apsp(torch.tensor(eis[0]), n, device=DEV)))
    F, A, _, _ = packed_reference(m, eis, node_off, x, "output", True)
    want = X.nam_features(f64(m.readout_nam.fs), F[:, :, 0])
    assert e.nodes is None and e.features.shape == want.shape
    assert G.rel_err(e.features.cpu().numpy(), want.numpy()) < TOL
    assert_sums(e)


def test_int16_hop_matrices_are_refused():
    from gnan_b200 import interpret
    from gnan_b200.preprocess import apsp
    from tests.test_gpu_wide import deep_graph
    ei, n = deep_graph(np.random.default_rng(3))
    hd = apsp(torch.tensor(ei), n, device=DEV)
    assert hd.wide
    m = build("gnanpy", 3, 2, 3, 64, True, True)
    with pytest.raises(NotImplementedError):
        interpret.explain(m, SimpleNamespace(x=torch.ones(n, 3), hop_data=hd))


# ---- real-size configurations (bench.py's workloads) ----------------------------------------------------------------------
@pytest.mark.parametrize("name,rows", [("cora", None), ("pubmed", 512)])
def test_real_size_node_configs(name, rows):
    """Cora shape (all 2 708 rows) and a 512-row block of the PubMed shape, as tests/test_gpu_configs.py builds them: sums and
    determinism on every row, float64 on a sample of rows. The sample is checked twice: end to end (shape functions in float64),
    and against a float64 aggregation of the GPU's own entry values, which holds the kernels to the aggregation's terms alone."""
    import bench
    from gnan_b200.GNAN import TensorGNAN
    from gnan_b200.preprocess import apsp
    wl = bench.make_node_workload(name)
    torch.manual_seed(0)
    m = TensorGNAN(wl.K, wl.C, bench.L, bench.H, normalize_rho=True, is_graph_task=False, device=DEV).to(DEV)
    m.fs.xavier_normal_(1.0); m.rho.xavier_normal_(1.0)
    R = wl.n if rows is None else rows
    hd = apsp(wl.edge_index, wl.n, device=DEV, row_begin=0, row_end=R)
    inputs = SimpleNamespace(x=wl.x, hop_data=hd)
    e = explain_checked(m, inputs)
    assert e.features.shape == (R, wl.K, wl.C)
    assert_sums(e)
    sample = [0, 1, R // 2, R - 1]
    hop = torch.tensor(oapsp.apsp(wl.edge_index.numpy(), wl.n)[sample] if rows is None else oapsp.apsp_rows(wl.edge_index.numpy(), wl.n, R)[sample]).long()
    cnt = hd.level_counts[sample].cpu().long()
    F, A, _, W = X.node_rows(f64(m.fs), f64(m.rho), wl.x, hop, cnt, "input")
    assert_close(e.features[sample], F, A, name)
    Yx = entry_values_dense(m, wl.x)
    assert_close(e.features[sample], torch.einsum("ijc,jkc->ikc", W, Yx), torch.einsum("ijc,jkc->ikc", W.abs(), Yx.abs()), name + " kernel")


def entry_values_dense(model, x):
    """f_k(x_jk) [N,K,C] in float64 as the GPU's entries forward computes it (the values explain aggregates)"""
    from gnan_b200 import sparse
    cx = sparse.compress_features(x.to(DEV), max_density=None)
    with torch.no_grad():
        Y = sparse.entry_values(cx, *model.fs.kernel_args()).double().cpu()
    grp_ptr, ent_row, ent_grp = cx.grp_ptr.cpu(), cx.ent_row.cpu(), cx.ent_grp.cpu().long()
    Yx = Y[grp_ptr[:-1]].unsqueeze(0).repeat(x.shape[0], 1, 1)
    exc = ent_row >= 0
    Yx[ent_row[exc], ent_grp[exc]] = Y[exc]
    return Yx


# ---- shapes at the edges of the rows kernel's launch -----------------------------------------------------------------------
@pytest.mark.parametrize("kind,C,rpf,norm", [("gnanpy", 7, True, True), ("models", 1, False, True), ("gnan", 3, True, True)])
def test_rows_wider_than_two_rows_of_shared_memory(kind, C, rpf, norm):
    """A row block of a 120 000-node graph: two staged hop rows exceed the CTA's shared memory, so the rows kernel runs one row per
    CTA. nbins is even and C is odd or 1: the layouts where 8-byte row metadata placed after the float arrays would sit at 4 mod 8."""
    from gnan_b200.ops import hop_ld
    from gnan_b200.preprocess import HopData
    rng = np.random.default_rng(C)
    N, R, nbins, K = 120_000, 5, 16, 4
    h = rng.integers(0, nbins - 1, size=(R, N))
    h[rng.random((R, N)) < 0.05] = -1                                        # unreachable pairs
    h[:, 0] = nbins - 2                                                      # every row reaches the last level
    hop = torch.full((R, hop_ld(N)), 255, dtype=torch.uint8)
    hop[:, :N] = torch.tensor(np.where(h < 0, 255, h).astype(np.uint8))
    hl = torch.tensor(h).long()
    cnt = torch.zeros(R, nbins, dtype=torch.long).scatter_add_(1, torch.where(hl < 0, nbins - 1, hl), torch.ones_like(hl))
    hd = HopData(hop.to(DEV), cnt.to(torch.int32).to(DEV), N)
    x = features_of(rng, N, K)
    m = build(kind, K, C, 3, 64, rpf, norm)
    ids = [4, 0, 4] if kind == "gnan" else None
    e = explain_checked(m, SimpleNamespace(x=x, hop_data=hd), ids)
    sel = torch.arange(R) if ids is None else torch.tensor(ids)
    F, A, _, _ = X.node_rows(f64(m.fs), f64(m.rho), x, hl[sel], cnt[sel], mode_of(kind, norm))
    assert e.features.shape == F.shape
    assert_close(e.features, F, A, f"{kind} {C}")
    assert_sums(e)


def test_batch_without_nodes_is_refused_like_the_forward():
    """an empty packed batch: the model's own forward refuses it (no shape-function rows), and explain reports that same error"""
    from gnan_b200 import interpret
    from gnan_b200.preprocess import PackedBatch
    K, C, nbins = 5, 2, 8
    m = build("models", K, C, 3, 64, True, False, graph=True)
    pk = PackedBatch(torch.zeros(0, K, device=DEV), torch.zeros(1, dtype=torch.uint8, device=DEV), torch.zeros(1, dtype=torch.int64, device=DEV),
                     torch.zeros(1, dtype=torch.int32, device=DEV), torch.zeros(0, nbins, dtype=torch.int32, device=DEV), max_nodes=1)
    with pytest.raises(ValueError):
        forward_fp32(m, pk)
    with pytest.raises(ValueError):
        interpret.explain(m, pk)
