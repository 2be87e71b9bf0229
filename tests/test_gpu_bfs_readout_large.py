"""GPU: deferred batches with graphs of 129..1024 nodes. The fused BFS + graph readout (gnan_bfs_graph_readout_fwd for uint8
endpoints up to 256 nodes, gnan_bfs_graph_readout_fwd_i16 up to 1024) runs graphs of at most 128 nodes on the v3 kernel and the
others on bfs_readout_large_kernel, one CTA each; the first read of `hop` / `level_rscale` materialises such a batch through the
CSR and apsp_batched_large_kernel's rscale output.

Checkers: the float64 restatement of tests/_readout_f64.py on the C oracle's distances (|err| <= 1e-5 * A per entry), the same
model on the materialised twin (2e-6 norm-wise), the count path of apsp_batched (bit-exact), and the kernel itself (bit-identical
reruns; the small graphs of a batch bit-identical with and without large graphs next to them)."""
import numpy as np
import pytest
import torch

from tests import _golden as G
from tests import _readout_f64 as R
from tests.test_gpu_batched_large_graphs import MIXED_SIZES, molecule_like_graphs, mutagenicity_sizes, random_graph

pytestmark = pytest.mark.gpu
DEV = "cuda"
RTOL = 1e-5
TOL = 2e-6
CCR = [(1, 1), (2, 1), (2, 2), (4, 1), (4, 4)]


class _Batch:
    """graphs (n, local [2,E]) -> global edge list, node offsets, oracle hops and the LocalEdges of a width"""

    def __init__(self, graphs):
        self.sizes = np.array([n for n, _ in graphs], dtype=np.int64)
        self.eis = [np.asarray(e, dtype=np.int64).reshape(2, -1) for _, e in graphs]
        self.node_off = np.concatenate([[0], np.cumsum(self.sizes)])
        self.N, self.B, self.max_n = int(self.node_off[-1]), len(graphs), int(self.sizes.max())
        self.ei = torch.from_numpy(np.concatenate([e + self.node_off[b] for b, e in enumerate(self.eis)], axis=1))
        self.node_off_d = torch.tensor(self.node_off, dtype=torch.int32, device=DEV)
        self._hops = None

    @property
    def hops(self):
        if self._hops is None:
            self._hops = R.oracle_hops(self.eis, self.sizes)
        return self._hops

    def edges(self, dtype):
        from gnan_b200.preprocess import LocalEdges
        return LocalEdges.from_edge_index(self.ei, self.node_off, dtype=dtype).to(DEV)


def _graph(rng, n, directed, k):
    """random graphs of average degree 4 (shallow enough for nbins = 64), every third one with isolated vertices"""
    return random_graph(rng, n, 4.0, directed, n_isolated=(1 + k % 4) if (n > 8 and k % 3 == 0) else 0)


def _mixed(seed, max_n=1024, directed=None):
    rng = np.random.default_rng(seed)
    sizes = [n for n in MIXED_SIZES if n <= max_n] + [int(v) for v in rng.integers(1, 129, size=40)]
    sizes = [sizes[k] for k in rng.permutation(len(sizes))]
    return _Batch([(n, _graph(rng, n, bool(k % 2) if directed is None else directed, k)) for k, n in enumerate(sizes)])


def _fused(bt, dtype, T, S, status=None):
    from gnan_b200 import ops
    status = torch.zeros(3, dtype=torch.int32, device=DEV) if status is None else status
    out, colw, Q = ops.bfs_graph_readout_fwd(bt.edges(dtype), bt.node_off_d, bt.max_n, T, S, status)
    return out, colw, Q, status


def _tensors(rng, bt, nbins, C, Cr):
    T = torch.tensor(rng.normal(size=(nbins, Cr))).float().to(DEV)
    S = torch.tensor(rng.normal(size=(bt.N, C))).float().to(DEV)
    return T, S


# ---- 1. out / colw / Q against float64, 4. reruns ---------------------------------------------------------------------------
@pytest.mark.parametrize("C,Cr", CCR)
@pytest.mark.parametrize("dtype,max_n", [(torch.uint8, 256), (torch.int16, 1024)])
def test_fused_large_matches_float64(C, Cr, dtype, max_n):
    bt = _mixed(100 + 10 * C + Cr + max_n, max_n)
    rng = np.random.default_rng(C * 7 + Cr)
    nbins = 64
    T, S = _tensors(rng, bt, nbins, C, Cr)
    out, colw, Q, st = _fused(bt, dtype, T, S)
    ref = R.readout_f64(bt.hops, nbins, T.cpu().numpy(), S.cpu().numpy())
    R.assert_entrywise("out", out.cpu().numpy(), ref.out, ref.a_out, RTOL)
    R.assert_entrywise("colw", colw.cpu().numpy(), ref.colw, ref.a_colw, RTOL, bt.node_off)
    R.assert_entrywise("Q", Q.cpu().numpy(), ref.Q, ref.a_Q, RTOL)
    assert st.tolist() == R.expected_status(bt.hops, nbins)
    again = _fused(bt, dtype, T, S)
    for a, b in zip((out, colw, Q, st), again):
        assert torch.equal(a, b)


@pytest.mark.parametrize("nbins", [2, 5, 33])
def test_fused_large_small_tables(nbins):
    """levels beyond the table: the overflow flag, and the bins below it still exact"""
    bt = _mixed(7 + nbins, 700)
    rng = np.random.default_rng(nbins)
    T, S = _tensors(rng, bt, nbins, 2, 2)
    out, colw, Q, st = _fused(bt, torch.int16, T, S)
    want = R.expected_status(bt.hops, nbins)
    assert st.tolist() == want
    if not want[1]:
        ref = R.readout_f64(bt.hops, nbins, T.cpu().numpy(), S.cpu().numpy())
        R.assert_entrywise("out", out.cpu().numpy(), ref.out, ref.a_out, RTOL)


# ---- 3. the graphs of at most 128 nodes do not notice the large ones; both widths agree ---------------------------------------
def test_small_graphs_are_untouched_and_widths_agree():
    rng = np.random.default_rng(5)
    small = [(int(n), _graph(rng, int(n), bool(k % 2), k)) for k, n in enumerate(rng.integers(1, 129, size=300))]
    large = [(n, _graph(rng, n, bool(k % 2), k)) for k, n in enumerate([129, 200, 256])]
    a, b = _Batch(small), _Batch(small + large)
    for C, Cr in [(1, 1), (2, 2), (4, 1)]:
        T = torch.tensor(rng.normal(size=(48, Cr))).float().to(DEV)
        S = torch.tensor(rng.normal(size=(b.N, C))).float().to(DEV)
        o1, c1, q1, s1 = _fused(a, torch.uint8, T, S[:a.N].contiguous())
        o2, c2, q2, s2 = _fused(b, torch.uint8, T, S)
        assert torch.equal(o1, o2[:a.B]) and torch.equal(c1, c2[:a.N]) and torch.equal(q1, q2[:a.B])
        o3, c3, q3, s3 = _fused(b, torch.int16, T, S)
        assert torch.equal(o2, o3) and torch.equal(c2, c3) and torch.equal(q2, q3) and torch.equal(s2, s3)
        o4, c4, q4, _ = _fused(a, torch.int16, T, S[:a.N].contiguous())
        assert torch.equal(o1, o4) and torch.equal(c1, c4) and torch.equal(q1, q4)


# ---- 2. the model on the deferred batch and on its materialised twin ------------------------------------------------------------
def _model(K, C, rho_per_feature):
    from gnan_b200.models import TensorGNAN
    torch.manual_seed(0)
    m = TensorGNAN(K, C, 3, 64, normalize_rho=True, is_graph_task=True, readout_n_layers=0, rho_per_feature=rho_per_feature,
                   device=DEV).to(DEV)
    m.fs.xavier_normal_(1.0); m.rho.xavier_normal_(1.0)
    return m


def _step(m, batch, w):
    m.zero_grad(set_to_none=True)
    out = m(batch)
    (out * w).sum().backward()
    return out.detach().clone(), [p.grad.clone() for p in m.parameters() if p.grad is not None]


@pytest.mark.parametrize("C,rho_per_feature,dtype", [(1, False, torch.int16), (3, True, torch.int16), (4, False, torch.int16),
                                                     (2, True, torch.uint8)])
def test_model_on_deferred_large_batch_matches_materialised(C, rho_per_feature, dtype):
    from gnan_b200.preprocess import apsp_batched, check_batched_status
    bt = _mixed(30 + C, 1024 if dtype == torch.int16 else 256)
    rng = np.random.default_rng(C)
    x = torch.tensor(rng.normal(size=(bt.N, 5))).float().to(DEV)
    le = bt.edges(dtype)
    pk = apsp_batched(le, bt.node_off, device=DEV, x=x, nbins=64, rscale=True)
    alias = apsp_batched(le, bt.node_off, device=DEV, x=x, nbins=64, pair_stats=True)
    assert pk.deferred and alias.deferred
    m = _model(5, C, rho_per_feature)
    w = torch.tensor(rng.normal(size=(bt.B, C))).float().to(DEV)
    fused = _step(m, pk, w)
    assert pk.deferred
    check_batched_status(pk.status)
    assert torch.equal(_step(m, alias, w)[0], fused[0])
    pk.hop
    assert not pk.deferred
    mat = _step(m, pk, w)
    assert G.rel_err(fused[0].cpu().numpy(), mat[0].cpu().numpy()) < TOL
    assert len(fused[1]) == len(mat[1]) > 0
    for a, b in zip(fused[1], mat[1]):
        assert G.rel_err(a.cpu().numpy(), b.cpu().numpy()) < TOL


# ---- 5. status words ----------------------------------------------------------------------------------------------------------
def test_status_words_of_large_graphs():
    from gnan_b200.preprocess import LocalEdges, check_batched_status
    rng = np.random.default_rng(2)
    T = torch.ones(64, 1, device=DEV)
    g300 = random_graph(rng, 300, 3.0, False)
    node_off = np.array([0, 20, 320])
    ring = np.stack([np.arange(20), (np.arange(20) + 1) % 20])
    base = np.concatenate([ring, ring[::-1], g300 + 20], axis=1)
    S = torch.ones(320, 1, device=DEV)
    from gnan_b200 import ops

    def run(ei, le=None):
        le = le if le is not None else LocalEdges.from_edge_index(torch.tensor(ei), node_off, dtype=torch.int16)
        st = torch.zeros(3, dtype=torch.int32, device=DEV)
        ops.bfs_graph_readout_fwd(le.to(DEV), torch.tensor(node_off, dtype=torch.int32, device=DEV), 300, T, S, st)
        return st

    st = run(base)
    hops = R.oracle_hops([np.concatenate([ring, ring[::-1]], axis=1), g300], [20, 300])
    assert st.tolist() == R.expected_status(hops, 64)                 # max_level = the oracle's largest hop
    check_batched_status(st)
    st = run(np.concatenate([base, base[:, -1:]], axis=1))            # a repeated edge inside the 300-node graph
    assert int(st[0]) == 2
    with pytest.raises(ValueError):
        check_batched_status(st)
    le = LocalEdges.from_edge_index(torch.tensor(base), node_off, dtype=torch.int16)
    le.dst[-1] = 300                                                  # one past the 300-node graph
    st = run(None, le)
    assert int(st[0]) & 1
    path = np.stack([np.arange(299), np.arange(1, 300)]) + 20          # a 300-node path: hops up to 299 > nbins - 2
    st = run(np.concatenate([ring, ring[::-1], path, path[::-1]], axis=1))
    assert int(st[1]) == 1 and int(st[2]) == 299
    with pytest.raises(ValueError):
        check_batched_status(st)


# ---- 6. materialising a deferred large batch -----------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.uint8, torch.int16])
def test_materialised_large_batch_matches_the_count_path(dtype):
    from gnan_b200 import ops
    from gnan_b200.preprocess import apsp_batched
    bt = _mixed(55, 1024 if dtype == torch.int16 else 256)
    pk = apsp_batched(bt.edges(dtype), bt.node_off, device=DEV, nbins=64, rscale=True)
    cnt = apsp_batched(bt.ei, bt.node_off, device=DEV, nbins=64)
    dense = apsp_batched(bt.ei, bt.node_off, device=DEV, nbins=64, rscale=True)      # the int64 input with rscale
    assert pk.deferred and not dense.deferred
    want = ops.level_rscale(cnt.level_counts)
    assert torch.equal(pk.hop, cnt.hop) and torch.equal(pk.level_rscale, want)
    assert torch.equal(dense.hop, cnt.hop) and torch.equal(dense.level_rscale, want)
    assert pk.status.tolist() == cnt.status.tolist() == dense.status.tolist()


def test_model_outside_the_fused_envelope_on_a_deferred_large_batch():
    """C = 5: the model materialises the batch and takes the general kernels; the same as on the count-path batch"""
    from gnan_b200.preprocess import apsp_batched
    bt = _mixed(66, 1024)
    rng = np.random.default_rng(66)
    x = torch.tensor(rng.normal(size=(bt.N, 4))).float().to(DEV)
    pk = apsp_batched(bt.edges(torch.int16), bt.node_off, device=DEV, x=x, nbins=64, rscale=True)
    ref = apsp_batched(bt.ei, bt.node_off, device=DEV, x=x, nbins=64)
    m = _model(4, 5, False)
    with torch.no_grad():
        got, want = m(pk), m(ref)
    assert not pk.deferred
    assert torch.equal(got, want)


# ---- 7. whole paths ---------------------------------------------------------------------------------------------------------
def test_captured_step_on_a_mutagenicity_shaped_batch_replays_the_eager_steps():
    from gnan_b200 import ops, trainer
    from gnan_b200.preprocess import LocalEdges, apsp_batched
    rng = np.random.default_rng(17)
    sizes = mutagenicity_sizes(rng, n_graphs=1024, n_tail=6)
    graphs = molecule_like_graphs(rng, sizes)
    node_off = np.concatenate([[0], np.cumsum(sizes)])
    ei = torch.cat([g.edge_index + int(node_off[i]) for i, g in enumerate(graphs)], dim=1)
    le = LocalEdges.from_edge_index(ei, node_off, dtype=torch.int16).to(DEV)
    no_d = torch.tensor(node_off, dtype=torch.int32, device=DEV)
    ho_d = torch.tensor(np.concatenate([[0], np.cumsum(sizes.astype(np.int64) ** 2)]), dtype=torch.int64, device=DEV)
    x = torch.cat([g.x for g in graphs]).to(DEV)
    y = torch.cat([g.y for g in graphs]).to(DEV)
    losses = {}
    for mode in ("eager", "graph"):
        m = _model(x.shape[1], 1, False)
        opt = torch.optim.Adam(m.parameters(), lr=1e-3, capturable=True)

        def closure():
            pk = apsp_batched(le, node_off, device=DEV, x=x, y=y, node_off_device=no_d, hop_off_device=ho_d, nbins=48, rscale=True)
            assert pk.deferred
            return ops.bce_with_logits(m(pk).flatten(), pk.y)
        if mode == "eager":
            out = []
            for _ in range(3 + 5):
                opt.zero_grad(set_to_none=True)
                l = closure(); l.backward(); opt.step()
                out.append(float(l.detach()))
            losses[mode] = out[3:]
        else:
            step = trainer.CapturedStep(closure, opt, warmup=2)
            losses[mode] = [float(step()) for _ in range(6)][1:]
    assert losses["eager"] == losses["graph"], losses


def test_explain_on_a_deferred_large_batch():
    from tests.test_gpu_explain import assert_close, assert_sums, build, explain_checked, features_of, packed_reference
    from gnan_b200.preprocess import apsp_batched
    bt = _mixed(77, 620, directed=False)
    x = features_of(np.random.default_rng(77), bt.N, 5).to(DEV)
    fused = apsp_batched(bt.edges(torch.int16), bt.node_off, device=DEV, x=x, nbins=64, rscale=True)
    m = build("models", 5, 1, 3, 64, False, True, graph=True)
    e = explain_checked(m, fused)
    assert fused.deferred
    F, A, nodes, An = packed_reference(m, bt.eis, bt.node_off, x.cpu(), "output", True)
    assert_close(e.features, F, A, "fused")
    assert_close(e.nodes, nodes, An, "fused nodes")
    assert_sums(e, fused.batch_vector)


def test_dense_1024_node_graph():
    """about 200 k edges in one graph: the in-neighbour bit matrix does not depend on the edge count"""
    rng = np.random.default_rng(3)
    n = 1024
    e = random_graph(rng, n, 230.0, True)
    bt = _Batch([(n, e), (50, _graph(rng, 50, False, 1)), (300, _graph(rng, 300, True, 2))])
    assert bt.ei.shape[1] > 180_000
    T, S = _tensors(rng, bt, 16, 2, 1)
    out, colw, Q, st = _fused(bt, torch.int16, T, S)
    ref = R.readout_f64(bt.hops, 16, T.cpu().numpy(), S.cpu().numpy())
    R.assert_entrywise("out", out.cpu().numpy(), ref.out, ref.a_out, RTOL)
    R.assert_entrywise("colw", colw.cpu().numpy(), ref.colw, ref.a_colw, RTOL, bt.node_off)
    R.assert_entrywise("Q", Q.cpu().numpy(), ref.Q, ref.a_Q, RTOL)
    assert st.tolist() == R.expected_status(bt.hops, 16)
