"""GPU: the two kernels of the output-normalised graph readout against the float64 reference of tests/_readout_f64.py on the
C oracle's hop matrices, graph by graph and entry by entry.

- gnan_bfs_graph_readout_fwd (csrc/apsp.cu, ops.bfs_graph_readout_fwd): the batched BFS of a LocalEdges batch fused with the
  readout; out / colw / Q, its status word, and dS / dT of agg_bd_graph_bwd through ops.bfs_graph_readout.
- agg_bd_graph_fwd_kernel (csrc/agg_bd.cu, ops.agg_bd_graph_fwd) on hop bytes and a normaliser table packed here from the
  oracle; dS / dT through ops.aggregate_blockdiag.

T, S and g are random float32 inputs; no model is involved, so any (C, Cr) runs. Tolerance, per entry:
|got - ref| <= 1e-5 * A + 1e-30, A = the sum of the absolute values of the entry's terms. Every kernel sum is a float32 sum of
terms whose exact values make up A (P[j,d] sums positive 1/count over the rows of a column in row order, colw and Q sum P
times T or S, out sums S times colw, the dT slabs sum g times Q); its rounding error is at most (length of the sequential
chain) * 2^-24 * A and grows like its square root for independent roundings. The longest chain is P over the 300 rows of the
largest graph here. Measured on a B200: worst |err| / A = 2.9e-6 for the one-pass kernel (300-node graphs), 1.5e-6 for the
fused kernel, 4e-7 on the molecule step's batch; a single wrong term in any entry of any graph of a batch of 32 768 exceeds
the bound. Empty bins (A = 0) must be exactly zero."""
import functools

import numpy as np
import pytest
import torch

from tests import _readout_f64 as R
from tests.test_gpu_parity import random_graph

pytestmark = pytest.mark.gpu
DEV = "cuda"
RTOL = 1e-5
CCR = [(1, 1), (2, 1), (2, 2), (3, 1), (3, 3), (4, 1), (4, 4)]          # instantiations CC = 1, 2, 4
NBINS = [2, 3, 5, 31, 32, 33, 47, 48, 63, 64]
SIZES = [1, 2, 31, 32, 33, 63, 64, 65, 95, 96, 97, 127, 128]               # every edge of the kernel's size classes


# ---- graphs (local ids, [2,E] int64, no self loops, no duplicate edges) -------------------------------------------------
def _clean(e):
    e = np.asarray(e, dtype=np.int64).reshape(2, -1)
    e = e[:, e[0] != e[1]]
    return np.unique(e, axis=1) if e.shape[1] else np.zeros((2, 0), np.int64)


def _sym(e):
    return np.concatenate([e, e[::-1]], axis=1)


def _edgeless(n):
    return np.zeros((2, 0), np.int64)


def _complete(n, directed):                                 # directed: i -> j for i < j (depth 1, the reverse unreachable)
    i, j = np.triu_indices(n, 1)
    e = np.stack([i, j])
    return e if directed else _sym(e)


def _star(n, directed, inward=False):                       # centre 0; directed: out-star (or in-star), depth 1
    e = np.stack([np.zeros(n - 1, np.int64), np.arange(1, n)])
    return (e[::-1] if inward else e) if directed else _sym(e)


def _path(n, directed):
    e = np.stack([np.arange(n - 1), np.arange(1, n)])
    return e if directed else _sym(e)


def _hub(rng, n, directed):                                 # vertex 0 with more than 8 out- (and in-) neighbours
    e = random_graph(rng, n, 3.0, directed)
    out_nb = rng.choice(np.arange(1, n), size=min(n - 1, 9 + n // 6), replace=False)
    in_nb = rng.choice(np.arange(1, n), size=min(n - 1, 9 + n // 8), replace=False)
    h = np.concatenate([np.stack([np.zeros_like(out_nb), out_nb]), np.stack([in_nb, np.zeros_like(in_nb)])], axis=1)
    return np.concatenate([e, h if directed else _sym(h)], axis=1)


def _random(rng, n, directed, isolated=0):                  # average degree 4: shallow enough for nbins >= 31
    return random_graph(rng, n, 4.0, directed, n_isolated=isolated)


def _remainders(rng, graphs, seed, max_n=128, make=None):
    """graphs of <= 32 nodes: a count = 1, 2 or 3 (mod 4); of 33..64 nodes: an odd count (partly filled work items)"""
    make = make or (lambda n, k: _random(rng, n, bool(k % 2)))
    small = lambda: sum(1 for n, _ in graphs if n <= 32)
    want = 1 + seed % 3
    while small() % 4 != want:
        n = int(rng.integers(1, min(32, max_n) + 1))
        graphs.append((n, make(n, len(graphs))))
    if max_n > 32 and sum(1 for n, _ in graphs if 32 < n <= 64) % 2 == 0:
        n = int(rng.integers(33, min(64, max_n) + 1))
        graphs.append((n, make(n, len(graphs))))
    return graphs


class _Batch:
    """a batch in both kernel inputs: LocalEdges (graphs of at most 128 nodes) and hop bytes packed from the oracle"""
    def __init__(self, graphs, rng=None, hops=None):
        from gnan_b200.preprocess import LocalEdges
        if rng is not None:                                       # size classes interleaved in memory
            graphs = [graphs[k] for k in rng.permutation(len(graphs))]
        self.sizes = np.array([n for n, _ in graphs], dtype=np.int64)
        self.eis = eis = [_clean(e) for _, e in graphs]
        self.hops = R.oracle_hops(eis, self.sizes) if hops is None else hops
        self.node_off = np.concatenate([[0], np.cumsum(self.sizes)])
        self.N, self.B = int(self.node_off[-1]), len(graphs)
        self.max_n = int(self.sizes.max()) if self.B else 1
        self.depth = max((int(h.max()) for h in self.hops), default=0)
        ei = np.concatenate([e + self.node_off[b] for b, e in enumerate(eis)], axis=1) if eis else np.zeros((2, 0), np.int64)
        self.edges = LocalEdges.from_edge_index(torch.from_numpy(ei), self.node_off).to(DEV) if self.max_n <= 128 else None
        self.node_off_d = torch.tensor(self.node_off, dtype=torch.int32, device=DEV)
        hop, hop_off, _ = R.pack_hops(self.hops)
        self.hop, self.hop_off = torch.from_numpy(hop).to(DEV), torch.from_numpy(hop_off).to(DEV)


def _shapes(rng, directed, max_n=128):
    """hubs, K_n, stars, isolated vertices, no edges at all"""
    m = max_n
    return [(min(40, m), _hub(rng, min(40, m), directed)), (m, _hub(rng, m, directed)), (m, _complete(m, directed)),
            (min(50, m), _star(min(50, m), directed)), (m, _star(m, directed, inward=True)),
            (min(70, m), _random(rng, min(70, m), directed, isolated=min(70, m) // 4)), (min(20, m), _edgeless(min(20, m))),
            (m, _edgeless(m))]


@functools.lru_cache(maxsize=None)
def _general(max_n=128, large=False, deep=False):
    """every class edge, random sizes, the special shapes in both forms (depth < 30: fits nbins >= 31); large: graphs of 150
    and 300 nodes; deep: paths of depth 99 and 199"""
    rng = np.random.default_rng(1000 + max_n + large + 2 * deep)
    sizes = [n for n in SIZES if n <= max_n] + [int(v) for v in rng.integers(1, max_n + 1, size=30)] + [max_n]
    graphs = [(n, _random(rng, n, bool(k % 2), isolated=(k % 3) if n > 8 else 0)) for k, n in enumerate(sizes)]
    graphs += _shapes(rng, False, max_n) + _shapes(rng, True, max_n)
    graphs = _remainders(rng, graphs, max_n, max_n)
    if large:                                                     # the one-pass kernel takes any n
        graphs += [(150, _random(rng, 150, False, isolated=3)), (300, _random(rng, 300, True)), (300, _hub(rng, 300, False))]
    if deep:
        graphs += [(100, _path(100, False)), (200, _path(200, True))]
    bt = _Batch(graphs, rng)
    assert (bt.depth > 64) if deep else (bt.depth <= 29), bt.depth
    return bt


@functools.lru_cache(maxsize=None)
def _shallow(nbins, large=False):
    """graphs of depth <= nbins - 2 for nbins <= 5: edgeless graphs; K_n and one-way stars (depth 1); stars (depth 2)"""
    rng = np.random.default_rng(2000 + nbins + large)

    def make(n, k):
        kinds = ["none"] + (["kdir", "ksym", "out", "in"] if nbins >= 3 else []) + (["star"] if nbins >= 4 else [])
        kind = kinds[k % len(kinds)]
        return {"none": _edgeless(n), "kdir": _complete(n, True), "ksym": _complete(n, False), "out": _star(n, True),
                "in": _star(n, True, inward=True), "star": _star(n, False)}[kind] if n > 1 else _edgeless(n)

    sizes = SIZES + [int(v) for v in rng.integers(1, 129, size=20)]
    graphs = _remainders(rng, [(n, make(n, k)) for k, n in enumerate(sizes)], nbins, 128, make)
    if large:
        graphs += [(150, make(150, 1)), (300, make(300, 0)), (300, make(300, 3 if nbins >= 3 else 0))]
    bt = _Batch(graphs, rng)
    assert bt.depth <= nbins - 2, (nbins, bt.depth)
    return bt


def _inputs(bt, nbins, C, Cr, seed):
    rng = np.random.default_rng(seed)
    f = lambda *s: torch.tensor(rng.normal(size=s), dtype=torch.float32, device=DEV)
    return f(nbins, Cr), f(bt.N, C), f(bt.B, C)


def _np(t):
    return t.detach().double().cpu().numpy()


def _check(ref, node_off, out, colw, Q, dS=None, dT=None):
    R.assert_entrywise("out", _np(out), ref.out, ref.a_out, RTOL)
    R.assert_entrywise("colw", _np(colw), ref.colw, ref.a_colw, RTOL, node_off)
    R.assert_entrywise("Q", _np(Q), ref.Q, ref.a_Q, RTOL)
    if dS is not None:
        R.assert_entrywise("dS", _np(dS), ref.dS, ref.a_dS, RTOL, node_off)
        R.assert_entrywise("dT", _np(dT), ref.dT, ref.a_dT, RTOL)


def _fused(bt, T, S, g):
    """fused forward twice (bit-identical), then autograd; returns (out, colw, Q), (dS, dT), status"""
    from gnan_b200 import ops
    runs = []
    for _ in range(2):
        status = torch.zeros(3, dtype=torch.int32, device=DEV)        # the kernel clears the CSR bits only
        runs.append(ops.bfs_graph_readout_fwd(bt.edges, bt.node_off_d, bt.max_n, T, S, status) + (status,))
    for a, b in zip(runs[0], runs[1]):
        assert torch.equal(a, b), "two calls of the fused kernel differ"
    Tg, Sg = T.clone().requires_grad_(True), S.clone().requires_grad_(True)
    out = ops.bfs_graph_readout(bt.edges, bt.node_off_d, bt.max_n, Tg, Sg, torch.zeros(3, dtype=torch.int32, device=DEV))
    assert torch.equal(out, runs[0][0])
    dT, dS = torch.autograd.grad(out, (Tg, Sg), grad_outputs=g)
    return runs[0][:3], (dS, dT), runs[0][3].tolist()


def _onepass(bt, T, S, g, rs):
    from gnan_b200 import ops
    fwd = ops.agg_bd_graph_fwd(bt.hop, bt.hop_off, bt.node_off_d, T, rs, S)
    assert all(torch.equal(a, b) for a, b in zip(fwd, ops.agg_bd_graph_fwd(bt.hop, bt.hop_off, bt.node_off_d, T, rs, S)))
    Tg, Sg = T.clone().requires_grad_(True), S.clone().requires_grad_(True)
    out = ops.aggregate_blockdiag(bt.hop, bt.hop_off, bt.node_off_d, Tg, Sg, rscale=rs, reduce_graph=True)
    assert torch.equal(out, fwd[0])
    dT, dS = torch.autograd.grad(out, (Tg, Sg), grad_outputs=g)
    return fwd, (dS, dT)


def _rscale(bt, nbins):
    return torch.from_numpy(R.rscale_f32(bt.hops, nbins)).to(DEV)


# ---- the fused BFS + readout kernel ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("nbins", NBINS)
@pytest.mark.parametrize("C,Cr", CCR)
def test_fused_readout_vs_float64(C, Cr, nbins):
    bt = _general() if nbins > 5 else _shallow(nbins)
    T, S, g = _inputs(bt, nbins, C, Cr, 10 * nbins + 3 * C + Cr)
    fwd, bwd, status = _fused(bt, T, S, g)
    assert status == R.expected_status(bt.hops, nbins)
    _check(R.readout_f64(bt.hops, nbins, _np(T), _np(S), _np(g)), bt.node_off, *fwd, *bwd)


@pytest.mark.parametrize("max_n", [27, 31, 32, 33, 64, 95])
@pytest.mark.parametrize("C,Cr,nbins", [(1, 1, 48), (2, 1, 33), (4, 4, 64)])
def test_fused_readout_by_largest_graph(C, Cr, nbins, max_n):
    """the shared-memory slices are sized from the largest graph of the batch"""
    bt = _general(max_n)
    assert bt.max_n == max_n
    T, S, g = _inputs(bt, nbins, C, Cr, max_n + C)
    fwd, bwd, status = _fused(bt, T, S, g)
    assert status == R.expected_status(bt.hops, nbins)
    _check(R.readout_f64(bt.hops, nbins, _np(T), _np(S), _np(g)), bt.node_off, *fwd, *bwd)


@pytest.mark.parametrize("over", [False, True])
@pytest.mark.parametrize("nbins", NBINS)
def test_fused_readout_at_the_depth_limit(nbins, over):
    """paths of eccentricity nbins - 2 (the deepest bin) and nbins - 1 (overflow: status only), symmetric and directed"""
    base = _shallow(nbins) if nbins <= 5 else _general()
    L = nbins - 1 if over else nbins - 2
    rng = np.random.default_rng(nbins)
    graphs = list(zip(base.sizes.tolist(), base.eis)) + [(L + 1, _path(L + 1, False)), (L + 1, _path(L + 1, True))]
    bt = _Batch(graphs, rng)
    T, S, g = _inputs(bt, nbins, 2, 1, nbins + over)
    fwd, bwd, status = _fused(bt, T, S, g)
    assert status == [0, int(over), max(L, base.depth)]
    if not over:
        _check(R.readout_f64(bt.hops, nbins, _np(T), _np(S), _np(g)), bt.node_off, *fwd, *bwd)


# ---- the one-pass kernel on packed hop bytes --------------------------------------------------------------------------------
@pytest.mark.parametrize("normalize", [True, False])
@pytest.mark.parametrize("nbins", NBINS)
@pytest.mark.parametrize("C,Cr", CCR)
def test_onepass_readout_vs_float64(C, Cr, nbins, normalize):
    """graphs of up to 300 nodes; without the normaliser, deeper hops than nbins - 2 share the last bin (the clamp)"""
    if normalize:
        bt = _general(large=True) if nbins > 5 else _shallow(nbins, large=True)
    else:
        bt = _general(large=True, deep=True)
    T, S, g = _inputs(bt, nbins, C, Cr, 7 * nbins + 3 * C + Cr + normalize)
    rs = _rscale(bt, nbins) if normalize else None
    fwd, bwd = _onepass(bt, T, S, g, rs)
    _check(R.readout_f64(bt.hops, nbins, _np(T), _np(S), _np(g), normalize=normalize), bt.node_off, *fwd, *bwd)


@functools.lru_cache(maxsize=None)
def _small_graphs(B):
    rng = np.random.default_rng(B)
    sizes = rng.integers(1, 25, size=B)
    return _Batch([(int(n), _random(rng, int(n), bool(k % 2), isolated=k % 2)) for k, n in enumerate(sizes)], rng)


@pytest.mark.parametrize("B", [1, 7, 8, 9, 8197])
@pytest.mark.parametrize("C,Cr", [(3, 1), (2, 2)])
def test_onepass_backward_by_batch_size(C, Cr, B):
    """the dT reduction: one slab (B <= 15), 1 024 slabs with an uneven last slab and empty slabs (B = 8 197)"""
    nbins = 33
    bt = _small_graphs(B)
    T, S, g = _inputs(bt, nbins, C, Cr, B + C)
    fwd, bwd = _onepass(bt, T, S, g, _rscale(bt, nbins))
    _check(R.readout_f64(bt.hops, nbins, _np(T), _np(S), _np(g)), bt.node_off, *fwd, *bwd)


@pytest.mark.parametrize("C,Cr", [(1, 1), (3, 1), (2, 2)])
def test_empty_batch(C, Cr):
    from gnan_b200 import ops
    from gnan_b200.preprocess import LocalEdges
    nbins = 48
    T = torch.randn(nbins, Cr, device=DEV).requires_grad_(True)
    S = torch.randn(0, C, device=DEV).requires_grad_(True)
    node_off = torch.zeros(1, dtype=torch.int32, device=DEV)
    empty8 = torch.zeros(0, dtype=torch.uint8, device=DEV)
    edges = LocalEdges(empty8, empty8, node_off.clone())
    status = torch.zeros(3, dtype=torch.int32, device=DEV)
    for out in (ops.bfs_graph_readout(edges, node_off, 1, T, S, status),
                ops.aggregate_blockdiag(torch.zeros(1, dtype=torch.uint8, device=DEV), torch.zeros(1, dtype=torch.int64, device=DEV),
                                        node_off, T, S, rscale=None)):
        assert tuple(out.shape) == (0, C)
        T.grad = None
        out.backward(torch.zeros(0, C, device=DEV))
        assert T.grad is not None and torch.equal(T.grad, torch.zeros(nbins, Cr, device=DEV))
    assert status.tolist() == [0, 0, 0]


# ---- the molecule step's own batch -------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def headline():
    """bench.py --workload mol's batch with the oracle's distances (computed once for the module)"""
    import bench
    wl = bench.make_mol_workload(seed=0)
    eis = R.split_edges(wl.edge_index.numpy(), wl.node_off.numpy())
    return _Batch(list(zip(wl.sizes.tolist(), eis)), hops=R.oracle_hops(eis, wl.sizes))


def test_headline_batch_vs_float64(headline):
    """the molecule step: 32 768 graphs of 10-100 nodes, nbins 48, C = 1; both kernels, forward and backward (1 024 dT slabs)"""
    bt, nbins = headline, 48
    T, S, g = _inputs(bt, nbins, 1, 1, 48)
    ref = R.readout_f64(bt.hops, nbins, _np(T), _np(S), _np(g))
    fwd, bwd, status = _fused(bt, T, S, g)
    assert status == R.expected_status(bt.hops, nbins)
    _check(ref, bt.node_off, *fwd, *bwd)
    fwd, bwd = _onepass(bt, T, S, g, _rscale(bt, nbins))
    _check(ref, bt.node_off, *fwd, *bwd)
