"""GPU: the batched BFS on graphs of 129..1024 nodes (apsp_batched_large_kernel, next to the 4-warp-group kernel for the graphs of at
most 128 nodes of the same batch), the per-graph path above that size, and what the packed datasets and models do with such
graphs. Hop blocks and level counts are compared bit-exactly with the C oracle or per-graph `apsp`; model outputs and gradients
norm-wise within 1e-5 of the per-graph forward."""
import re
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import apsp as oapsp
from tests import _golden as G

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5
MIXED_SIZES = [1, 5, 31, 64, 100, 128, 129, 200, 256, 257, 300, 417, 512, 620, 1000, 1024]


def random_graph(rng, n, avg_deg=2.2, directed=False, n_isolated=0):
    """int64 [2,E] local edge list: random edges among the first n - n_isolated nodes (the rest isolated), no self loops, no repeats"""
    m = n - n_isolated
    E = int(m * avg_deg / (1 if directed else 2))
    src = rng.integers(0, max(m, 1), size=E); dst = rng.integers(0, max(m, 1), size=E)
    keep = src != dst
    e = np.unique(np.stack([src[keep], dst[keep]], 1), axis=0)
    if not directed:
        e = np.unique(np.concatenate([e, e[:, ::-1]]), axis=0)
    return e.T.astype(np.int64).reshape(2, -1)


def varied_graph(rng, n, directed):
    """Two components, three isolated vertices and hubs of 40 and 12 neighbours (graphs of more than 45 nodes)"""
    if n <= 45:
        return random_graph(rng, n, 2.2, directed, n_isolated=1 if n > 4 else 0)
    m = n - 3
    h = m // 2
    e = np.concatenate([random_graph(rng, h, 2.2, directed), random_graph(rng, m - h, 2.2, directed) + h], axis=1)
    hubs = [np.stack([np.zeros(40, np.int64), rng.choice(np.arange(1, h), 40, replace=False) if h > 41 else rng.integers(1, m, 40)]),
            np.stack([np.full(12, m - 1, np.int64), h + rng.integers(0, m - h - 1, 12)])]
    e = np.concatenate([e] + hubs + ([] if directed else [hb[::-1] for hb in hubs]), axis=1)
    e = e[:, e[0] != e[1]]
    return np.unique(e.T, axis=0).T.copy()


def molecule_like_graphs(rng, sizes, k=15):
    """Graphs shaped like bench.py's Mutagenicity workload: a random tree + ceil(n/10) extra edges, both directions, one-hot x"""
    out = []
    for n in sizes:
        n = int(n)
        par = np.array([rng.integers(0, v) for v in range(1, n)], dtype=np.int64)
        e = set(zip(par.tolist(), range(1, n)))
        extra = int(np.ceil(n / 10))
        while extra > 0 and n > 2:
            a, b = int(rng.integers(0, n)), int(rng.integers(0, n))
            if a != b and (min(a, b), max(a, b)) not in e:
                e.add((min(a, b), max(a, b))); extra -= 1
        e = np.array(sorted(e), dtype=np.int64).reshape(-1, 2)
        ei = np.concatenate([e, e[:, ::-1]]).T.copy()
        x = np.zeros((n, k - 1), np.float32)
        x[np.arange(n), rng.integers(0, k - 1, size=n)] = 1.0
        out.append(SimpleNamespace(x=torch.tensor(x), edge_index=torch.tensor(ei), y=torch.tensor([float(rng.integers(0, 2))])))
    return out


def mutagenicity_sizes(rng, n_graphs=4337, n_tail=20):
    """bench.py's size draw (clip(round(N(30.3, 20)), 4, 120)) with the last n_tail graphs redrawn in 257..417"""
    sizes = np.clip(np.round(rng.normal(30.3, 20.0, size=n_graphs)), 4, 120).astype(np.int64)
    if n_tail:
        sizes[-n_tail:] = rng.integers(257, 418, size=n_tail)
        sizes[-1] = 417
    return sizes


def concat(eis):
    sizes = [int(e[1]) for e in eis]
    node_off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    ei = np.concatenate([e[0] + node_off[i] for i, e in enumerate(eis)], axis=1) if eis else np.zeros((2, 0), np.int64)
    return torch.tensor(ei), node_off


def widened(want_cnt, width):
    full = np.zeros((want_cnt.shape[0], width), dtype=np.int32)
    full[:, :want_cnt.shape[1] - 1] = want_cnt[:, :-1]
    full[:, -1] = want_cnt[:, -1]
    return full


def assert_batch_equals_oracle(pk, graphs, node_off):
    hop, cnt, ho = pk.hop.cpu().numpy(), pk.level_counts.cpu().numpy(), pk.hop_off.cpu().numpy()
    dmax = 0
    for i, (e, n) in enumerate(graphs):
        want = oapsp.apsp(e, n)
        got = hop[ho[i]:ho[i + 1]].reshape(n, n).astype(np.int32)
        got[got == 255] = -1
        assert np.array_equal(got, want), (i, n)
        wc = oapsp.level_counts(want)
        assert np.array_equal(cnt[node_off[i]:node_off[i + 1]], widened(wc, cnt.shape[1])), (i, n)
        dmax = max(dmax, int(want.max()))
    return dmax


def mixed_batch(directed, seed=5):
    rng = np.random.default_rng(seed + int(directed))
    sizes = MIXED_SIZES + [int(v) for v in rng.integers(1, 129, size=200)]
    sizes = [sizes[i] for i in rng.permutation(len(sizes))]
    return [(varied_graph(rng, n, directed), n) for n in sizes]


@pytest.mark.parametrize("directed,cap", [(False, 1024), (True, 1024), (False, 256), (True, 256)],
                         ids=["False", "True", "False-256", "True-256"])
def test_mixed_batch_exact_free_and_fixed_width(directed, cap):
    """cap: the batch keeps the graphs of mixed_batch with at most cap nodes (256: the largest graph has 129..256 nodes)"""
    from gnan_b200.preprocess import apsp_batched, check_batched_status
    graphs = [(e, n) for e, n in mixed_batch(directed) if n <= cap]
    ei, node_off = concat(graphs)
    pk = apsp_batched(ei, node_off, device=DEV)
    dmax = assert_batch_equals_oracle(pk, graphs, node_off)
    assert pk.level_counts.shape[1] == dmax + 2
    pk = apsp_batched(ei, node_off, device=DEV, nbins=256)
    assert pk.level_counts.shape[1] == 256
    assert_batch_equals_oracle(pk, graphs, node_off)
    check_batched_status(pk.status)
    assert int(pk.status[2]) == dmax


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.key for e in prof.key_averages()}


def _has(names, kernel):
    return any(re.search(r"\b" + kernel + r"\b", k) for k in names)


def test_routing_of_large_and_small_graphs():
    """Each graph runs by its own size: at most 128 nodes on the v3 kernel, more on the large kernel, whatever the rest of the batch"""
    from gnan_b200.preprocess import apsp_batched
    graphs = mixed_batch(False)
    batches = {"up to 1024": (graphs, True, True), "up to 256": ([g for g in graphs if g[1] <= 256], True, True),
               "129..256 only": ([g for g in graphs if 128 < g[1] <= 256], False, True),
               "up to 128": ([g for g in graphs if g[1] <= 128], True, False)}
    for name, (gs, v3, large) in batches.items():
        ei, node_off = concat(gs)
        apsp_batched(ei, node_off, device=DEV)                              # warm-up (module load, attribute setting)
        names = _kernel_names(lambda: apsp_batched(ei, node_off, device=DEV))
        assert _has(names, "bv3_classify_kernel"), (name, names)
        assert not v3 or _has(names, "apsp_batched_v3_kernel"), (name, names)
        assert _has(names, "apsp_batched_large_kernel") == large, (name, names)
        assert not _has(names, "apsp_batched_kernel"), (name, names)


def test_deep_large_graph_redo_and_hop_overflow():
    from gnan_b200.preprocess import apsp_batched
    rng = np.random.default_rng(3)
    path = np.stack([np.arange(120), np.arange(1, 121)])                     # 121-node path + 179 leaves hung on it
    leaves = np.stack([rng.integers(0, 121, size=179), np.arange(121, 300)])
    e = np.concatenate([path, leaves], axis=1)
    e = np.concatenate([e, e[::-1]], axis=1)
    graphs = [(random_graph(rng, 40), 40), (e, 300), (random_graph(rng, 100), 100), (random_graph(rng, 260), 260)]
    ei, node_off = concat(graphs)
    pk = apsp_batched(ei, node_off, device=DEV)                              # deeper than the 48-column first try
    dmax = assert_batch_equals_oracle(pk, graphs, node_off)
    assert dmax >= 120 and pk.level_counts.shape[1] == dmax + 2
    p400 = np.stack([np.arange(399), np.arange(1, 400)])
    ei, node_off = concat([(random_graph(rng, 30), 30), (np.concatenate([p400, p400[::-1]], axis=1), 400)])
    with pytest.raises(NotImplementedError, match="uint8 hop matrix"):
        apsp_batched(ei, node_off, device=DEV)


def test_graph_above_the_cap_takes_the_per_graph_path():
    from gnan_b200 import _lib
    from gnan_b200.preprocess import apsp_batched
    rng = np.random.default_rng(9)
    graphs = [(random_graph(rng, 20), 20), (random_graph(rng, 1500, 2.5, n_isolated=2), 1500), (random_graph(rng, 300), 300)]
    ei, node_off = concat(graphs)
    pk = apsp_batched(ei, node_off, device=DEV)
    assert_batch_equals_oracle(pk, graphs, node_off)
    with pytest.raises(ValueError, match=str(_lib.APSP_BATCHED_MAX_NODES)):
        apsp_batched(ei, node_off, device=DEV, nbins=64)


def test_duplicate_edges_in_a_large_graph_match_per_graph_apsp():
    from gnan_b200.preprocess import apsp, apsp_batched
    rng = np.random.default_rng(11)
    e = random_graph(rng, 417, 2.4)
    dup = e[:, rng.choice(e.shape[1], 25, replace=False)]
    e_dup = np.concatenate([e, dup, dup[:, :5]], axis=1)                    # some pairs listed twice, some three times
    graphs = [(random_graph(rng, 50), 50), (e_dup, 417), (random_graph(rng, 300), 300)]
    ei, node_off = concat(graphs)
    pk = apsp_batched(ei, node_off, device=DEV)
    hop, cnt, ho = pk.hop.cpu().numpy(), pk.level_counts.cpu().numpy(), pk.hop_off.cpu().numpy()
    for i, (eg, n) in enumerate(graphs):
        hd = apsp(torch.tensor(eg), n, device=DEV)
        assert np.array_equal(hop[ho[i]:ho[i + 1]].reshape(n, n), hd.hop[:, :n].cpu().numpy()), i
        assert np.array_equal(cnt[node_off[i]:node_off[i + 1]], widened(hd.level_counts.cpu().numpy(), cnt.shape[1])), i


def test_packed_dataset_with_mutagenicity_and_larger_graphs(tmp_path):
    from gnan_b200.packed import PackedDataset
    from gnan_b200.preprocess import apsp
    rng = np.random.default_rng(4337)
    sizes = mutagenicity_sizes(rng)
    graphs = molecule_like_graphs(rng, sizes)
    ds = PackedDataset.from_graphs(graphs, device=DEV)
    assert len(ds) == 4337 and ds.max_nodes == 417
    hop, cnt = ds.hop.cpu().numpy(), ds.level_counts.cpu().numpy()
    no, ho = ds.node_off.cpu().numpy(), ds.hop_off.cpu().numpy()
    for i, g in enumerate(graphs):
        n = int(sizes[i])
        hd = apsp(g.edge_index, n, device=DEV)
        assert np.array_equal(hop[ho[i]:ho[i + 1]].reshape(n, n), hd.hop[:, :n].cpu().numpy()), i
        assert np.array_equal(cnt[no[i]:no[i + 1]], widened(hd.level_counts.cpu().numpy(), cnt.shape[1])), i
    path = tmp_path / "mutag_like.gnan_b200.pt"
    ds.save(str(path))
    back = PackedDataset.load(str(path), device=DEV)
    for a, b in ((ds.x, back.x), (ds.node_off, back.node_off), (ds.hop, back.hop), (ds.hop_off, back.hop_off),
                 (ds.level_counts, back.level_counts), (ds.y, back.y)):
        assert torch.equal(a, b)
    ids = [4336, 3, 4320, 17, 4336, 0]                                      # large and small graphs, one repeated
    bt = ds.batch(ids)
    bh, bo = bt.hop.cpu().numpy(), bt.hop_off.cpu().numpy()
    bno = bt.node_off.cpu().numpy()
    for k, i in enumerate(ids):
        assert np.array_equal(bh[bo[k]:bo[k + 1]], hop[ho[i]:ho[i + 1]]), (k, i)
        assert np.array_equal(bt.level_counts[bno[k]:bno[k + 1]].cpu().numpy(), cnt[no[i]:no[i + 1]]), (k, i)
        assert torch.equal(bt.x[bno[k]:bno[k + 1]], ds.x[no[i]:no[i + 1]])


@pytest.mark.parametrize("family", ["models", "GNAN"])
def test_model_on_large_graphs_equals_per_graph_forward(family):
    """Output-normalised models.TensorGNAN and input-normalised GNAN.TensorGNAN (graph task): forward_packed + backward on a batch
    with graphs of 300..1000 nodes against the per-graph forward on `apsp` hop data."""
    from gnan_b200.preprocess import apsp, apsp_batched
    if family == "models":
        from gnan_b200.models import TensorGNAN
    else:
        from gnan_b200.GNAN import TensorGNAN
    rng = np.random.default_rng(31)
    sizes = [300, 17, 1000, 45, 517, 128, 129]
    K, C = 6, 2
    graphs = [(random_graph(rng, n, 2.2, n_isolated=2 if n > 100 else 0), n) for n in sizes]
    ei, node_off = concat(graphs)
    x = torch.tensor(rng.normal(size=(int(node_off[-1]), K))).float()
    torch.manual_seed(2)
    m = TensorGNAN(K, C, 3, 64, is_graph_task=True, normalize_rho=True).to(DEV)
    m.fs.xavier_normal_(1.0); m.rho.xavier_normal_(1.0)
    pk = apsp_batched(ei, node_off, device=DEV)
    pk.x = x.to(DEV)
    w = torch.tensor(rng.normal(size=(len(sizes), C))).float().to(DEV)
    out = m(pk)
    assert tuple(out.shape) == (len(sizes), C)
    params = list(m.parameters())
    g_pk = torch.autograd.grad((out * w).sum(), params)
    ref = []
    for i, (e, n) in enumerate(graphs):
        d = SimpleNamespace(x=x[node_off[i]:node_off[i + 1]], hop_data=apsp(torch.tensor(e), n, device=DEV))
        ref.append(m.forward(d).T)
    ref = torch.cat(ref)
    g_ref = torch.autograd.grad((ref * w).sum(), params)
    assert G.rel_err(out.detach().cpu().numpy(), ref.detach().cpu().numpy()) < TOL
    for a, b in zip(g_pk, g_ref):
        assert G.rel_err(a.cpu().numpy(), b.cpu().numpy()) < TOL
