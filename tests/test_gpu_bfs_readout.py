"""GPU: the batched BFS fused with the output-normalised graph readout (gnan_bfs_graph_readout_fwd, ops.bfs_graph_readout) and the
deferred batches of preprocess.apsp_batched that feed it.

Checker: the same model on the same batch after its distances were materialised (first read of `hop`), i.e. the hop bytes +
normaliser table + one-pass readout kernel path. The two forwards sum in different orders: 2e-6 norm-wise."""
import numpy as np
import pytest
import torch

from tests import _golden as G
from tests.test_gpu_parity import random_graph

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 2e-6
SIZES = [1, 2, 32, 33, 64, 65, 96, 97, 128]


def _edges(rng, sizes, directed):
    node_off = np.concatenate([[0], np.cumsum(sizes)])
    eis = [random_graph(rng, n, 2.2, directed, n_isolated=(1 + i % 3) if (n > 8 and i % 2) else 0) for i, n in enumerate(sizes)]
    return torch.tensor(np.concatenate([e + node_off[i] for i, e in enumerate(eis)], axis=1)), node_off


def _model(K, C, rho_per_feature):
    from gnan_b200.models import TensorGNAN
    torch.manual_seed(0)
    m = TensorGNAN(K, C, 3, 64, normalize_rho=True, is_graph_task=True, readout_n_layers=0, rho_per_feature=rho_per_feature,
                   device=DEV).to(DEV)
    m.fs.xavier_normal_(1.0); m.rho.xavier_normal_(1.0)
    return m


def _fused_vs_materialised(directed, C, rho_per_feature, seed):
    from gnan_b200.preprocess import LocalEdges, apsp_batched, check_batched_status
    rng = np.random.default_rng(seed)
    sizes = SIZES + [int(v) for v in rng.integers(1, 129, size=120)]
    ei, node_off = _edges(rng, sizes, directed)
    x = torch.tensor(rng.normal(size=(node_off[-1], 5))).float().to(DEV)
    le = LocalEdges.from_edge_index(ei, node_off)
    pk = apsp_batched(le, node_off, device=DEV, x=x, nbins=48, rscale=True)
    alias = apsp_batched(le, node_off, device=DEV, x=x, nbins=48, pair_stats=True)     # the same deferred batch
    assert pk.deferred and alias.deferred and pk.nbins == alias.nbins == 48
    m = _model(5, C, rho_per_feature)
    w = torch.tensor(rng.normal(size=(len(sizes), C))).float().to(DEV)

    def step(batch):
        m.zero_grad(set_to_none=True)
        out = m(batch)
        (out * w).sum().backward()
        return out.detach().clone(), [p.grad.clone() for p in m.parameters() if p.grad is not None]

    res = [step(pk)]                                 # fused (distances never materialised)
    via_alias = step(alias)
    for b in (pk, alias):
        assert b.deferred
        check_batched_status(b.status)
    assert torch.equal(via_alias[0], res[0][0]) and len(via_alias[1]) == len(res[0][1])
    for a, b in zip(via_alias[1], res[0][1]):
        assert G.rel_err(a.cpu().numpy(), b.cpu().numpy()) < TOL
    pk.hop                                           # materialise: the next forward reads the hop bytes + normaliser table
    assert not pk.deferred and pk.level_rscale is not None
    res.append(step(pk))                             # the hop-byte path on the same batch
    assert len(res[0][1]) == len(res[1][1]) > 0
    assert G.rel_err(res[0][0].cpu().numpy(), res[1][0].cpu().numpy()) < TOL
    for a, b in zip(res[0][1], res[1][1]):
        assert G.rel_err(a.cpu().numpy(), b.cpu().numpy()) < TOL


@pytest.mark.parametrize("C,rho_per_feature", [(1, False), (3, False), (3, True), (4, True)])
def test_fused_readout_matches_the_materialised_path(C, rho_per_feature):
    _fused_vs_materialised(False, C, rho_per_feature, 10 + C)


@pytest.mark.parametrize("C,rho_per_feature", [(1, False), (3, True)])
def test_fused_readout_on_directed_graphs(C, rho_per_feature):
    """non-symmetric edge lists take the per-graph asymmetric path inside the kernel: same results"""
    _fused_vs_materialised(True, C, rho_per_feature, 20 + C)


def _forward_status(le, node_off):
    from gnan_b200.preprocess import apsp_batched
    x = torch.ones(int(node_off[-1]), 3, device=DEV)
    pk = apsp_batched(le, node_off, device=DEV, x=x, nbins=48, rscale=True)
    with torch.no_grad():
        _model(3, 1, False)(pk)
    assert pk.deferred
    return pk.status


def test_fused_readout_reports_bad_batches():
    from gnan_b200.preprocess import LocalEdges, check_batched_status
    node_off = np.array([0, 5, 65])
    path = np.stack([np.arange(5, 64), np.arange(6, 65)])                    # graph 1: a path of 60 nodes (hop 59 > nbins - 2)
    ring = np.array([[0, 1, 2, 3, 4], [1, 2, 3, 4, 0]])
    ok = np.concatenate([ring, ring[::-1], path, path[::-1]], axis=1)
    st = _forward_status(LocalEdges.from_edge_index(torch.tensor(ok), node_off), node_off)
    assert int(st[0]) == 0 and int(st[1]) != 0 and int(st[2]) >= 47
    with pytest.raises(ValueError):
        check_batched_status(st)

    short = np.array([0, 5, 10])
    dup = np.concatenate([ring, ring[::-1], ring + 5, ring[::-1] + 5, ring[:, :1]], axis=1)    # edge (0,1) listed twice
    st = _forward_status(LocalEdges.from_edge_index(torch.tensor(dup), short), short)
    assert int(st[0]) == 2 and int(st[1]) == 0
    with pytest.raises(ValueError):
        check_batched_status(st)

    le = LocalEdges.from_edge_index(torch.tensor(np.concatenate([ring, ring[::-1], ring + 5, ring[::-1] + 5], axis=1)), short)
    le.dst[3] = 7                                                           # an endpoint outside its 5-node graph
    st = _forward_status(le, short)
    assert int(st[0]) & 1
    with pytest.raises(ValueError):
        check_batched_status(st)


def test_captured_step_on_a_deferred_batch_replays_the_eager_steps():
    """a training step that preprocesses its batch (apsp_batched on LocalEdges inside the step, as bench.py's molecule step)
    captured with trainer.CapturedStep follows the eager trajectory"""
    from gnan_b200 import ops, trainer
    from gnan_b200.preprocess import LocalEdges, apsp_batched
    rng = np.random.default_rng(3)
    sizes = SIZES + [int(v) for v in rng.integers(10, 101, size=200)]
    ei, node_off = _edges(rng, sizes, False)
    le = LocalEdges.from_edge_index(ei, node_off).to(DEV)
    no_d = torch.tensor(node_off, dtype=torch.int32, device=DEV)
    ho_d = torch.tensor(np.concatenate([[0], np.cumsum(np.asarray(sizes) ** 2)]), dtype=torch.int64, device=DEV)
    x = torch.tensor(rng.normal(size=(node_off[-1], 5))).float().to(DEV)
    y = torch.tensor(rng.integers(0, 2, size=len(sizes))).float().to(DEV)
    losses = {}
    for mode in ("eager", "graph"):
        m = _model(5, 1, False)
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
    assert np.allclose(losses["eager"], losses["graph"], rtol=1e-6, atol=0), losses
