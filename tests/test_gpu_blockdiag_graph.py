"""GPU: the one-pass graph-readout aggregation (csrc/agg_bd.cu) and the round-2 changes of the molecule path
(fused 1/count output of the batched BFS, block-per-segment sums, thread-per-row duplicate detection).

Checker: a float64 restatement of models.py:366-384 / batched_pyg_main.py:154-181 per graph (plain loops over the packed
blocks), and the general block-diagonal kernels of csrc/agg.cu. Tolerance 1e-5 norm-wise; integer outputs bit-exact."""
import numpy as np
import pytest
import torch

from tests import _golden as G
from tests.test_gpu_parity import random_graph

pytestmark = pytest.mark.gpu
TOL = 1e-5
DEV = "cuda"


def _batch(rng, sizes, iso=True):
    from gnan_b200.preprocess import apsp_batched
    node_off = np.concatenate([[0], np.cumsum(sizes)])
    eis = [random_graph(rng, n, 2.3, False, n_isolated=1 if (iso and n > 8) else 0) for n in sizes]
    ei = np.concatenate([e + node_off[i] for i, e in enumerate(eis)], axis=1)
    return apsp_batched(torch.tensor(ei), torch.tensor(node_off), device=DEV), node_off, ei


def _oracle_f64(pk, node_off, T, S, rs):
    """out[b,c] = sum_{i,j} T[d_ij,c'] rs[i,d_ij] S[j,c] in float64, graph by graph (differentiable)."""
    hop, ho = pk.hop.cpu().long(), pk.hop_off.cpu().numpy()
    nb, Cr = T.shape
    outs = []
    for b in range(len(node_off) - 1):
        n0, n1 = int(node_off[b]), int(node_off[b + 1])
        n = n1 - n0
        d = hop[ho[b]:ho[b + 1]].reshape(n, n).clamp(max=nb - 1)
        W = T[d]                                                      # [n,n,Cr]
        if rs is not None:
            W = W * torch.gather(rs[n0:n1], 1, d).unsqueeze(-1)
        outs.append((W * S[n0:n1].unsqueeze(0)).sum(dim=(0, 1)) if Cr > 1 else (W[..., 0] @ S[n0:n1]).sum(0))
    return torch.stack(outs)


@pytest.mark.parametrize("C,Cr", [(1, 1), (2, 2), (3, 1), (3, 3), (4, 4)])
@pytest.mark.parametrize("normalise", [True, False])
@pytest.mark.parametrize("pad_bins", [0, 48])
def test_graph_readout_kernels_vs_float64_and_general_kernels(C, Cr, normalise, pad_bins):
    from gnan_b200 import ops
    rng = np.random.default_rng(100 * C + 10 * Cr + normalise)
    sizes = [4, 33, 9, 64, 100, 1, 128, 31, 32, 57]
    pk, node_off, _ = _batch(rng, sizes)
    cnt = pk.level_counts
    if pad_bins:                                                      # fixed-width table (multiple of 4: the float4 staging path)
        wide = torch.zeros(cnt.shape[0], pad_bins, dtype=torch.int32, device=DEV)
        wide[:, :cnt.shape[1] - 1] = cnt[:, :-1]; wide[:, -1] = cnt[:, -1]
        cnt = wide
    nb = cnt.shape[1]
    T = torch.tensor(rng.normal(size=(nb, Cr))).float().to(DEV).requires_grad_(True)
    S = torch.tensor(rng.normal(size=(node_off[-1], C))).float().to(DEV).requires_grad_(True)
    rs = ops.level_rscale(cnt) if normalise else None
    w = torch.tensor(rng.normal(size=(len(sizes), C))).float().to(DEV)

    assert ops.load().gnan_aggregate_blockdiag_graph_supported(nb, Cr, C)
    out = ops.aggregate_blockdiag(pk.hop, pk.hop_off, pk.node_off, T, S, rscale=rs, reduce_graph=True)
    gT, gS = torch.autograd.grad((out * w).sum(), (T, S))

    T64 = T.detach().double().cpu().requires_grad_(True)
    S64 = S.detach().double().cpu().requires_grad_(True)
    want = _oracle_f64(pk, node_off, T64, S64, None if rs is None else rs.double().cpu())
    wT, wS = torch.autograd.grad((want * w.double().cpu()).sum(), (T64, S64))
    assert G.rel_err(out.detach().cpu().numpy(), want.detach().numpy()) < TOL
    assert G.rel_err(gT.cpu().numpy(), wT.numpy()) < TOL
    assert G.rel_err(gS.cpu().numpy(), wS.numpy()) < TOL

    ops.BLOCKDIAG_GRAPH_KERNEL = False                               # the general kernels on the same inputs
    try:
        ref = ops.aggregate_blockdiag(pk.hop, pk.hop_off, pk.node_off, T, S, rscale=rs, reduce_graph=True)
        rT, rS = torch.autograd.grad((ref * w).sum(), (T, S))
    finally:
        ops.BLOCKDIAG_GRAPH_KERNEL = True
    assert G.rel_err(out.detach().cpu().numpy(), ref.detach().cpu().numpy()) < TOL
    assert G.rel_err(gT.cpu().numpy(), rT.cpu().numpy()) < TOL and G.rel_err(gS.cpu().numpy(), rS.cpu().numpy()) < TOL


def test_graph_readout_is_deterministic_and_handles_empty_batches():
    from gnan_b200 import ops
    rng = np.random.default_rng(5)
    pk, node_off, _ = _batch(rng, list(rng.integers(1, 101, size=300)))
    nb = pk.nbins
    T = torch.tensor(rng.normal(size=(nb, 1))).float().to(DEV).requires_grad_(True)
    S = torch.tensor(rng.normal(size=(node_off[-1], 1))).float().to(DEV).requires_grad_(True)
    rs = ops.level_rscale(pk.level_counts)
    runs = []
    for _ in range(3):                                               # graphs are handed out dynamically: results must not depend on it
        out = ops.aggregate_blockdiag(pk.hop, pk.hop_off, pk.node_off, T, S, rscale=rs)
        gT, gS = torch.autograd.grad(out.square().sum(), (T, S))
        runs.append((out.detach().clone(), gT.clone(), gS.clone()))
    for r in runs[1:]:
        assert all(torch.equal(a, b) for a, b in zip(r, runs[0]))
    e = torch.zeros(1, dtype=torch.int32, device=DEV)
    out = ops.aggregate_blockdiag(torch.zeros(1, dtype=torch.uint8, device=DEV), torch.zeros(1, dtype=torch.int64, device=DEV), e,
                                  T, torch.zeros(0, 1, device=DEV), rscale=None)
    assert tuple(out.shape) == (0, 1)


def test_batched_bfs_fused_normaliser_equals_level_rscale():
    """apsp_batched(..., rscale=True) writes 1/level_counts itself: bit-identical to gnan_level_rscale of the counts."""
    from gnan_b200 import ops
    from gnan_b200.preprocess import apsp_batched, check_batched_status
    rng = np.random.default_rng(8)
    sizes = list(rng.integers(1, 101, size=200)) + [128, 127, 2]
    node_off = np.concatenate([[0], np.cumsum(sizes)])
    eis = [random_graph(rng, n, 2.2, False, n_isolated=1 if n > 8 else 0) for n in sizes]
    ei = torch.tensor(np.concatenate([e + node_off[i] for i, e in enumerate(eis)], axis=1))
    a = apsp_batched(ei, node_off, device=DEV, nbins=48)
    b = apsp_batched(ei, node_off, device=DEV, nbins=48, rscale=True)
    check_batched_status(a.status); check_batched_status(b.status)
    assert b.level_counts is None and b.nbins == 48
    assert torch.equal(a.hop, b.hop)
    assert torch.equal(ops.level_rscale(a.level_counts), b.level_rscale)


def test_molecule_step_with_fused_normaliser_matches_the_counts_path():
    """models.TensorGNAN on a packed batch: level_rscale from the BFS == level_counts converted by the module (outputs and all
    parameter gradients identical)."""
    from gnan_b200.models import TensorGNAN
    from gnan_b200.preprocess import apsp_batched
    rng = np.random.default_rng(12)
    sizes = list(rng.integers(10, 101, size=64))
    node_off = np.concatenate([[0], np.cumsum(sizes)])
    eis = [random_graph(rng, n, 2.2, False) for n in sizes]
    ei = torch.tensor(np.concatenate([e + node_off[i] for i, e in enumerate(eis)], axis=1))
    x = torch.tensor(rng.normal(size=(node_off[-1], 5))).float().to(DEV)
    torch.manual_seed(0)
    m = TensorGNAN(5, 1, 3, 64, normalize_rho=True, is_graph_task=True, readout_n_layers=0, device=DEV).to(DEV)
    m.fs.xavier_normal_(1.0); m.rho.xavier_normal_(1.0)
    res = []
    for fused in (False, True):
        pk = apsp_batched(ei, node_off, device=DEV, x=x, nbins=48, rscale=fused)
        m.zero_grad(set_to_none=True)
        out = m(pk)
        out.square().sum().backward()
        res.append((out.detach().clone(), [p.grad.clone() for p in m.parameters() if p.grad is not None]))
    assert torch.equal(res[0][0], res[1][0])
    for a, b in zip(res[0][1], res[1][1]):       # same inputs to every kernel; some weight-gradient reductions are not run-to-run bit-stable
        assert float((a - b).norm()) <= 1e-6 * float(b.norm()) + 1e-12


def test_gather_segment_sum_few_long_segments():
    """the block-per-segment variant (a handful of segments with ~1e5 rows each: one-hot columns) against float64"""
    from gnan_b200 import ops
    g = torch.Generator(device=DEV).manual_seed(3)
    for nseg, C in ((3, 1), (30, 1), (7, 3)):
        lens = torch.randint(0, 90000, (nseg,), generator=torch.Generator().manual_seed(nseg))
        lens[0] = 0 if nseg > 3 else lens[0]
        seg_ptr = torch.cat([torch.zeros(1, dtype=torch.long), lens.cumsum(0)]).to(DEV)
        n = int(seg_ptr[-1])
        src = torch.randn(n, C, device=DEV, generator=g)
        order = torch.randperm(n, device=DEV, generator=g)
        for od in (None, order):
            got = ops.gather_segment_sum(src, od, seg_ptr)
            s64 = (src if od is None else src[od]).double()
            want = torch.stack([s64[int(seg_ptr[i]):int(seg_ptr[i + 1])].sum(0) for i in range(nseg)])
            assert float((got.double() - want).abs().max()) < 1e-5 * max(1.0, float(want.abs().max()))
            assert torch.equal(got, ops.gather_segment_sum(src, od, seg_ptr))


def test_duplicate_detection_short_and_long_rows():
    """csr.cu: rows of up to 16 neighbours are checked by one thread, longer rows by a warp from a queue"""
    from gnan_b200.preprocess import build_csr
    rng = np.random.default_rng(4)
    n = 3000
    ei = random_graph(rng, n, 2.5, True)
    hub = np.stack([np.full(400, 7), rng.choice(np.setdiff1d(np.arange(n), ei[1][ei[0] == 7]), 400, replace=False)])
    base = np.concatenate([ei, hub], axis=1)                          # node 7: a row of > 400 distinct neighbours
    assert int(build_csr(torch.tensor(base), n, DEV)[2].item()) == 0
    assert int(build_csr(torch.tensor(np.concatenate([base, hub[:, 123:124]], axis=1)), n, DEV)[2].item()) == 2    # long row
    short = ei[:, ei[0] != 7][:, 5:6]
    assert int(build_csr(torch.tensor(np.concatenate([base, short], axis=1)), n, DEV)[2].item()) == 2             # short row


# ---- the tail of the training step (csrc/train.cu): fused losses and the one-launch Adam ----------------------------------
@pytest.mark.parametrize("N,C,frac", [(2708, 7, 0.05), (300, 40, 1.0), (5, 3, 0.6)])
def test_fused_cross_entropy_rows_vs_torch(N, C, frac):
    from gnan_b200 import ops
    g = torch.Generator(device=DEV).manual_seed(N)
    logits = (torch.randn(N, C, device=DEV, generator=g) * 3).requires_grad_(True)
    rows = torch.nonzero(torch.rand(N, device=DEV, generator=g) < frac).flatten()
    if rows.numel() == 0:
        rows = torch.tensor([0], device=DEV)
    labels = torch.randint(0, C, (rows.numel(),), device=DEV, generator=g)
    for reduction in ("mean", "sum"):
        ref = torch.nn.functional.cross_entropy(logits.double()[rows], labels, reduction=reduction)
        (gref,) = torch.autograd.grad(ref * 1.7, logits)
        got, bad = ops.cross_entropy_rows(logits, labels, rows=rows, reduction=reduction, return_flag=True)
        (ggot,) = torch.autograd.grad(got * 1.7, logits)
        assert int(bad.item()) == 0
        assert abs(float(got) - float(ref)) < 1e-5 * max(1.0, abs(float(ref)))
        assert G.rel_err(ggot.cpu().numpy(), gref.cpu().numpy()) < TOL
    full = ops.cross_entropy_rows(logits, torch.randint(0, C, (N,), device=DEV, generator=g))         # every row, no index list
    assert torch.isfinite(full)
    _, bad = ops.cross_entropy_rows(logits, torch.full((1,), C, device=DEV), rows=torch.zeros(1, dtype=torch.long, device=DEV), return_flag=True)
    assert int(bad.item()) == 1                                                                       # label out of range is reported


def test_fused_bce_with_logits_vs_torch():
    from gnan_b200 import ops
    g = torch.Generator(device=DEV).manual_seed(1)
    x = (torch.randn(4337, device=DEV, generator=g) * 4).requires_grad_(True)
    t = (torch.rand(4337, device=DEV, generator=g) < 0.4).float()
    for reduction in ("mean", "sum"):
        ref = torch.nn.functional.binary_cross_entropy_with_logits(x.double(), t.double(), reduction=reduction)
        (gref,) = torch.autograd.grad(ref, x)
        got = ops.bce_with_logits(x, t, reduction=reduction)
        (ggot,) = torch.autograd.grad(got, x)
        assert abs(float(got) - float(ref)) < 1e-5 * max(1.0, abs(float(ref)))
        assert G.rel_err(ggot.cpu().numpy(), gref.cpu().numpy()) < TOL


@pytest.mark.parametrize("wd", [0.0, 5e-4])
def test_one_launch_adam_follows_torch_adam(wd):
    """gnan_b200.optim.Adam against torch.optim.Adam over 25 steps on tensors of odd sizes (incl. > 24 tensors: two launches)."""
    from gnan_b200.optim import Adam
    g = torch.Generator(device=DEV).manual_seed(3)
    shapes = [(1434, 64), (64,), (1, 1434, 64, 64)[1:], (7,), (3, 5, 1025)] + [(k + 1,) for k in range(26)]
    pa = [torch.randn(*s, device=DEV, generator=g).requires_grad_(True) for s in shapes]
    pb = [p.detach().clone().requires_grad_(True) for p in pa]
    oa, ob = Adam(pa, lr=3e-3, weight_decay=wd), torch.optim.Adam(pb, lr=3e-3, weight_decay=wd)
    for step in range(25):
        for a, b in zip(pa, pb):
            gr = torch.randn(a.shape, device=DEV, generator=g) * (0.1 + step % 3)
            a.grad = gr.clone(); b.grad = gr.clone()
        oa.step(); ob.step()
    for a, b in zip(pa, pb):
        assert G.rel_err(a.detach().cpu().numpy(), b.detach().cpu().numpy()) < 2e-6
    assert float(oa.param_groups[0]["state_buf"][0]) == 25.0
