"""GPU: the general block-diagonal kernels of csrc/agg.cu (gnan_aggregate_blockdiag_fwd/bwd) against float64 on every launch
branch. They serve every packed batch with per-row tables, every node-level packed batch and every graph readout outside the
one-pass kernel's envelope (C <= 4, nbins <= 64), so they are called here directly, also inside that envelope.

Branches, by (table, nbins * Cr): forward rows kernel <1>/<2>/<4> (channel-chunk remainder at C = 5, 7, 9) and the v1 kernel
of a global table past 12 288 entries; backward with lane-private accumulators (global, <= 199 entries), with shared-memory
bins (global fallback, per-row with 8, 4, ... warps per CTA, above 48 KB) and with bins in dT itself past 227 KB.

Checker: a float64 restatement vectorised over the pair list of the packed batch, gradients by autograd. Each entry of out, dS
and dT is held to 1e-5 of the sum of |terms| of its own sum (a single wrong graph among thousands fails), and each tensor to
1e-5 norm-wise."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from tests import _golden as G
from tests.test_gpu_parity import random_graph

pytestmark = pytest.mark.gpu
TOL = 1e-5
DEV = "cuda"

MIXED = [1, 2, 31, 32, 33, 63, 64, 65, 257]          # around the 32-lane strides of both kernels
# (C, Cr, nbins, per_row)
CASES = [
    (1, 1, 9, False), (3, 1, 66, False), (5, 5, 39, False),            # lane-private backward
    (5, 5, 40, False), (7, 7, 256, False), (9, 1, 256, False),          # shared-memory fallback backward, channel remainder
    (64, 64, 200, False),                                               # v1 forward, fallback backward above 48 KB
    (256, 256, 256, False),                                             # v1 forward, bins in dT
    (2, 2, 12, True), (40, 40, 38, True),                               # per-row, 8 warps within 48 KB
    (40, 40, 39, True), (16, 16, 256, True),                            # per-row, 8 warps above 48 KB
    (40, 40, 182, True),                                                # per-row, 4 warps
    (5, 1, 256, True),
    (256, 256, 256, True),                                              # per-row, bins in dT
]


def _case_id(case):
    C, Cr, nbins, per_row = case
    return f"{'row' if per_row else 'global'}-C{C}-Cr{Cr}-nb{nbins}"


def _sizes(rng, C, Cr, nbins, per_row):
    """MIXED, a 1024-node graph where pairs x C stay small, and 12 000 graphs of 1-12 nodes (more than the resident warps of
    either grid on a B200: forward 8 x 148 CTAs x 8 warps, backward 4 x 148 x 8) where the tables stay small; shuffled"""
    sizes = list(MIXED)
    if C <= 5:
        sizes.append(1024)
    if C <= 64 and (not per_row or 80_000 * nbins * Cr <= 3e7):
        sizes += rng.integers(1, 13, size=12_000).tolist()
    rng.shuffle(sizes)
    return sizes


def _packed(rng, sizes, nbins):
    """A packed batch written directly: random levels, 255 for unreachable pairs, levels past nbins - 1 (the clamp), 0 on
    the diagonal; node_off int32 and hop_off int64 as preprocess.apsp_batched makes them. Also the pair list (graph, global
    row, global column, bin) of the reference."""
    n = torch.tensor(sizes, dtype=torch.int64)
    node_off = torch.zeros(len(sizes) + 1, dtype=torch.int64)
    node_off[1:] = n.cumsum(0)
    hop_off = torch.zeros_like(node_off)
    hop_off[1:] = (n * n).cumsum(0)
    P = int(hop_off[-1])
    b = torch.repeat_interleave(torch.arange(len(sizes)), n * n)
    k = torch.arange(P) - hop_off[b]
    i, j = k // n[b], k % n[b]
    h = torch.tensor(rng.integers(1, min(nbins + 2, 255), size=P))
    h[torch.tensor(rng.random(P) < 0.05)] = 255
    h[i == j] = 0
    return SimpleNamespace(hop=h.to(torch.uint8).to(DEV), hop_off=hop_off.to(DEV), node_off=node_off.to(torch.int32).to(DEV),
                           B=len(sizes), N=int(node_off[-1]), b=b.to(DEV), gi=(node_off[b] + i).to(DEV),
                           gj=(node_off[b] + j).to(DEV), d=h.clamp(max=nbins - 1).to(DEV))


def _reference(pk, T, rs, S, g, per_row, reduce_graph):
    """float64 (out, dS, dT), each with the sums of |terms| of its entries"""
    nbins, Cr = T.shape[-2:]
    T64, S64 = T.double().requires_grad_(True), S.double().requires_grad_(True)
    r = None if rs is None else rs.double()[pk.gi, pk.d].unsqueeze(1)            # [P,1]
    w = T64[pk.gi, pk.d] if per_row else T64[pk.d]                                 # [P,Cr]
    if r is not None:
        w = w * r
    terms = w * S64[pk.gj]                                                         # [P,C]
    dst = pk.b if reduce_graph else pk.gi
    out = torch.zeros(pk.B if reduce_graph else pk.N, S.shape[1], dtype=torch.float64, device=DEV).index_add(0, dst, terms)
    g64 = g.double()
    dT, dS = torch.autograd.grad((out * g64).sum(), (T64, S64))
    with torch.no_grad():
        gp = g64[dst]
        out_abs = torch.zeros_like(out).index_add_(0, dst, terms.abs())
        dS_abs = torch.zeros_like(dS).index_add_(0, pk.gj, (w * gp).abs())
        tt = (gp * S64[pk.gj]).abs()
        if r is not None:
            tt = tt * r
        if Cr == 1:
            tt = tt.sum(1, keepdim=True)
        slot = pk.gi * nbins + pk.d if per_row else pk.d
        dT_abs = torch.zeros(T.numel() // Cr, Cr, dtype=torch.float64, device=DEV).index_add_(0, slot, tt).view(T.shape)
    return (out.detach(), out_abs), (dS, dS_abs), (dT, dT_abs)


def _check(got, want, bound, what):
    """every entry within 1e-5 of its sum of |terms|, and the whole within 1e-5 norm-wise, or within 1e-6 of the norm of
    the sums of |terms| where its entries cancel by more than 10x (a global-table dT of a graph readout without rscale sums
    ~1e5 pairs of one 1024-node graph per bin with 50-70x cancellation: fp32 accumulation reaches 2e-5 norm-wise there,
    2.5e-7 of the sums of |terms|)"""
    err = (got.double() - want).abs()
    bad = err > TOL * bound
    if bad.any():
        k = int(torch.argmax((err - TOL * bound).flatten()))
        idx = np.unravel_index(k, tuple(want.shape))
        raise AssertionError(f"{what}: {int(bad.sum())} of {want.numel()} entries off; worst at {idx}: got "
                             f"{float(got[idx]):.9g}, want {float(want[idx]):.9g}, 1e-5 * sum|terms| = {float(TOL * bound[idx]):.3g}")
    cancellation = float(bound.norm() / want.norm().clamp_min(1e-300))
    assert G.rel_err(got.cpu().numpy(), want.cpu().numpy()) < TOL * max(1.0, cancellation / 10), (what, cancellation)


@pytest.mark.parametrize("reduce_graph", [True, False])
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_general_blockdiag_kernels_vs_float64(case, reduce_graph):
    from gnan_b200 import ops
    C, Cr, nbins, per_row = case
    seed = CASES.index(case)
    rng = np.random.default_rng(1000 + 2 * seed + reduce_graph)
    pk = _packed(rng, _sizes(rng, *case), nbins)
    T = torch.tensor(rng.normal(size=(pk.N, nbins, Cr) if per_row else (nbins, Cr))).float().to(DEV)
    S = torch.tensor(rng.normal(size=(pk.N, C))).float().to(DEV)
    rs = torch.tensor(rng.random((pk.N, nbins)) + 0.1).float().to(DEV) if (seed + reduce_graph) % 2 == 0 else None
    g = torch.tensor(rng.normal(size=(pk.B if reduce_graph else pk.N, C))).float().to(DEV)

    Tg, Sg = T.clone().requires_grad_(True), S.clone().requires_grad_(True)
    out = ops.agg_blockdiag_fwd(pk.hop, pk.hop_off, pk.node_off, Tg, rs, Sg, per_row, reduce_graph)
    dT, dS = torch.autograd.grad((out * g).sum(), (Tg, Sg))
    (want, out_abs), (wS, dS_abs), (wT, dT_abs) = _reference(pk, T, rs, S, g, per_row, reduce_graph)
    _check(out.detach(), want, out_abs, "out")
    _check(dS, wS, dS_abs, "dS")
    _check(dT, wT, dT_abs, "dT")
    with torch.no_grad():                   # the forward has no atomics: bit-identical on a second run
        assert torch.equal(ops.agg_blockdiag_fwd(pk.hop, pk.hop_off, pk.node_off, T, rs, S, per_row, reduce_graph), out.detach())


@pytest.mark.parametrize("per_row", [False, True])
@pytest.mark.parametrize("reduce_graph", [True, False])
def test_general_blockdiag_kernels_empty_batch(per_row, reduce_graph):
    from gnan_b200 import ops
    nbins, C = 9, 3
    T = torch.randn((0, nbins, C) if per_row else (nbins, C), device=DEV, requires_grad=True)
    S = torch.zeros(0, C, device=DEV, requires_grad=True)
    hop = torch.zeros(0, dtype=torch.uint8, device=DEV)
    hop_off = torch.zeros(1, dtype=torch.int64, device=DEV)
    node_off = torch.zeros(1, dtype=torch.int32, device=DEV)
    out = ops.agg_blockdiag_fwd(hop, hop_off, node_off, T, None, S, per_row, reduce_graph)
    assert tuple(out.shape) == (0, C)
    dT, dS = torch.autograd.grad(out.sum(), (T, S))
    assert dT.shape == T.shape and dS.shape == S.shape and not dT.any()


@pytest.mark.parametrize("graph_task", [False, True])
def test_packed_model_with_wide_per_row_tables_equals_per_graph_forward(graph_task):
    """GNAN.TensorGNAN (input-normalised rho: a per-row table) with 40 outputs on a batch holding a 45-node chain, so the
    per-row backward's 8 warps of nbins * C bins need more than 48 KB of shared memory: the packed call equals the per-graph
    forward, outputs and parameter gradients."""
    from gnan_b200.GNAN import TensorGNAN
    from gnan_b200.preprocess import apsp, apsp_batched
    rng = np.random.default_rng(41 + graph_task)
    K, C, chain = 5, 40, 45
    a = np.arange(chain - 1)
    path = np.concatenate([np.stack([a, a + 1]), np.stack([a + 1, a])], axis=1)
    graphs = [(random_graph(rng, 17, 2.2, n_isolated=1), 17), (path, chain), (random_graph(rng, 1, 0.0), 1),
              (random_graph(rng, 33, 2.5, n_isolated=2), 33)]
    sizes = [n for _, n in graphs]
    node_off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    ei = np.concatenate([e + node_off[i] for i, (e, _) in enumerate(graphs)], axis=1)
    x = torch.tensor(rng.normal(size=(int(node_off[-1]), K))).float()
    torch.manual_seed(3)
    m = TensorGNAN(K, C, 3, 64, is_graph_task=graph_task, normalize_rho=True).to(DEV)
    m.fs.xavier_normal_(1.0); m.rho.xavier_normal_(1.0)
    pk = apsp_batched(torch.tensor(ei), torch.tensor(node_off), device=DEV)
    assert pk.nbins >= chain and pk.nbins * C * 4 * 8 > 48 * 1024
    pk.x = x.to(DEV)
    out = m(pk)
    w = torch.tensor(rng.normal(size=tuple(out.shape))).float().to(DEV)
    params = list(m.parameters())
    g_pk = torch.autograd.grad((out * w).sum(), params)
    ref = []
    for i, (e, n) in enumerate(graphs):
        o = m.forward(SimpleNamespace(x=x[node_off[i]:node_off[i + 1]], hop_data=apsp(torch.tensor(e), n, device=DEV)))
        ref.append(o.T if graph_task else o)
    ref = torch.cat(ref)
    g_ref = torch.autograd.grad((ref * w).sum(), params)
    assert G.rel_err(out.detach().cpu().numpy(), ref.detach().cpu().numpy()) < TOL
    for p, q in zip(g_pk, g_ref):
        assert G.rel_err(p.cpu().numpy(), q.cpu().numpy()) < TOL
