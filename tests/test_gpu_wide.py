"""GPU: deep graphs (hop distances > 254) through the int16 path of csrc/wide.cu — BFS + level histogram bit-exact against the C
oracle, the aggregation and its backward against float64, and a whole module step against the float64 restatement of
GNAN.py:55-79 (1e-5 norm-wise)."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import apsp as oapsp
from oracle import gnan_lut, gnan_port, params as P
from tests import _golden as G

pytestmark = pytest.mark.gpu
TOL = 1e-5
DEV = "cuda"


def deep_graph(rng, n_chain=420, n_extra=180, directed=False):
    """a long chain (diameter > 254) with short random side branches and one far isolated pair"""
    a = np.arange(n_chain - 1)
    e = [np.stack([a, a + 1])]
    nxt = n_chain
    for _ in range(n_extra):
        e.append(np.array([[int(rng.integers(0, nxt))], [nxt]]))
        nxt += 1
    e.append(np.array([[nxt], [nxt + 1]]))                      # a component of its own: unreachable pairs
    n = nxt + 2
    ei = np.concatenate(e, axis=1)
    if not directed:
        ei = np.concatenate([ei, ei[::-1]], axis=1)
    return ei.astype(np.int64), n


@pytest.mark.parametrize("directed", [False, True])
def test_deep_graph_bfs_bit_exact_vs_oracle(directed):
    from gnan_b200.preprocess import apsp, from_reference_format
    rng = np.random.default_rng(3 + directed)
    ei, n = deep_graph(rng, directed=directed)
    hd = apsp(torch.tensor(ei), n, device=DEV)
    want = oapsp.apsp(ei, n)                                     # int32, -1 = unreachable
    assert hd.wide and int(want.max()) > 254
    assert np.array_equal(hd.hop[:, :n].cpu().numpy().astype(np.int32), want)
    assert np.array_equal(hd.level_counts.cpu().numpy(), oapsp.level_counts(want, hd.nbins))
    part = apsp(torch.tensor(ei), n, device=DEV, row_begin=100, row_end=333)                         # a row shard
    assert np.array_equal(part.hop[:, :n].cpu().numpy().astype(np.int32), want[100:333])
    nd, nm = hd.reference_format()                                                                    # the reference's fp32 matrices
    wnd, wnm = oapsp.reference_format(want, oapsp.level_counts(want))
    assert np.array_equal(nd.cpu().numpy(), wnd) and np.array_equal(nm.cpu().numpy(), wnm)
    back = from_reference_format(nd, nm)
    assert back.wide and torch.equal(back.hop[:, :n], hd.hop[:, :n]) and torch.equal(back.level_counts, hd.level_counts)


@pytest.mark.parametrize("R,N,C,Cr,nbins,per_row,scale", [(70, 900, 3, 3, 700, True, True), (33, 515, 5, 1, 300, False, True),
                                                          (64, 1000, 7, 7, 1200, False, False), (9, 260, 1, 1, 270, True, False)])
def test_wide_aggregation_vs_float64(R, N, C, Cr, nbins, per_row, scale):
    from gnan_b200 import ops
    rng = np.random.default_rng(R + N)
    h = rng.integers(0, nbins - 1, size=(R, N))
    h[rng.random((R, N)) < 0.02] = -1                            # unreachable pairs -> last bin
    hop = torch.full((R, ops.hop_ld(N)), -1, dtype=torch.int16, device=DEV)
    hop[:, :N] = torch.tensor(h.astype(np.int16), device=DEV)
    T = torch.tensor(rng.normal(size=((R, nbins, Cr) if per_row else (nbins, Cr)))).float()
    S = torch.tensor(rng.normal(size=(N, C))).float()
    rs = torch.tensor(rng.random(size=(R, nbins)) + 0.1).float() if scale else None
    gO = torch.tensor(rng.normal(size=(R, C))).float()
    gO[::3] = 0.0                                                # rows without a loss are skipped
    idx = torch.tensor(np.where(h < 0, nbins - 1, h))
    Td, Sd = T.double().requires_grad_(True), S.double().requires_grad_(True)
    W = (torch.gather(Td, 1, idx.unsqueeze(-1).expand(-1, -1, Cr)) if per_row else Td[idx])
    if scale:
        W = W * torch.gather(rs.double(), 1, idx).unsqueeze(-1)
    want = (W * Sd.unsqueeze(0)).sum(1)
    (want * gO.double()).sum().backward()
    Tg, Sg = T.to(DEV).requires_grad_(True), S.to(DEV).requires_grad_(True)
    got = ops.aggregate_rows(hop, Tg, Sg, rscale=None if rs is None else rs.to(DEV), per_row=per_row)
    (got * gO.to(DEV)).sum().backward()
    assert G.rel_err(got.detach().cpu().numpy(), want.detach().numpy()) < TOL
    assert G.rel_err(Sg.grad.cpu().numpy(), Sd.grad.numpy()) < TOL
    assert G.rel_err(Tg.grad.cpu().numpy(), Td.grad.numpy()) < TOL


@pytest.mark.parametrize("variant,n_chain,C", [
    pytest.param("GNAN.TensorGNAN", 300, 3, id="GNAN.TensorGNAN"), pytest.param("models.TensorGNAN", 300, 3, id="models.TensorGNAN"),
    # diameter 209-254: still uint8 hops, nbins > 210 on the CUDA-core row kernels with 4-channel chunks
    pytest.param("GNAN.TensorGNAN", 230, 5, id="GNAN.TensorGNAN-uint8"),
    pytest.param("models.TensorGNAN", 230, 5, id="models.TensorGNAN-uint8")])
def test_deep_graph_module_step_vs_float64_restatement(variant, n_chain, C):
    """A whole forward + backward on a graph of diameter > 254 (int16 hops), or 209-254 (uint8 hops, nbins > 210), with input-
    and output-normalised rho, against oracle/gnan_lut.py."""
    from gnan_b200.preprocess import apsp
    rng = np.random.default_rng(11)
    ei, n = deep_graph(rng, n_chain=n_chain, n_extra=60)
    K, H, L = 5, 64, 3
    x = torch.tensor(rng.normal(size=(n, K))).float()
    w = torch.tensor(rng.normal(size=(n, C))).float()
    torch.manual_seed(0)
    if variant == "GNAN.TensorGNAN":
        from gnan_b200.GNAN import TensorGNAN
        m = TensorGNAN(K, C, L, H, normalize_rho=True, is_graph_task=False).to(DEV)
        mode, rl = "input", 2
    else:
        from gnan_b200.models import TensorGNAN
        m = TensorGNAN(K, C, L, H, normalize_rho=True, is_graph_task=False, rho_per_feature=True, readout_n_layers=0).to(DEV)
        mode, rl = "output", 2
    m.fs.xavier_normal_(1.0); m.rho.xavier_normal_(1.0)
    hd = apsp(torch.tensor(ei), n, device=DEV)
    assert hd.wide if n_chain > 256 else (not hd.wide and hd.nbins > 210)
    out = m.forward(SimpleNamespace(x=x, hop_data=hd))
    (out * w.to(DEV)).sum().backward()
    hop = torch.tensor(oapsp.apsp(ei, n)).long()
    cnt = gnan_lut.counts_from_hops(hop)
    sd = {k: v.detach().cpu().numpy() for k, v in m.state_dict().items()}
    fs = gnan_port.to_torch(P.stack_mlps(sd, [f"fs.{k}" for k in range(K)], L, 3), torch.float64, True)
    rho = gnan_port.to_torch(P.stack_mlps(sd, ["rho"], L, rl), torch.float64, True)
    want = gnan_lut.forward_rows(fs, rho, x.double(), hop, cnt, mode)
    (want * w.double()).sum().backward()
    rel = lambda a, b: float((a.double().cpu() - b).norm() / b.norm())
    assert rel(out.detach(), want.detach()) < TOL
    for name in ("wh", "wo", "w1"):
        assert rel(getattr(m.fs, name).grad, fs[name].grad) < TOL, name
        assert rel(getattr(m.rho, name).grad, rho[name].grad) < TOL, name
