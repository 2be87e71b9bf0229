"""CPU: the float64 graph-readout reference of tests/_readout_f64.py (the checker of tests/test_gpu_graph_readout_f64.py)
against plain loops over the pairs, against the port of the unmodified reference (oracle.gnan_port.tensor_gnan_models,
models.py:358-384) fed the same table and feature sums, and its status words at the depth limit."""
import numpy as np
import pytest
import torch

from oracle import apsp as oapsp
from oracle import gnan_port
from tests import _readout_f64 as R
from tests.test_gpu_parity import random_graph


def _graphs(rng, sizes, directed=False, isolated=False):
    return [random_graph(rng, n, 2.5, directed, n_isolated=(1 + n // 6) if (isolated and n > 3) else 0) for n in sizes]


def _loops(hops, nbins, T, S, g, normalize):
    """the definition, one pair at a time"""
    B, Cr, C = len(hops), T.shape[1], S.shape[1]
    N = sum(h.shape[0] for h in hops)
    out, a_out = np.zeros((B, C)), np.zeros((B, C))
    colw, Q = np.zeros((N, Cr)), np.zeros((B, nbins, C))
    dS, dT = np.zeros((N, C)), np.zeros((nbins, Cr))
    n0 = 0
    for b, hop in enumerate(hops):
        n = hop.shape[0]
        dd = lambda i, j: nbins - 1 if hop[i, j] < 0 else min(int(hop[i, j]), nbins - 1)
        cnt = np.zeros((n, nbins))
        for i in range(n):
            for j in range(n):
                cnt[i, dd(i, j)] += 1
        for i in range(n):
            for j in range(n):
                d = dd(i, j)
                r = 1.0 / cnt[i, d] if normalize else 1.0
                for c in range(C):
                    cr = 0 if Cr == 1 else c
                    t = T[d, cr] * r * S[n0 + j, c]
                    out[b, c] += t
                    a_out[b, c] += abs(t)
                    Q[b, d, c] += r * S[n0 + j, c]
                    dT[d, cr] += g[b, c] * r * S[n0 + j, c]
                for cr in range(Cr):
                    colw[n0 + j, cr] += T[d, cr] * r
        for j in range(n):
            for c in range(C):
                dS[n0 + j, c] = g[b, c] * colw[n0 + j, 0 if Cr == 1 else c]
        n0 += n
    return out, a_out, colw, Q, dS, dT


@pytest.mark.parametrize("C,Cr", [(1, 1), (3, 1), (2, 2)])
@pytest.mark.parametrize("normalize", [True, False])
@pytest.mark.parametrize("nbins", [3, 6, 16])
def test_reference_matches_plain_loops(C, Cr, normalize, nbins):
    rng = np.random.default_rng(7 * C + Cr + 100 * nbins + normalize)
    sizes = [1, 2, 5, 9, 14]
    hops = R.oracle_hops(_graphs(rng, sizes, directed=bool(nbins % 2), isolated=True), sizes)
    N = sum(sizes)
    T, S, g = rng.normal(size=(nbins, Cr)), rng.normal(size=(N, C)), rng.normal(size=(len(sizes), C))
    ref = R.readout_f64(hops, nbins, T, S, g, normalize=normalize)
    out, a_out, colw, Q, dS, dT = _loops(hops, nbins, T, S, g, normalize)
    for got, want in ((ref.out, out), (ref.a_out, a_out), (ref.colw, colw), (ref.Q, Q), (ref.dS, dS), (ref.dT, dT)):
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12)
    assert np.all(ref.a_out >= np.abs(ref.out)) and np.all(ref.a_dT >= np.abs(ref.dT) - 1e-12)


def test_folded_counts_are_the_bincount_of_the_bins():
    rng = np.random.default_rng(3)
    for n, nbins in ((1, 2), (7, 2), (40, 4), (40, 48), (100, 9)):
        hop = R.oracle_hops(_graphs(rng, [n], isolated=True), [n])[0]
        cnt = R.folded_counts(hop, nbins)
        d = R.bins(hop, nbins)
        want = np.stack([np.bincount(row, minlength=nbins) for row in d])
        assert np.array_equal(cnt, want) and np.all(cnt.sum(axis=1) == n)


def _port(monkeypatch, hop, nbins, T, S, normalize):
    """tensor_gnan_models on one graph with rho(node_distances) = T[d_ij] and the shape functions' sum = S (one feature):
    the reference's own normalisation, matmul and sums, float64, autograd for dT / dS"""
    unreach = nbins - 1

    def rho_lookup(p, g, t):
        nd = t.view(-1)
        idx = torch.where(nd == 0, torch.full_like(nd, unreach), torch.round(1.0 / nd) - 1).long()   # nd = 1 / (hop + 1), 0
        return p["wo"][idx]

    monkeypatch.setattr(gnan_port, "scalar_mlp", rho_lookup)
    monkeypatch.setattr(gnan_port, "shape_functions", lambda p, x: p["S"].unsqueeze(1))
    cnt = oapsp.level_counts(hop, nbins)                 # the reference's counts (no hop >= nbins - 1 in these graphs)
    nd, nm = oapsp.reference_format(hop, cnt)
    return gnan_port.tensor_gnan_models({"S": S}, {"wo": T}, S, torch.tensor(nd, dtype=torch.float64),
                                        torch.tensor(nm, dtype=torch.float64), normalize_rho=normalize, is_graph_task=True)[:, 0]


@pytest.mark.parametrize("Cr", [1, 3])
@pytest.mark.parametrize("normalize", [True, False])
@pytest.mark.parametrize("connected", [True, False])
def test_reference_matches_the_ported_reference_model(monkeypatch, Cr, normalize, connected):
    C, nbins = 3, 24
    rng = np.random.default_rng(10 * Cr + 2 * normalize + connected)
    sizes = [1, 3, 17, 30, 41]
    eis = _graphs(rng, sizes, directed=False, isolated=not connected)
    if connected:                                         # a path through all nodes makes every graph connected
        eis = [np.concatenate([e, np.stack([np.arange(n - 1), np.arange(1, n)]), np.stack([np.arange(1, n), np.arange(n - 1)])],
                              axis=1) for e, n in zip(eis, sizes)]
    hops = R.oracle_hops(eis, sizes)
    assert all((h.min() >= 0) == connected for h in hops[2:]) and max(int(h.max()) for h in hops) <= nbins - 2
    N = sum(sizes)
    T, S, g = rng.normal(size=(nbins, Cr)), rng.normal(size=(N, C)), rng.normal(size=(len(sizes), C))
    ref = R.readout_f64(hops, nbins, T, S, g, normalize=normalize)
    T64 = torch.tensor(T, requires_grad=True)
    S64 = torch.tensor(S, requires_grad=True)
    outs, n0 = [], 0
    for hop in hops:
        n = hop.shape[0]
        outs.append(_port(monkeypatch, hop, nbins, T64, S64[n0:n0 + n], normalize))
        n0 += n
    out = torch.stack(outs)
    dT, dS = torch.autograd.grad(out, (T64, S64), grad_outputs=torch.tensor(g))
    np.testing.assert_allclose(ref.out, out.detach().numpy(), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(ref.dT, dT.numpy(), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(ref.dS, dS.numpy(), rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("nbins", [2, 3, 5, 33, 48, 64])
def test_expected_status_of_paths_around_the_depth_limit(nbins):
    """a path of L + 1 nodes has eccentricity L: bins 0..nbins-2 hold L <= nbins - 2, L = nbins - 1 overflows"""
    for L in range(max(0, nbins - 3), nbins + 1):
        n = L + 1
        path = np.stack([np.arange(n - 1), np.arange(1, n)])
        for ei in (path, np.concatenate([path, path[::-1]], axis=1)):
            hops = R.oracle_hops([ei], [n]) + R.oracle_hops([np.zeros((2, 0), np.int64)], [3])
            assert R.expected_status(hops, nbins) == [0, int(L >= nbins - 1), L], (nbins, L)


def test_pack_hops_and_rscale():
    rng = np.random.default_rng(1)
    sizes = [3, 1, 12]
    hops = R.oracle_hops(_graphs(rng, sizes, directed=True, isolated=True), sizes)
    buf, hop_off, node_off = R.pack_hops(hops)
    assert list(node_off) == [0, 3, 4, 16] and list(hop_off) == [0, 9, 10, 154]
    back = buf[hop_off[2]:hop_off[3]].astype(np.int32).reshape(12, 12)
    back[back == 255] = -1
    assert np.array_equal(back, hops[2])
    rs = R.rscale_f32(hops, 5)
    cnt = np.concatenate([R.folded_counts(h, 5) for h in hops])
    assert rs.dtype == np.float32 and np.array_equal(rs == 0, cnt == 0)
    assert np.array_equal(rs[cnt > 0], (1.0 / cnt[cnt > 0]).astype(np.float32))

