"""Float64 reference of the output-normalised graph readout with a global distance table (models.py:366-384 with
is_graph_task), graph by graph, on hop matrices of the C oracle (oracle/apsp_oracle.c; -1 = unreachable).

For a batch of B graphs, a table T [nbins, Cr] (Cr = 1 or C) and feature sums S [sum n, C]:
    d_ij = min(hop_ij, nbins - 1), unreachable pairs -> nbins - 1
    r[i,d] = 1 / cnt[i,d]   (cnt = the oracle's level counts folded to nbins columns; r = 1 without the normaliser)
    P[j,d] = sum_{i: d_ij = d} r[i,d]
    colw[j,c'] = sum_d T[d,c'] P[j,d]      Q[b,d,c] = sum_{j in b} S[j,c] P[j,d]      out[b,c] = sum_j colw[j,c'] S[j,c]
    dS[j,c] = g[b,c] colw[j,c']            dT[d,c'] = sum_b sum_c g[b,c] Q[b,d,c]  (sum over c only when Cr = 1; else c = c')
Every result comes with A, the sum of the absolute values of its terms (T, S and g enter with their absolute values; r and
P are positive), which scales the per-entry error bound of a float32 kernel."""
from types import SimpleNamespace

import numpy as np

from oracle import apsp as oapsp


def split_edges(edge_index, node_off):
    """[2,E] global edge list -> per-graph [2,E_b] int64 lists of local ids (edges grouped by the graph of their source)."""
    ei = np.asarray(edge_index, dtype=np.int64)
    no = np.asarray(node_off, dtype=np.int64)
    g = np.searchsorted(no, ei[0], side="right") - 1
    order = np.argsort(g, kind="stable")
    ei, g = ei[:, order], g[order]
    cut = np.searchsorted(g, np.arange(len(no)))
    return [ei[:, cut[b]:cut[b + 1]] - no[b] for b in range(len(no) - 1)]


def oracle_hops(edge_lists, sizes, dtype=np.int16):
    """the oracle's hop matrix of every graph (int16 keeps a 32 768-graph batch small; -1 = unreachable)"""
    return [oapsp.apsp(e, int(n)).astype(dtype) for e, n in zip(edge_lists, sizes)]


def folded_counts(hop, nbins):
    """oracle.apsp.level_counts at the graph's own width (levels 0..max, then unreachable), folded to nbins columns: levels
    >= nbins - 1 join the unreachable column, as d_ij does"""
    nat = oapsp.level_counts(hop)
    w = nat.shape[1]
    cnt = np.zeros((hop.shape[0], nbins), dtype=np.int64)
    keep = min(w - 1, nbins - 1)
    cnt[:, :keep] = nat[:, :keep]
    cnt[:, nbins - 1] = nat[:, keep:].sum(axis=1)
    return cnt


def bins(hop, nbins):
    hop = np.asarray(hop)
    return np.where(hop < 0, nbins - 1, np.minimum(hop, nbins - 1)).astype(np.int64)


def expected_status(hops, nbins):
    """the batch's status word: CSR status bits, overflow (a finite hop >= nbins - 1), largest finite hop"""
    largest = max((int(h.max()) for h in hops), default=0)
    return [0, int(largest >= nbins - 1), largest]


def readout_f64(hops, nbins, T, S, g=None, normalize=True):
    """out [B,C], colw [N,Cr], Q [B,nbins,C] and, for g [B,C], dS [N,C] and dT [nbins,Cr]; each X with its A_X"""
    T = np.asarray(T, dtype=np.float64)
    S = np.asarray(S, dtype=np.float64)
    Cr, C, B = T.shape[1], S.shape[1], len(hops)
    aT, aS = np.abs(T), np.abs(S)
    N = sum(h.shape[0] for h in hops)
    assert S.shape[0] == N and T.shape[0] == nbins and Cr in (1, C)
    out, a_out = np.zeros((B, C)), np.zeros((B, C))
    colw, a_colw = np.zeros((N, Cr)), np.zeros((N, Cr))
    Q, a_Q = np.zeros((B, nbins, C)), np.zeros((B, nbins, C))
    n0 = 0
    for b, hop in enumerate(hops):
        n = hop.shape[0]
        d = bins(hop, nbins)
        if normalize:
            r = 1.0 / np.maximum(folded_counts(hop, nbins), 1)         # bins with a zero count are never read
            w = np.take_along_axis(r, d, axis=1).ravel()
        else:
            w = None
        P = np.bincount((d * n + np.arange(n)).ravel(), weights=w, minlength=nbins * n).reshape(nbins, n)     # P[d, j]
        s, a_s = S[n0:n0 + n], aS[n0:n0 + n]
        cw, acw = P.T @ T, P.T @ aT
        colw[n0:n0 + n], a_colw[n0:n0 + n] = cw, acw
        Q[b], a_Q[b] = P @ s, P @ a_s
        out[b], a_out[b] = (s * cw).sum(axis=0), (a_s * acw).sum(axis=0)
        n0 += n
    res = SimpleNamespace(out=out, a_out=a_out, colw=colw, a_colw=a_colw, Q=Q, a_Q=a_Q)
    if g is not None:
        g = np.asarray(g, dtype=np.float64)
        sizes = np.array([h.shape[0] for h in hops], dtype=np.int64)
        gj, agj = np.repeat(g, sizes, axis=0), np.repeat(np.abs(g), sizes, axis=0)      # g of each node's graph [N,C]
        res.dS, res.a_dS = gj * colw, agj * a_colw
        if Cr == 1:
            res.dT = np.einsum("bdc,bc->d", Q, g)[:, None]
            res.a_dT = np.einsum("bdc,bc->d", a_Q, np.abs(g))[:, None]
        else:
            res.dT = np.einsum("bdc,bc->dc", Q, g)
            res.a_dT = np.einsum("bdc,bc->dc", a_Q, np.abs(g))
    return res


def pack_hops(hops):
    """the packed hop bytes of a batch (row-major blocks, 255 = unreachable), hop_off int64 [B+1], node_off int32 [B+1]"""
    sizes = np.array([h.shape[0] for h in hops], dtype=np.int64)
    hop_off = np.zeros(len(hops) + 1, dtype=np.int64)
    np.cumsum(sizes * sizes, out=hop_off[1:])
    node_off = np.zeros(len(hops) + 1, dtype=np.int32)
    np.cumsum(sizes, out=node_off[1:])
    buf = np.empty(max(int(hop_off[-1]), 1), dtype=np.uint8)
    for b, h in enumerate(hops):
        assert int(h.max()) < 255, "a hop of 255 or more does not fit the hop bytes"
        buf[hop_off[b]:hop_off[b + 1]] = np.where(h < 0, 255, h).ravel()
    return buf, hop_off, node_off


def rscale_f32(hops, nbins):
    """the normaliser table [sum n, nbins] as float32 1/cnt (0 for empty bins), from the oracle's counts"""
    cnt = np.concatenate([folded_counts(h, nbins) for h in hops]) if hops else np.zeros((0, nbins), np.int64)
    rs = np.zeros(cnt.shape, dtype=np.float32)
    nz = cnt > 0
    rs[nz] = np.float32(1.0) / cnt[nz].astype(np.float32)
    return rs


def assert_entrywise(name, got, ref, a, rtol, node_off=None):
    """|got - ref| <= rtol * A + 1e-30 for every entry; the message names the first failing graph (rows of node-indexed
    arrays are mapped to graphs through node_off)."""
    got = np.asarray(got, dtype=np.float64)
    assert got.shape == ref.shape, (name, got.shape, ref.shape)
    err = np.abs(got - ref)
    bad = ~(err <= rtol * a + 1e-30)
    if bad.any():
        idx = np.argwhere(bad)
        first = tuple(int(v) for v in idx[0])
        where = f"entry {first}"
        if node_off is not None:
            where += f" (graph {int(np.searchsorted(node_off, first[0], side='right') - 1)})"
        ratio = err[bad] / np.maximum(a[bad], 1e-300)
        raise AssertionError(f"{name}: {int(bad.sum())} of {bad.size} entries outside {rtol:g} * A; first at {where}: got "
                             f"{got[first]!r}, want {ref[first]!r}, A {a[first]!r}; worst |err| / A = {float(ratio.max()):.3g}")
