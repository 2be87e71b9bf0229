"""GPU: parity of the CUDA path (through the C ABI) against the golden vectors of the unmodified reference and
against the oracle on seeded inputs. Tolerances (norm-wise relative, SURVEY.md §8c): 1e-5 for fp32 outputs and
gradients; hop distances, level counts and the reference-format matrices are compared bit-exactly."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import apsp as oapsp
from oracle import gnan_lut, gnan_port
from tests import _golden as G
from tests._build import build_module

pytestmark = pytest.mark.gpu
TOL = 1e-5
TOL_TF32X3 = 3e-5   # end-to-end bound of the 3xTF32 tensor-core mode (kernel-level tests of that mode still hold 1e-5)
DEV = "cuda"


def grads_of(stacked):
    out = {}
    for n in ("w1", "b1", "wh", "bh", "wo", "bo"):
        p = getattr(stacked, n)
        out[n] = None if not isinstance(p, torch.nn.Parameter) or p.grad is None else p.grad.detach().cpu().numpy()
    return out


def check_grads(z, got, want, tag, tol=TOL):
    for k in ("w1", "b1", "wh", "bh", "wo", "bo"):
        w = want[k]
        if w is None or w.size == 0 or got[k] is None:
            continue
        if np.linalg.norm(w) == 0:
            assert np.abs(got[k]).max() < 1e-6, (z["name"], tag, k)
        else:
            assert G.rel_err(got[k], w) < tol, (z["name"], tag, k, G.rel_err(got[k], w))


def run_case(z, compact, precision="fp32"):
    m = build_module(z, DEV).eval()
    m.precision = precision
    w = torch.tensor(z["out_weight"], device=DEV)
    if z["variant"] == "batched":
        if compact:
            from gnan_b200.batched import pack_dense
            pk = pack_dense(torch.tensor(z["x"], device=DEV), torch.tensor(z["dist_batch"], device=DEV),
                            torch.tensor(z["batch_vector"], device=DEV))
            out = m(pk)
        else:
            out = m(torch.tensor(z["x"]), torch.tensor(z["dist_batch"]), torch.tensor(z["batch_vector"]))
    else:
        if compact:
            from gnan_b200.preprocess import apsp
            hd = apsp(torch.tensor(z["edge_index"]), z["N"], device=DEV)
            data = SimpleNamespace(x=torch.tensor(z["x"]), edge_index=torch.tensor(z["edge_index"]), hop_data=hd)
        else:
            data = SimpleNamespace(x=torch.tensor(z["x"]), edge_index=torch.tensor(z["edge_index"]),
                                   node_distances=torch.tensor(z["node_distances"]),
                                   normalization_matrix=torch.tensor(z["normalization_matrix"]))
        if z["variant"] == "gnan_loop" and "node_ids" in z:
            out = m.forward(data, z["node_ids"].tolist())
        else:
            out = m.forward(data)
    (out * w).sum().backward()
    return m, out


RUNNABLE = G.MODEL_CASES + G.BATCHED_CASES


@pytest.mark.parametrize("precision", ["fp32", "tf32x3"])
@pytest.mark.parametrize("compact", [False, True], ids=["reference_inputs", "compact_inputs"])
@pytest.mark.parametrize("name", RUNNABLE)
def test_module_matches_reference_golden(name, compact, precision):
    """Both kernel paths against the unmodified reference's outputs and gradients (the tcgen05 path covers H = 64, 3 layers,
    C <= 8; other golden shapes run the fp32 kernels under either setting).

    fp32 kernels: 1e-5 (measured worst over the cases 1.5e-6). 3xTF32 tcgen05 kernels: each product carries ~2^-22 instead of
    2^-24 relative error, so module-level errors are ~10x the fp32 ones: typically 1-3e-6, 1.1e-5 on the worst-conditioned
    case (gnan_loop_shared_rho, 1/count normalisation with heavy cancellation, where the fp32 kernels are at 1.5e-6 too).
    The stated bound for that mode is 3e-5 (tests/tools/debug_golden_tc.py prints the per-case numbers)."""
    tol = TOL if precision == "fp32" else TOL_TF32X3
    z = G.load(name)
    m, out = run_case(z, compact, precision)
    assert tuple(out.shape) == z["out"].shape
    assert G.rel_err(out.detach().cpu().numpy(), z["out"]) < tol
    check_grads(z, grads_of(m.fs), z["grad_fs"], "fs", tol)
    check_grads(z, grads_of(m.rho), z["grad_rho"], "rho", tol)
    if "grad_readout" in z:                                   # models.py NAM readout (readout_n_layers > 0)
        check_grads(z, grads_of(m.readout_nam.fs), z["grad_readout"], "readout", tol)


@pytest.mark.parametrize("name", G.PREPROCESS_CASES)
def test_apsp_bit_exact_vs_reference_golden(name):
    from gnan_b200.preprocess import apsp, from_reference_format
    z = G.load(name)
    n = int(z["meta"][0])
    hd = apsp(torch.tensor(z["edge_index"].reshape(2, -1)), n, device=DEV)
    nd, nm = hd.reference_format()
    assert np.array_equal(nd.cpu().numpy(), z["node_distances"])
    assert np.array_equal(nm.cpu().numpy(), z["normalization_matrix"])
    back = from_reference_format(torch.tensor(z["node_distances"], device=DEV), torch.tensor(z["normalization_matrix"], device=DEV))
    assert torch.equal(back.hop[:, :n], hd.hop[:, :n]) and torch.equal(back.level_counts, hd.level_counts)


def random_graph(rng, n, avg_deg=3.0, directed=False, n_isolated=0):
    m = n - n_isolated
    E = int(m * avg_deg / (1 if directed else 2))
    src = rng.integers(0, max(m, 1), size=E); dst = rng.integers(0, max(m, 1), size=E)
    keep = src != dst
    e = np.unique(np.stack([src[keep], dst[keep]], 1), axis=0)
    if not directed:
        e = np.unique(np.concatenate([e, e[:, ::-1]]), axis=0)
    return e.T.astype(np.int64).reshape(2, -1)


@pytest.mark.parametrize("method", ["warp", "msbfs"])
@pytest.mark.parametrize("n,deg,directed", [(1, 0, False), (2, 1, False), (257, 2.2, False), (1000, 3.0, True), (3001, 2.5, False),
                                            (5000, 1.6, True)])
def test_apsp_vs_oracle_random(n, deg, directed, method):
    from gnan_b200.preprocess import apsp
    rng = np.random.default_rng(n)
    ei = random_graph(rng, n, deg, directed, n_isolated=min(3, n - 1))
    hop = oapsp.apsp(ei, n)
    cnt = oapsp.level_counts(hop)
    hd = apsp(torch.tensor(ei), n, device=DEV, method=method)
    got = hd.hop[:, :n].cpu().numpy().astype(np.int32)
    got[got == 255] = -1
    assert np.array_equal(got, hop)
    assert np.array_equal(hd.level_counts.cpu().numpy(), cnt)
    # row-sharded call == slice of the full matrix
    if n > 10:
        part = apsp(torch.tensor(ei), n, device=DEV, row_begin=n // 3, row_end=n // 3 + 7, method=method)
        assert torch.equal(part.hop[:, :n], hd.hop[n // 3:n // 3 + 7, :n])
        assert torch.equal(part.level_counts[:, :-1], hd.level_counts[n // 3:n // 3 + 7, :part.level_counts.shape[1] - 1])


@pytest.mark.parametrize("method", ["warp", "msbfs"])
def test_apsp_path_graph_depth_limit(method):
    """uint8 hop matrix: depth 254 is the last one it represents; a deeper graph comes back in the int16 form (csrc/wide.cu; the
    reference has no depth limit)."""
    from gnan_b200.preprocess import apsp

    def path(n):
        a = np.arange(n - 1)
        return torch.tensor(np.stack([np.concatenate([a, a + 1]), np.concatenate([a + 1, a])]))
    hd = apsp(path(255), 255, device=DEV, method=method)
    i = torch.arange(255, device=DEV)
    assert torch.equal(hd.hop[:, :255].long(), (i[:, None] - i[None, :]).abs())
    assert hd.nbins == 256 and int(hd.level_counts[0, 254]) == 1 and int(hd.level_counts[:, -1].sum()) == 0
    deep = apsp(path(256), 256, device=DEV, method=method)
    j = torch.arange(256, device=DEV)
    assert deep.wide and deep.hop.dtype == torch.int16 and deep.nbins == 257
    assert torch.equal(deep.hop[:, :256].long(), (j[:, None] - j[None, :]).abs())
    assert int(deep.level_counts[0, 255]) == 1 and int(deep.level_counts[:, -1].sum()) == 0


@pytest.mark.parametrize("G_,H,C,L", [(5, 64, 3, 3), (7, 16, 2, 2), (3, 32, 4, 4), (4, 8, 2, 1)])
def test_mlp_input_gradient_vs_oracle(G_, H, C, L):
    """du of gnan_mlp_bwd (needed by the NAM readout, whose inputs are computed values) against autograd of the port."""
    from gnan_b200 import ops
    gen = torch.Generator().manual_seed(G_ * 100 + H)
    R = 300
    nh, Hh = max(L - 2, 0), (H if L >= 2 else 1)
    p = dict(w1=torch.randn(G_, Hh, generator=gen), b1=torch.randn(G_, Hh, generator=gen),
             wh=torch.randn(nh, G_, Hh, Hh, generator=gen) / Hh ** 0.5, bh=torch.randn(nh, G_, Hh, generator=gen) * 0.1,
             wo=torch.randn(G_, C, Hh, generator=gen) / Hh ** 0.5, bo=torch.randn(G_, C, generator=gen))
    if L == 1:
        p.update(w1=torch.zeros(0), b1=torch.zeros(0), wh=torch.zeros(0), bh=torch.zeros(0))
    u = torch.randn(R, G_, generator=gen)
    w = torch.randn(R, C, generator=gen)
    uo = u.clone().requires_grad_(True)
    q = {k: v.clone() for k, v in p.items()}
    if L == 1:
        q["w1"] = None
    want = gnan_port.shape_functions(q, uo).sum(dim=1)
    (want * w).sum().backward()
    ud = u.to(DEV).requires_grad_(True)
    d = {k: v.to(DEV).requires_grad_(True) for k, v in p.items()}
    got = ops.mlp(ud, d["w1"], d["b1"], d["wh"], d["bh"], d["wo"], d["bo"], L)
    (got * w.to(DEV)).sum().backward()
    assert G.rel_err(got.detach().cpu().numpy(), want.detach().numpy()) < TOL
    assert G.rel_err(ud.grad.cpu().numpy(), uo.grad.numpy()) < TOL


def test_build_csr_counting_sort():
    """csrc/csr.cu: rowptr exact, every row holds the right neighbour SET (order unspecified), status bits."""
    from gnan_b200.preprocess import build_csr
    rng = np.random.default_rng(3)
    n = 5000
    ei = random_graph(rng, n, 3.1, True, n_isolated=40)
    rowptr, col, st = build_csr(torch.tensor(ei), n, DEV)
    rp, cl = rowptr.cpu().numpy(), col.cpu().numpy()
    assert int(st.item()) == 0
    deg = np.bincount(ei[0], minlength=n)
    assert np.array_equal(rp, np.concatenate([[0], np.cumsum(deg)]))
    order = np.lexsort((ei[1], ei[0]))
    want = ei[1][order]
    got = np.concatenate([np.sort(cl[rp[i]:rp[i + 1]]) for i in range(n)])
    assert np.array_equal(got, want)
    dup = np.concatenate([ei, ei[:, 7:8]], axis=1)
    assert int(build_csr(torch.tensor(dup), n, DEV)[2].item()) == 2
    bad = ei.copy(); bad[1, 3] = n
    assert int(build_csr(torch.tensor(bad), n, DEV)[2].item()) & 1
    rowptr, col, st = build_csr(torch.zeros(2, 0, dtype=torch.long), 4, DEV)
    assert rowptr.tolist() == [0, 0, 0, 0, 0] and int(st.item()) == 0


@pytest.mark.parametrize("batched", [False, True])
def test_duplicate_edges_follow_the_reference_weighted_dijkstra(batched):
    """pre_process_datasets.py:109-110: the COO -> LIL conversion SUMS duplicate edges, Dijkstra then runs on weights 2, 3, ...
    Checked against scipy on the summed matrix (the reference's own two calls)."""
    import scipy.sparse as sp
    from scipy.sparse.csgraph import dijkstra
    from gnan_b200.preprocess import apsp, apsp_batched
    rng = np.random.default_rng(9)

    def graph(n):
        ei = random_graph(rng, n, 2.2, False, n_isolated=1)
        pick = rng.choice(ei.shape[1], size=max(2, ei.shape[1] // 6), replace=False)
        extra = np.concatenate([ei[:, pick], ei[:, pick[:2]]], axis=1)          # some edges twice, two of them three times
        return np.concatenate([ei, extra], axis=1)

    def want_of(ei, n):
        adj = sp.lil_matrix(sp.coo_matrix((np.ones(ei.shape[1]), (ei[0], ei[1])), shape=(n, n)))
        d = dijkstra(adj)
        return np.where(np.isinf(d), -1, d).astype(np.int32)

    if not batched:
        n = 300
        ei = graph(n)
        hd = apsp(torch.tensor(ei), n, device=DEV)
        got = hd.hop[:, :n].cpu().numpy().astype(np.int32); got[got == 255] = -1
        want = want_of(ei, n)
        assert np.array_equal(got, want)
        assert np.array_equal(hd.level_counts.cpu().numpy(), oapsp.level_counts(want, hd.nbins))
        nd, nm = hd.reference_format()
        wnd, wnm = oapsp.reference_format(want, oapsp.level_counts(want))
        assert np.array_equal(nd.cpu().numpy(), wnd) and np.array_equal(nm.cpu().numpy(), wnm)
    else:
        sizes = [12, 40, 7]
        node_off = np.concatenate([[0], np.cumsum(sizes)])
        eis = [graph(n) for n in sizes]
        ei = np.concatenate([e + node_off[i] for i, e in enumerate(eis)], axis=1)
        pk = apsp_batched(torch.tensor(ei), node_off, device=DEV)
        hop, ho = pk.hop.cpu().numpy(), pk.hop_off.cpu().numpy()
        for i, n in enumerate(sizes):
            got = hop[ho[i]:ho[i + 1]].reshape(n, n).astype(np.int32); got[got == 255] = -1
            assert np.array_equal(got, want_of(eis[i], n)), i


@pytest.mark.parametrize("directed", [False, True])
def test_apsp_batched_small_graph_kernel_vs_oracle(directed):
    """graphs of <= 128 nodes take the bit-parallel-over-sources kernel (hop block assembled in shared memory, written once);
    includes a path deeper than the narrow first-try level table (redo with the full width) and ragged block alignments."""
    from gnan_b200.preprocess import apsp_batched
    rng = np.random.default_rng(17)
    sizes = [1, 2, 5, 31, 32, 33, 64, 100, 17, 128, 3, 70, 9]
    node_off = np.concatenate([[0], np.cumsum(sizes)])
    eis = [random_graph(rng, n, 2.2, directed, n_isolated=1 if n > 4 else 0) for n in sizes]
    for deep in (False, True):
        if deep:                                            # graph 6 (64 nodes) becomes a path: hop distances up to 63
            eis[6] = np.stack([np.arange(63), np.arange(1, 64)]) if directed else np.concatenate(
                [np.stack([np.arange(63), np.arange(1, 64)]), np.stack([np.arange(1, 64), np.arange(63)])], axis=1)
        ei = np.concatenate([e + node_off[i] for i, e in enumerate(eis)], axis=1)
        pk = apsp_batched(torch.tensor(ei), node_off, device=DEV)
        hop, cnt, ho = pk.hop.cpu().numpy(), pk.level_counts.cpu().numpy(), pk.hop_off.cpu().numpy()
        assert not deep or cnt.shape[1] == 65
        for i, n in enumerate(sizes):
            want = oapsp.apsp(eis[i], n)
            got = hop[ho[i]:ho[i + 1]].reshape(n, n).astype(np.int32)
            got[got == 255] = -1
            assert np.array_equal(got, want), (i, deep)
            wc = oapsp.level_counts(want)
            full = np.zeros((n, cnt.shape[1]), dtype=np.int32)
            full[:, :wc.shape[1] - 1] = wc[:, :-1]; full[:, -1] = wc[:, -1]
            assert np.array_equal(cnt[node_off[i]:node_off[i + 1]], full), (i, deep)


@pytest.mark.parametrize("max_n", [31, 95, 27])
def test_apsp_batched_odd_maximum_sizes(max_n):
    """odd max_n with an odd number of source words (31 -> 1 word, 95 -> 3 words): the per-warp shared-memory slices of the
    small-graph kernel must stay 16-byte aligned (a Mutagenicity-shaped batch whose largest graph had 95 nodes faulted)."""
    from gnan_b200.preprocess import apsp_batched
    rng = np.random.default_rng(max_n)
    sizes = [max_n] + [int(v) for v in rng.integers(1, max_n + 1, size=40)]
    node_off = np.concatenate([[0], np.cumsum(sizes)])
    eis = [random_graph(rng, n, 2.2, False, n_isolated=1 if n > 4 else 0) for n in sizes]
    ei = np.concatenate([e + node_off[i] for i, e in enumerate(eis)], axis=1)
    pk = apsp_batched(torch.tensor(ei), node_off, device=DEV)
    hop, ho = pk.hop.cpu().numpy(), pk.hop_off.cpu().numpy()
    for i, n in enumerate(sizes):
        got = hop[ho[i]:ho[i + 1]].reshape(n, n).astype(np.int32)
        got[got == 255] = -1
        assert np.array_equal(got, oapsp.apsp(eis[i], n)), i


@pytest.mark.parametrize("directed,lo,hi", [(False, 1, 128), (True, 1, 128), (False, 1, 32), (False, 30, 64), (False, 60, 100)])
def test_apsp_batched_grouped_warps_many_graphs(directed, lo, hi):
    """The 4-warp-group kernel (graphs of 65..128 nodes on a whole group, 33..64 on warp pairs, <= 32 on single warps) on a batch
    with odd class sizes, hubs of more than 8 neighbours and isolated vertices: hop blocks and level sizes against the C oracle,
    and the fused 1/count table (fixed-width mode) against the counts."""
    from gnan_b200.preprocess import apsp_batched, check_batched_status
    rng = np.random.default_rng(lo * 1000 + hi + int(directed))
    sizes = [int(v) for v in rng.integers(lo, hi + 1, size=301)] + [hi, lo]
    node_off = np.concatenate([[0], np.cumsum(sizes)])
    eis = []
    for n in sizes:
        e = random_graph(rng, n, 2.6, directed, n_isolated=1 if n > 4 else 0)
        if n > 12:                                                  # a hub: vertex 0 linked to 11 others (rows longer than the register cache)
            tgt = rng.choice(np.arange(1, n), size=11, replace=False)
            hub = np.stack([np.zeros(11, dtype=np.int64), tgt])
            e = np.unique(np.concatenate([e, hub, hub[::-1]] if not directed else [e, hub], axis=1).T, axis=0).T
        eis.append(e)
    ei = torch.tensor(np.concatenate([e + node_off[i] for i, e in enumerate(eis)], axis=1))
    pk = apsp_batched(ei, node_off, device=DEV)
    hop, cnt, ho = pk.hop.cpu().numpy(), pk.level_counts.cpu().numpy(), pk.hop_off.cpu().numpy()
    for i, n in enumerate(sizes):
        want = oapsp.apsp(eis[i], n)
        got = hop[ho[i]:ho[i + 1]].reshape(n, n).astype(np.int32)
        got[got == 255] = -1
        assert np.array_equal(got, want), i
        wc = oapsp.level_counts(want)
        full = np.zeros((n, cnt.shape[1]), dtype=np.int32)
        full[:, :wc.shape[1] - 1] = wc[:, :-1]; full[:, -1] = wc[:, -1]
        assert np.array_equal(cnt[node_off[i]:node_off[i + 1]], full), i
    fx = apsp_batched(ei, node_off, device=DEV, nbins=130, rscale=True)
    check_batched_status(fx.status)
    assert torch.equal(fx.hop, pk.hop)
    wide = torch.zeros(cnt.shape[0], 130, dtype=torch.float32)
    c = torch.tensor(cnt).float()
    wide[:, :cnt.shape[1] - 1] = c[:, :-1]; wide[:, -1] = c[:, -1]
    want_rs = torch.where(wide > 0, 1.0 / wide, torch.zeros_like(wide))
    assert torch.equal(fx.level_rscale.cpu(), want_rs)
    # the same batch from its transfer form (no CSR: adjacency bit matrices built in shared memory from the edge segments)
    from gnan_b200.preprocess import LocalEdges
    le = LocalEdges.from_edge_index(ei, node_off).to(DEV)
    lp = apsp_batched(le, node_off, device=DEV)
    assert torch.equal(lp.hop, pk.hop) and torch.equal(lp.level_counts, pk.level_counts)
    lf = apsp_batched(le, node_off, device=DEV, nbins=130, rscale=True)
    check_batched_status(lf.status)
    assert torch.equal(lf.hop, pk.hop) and torch.equal(lf.level_rscale, fx.level_rscale)


def test_apsp_batched_local_edges_flags_duplicates_and_bad_endpoints():
    """gnan_apsp_bfs_batched_local reports gnan_build_csr's status bits: a repeated (src,dst) pair (the caller then takes the
    multi-edge path and reproduces the reference's summed weights) and an endpoint outside the graph (edge dropped)."""
    from gnan_b200.preprocess import LocalEdges, apsp_batched
    rng = np.random.default_rng(12)
    sizes = [12, 40, 7, 100]
    node_off = np.concatenate([[0], np.cumsum(sizes)])
    eis = [random_graph(rng, n, 2.2, False, n_isolated=1) for n in sizes]
    eis[1] = np.concatenate([eis[1], eis[1][:, :3]], axis=1)                      # three edges of graph 1 twice
    ei = torch.tensor(np.concatenate([e + node_off[i] for i, e in enumerate(eis)], axis=1))
    a = apsp_batched(ei, node_off, device=DEV)
    b = apsp_batched(LocalEdges.from_edge_index(ei, node_off), node_off, device=DEV)
    assert torch.equal(a.hop, b.hop) and torch.equal(a.level_counts, b.level_counts)
    fx = apsp_batched(LocalEdges.from_edge_index(ei, node_off), node_off, device=DEV, nbins=48)
    assert int(fx.status[0]) & 2                                                  # duplicates flagged in the sync-free mode
    clean = torch.tensor(np.concatenate([e + node_off[i] for i, e in enumerate(eis) if i != 1], axis=1))
    le = LocalEdges.from_edge_index(clean, node_off)
    le.dst[0] = 200                                                               # endpoint beyond its graph's 12 nodes
    fx = apsp_batched(le, node_off, device=DEV, nbins=48)
    assert int(fx.status[0]) == 1


def test_apsp_batched_vs_oracle():
    from gnan_b200.preprocess import apsp_batched
    rng = np.random.default_rng(5)
    sizes = [1, 2, 5, 31, 32, 33, 64, 100, 17, 256, 3]
    node_off = np.concatenate([[0], np.cumsum(sizes)])
    eis = [random_graph(rng, n, 2.4, False, n_isolated=1 if n > 4 else 0) + node_off[i] for i, n in enumerate(sizes)]
    ei = np.concatenate(eis, axis=1)
    pk = apsp_batched(torch.tensor(ei), torch.tensor(node_off), device=DEV)
    hop = pk.hop.cpu().numpy(); cnt = pk.level_counts.cpu().numpy(); ho = pk.hop_off.cpu().numpy()
    for i, n in enumerate(sizes):
        want = oapsp.apsp(eis[i] - node_off[i], n)
        got = hop[ho[i]:ho[i + 1]].reshape(n, n).astype(np.int32)
        got[got == 255] = -1
        assert np.array_equal(got, want), i
        wc = oapsp.level_counts(want, cnt.shape[1]) if want.max() + 2 <= cnt.shape[1] else None
        wc = oapsp.level_counts(want)
        full = np.zeros((n, cnt.shape[1]), dtype=np.int32)
        full[:, :wc.shape[1] - 1] = wc[:, :-1]; full[:, -1] = wc[:, -1]
        assert np.array_equal(cnt[node_off[i]:node_off[i + 1]], full), i


# ---- kernel-level: grouped MLP ------------------------------------------------------------------------------------------
def rand_mlp(rng, G_, H, C, L, bias=True):
    g = lambda *s: torch.tensor(rng.normal(size=s)).float()
    if L == 1:
        return dict(w1=torch.zeros(0), b1=torch.zeros(0), wh=torch.zeros(0), bh=torch.zeros(0), wo=g(G_, C, 1), bo=g(G_, C) * 0.3 * bias)
    nh = L - 2
    return dict(w1=g(G_, H), b1=g(G_, H) * 0.3 * bias, wh=g(nh, G_, H, H) / H ** 0.5 * 1.3, bh=g(nh, G_, H) * 0.3 * bias,
                wo=g(G_, C, H) / H ** 0.5, bo=g(G_, C) * 0.3 * bias)


def relu_margin(p, u):
    """smallest |pre-activation| over all rows, groups, layers and units, in float64"""
    h = u.double().unsqueeze(-1) * p["w1"].double() + p["b1"].double()
    m = float(h.abs().min())
    h = torch.relu(h)
    for l in range(p["wh"].shape[0]):
        h = torch.einsum("nki,kji->nkj", h, p["wh"][l].double()) + p["bh"][l].double()
        m = min(m, float(h.abs().min()))
        h = torch.relu(h)
    return m


def preact_margin_per_input(p, u):
    """[R,G] smallest |pre-activation| over layers and units for every scalar input, in float64"""
    h = u.double().unsqueeze(-1) * p["w1"].double() + p["b1"].double()
    m = h.abs().amin(-1)
    h = torch.relu(h)
    for l in range(p["wh"].shape[0]):
        h = torch.einsum("nki,kji->nkj", h, p["wh"][l].double()) + p["bh"][l].double()
        m = torch.minimum(m, h.abs().amin(-1))
        h = torch.relu(h)
    return m


def kink_free_inputs(rng, p, R, G_, margin, L):
    """Inputs u [R,G] (30 % exact zeros) none of whose float64 pre-activations is within `margin` of a ReLU kink: a
    pre-activation inside the rounding noise of 0 flips a mask between two correct implementations and moves a gradient by
    a whole term (the reference has the same property), so parity is only well-posed away from kinks. Offending entries
    are redrawn individually."""
    u = torch.tensor(rng.normal(size=(R, G_)) * (rng.random((R, G_)) < 0.7)).float()
    if L == 1:
        return u
    for _ in range(100):
        bad = preact_margin_per_input(p, u) <= margin
        n = int(bad.sum())
        if n == 0:
            return u
        u[bad] = torch.tensor(rng.normal(size=n)).float()
    raise AssertionError("could not build kink-free inputs")


def dropout_masks(seed, p_drop, layer, G_, R, H):
    """numpy port of gnan_dropout_mul (csrc/common.cuh): splitmix64 over key = ((layer*G+g)*R+row)*H+unit -> [R,G,H] multipliers"""
    with np.errstate(over="ignore"):
        g, r, h = np.meshgrid(np.arange(G_, dtype=np.uint64), np.arange(R, dtype=np.uint64), np.arange(H, dtype=np.uint64), indexing="ij")
        key = ((np.uint64(layer) * np.uint64(G_) + g) * np.uint64(R) + r) * np.uint64(H) + h
        z = np.uint64(seed) + key * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
        bits = (z >> np.uint64(32)).astype(np.uint64)
    thresh = np.uint64(min(max(int(float(np.float32(p_drop)) * 4294967296.0), 0), 4294967295))
    keep = bits >= thresh
    scale = float(np.float32(1.0) / (np.float32(1.0) - np.float32(p_drop)))
    return torch.tensor(np.transpose(keep, (1, 0, 2)).astype(np.float64) * scale)      # [R,G,H]


def oracle_params(p, L):
    q = {k: v.double().clone().requires_grad_(v.numel() > 0) for k, v in p.items()}
    if L == 1:
        q["w1"] = None
    return q


@pytest.mark.parametrize("R,G_,H,C,L", [
    (1, 1, 64, 1, 3), (127, 3, 64, 7, 3), (300, 15, 64, 1, 3), (1000, 40, 64, 3, 3), (257, 5, 32, 4, 3),
    (130, 4, 16, 8, 2), (64, 3, 8, 2, 4), (90, 3, 64, 40, 3), (77, 6, 16, 9, 5), (50, 4, 64, 3, 1),
    (4000, 70, 64, 7, 3)])
def test_mlp_kernel_vs_oracle(R, G_, H, C, L):
    from gnan_b200 import ops
    rng = np.random.default_rng(R * 7 + G_)
    p = rand_mlp(rng, G_, H, C, L)
    u = kink_free_inputs(rng, p, R, G_, 2e-6, L)
    dS = torch.tensor(rng.normal(size=(R, C))).float()
    q = oracle_params(p, L)
    want = gnan_lut.feature_sums(q, u.double())
    (want * dS.double()).sum().backward()
    d = {k: v.to(DEV).requires_grad_(v.numel() > 0) for k, v in p.items()}
    got = ops.mlp(u.to(DEV), d["w1"], d["b1"], d["wh"], d["bh"], d["wo"], d["bo"], L)
    (got * dS.to(DEV)).sum().backward()
    assert G.rel_err(got.detach().cpu().numpy(), want.detach().numpy()) < TOL
    for k in p:
        if p[k].numel() and q[k] is not None:
            gk, wk = d[k].grad.cpu().numpy(), q[k].grad.numpy()
            if k == "bo":       # d bo = column sums of dS, which may cancel to ~0: scale the error by the summands, not the sum
                assert np.linalg.norm(gk - wk) < TOL * max(np.linalg.norm(wk), float(dS.norm())), k
            else:
                assert G.rel_err(gk, wk) < TOL, k


@pytest.mark.parametrize("precision", ["fp32", "tf32x3"])
def test_mlp_dropout_matches_oracle_with_the_same_masks(precision):
    """The counter-based masks are reproducible on the host (splitmix64), so dropout is checked exactly: float64 oracle with
    the same masks, forward and backward, both kernel paths."""
    from gnan_b200 import ops
    rng = np.random.default_rng(12)
    R, G_, H, C, L, pd, seed = 300, 4, 64, 3, 3, 0.5, 1234
    p = rand_mlp(rng, G_, H, C, L)
    m0 = dropout_masks(seed, pd, 0, G_, R, H); m1 = dropout_masks(seed, pd, 1, G_, R, H)
    assert 0.45 < float((m0 > 0).double().mean()) < 0.55

    def oracle(q, u):
        h = torch.relu(u.double().unsqueeze(-1) * q["w1"] + q["b1"]) * m0
        z = torch.einsum("nki,kji->nkj", h, q["wh"][0]) + q["bh"][0]
        return torch.einsum("nkj,kcj->nc", torch.relu(z) * m1, q["wo"]) + q["bo"].sum(0), z

    u = torch.tensor(rng.normal(size=(R, G_))).float()
    for _ in range(100):                                   # keep z2 away from its kinks (layer-1 kinks: |x w1 + b1|)
        q = oracle_params(p, L)
        _, z = oracle(q, u)
        z1 = u.double().unsqueeze(-1) * q["w1"] + q["b1"]
        bad = (torch.minimum(z.abs().amin(-1), z1.abs().amin(-1)) <= 2e-5).detach()
        if not bad.any():
            break
        u[bad] = torch.tensor(rng.normal(size=int(bad.sum()))).float()
    dS = torch.tensor(rng.normal(size=(R, C))).float()
    q = oracle_params(p, L)
    want, _ = oracle(q, u)
    (want * dS.double()).sum().backward()
    d = {k: v.to(DEV).requires_grad_(True) for k, v in p.items()}
    got = ops.mlp(u.to(DEV), d["w1"], d["b1"], d["wh"], d["bh"], d["wo"], d["bo"], L, dropout_p=pd, seed=seed, precision=precision)
    (got * dS.to(DEV)).sum().backward()
    assert G.rel_err(got.detach().cpu().numpy(), want.detach().numpy()) < TOL
    for k in p:
        assert G.rel_err(d[k].grad.cpu().numpy(), q[k].grad.numpy()) < TOL, k
    again = ops.mlp(u.to(DEV), d["w1"], d["b1"], d["wh"], d["bh"], d["wo"], d["bo"], L, dropout_p=pd, seed=seed, precision=precision)
    other = ops.mlp(u.to(DEV), d["w1"], d["b1"], d["wh"], d["bh"], d["wo"], d["bo"], L, dropout_p=pd, seed=seed + 1, precision=precision)
    assert torch.equal(again, got) and not torch.equal(other, got)


# ---- kernel-level: aggregation -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("R,N,C,Cr,nbins,per_row,scale", [
    (5, 7, 1, 1, 3, False, False), (37, 100, 3, 3, 6, True, False), (64, 2500, 7, 7, 12, False, True),
    (33, 4099, 4, 1, 40, False, True), (20, 300, 2, 2, 70, True, True), (129, 515, 40, 40, 9, False, False),
    (300, 300, 5, 1, 5, True, False),
    # nbins 210 / 211 / 256 with 4-channel chunks: two lane-private bin copies per warp up to 210, one from 211 on
    (24, 300, 4, 4, 210, False, True), (24, 300, 4, 1, 211, True, True), (12, 4099, 4, 4, 256, False, True),
    (17, 530, 5, 5, 211, False, True), (17, 530, 5, 1, 256, True, True),
    (9, 260, 40, 40, 210, True, True), (9, 260, 40, 40, 211, False, True), (9, 260, 40, 40, 256, True, True)])
def test_aggregate_rows_vs_oracle(R, N, C, Cr, nbins, per_row, scale):
    from gnan_b200 import ops
    rng = np.random.default_rng(R + N)
    h = rng.integers(0, nbins, size=(R, N))
    hop = ops.alloc_hop(R, N, DEV)
    hb = h.copy(); hb[hb == nbins - 1] = 255
    hop[:, :N] = torch.tensor(hb.astype(np.uint8), device=DEV)
    T = torch.tensor(rng.normal(size=((R, nbins, Cr) if per_row else (nbins, Cr)))).float()
    S = torch.tensor(rng.normal(size=(N, C))).float()
    rs = torch.tensor(rng.random(size=(R, nbins)) + 0.1).float() if scale else None
    gO = torch.tensor(rng.normal(size=(R, C))).float()
    Td, Sd = T.double().requires_grad_(True), S.double().requires_grad_(True)
    idx = torch.tensor(h)
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
    with torch.no_grad():                                   # inference path (no bin sums saved)
        assert torch.equal(ops.aggregate_rows(hop, Tg, Sg, rscale=None if rs is None else rs.to(DEV), per_row=per_row), got.detach())
        # backward without saved bin sums: rebuilt by one extra forward pass
        dS, dT = ops.agg_rows_bwd(hop, Tg, None if rs is None else rs.to(DEV), Sg, per_row, gO.to(DEV), torch.empty(0, device=DEV))
    assert G.rel_err(dS.cpu().numpy(), Sd.grad.numpy()) < TOL
    assert G.rel_err(dT.cpu().numpy(), Td.grad.numpy()) < TOL


# tensor-core form (csrc/agg_tc.cu): TMA-streamed hop tiles, on-the-fly 0/1 operand in TMEM, tcgen05 kind::i8 against the
# digit matrix of S. NB = 8 / 16 / 32 bin slots, 1 / 2 / 4 generator groups (by accumulator width), ragged R and N.
@pytest.mark.parametrize("R,N,C,Cr,nbins,per_row,scale", [
    (37, 300, 3, 3, 6, True, False), (64, 2500, 7, 7, 12, False, True), (33, 4099, 4, 1, 16, False, True),
    (20, 1000, 2, 2, 17, True, True), (129, 515, 40, 40, 9, False, False), (300, 700, 5, 1, 32, True, False),
    (50, 260, 1, 1, 3, False, False), (70, 900, 64, 64, 14, True, True), (1, 256, 3, 3, 8, True, False),
    # 10 / 12 / 14 lanes per row (tensor-bound shapes: >= 64 digit columns), 1-3 generator groups, ragged row tiles
    (200, 3000, 40, 40, 12, True, False), (91, 1500, 16, 16, 11, False, True), (45, 700, 20, 1, 13, True, True),
    (23, 1029, 33, 33, 10, True, False)])
def test_aggregate_rows_tensor_core_vs_oracle(R, N, C, Cr, nbins, per_row, scale):
    from gnan_b200 import ops
    rng = np.random.default_rng(R * 7 + N)
    h = rng.integers(0, nbins, size=(R, N))
    hop = torch.randint(0, 256, (R, ops.hop_ld(N)), dtype=torch.uint8, device=DEV)      # padding columns hold garbage
    hb = h.copy(); hb[hb == nbins - 1] = 255
    hop[:, :N] = torch.tensor(hb.astype(np.uint8), device=DEV)
    T = torch.tensor(rng.normal(size=((R, nbins, Cr) if per_row else (nbins, Cr)))).float()
    S = torch.tensor(rng.normal(size=(N, C)) * np.exp(rng.normal(size=(N, 1)) * 2)).float()   # magnitudes over ~4 decades
    rs = torch.tensor(rng.random(size=(R, nbins)) + 0.1).float() if scale else None
    gO = torch.tensor(rng.normal(size=(R, C))).float()
    Td, Sd = T.double().requires_grad_(True), S.double().requires_grad_(True)
    idx = torch.tensor(h)
    W = (torch.gather(Td, 1, idx.unsqueeze(-1).expand(-1, -1, Cr)) if per_row else Td[idx])
    if scale:
        W = W * torch.gather(rs.double(), 1, idx).unsqueeze(-1)
    want = (W * Sd.unsqueeze(0)).sum(1)
    (want * gO.double()).sum().backward()
    Tg, Sg = T.to(DEV).requires_grad_(True), S.to(DEV).requires_grad_(True)
    got = ops.aggregate_rows(hop, Tg, Sg, rscale=None if rs is None else rs.to(DEV), per_row=per_row, algo="tc")
    (got * gO.to(DEV)).sum().backward()
    assert G.rel_err(got.detach().cpu().numpy(), want.detach().numpy()) < TOL
    assert G.rel_err(Sg.grad.cpu().numpy(), Sd.grad.numpy()) < TOL
    assert G.rel_err(Tg.grad.cpu().numpy(), Td.grad.numpy()) < TOL
    # exact integer accumulation: bit-identical on a second run and under a column permutation of (hop, S)
    with torch.no_grad():
        again = ops.aggregate_rows(hop, Tg, Sg, rscale=None if rs is None else rs.to(DEV), per_row=per_row, algo="tc")
        assert torch.equal(again, got.detach())
        perm = torch.randperm(N, device=DEV)
        hop_p = hop.clone(); hop_p[:, :N] = hop[:, :N][:, perm]
        permuted = ops.aggregate_rows(hop_p, Tg, Sg[perm].contiguous(), rscale=None if rs is None else rs.to(DEV), per_row=per_row, algo="tc")
        assert torch.equal(permuted, got.detach())


@pytest.mark.parametrize("C", [5, 40])
def test_aggregate_rows_tensor_core_backward_keeps_weight_gradient_accuracy(C):
    """The quantisation error of T*g is shared by every column of a hop level, so sums of dS over many columns (what every
    shape-function weight gradient is: d bo = sum_j dS[j]) amplify it by the level size. With 3 digits this was 1.4e-4 at
    C = 5; the backward carries 4 digits. Checked: dS norm-wise AND its column sums against float64."""
    from gnan_b200 import ops
    rng = np.random.default_rng(C)
    R = N = 3000
    nbins = 9
    p = np.array([0.0004, 0.004, 0.03, 0.15, 0.4, 0.3, 0.1, 0.0156, 0.0])        # level sizes like a small-world graph
    h = rng.choice(nbins, size=(R, N), p=p / p.sum())
    hop = ops.alloc_hop(R, N, DEV)
    hop[:, :N] = torch.tensor(h.astype(np.uint8), device=DEV)
    T = torch.tensor(rng.normal(size=(R, nbins, C))).float()
    S = torch.tensor(rng.normal(size=(N, C))).float()
    gO = torch.tensor(rng.normal(size=(R, C))).float()
    gO[torch.tensor(rng.random(R) > 0.1)] = 0.0                                      # a 10 % train mask
    idx = torch.tensor(h)
    act = gO.abs().sum(1) > 0
    W = torch.gather(T[act].double(), 1, idx[act].unsqueeze(-1).expand(-1, -1, C))   # [Ract, N, C]
    dS64 = (W * gO[act].double().unsqueeze(1)).sum(0)                                # [N, C]
    Tg, Sg = T.to(DEV).requires_grad_(True), S.to(DEV).requires_grad_(True)
    got = ops.aggregate_rows(hop, Tg, Sg, per_row=True, algo="tc")
    (got * gO.to(DEV)).sum().backward()
    dS = Sg.grad.double().cpu()
    W0 = torch.gather(T[:200].double(), 1, idx[:200].unsqueeze(-1).expand(-1, -1, C))
    out64 = (W0 * S.double().unsqueeze(0)).sum(1)                                    # forward (3 digits of S at C = 5, 40), first rows
    assert G.rel_err(got[:200].detach().double().cpu().numpy(), out64.numpy()) < TOL
    assert G.rel_err(dS.numpy(), dS64.numpy()) < TOL
    assert G.rel_err(dS.sum(0).numpy(), dS64.sum(0).numpy()) < TOL
    wts = torch.tensor(rng.random(size=(N, 1))).double()                              # a positive-weight functional (like d wo)
    assert G.rel_err((dS * wts).sum(0).numpy(), (dS64 * wts).sum(0).numpy()) < TOL


def test_aggregate_rows_tensor_core_refuses_uncovered_shapes():
    from gnan_b200 import ops
    hop = ops.alloc_hop(8, 300, DEV)
    with pytest.raises(NotImplementedError):
        ops.aggregate_rows(hop, torch.zeros(40, 1, device=DEV), torch.zeros(300, 1, device=DEV), algo="tc")     # nbins > 32
    out = ops.aggregate_rows(hop, torch.ones(40, 1, device=DEV), torch.ones(300, 1, device=DEV))                  # auto -> CUDA cores
    assert float(out[0, 0]) == 300.0


def test_blockdiag_equals_per_graph_dense_rows():
    """Property (SURVEY §4): the block-diagonal batch equals looping the dense-row kernel over graphs."""
    from gnan_b200 import ops
    from gnan_b200.preprocess import apsp, apsp_batched
    rng = np.random.default_rng(11)
    sizes = [4, 30, 9, 64, 120, 1]
    node_off = np.concatenate([[0], np.cumsum(sizes)])
    eis = [random_graph(rng, n, 2.3, False, n_isolated=1 if n > 8 else 0) for n in sizes]
    ei = np.concatenate([e + node_off[i] for i, e in enumerate(eis)], axis=1)
    pk = apsp_batched(torch.tensor(ei), torch.tensor(node_off), device=DEV)
    C, nb = 3, pk.nbins
    T = torch.tensor(rng.normal(size=(nb, C))).float().to(DEV).requires_grad_(True)
    S = torch.tensor(rng.normal(size=(node_off[-1], C))).float().to(DEV).requires_grad_(True)
    rs = ops.level_rscale(pk.level_counts)
    for reduce_graph in (True, False):
        out = ops.aggregate_blockdiag(pk.hop, pk.hop_off, pk.node_off, T, S, rscale=rs, reduce_graph=reduce_graph)
        w = torch.tensor(rng.normal(size=tuple(out.shape))).float().to(DEV)
        gT, gS = torch.autograd.grad((out * w).sum(), (T, S))
        ref = []
        for i, n in enumerate(sizes):
            hd = apsp(torch.tensor(eis[i]), n, device=DEV)
            cnt = torch.zeros(n, nb, dtype=torch.int32, device=DEV)
            cnt[:, :hd.nbins - 1] = hd.level_counts[:, :-1]; cnt[:, -1] = hd.level_counts[:, -1]
            o = ops.aggregate_rows(hd.hop, T, S[node_off[i]:node_off[i + 1]].contiguous(), rscale=ops.level_rscale(cnt))
            ref.append(o.sum(0, keepdim=True) if reduce_graph else o)
        ref = torch.cat(ref)
        rT, rS = torch.autograd.grad((ref * w).sum(), (T, S))
        assert G.rel_err(out.detach().cpu().numpy(), ref.detach().cpu().numpy()) < TOL
        assert G.rel_err(gT.cpu().numpy(), rT.cpu().numpy()) < TOL and G.rel_err(gS.cpu().numpy(), rS.cpu().numpy()) < TOL


def test_readout_packed_batch_equals_per_graph_forward():
    """models.TensorGNAN with the NAM readout: the packed many-graph call equals the reference-shaped per-graph forward
    (rows of the [B,C] result == each graph's out.T), outputs and parameter gradients."""
    from gnan_b200.models import TensorGNAN
    from gnan_b200.preprocess import apsp, apsp_batched
    rng = np.random.default_rng(21)
    sizes = [5, 17, 40, 3, 26]
    K, C = 6, 3
    node_off = np.concatenate([[0], np.cumsum(sizes)])
    eis = [random_graph(rng, n, 2.2, False, n_isolated=1 if n > 8 else 0) for n in sizes]
    ei = np.concatenate([e + node_off[i] for i, e in enumerate(eis)], axis=1)
    x = torch.tensor(rng.normal(size=(node_off[-1], K))).float()
    torch.manual_seed(1)
    m = TensorGNAN(K, C, 3, 64, is_graph_task=True, readout_n_layers=2).to(DEV)
    m.fs.xavier_normal_(1.0); m.rho.xavier_normal_(1.0); m.readout_nam.fs.xavier_normal_(1.0)
    pk = apsp_batched(torch.tensor(ei), torch.tensor(node_off), device=DEV)
    pk.x = x.to(DEV)
    w = torch.tensor(rng.normal(size=(len(sizes), C))).float().to(DEV)
    out = m(pk)
    assert tuple(out.shape) == (len(sizes), C)
    params = list(m.parameters())
    g_pk = torch.autograd.grad((out * w).sum(), params)
    ref = []
    for i, n in enumerate(sizes):
        d = SimpleNamespace(x=x[node_off[i]:node_off[i + 1]], hop_data=apsp(torch.tensor(eis[i]), n, device=DEV))
        o = m.forward(d)
        assert tuple(o.shape) == (C, 1)
        ref.append(o.T)
    ref = torch.cat(ref)
    g_ref = torch.autograd.grad((ref * w).sum(), params)
    assert G.rel_err(out.detach().cpu().numpy(), ref.detach().cpu().numpy()) < TOL
    for a, b in zip(g_pk, g_ref):
        assert G.rel_err(a.cpu().numpy(), b.cpu().numpy()) < TOL


def test_node_order_permutation_equivariance():
    """Property: relabelling nodes permutes the node-level output rows and leaves parameter gradients unchanged."""
    from gnan_b200.GNAN import TensorGNAN
    from gnan_b200.preprocess import apsp
    rng = np.random.default_rng(3)
    n, K, C = 150, 6, 4
    ei = random_graph(rng, n, 2.5, False, n_isolated=2)
    x = torch.tensor(rng.normal(size=(n, K))).float()
    perm = rng.permutation(n); inv = np.argsort(perm)
    torch.manual_seed(0)
    m = TensorGNAN(K, C, 3, 64).to(DEV)
    m.fs.xavier_normal_(1.0); m.rho.xavier_normal_(1.0)
    d1 = SimpleNamespace(x=x, hop_data=apsp(torch.tensor(ei), n, device=DEV))
    d2 = SimpleNamespace(x=x[perm], hop_data=apsp(torch.tensor(inv[ei]), n, device=DEV))
    o1 = m.forward(d1); o2 = m.forward(d2)
    assert G.rel_err(o2.detach().cpu().numpy(), o1.detach().cpu().numpy()[perm]) < TOL


def test_large_row_block_vs_lut_oracle():
    """PubMed-like row block (the shipped forward cannot run at this shape: SURVEY §8c) against the float64 LUT oracle."""
    from gnan_b200.models import GNAN
    from gnan_b200.preprocess import apsp
    rng = np.random.default_rng(8)
    n, K, C = 5000, 33, 3
    ei = random_graph(rng, n, 2.4, True, n_isolated=20)
    x = torch.tensor(rng.random(size=(n, K)) * (rng.random((n, K)) < 0.1)).float()
    torch.manual_seed(1)
    m = GNAN(K, C, num_layers=3, hidden_channels=64, rho_per_feature=True).to(DEV)
    ids = list(range(100, 164))
    hd = apsp(torch.tensor(ei), n, device=DEV)
    out = m.forward(SimpleNamespace(x=x, hop_data=hd), ids)
    w = torch.tensor(rng.normal(size=tuple(out.shape))).float()
    (out * w.to(DEV)).sum().backward()
    hop = torch.tensor(oapsp.apsp(ei, n)).long()
    cnt = gnan_lut.counts_from_hops(hop)
    assert torch.equal(cnt.int(), hd.level_counts.cpu())
    from oracle import params as P
    sd = {k: v.detach().cpu().numpy() for k, v in m.state_dict().items()}
    fs = gnan_port.to_torch(P.stack_mlps(sd, [f"fs.{k}" for k in range(K)], 3, 3), torch.float64, True)
    rho = gnan_port.to_torch(P.stack_mlps(sd, ["rho"], 3, 2), torch.float64, True)
    want = gnan_lut.forward_rows(fs, rho, x.double(), hop[ids], cnt[ids], "output")
    (want * w.double()).sum().backward()
    assert G.rel_err(out.detach().cpu().numpy(), want.detach().numpy()) < TOL
    assert G.rel_err(m.fs.wh.grad.cpu().numpy(), fs["wh"].grad.numpy()) < TOL
    assert G.rel_err(m.rho.wo.grad.cpu().numpy(), rho["wo"].grad.numpy()) < TOL


# ---- tensor-core (tcgen05) path of the grouped MLP -------------------------------------------------------------------
@pytest.mark.parametrize("precision,tol,gtol", [("tf32x3", 1e-5, 1e-5), ("tf32", 5e-3, 5e-2)])
@pytest.mark.parametrize("R,G_,C", [(1, 1, 1), (128, 2, 3), (129, 9, 7), (300, 15, 1), (1000, 40, 4), (1100, 6, 7), (5000, 3, 8),
                                    (700, 5, 9), (513, 4, 16), (900, 3, 40), (1300, 9, 33), (300, 2, 64)])
def test_mlp_tensor_core_vs_oracle(R, G_, C, precision, tol, gtol):
    """Forward and backward on tcgen05. The 3xTF32 split keeps fp32-level accuracy: bound 1e-5 for outputs AND gradients
    (measured 7e-7 / 3e-6). Single-pass tf32 has the stated looser bounds 5e-3 (outputs) / 5e-2 (gradients: its 1e-3
    forward noise flips ReLU masks). Inputs are drawn with every float64 pre-activation at least 2e-5 from zero so that
    no mask flips under the 1e-6 rounding differences of the split. C > 8: forward with an N = 16..64 output-layer MMA (separate
    hi / lo operand blocks), backward in ONE pass with the output layer as two plain GEMMs around the kernel (gnan_mlp_bwd_ext)."""
    from gnan_b200 import ops
    H, L = 64, 3
    rng = np.random.default_rng(R * 11 + G_)
    p = rand_mlp(rng, G_, H, C, L)
    u = kink_free_inputs(rng, p, R, G_, 2e-5, L)
    dS = torch.tensor(rng.normal(size=(R, C))).float()
    q = oracle_params(p, L)
    want = gnan_lut.feature_sums(q, u.double())
    (want * dS.double()).sum().backward()
    d = {k: v.to(DEV).requires_grad_(v.numel() > 0) for k, v in p.items()}
    got = ops.mlp(u.to(DEV), d["w1"], d["b1"], d["wh"], d["bh"], d["wo"], d["bo"], L, precision=precision)
    (got * dS.to(DEV)).sum().backward()
    assert G.rel_err(got.detach().cpu().numpy(), want.detach().numpy()) < tol
    for k in p:
        assert G.rel_err(d[k].grad.cpu().numpy(), q[k].grad.numpy()) < gtol, k


def test_mlp_tensor_core_cora_sized_multi_tile():
    """Cora-sized rows (22 tiles per CTA, partial-gradient chunks), 12 M pre-activations, all parameters to 1e-5."""
    from gnan_b200 import ops
    R, G_, C, H, L = 2708, 70, 7, 64, 3
    rng = np.random.default_rng(2)
    p = rand_mlp(rng, G_, H, C, L)
    u = kink_free_inputs(rng, p, R, G_, 2e-5, L)
    dS = torch.tensor(rng.normal(size=(R, C))).float()
    q = oracle_params(p, L)
    want = gnan_lut.feature_sums(q, u.double())
    (want * dS.double()).sum().backward()
    d = {k: v.to(DEV).requires_grad_(True) for k, v in p.items()}
    got = ops.mlp(u.to(DEV), d["w1"], d["b1"], d["wh"], d["bh"], d["wo"], d["bo"], L, precision="tf32x3")
    (got * dS.to(DEV)).sum().backward()
    assert G.rel_err(got.detach().cpu().numpy(), want.detach().numpy()) < TOL
    for k in p:
        assert G.rel_err(d[k].grad.cpu().numpy(), q[k].grad.numpy()) < TOL, k


def test_mlp_tensor_core_dropout_masks_match_fp32_path():
    from gnan_b200 import ops
    rng = np.random.default_rng(4)
    R, G_, H, C, L = 700, 5, 64, 3, 3
    p = {k: v.to(DEV) for k, v in rand_mlp(rng, G_, H, C, L).items()}
    u = torch.tensor(rng.normal(size=(R, G_))).float().to(DEV)
    a = ops.mlp(u, p["w1"], p["b1"], p["wh"], p["bh"], p["wo"], p["bo"], L, dropout_p=0.4, seed=77, precision="fp32")
    b = ops.mlp(u, p["w1"], p["b1"], p["wh"], p["bh"], p["wo"], p["bo"], L, dropout_p=0.4, seed=77, precision="tf32x3")
    assert G.rel_err(b.cpu().numpy(), a.cpu().numpy()) < 1e-4      # same masks; a ReLU kink may flip under a different rounding


def test_mlp_tensor_core_backward_with_dropout_matches_fp32_path():
    from gnan_b200 import ops
    rng = np.random.default_rng(6)
    R, G_, H, C, L = 900, 6, 64, 7, 3
    p = rand_mlp(rng, G_, H, C, L)
    u = torch.tensor(rng.normal(size=(R, G_))).float().to(DEV)
    dS = torch.tensor(rng.normal(size=(R, C))).float().to(DEV)
    grads = {}
    for prec in ("fp32", "tf32x3"):
        d = {k: v.to(DEV).requires_grad_(True) for k, v in p.items()}
        out = ops.mlp(u, d["w1"], d["b1"], d["wh"], d["bh"], d["wo"], d["bo"], L, dropout_p=0.3, seed=5, precision=prec)
        (out * dS).sum().backward()
        grads[prec] = {k: v.grad.cpu().numpy() for k, v in d.items()}
    for k in p:
        assert G.rel_err(grads["tf32x3"][k], grads["fp32"][k]) < 2e-4, k     # same masks; a kink may flip under different rounding


@pytest.mark.parametrize("R,G_,C", [(700, 5, 9), (900, 3, 40), (300, 2, 64)])
def test_mlp_tensor_core_backward_channel_slices_match_one_pass(R, G_, C, monkeypatch):
    """C > 8 has two tensor-core backward routes: gnan_mlp_bwd_ext (one pass, output layer as GEMMs outside; the default) and
    gnan_mlp_bwd's ceil(C/8) channel-slice passes (taken when the dh / a1 buffers would exceed ops.MLP_EXT_MAX_BYTES). Both
    against the float64 oracle at 1e-5, and against each other."""
    from gnan_b200 import ops
    H, L = 64, 3
    rng = np.random.default_rng(R + C)
    p = rand_mlp(rng, G_, H, C, L)
    u = kink_free_inputs(rng, p, R, G_, 2e-5, L)
    dS = torch.tensor(rng.normal(size=(R, C))).float()
    q = oracle_params(p, L)
    (gnan_lut.feature_sums(q, u.double()) * dS.double()).sum().backward()
    grads = {}
    for route, cap in (("ext", ops.MLP_EXT_MAX_BYTES), ("slices", 0)):
        monkeypatch.setattr(ops, "MLP_EXT_MAX_BYTES", cap)
        d = {k: v.to(DEV).requires_grad_(True) for k, v in p.items()}
        out = ops.mlp(u.to(DEV), d["w1"], d["b1"], d["wh"], d["bh"], d["wo"], d["bo"], L, precision="tf32x3")
        (out * dS.to(DEV)).sum().backward()
        grads[route] = {k: v.grad.cpu().numpy() for k, v in d.items()}
        for k in p:
            assert G.rel_err(grads[route][k], q[k].grad.numpy()) < TOL, (route, k)
    for k in p:
        assert G.rel_err(grads["ext"][k], grads["slices"][k]) < TOL, k


def test_mlp_tensor_core_one_pass_backward_with_dropout_matches_fp32_path():
    """gnan_mlp_bwd_ext with dropout: a1 leaves the kernel AFTER the mask, so dWo = dS^T a1 sees the same masks as the fp32 kernels"""
    from gnan_b200 import ops
    rng = np.random.default_rng(16)
    R, G_, H, C, L = 900, 6, 64, 40, 3
    p = rand_mlp(rng, G_, H, C, L)
    u = torch.tensor(rng.normal(size=(R, G_))).float().to(DEV)
    dS = torch.tensor(rng.normal(size=(R, C))).float().to(DEV)
    grads = {}
    for prec in ("fp32", "tf32x3"):
        d = {k: v.to(DEV).requires_grad_(True) for k, v in p.items()}
        out = ops.mlp(u, d["w1"], d["b1"], d["wh"], d["bh"], d["wo"], d["bo"], L, dropout_p=0.3, seed=5, precision=prec)
        (out * dS).sum().backward()
        grads[prec] = {k: v.grad.cpu().numpy() for k, v in d.items()}
    for k in p:
        assert G.rel_err(grads["tf32x3"][k], grads["fp32"][k]) < 2e-4, k     # same masks; a kink may flip under different rounding


@pytest.mark.parametrize("G_,C,bias,precision", [(200, 7, True, "fp32"), (64, 1, True, "tf32x3"), (33, 8, False, "fp32"), (120, 3, True, "tf32x3")])
def test_mlp_entries_small_groups_vs_float64(G_, C, bias, precision):
    """Entries mode with a few dozen rows per feature (bag-of-words columns): forward + the CTA-per-feature fp32 backward
    (mlp_entries_bwd_small_kernel, taken in both precision modes when a feature has <= 96 entries on average), incl. single-entry
    groups, groups longer than one 32-row tile and an empty tail, against float64 on kink-free inputs: 1e-5."""
    from gnan_b200 import sparse
    H, L = 64, 3
    rng = np.random.default_rng(G_ * 10 + C)
    p = rand_mlp(rng, G_, H, C, L, bias=bias)
    R = 140
    u = kink_free_inputs(rng, p, R, G_, 2e-5, L)
    sizes = rng.integers(1, 91, size=G_)
    sizes[0], sizes[1], sizes[2] = 1, 140, 33
    rows = [np.sort(rng.choice(R, size=int(n), replace=False)) for n in sizes]
    grp_ptr = torch.tensor(np.concatenate([[0], np.cumsum(sizes)]), dtype=torch.int64)
    val = torch.cat([u[torch.tensor(r), g] for g, r in enumerate(rows)])
    E = val.numel()
    dY = torch.tensor(rng.normal(size=(E, C))).float()
    # float64 restatement per entry
    q = oracle_params(p, L)
    grp = torch.repeat_interleave(torch.arange(G_), torch.tensor(sizes))
    a0 = torch.relu(val.double().unsqueeze(1) * q["w1"][grp] + q["b1"][grp])
    a1 = torch.relu(torch.einsum("ei,eji->ej", a0, q["wh"][0][grp]) + q["bh"][0][grp])
    want = torch.einsum("ej,ecj->ec", a1, q["wo"][grp]) + q["bo"][grp]
    (want * dY.double()).sum().backward()
    from gnan_b200._lib import PRECISIONS
    d = {k: v.to(DEV).requires_grad_(True) for k, v in p.items()}
    items = sparse._tiles_of(torch.tensor(sizes).to(DEV), G_, DEV)
    got = sparse.mlp_entries_fwd(val.to(DEV), grp_ptr.to(DEV), items, d["w1"], d["b1"], d["wh"], d["bh"], d["wo"], d["bo"], L, int(sizes.max()),
                                 PRECISIONS[precision])
    (got * dY.to(DEV)).sum().backward()
    assert G.rel_err(got.detach().cpu().numpy(), want.detach().numpy()) < TOL
    for k in p:
        if bias or k in ("w1", "wh", "wo"):
            assert G.rel_err(d[k].grad.cpu().numpy(), q[k].grad.numpy()) < TOL, k


# ---- compact transfer forms (what crosses PCIe in bench.py's end-to-end leg) -------------------------------------------
def test_local_edges_expand_rebuilds_edge_index():
    """preprocess.LocalEdges: uint8 local endpoints + per-graph edge offsets -> gnan_edges_from_local -> the int64 edge_index,
    bit-exact (edge groups in graph order), and the batched BFS of it equals the BFS of the original list."""
    from gnan_b200.preprocess import LocalEdges, apsp_batched
    rng = np.random.default_rng(3)
    sizes = rng.integers(1, 257, size=300)
    sizes[5] = 256; sizes[6] = 1
    node_off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    src, dst = [], []
    for b, n in enumerate(sizes):
        m = int(rng.integers(0, 3 * n))
        src.append(node_off[b] + rng.integers(0, n, m)); dst.append(node_off[b] + rng.integers(0, n, m))
    ei = np.stack([np.concatenate(src), np.concatenate(dst)])
    und = np.unique(ei[:, ei[0] != ei[1]].T, axis=0).T                         # simple directed graph, sorted by source
    perm = rng.permutation(und.shape[1])                                       # shuffled: from_edge_index regroups it
    le = LocalEdges.from_edge_index(torch.tensor(und[:, perm]), node_off)
    no_d = torch.tensor(node_off, dtype=torch.int32, device=DEV)
    got = le.to(DEV).expand(no_d)
    assert got.dtype == torch.int64 and got.shape == (2, und.shape[1])
    g = np.searchsorted(node_off, und[0, perm], side="right") - 1
    want = und[:, perm][:, np.argsort(g, kind="stable")]
    assert np.array_equal(got.cpu().numpy(), want)
    out = torch.zeros_like(got)
    assert le.to(DEV).expand(no_d, out=out) is out and torch.equal(out, got)
    small = sizes <= 128                                                        # BFS equality on the graphs the batched kernel takes
    keep_g = np.nonzero(small)[0][:40]
    sel = np.isin(g, keep_g)
    remap = np.concatenate([[0], np.cumsum(sizes[keep_g])])
    def sub(e):
        gg = np.searchsorted(node_off, e[0], side="right") - 1
        pos = np.searchsorted(keep_g, gg)
        return torch.tensor(e - node_off[gg] + remap[pos])
    a = apsp_batched(sub(und[:, perm][:, sel]), remap, device=DEV)
    le2 = LocalEdges.from_edge_index(sub(und[:, perm][:, sel]), remap).to(DEV)
    b = apsp_batched(le2.expand(torch.tensor(remap, dtype=torch.int32, device=DEV)), remap, device=DEV)
    assert torch.equal(a.hop, b.hop) and torch.equal(a.level_counts, b.level_counts)


def test_compact_compressed_features_refresh_static_inputs():
    """CompressedFeatures.compact_host() (narrow index types, per-entry values dropped when values are shared) moved raw to the
    device and widened by copy_tensors_ into a step's static tensors: every tensor equals the original; .to(device) alone too."""
    from gnan_b200.sparse import compress_features
    rng = np.random.default_rng(8)
    N, K = 5000, 15
    x = np.zeros((N, K), np.float32)
    x[np.arange(N), rng.integers(0, 14, N)] = 1.0
    x[:, 14] = 1.0
    cx = compress_features(torch.tensor(x).to(DEV))
    assert cx.shared is not None
    ch = cx.compact_host()
    assert ch.val.numel() == 0 and ch.shared.inv.dtype == torch.uint8 and ch.nbytes() < 0.55 * cx.nbytes()
    static = cx.clone_tensors()
    for t in static._tensors():
        t.zero_()
    static.copy_tensors_(ch.to(DEV, raw=True))
    wide = ch.to(DEV)
    for a, b, c in zip(static._tensors(), cx._tensors(), wide._tensors()):
        assert a.dtype == b.dtype == c.dtype and torch.equal(a, b) and torch.equal(c, b)


# ---- training loop around the path (SURVEY §8f-1) ----------------------------------------------------------------------
def _trainer_items(z, graph_task, n_items):
    from gnan_b200.preprocess import apsp
    items = []
    for i in range(n_items):
        x = torch.tensor(z[f"item{i}.x"])
        ei = torch.tensor(z[f"item{i}.edge_index"])
        d = SimpleNamespace(x=x.to(DEV), edge_index=ei, hop_data=apsp(ei, x.shape[0], device=DEV), y=torch.tensor(z[f"item{i}.y"]))
        if not graph_task:
            for m in ("train_mask", "val_mask", "test_mask"):
                setattr(d, m, torch.tensor(z[f"item{i}.{m}"]))
        items.append(d)
    return items


@pytest.mark.parametrize("name", ["trainer_graph_bce", "trainer_node_ce"])
def test_trainer_epochs_match_reference_trainer(name):
    """gnan_b200.trainer.train_epoch / test_epoch against the UNMODIFIED trainer.py driving models.TensorGNAN + Adam
    (tests/golden/trainer_*.npz): the per-epoch (loss, accuracy, auc) tuples and the weights after the last epoch.
    Losses 1e-4 relative (Adam divides by sqrt(v): early steps amplify 1e-6 gradient differences); weights 2e-3."""
    from gnan_b200 import trainer
    from gnan_b200.models import TensorGNAN
    z = dict(np.load(f"{G.GOLDEN_DIR}/{name}.npz"))
    graph_task, n_items, K, C, H, epochs, compute_auc, _ = [int(t) for t in z["meta"]]
    lr, wd = [float(t) for t in z["hyper"]]
    m = TensorGNAN(K, C, 3, H, is_graph_task=bool(graph_task), readout_n_layers=0)
    m.load_state_dict({k[4:]: torch.tensor(v) for k, v in z.items() if k.startswith("sd0.")}, strict=True)
    m = m.to(DEV)
    items = _trainer_items(z, bool(graph_task), n_items)
    loss_fn = torch.nn.BCEWithLogitsLoss() if graph_task else torch.nn.CrossEntropyLoss()
    opt = torch.optim.Adam(params=m.parameters(), lr=lr, weight_decay=wd)
    hist = []
    for _ in range(epochs):
        tr = trainer.train_epoch(m, dloader=items, loss_fn=loss_fn, optimizer=opt, classify=True, device=DEV,
                                 compute_auc=bool(compute_auc), is_graph_task=bool(graph_task))
        va = trainer.test_epoch(m, dloader=items, loss_fn=loss_fn, classify=True, device=DEV, val_mask=True,
                                compute_auc=bool(compute_auc), is_graph_task=bool(graph_task))
        m.train()
        hist.append(list(tr) + list(va))
    hist = np.array(hist, dtype=np.float64)
    want = z["history"]
    assert hist.shape == want.shape
    assert np.allclose(hist[:, [0, 3]], want[:, [0, 3]], rtol=1e-4, atol=0), (hist[:, [0, 3]], want[:, [0, 3]])   # losses
    assert np.allclose(hist[:, [1, 4]], want[:, [1, 4]], atol=1e-6)                                              # accuracies
    assert np.allclose(hist[:, [2, 5]], want[:, [2, 5]], atol=1e-6)                                              # auc / -1
    sd = m.state_dict()
    for k, v in z.items():
        if k.startswith("sd1."):
            assert G.rel_err(sd[k[4:]].cpu().numpy(), v) < 2e-3, k


def test_captured_step_equals_eager_steps():
    """trainer.CapturedStep (whole step replayed as one CUDA graph) follows the same trajectory as eager steps."""
    from gnan_b200 import trainer
    from gnan_b200.GNAN import TensorGNAN
    from gnan_b200.preprocess import apsp
    rng = np.random.default_rng(8)
    n, K, C = 300, 9, 4
    ei = torch.tensor(random_graph(rng, n, 2.5, False, n_isolated=3))
    x = torch.tensor(rng.normal(size=(n, K))).float().to(DEV)
    y = torch.tensor(rng.integers(0, C, size=n)).to(DEV)
    hd = apsp(ei, n, device=DEV)
    data = SimpleNamespace(x=x, hop_data=hd)
    losses = {}
    for mode in ("eager", "graph"):
        torch.manual_seed(0)
        m = TensorGNAN(K, C, 3, 64).to(DEV)
        m.fs.xavier_normal_(1.0); m.rho.xavier_normal_(1.0)
        opt = torch.optim.Adam(m.parameters(), lr=1e-3, capturable=True)
        closure = lambda: torch.nn.functional.cross_entropy(m.forward(data), y)
        if mode == "eager":
            out = []
            for _ in range(3 + 5):
                opt.zero_grad(set_to_none=True)
                l = closure(); l.backward(); opt.step()
                out.append(float(l.detach()))
            losses[mode] = out[3:]
        else:
            step = trainer.CapturedStep(closure, opt, warmup=2)      # 2 warm-up steps + 1 captured (capture does not execute)
            assert step.kernel_launches > 0
            losses[mode] = [float(step()) for _ in range(6)][1:]
    assert np.allclose(losses["eager"], losses["graph"], rtol=1e-5), losses


def test_captured_step_sees_inputs_refreshed_in_place():
    """ADVICE round 1: the implicit shared-evaluation caches (compressed features keyed on x, value -> row mapping of the
    per-row rho inputs keyed on the level counts) must not be baked into a captured step: after x.copy_() /
    level_counts.copy_() the replay has to compute on the NEW values."""
    from gnan_b200 import trainer
    from gnan_b200.GNAN import TensorGNAN
    from gnan_b200.preprocess import HopData, apsp
    rng = np.random.default_rng(21)
    n, K, C = 600, 120, 3                                               # 72 000 (row, feature) pairs: above the auto-dedup threshold
    mk = lambda: torch.tensor((rng.random((n, K)) < 0.1) * rng.integers(1, 4, size=(n, K))).float().to(DEV)
    x_a, x_b = mk(), mk()
    hd_a = apsp(torch.tensor(random_graph(rng, n, 2.5, False, n_isolated=3)), n, device=DEV)
    hd_b = apsp(torch.tensor(random_graph(rng, n, 3.5, False, n_isolated=9)), n, device=DEV)
    nb = max(hd_a.nbins, hd_b.nbins)

    def padded(hd):                                                     # same level-table width for both graphs
        cnt = torch.zeros(n, nb, dtype=torch.int32, device=DEV)
        cnt[:, :hd.nbins - 1] = hd.level_counts[:, :-1]; cnt[:, -1] = hd.level_counts[:, -1]
        return HopData(hd.hop.clone(), cnt, n)
    hd_a, hd_b = padded(hd_a), padded(hd_b)
    y = torch.tensor(rng.integers(0, C, size=n)).to(DEV)
    torch.manual_seed(0)
    m = TensorGNAN(K, C, 3, 64).to(DEV)
    m.fs.xavier_normal_(1.0); m.rho.xavier_normal_(1.0)
    opt = torch.optim.SGD(m.parameters(), lr=0.0)                       # weights stay put: the loss depends on the inputs only
    static = SimpleNamespace(x=x_a.clone(), hop_data=HopData(hd_a.hop.clone(), hd_a.level_counts.clone(), n))
    closure = lambda: torch.nn.functional.cross_entropy(m.forward(static), y)
    step = trainer.CapturedStep(closure, opt, warmup=2)
    loss_a = float(step())
    static.x.copy_(x_b); static.hop_data.hop.copy_(hd_b.hop); static.hop_data.level_counts.copy_(hd_b.level_counts)
    loss_b = float(step())
    with torch.no_grad():
        want_a = float(torch.nn.functional.cross_entropy(m.forward(SimpleNamespace(x=x_a, hop_data=hd_a)), y))
        want_b = float(torch.nn.functional.cross_entropy(m.forward(SimpleNamespace(x=x_b, hop_data=hd_b)), y))
    assert abs(want_a - want_b) > 1e-4 * abs(want_a)                    # the two inputs really differ
    assert abs(loss_a - want_a) < 1e-5 * abs(want_a) and abs(loss_b - want_b) < 1e-5 * abs(want_b), (loss_a, want_a, loss_b, want_b)


# ---- packed dataset format and loader (SURVEY §8f-2) ---------------------------------------------------------------------
GRAPH_PRE = ["preprocess_tree_undirected", "preprocess_isolated_undirected", "preprocess_directed", "preprocess_single_node"]


def test_packed_dataset_matches_reference_preprocess_bit_exactly(tmp_path):
    """One batched GPU BFS over several graphs -> packed format -> the reference's per-graph fp32 tensors, compared
    bit-for-bit with what the unmodified pre_process() produced (tests/golden/preprocess_*.npz); and the way back."""
    from gnan_b200.packed import PackedDataset
    zs = [G.load(n) for n in GRAPH_PRE]
    graphs = [SimpleNamespace(x=torch.tensor(z["x"]), edge_index=torch.tensor(z["edge_index"].reshape(2, -1)),
                              y=torch.tensor([i % 2])) for i, z in enumerate(zs)]
    ds = PackedDataset.from_graphs(graphs, device=DEV)
    assert len(ds) == len(zs) and ds.y.tolist() == [0, 1, 0, 1]
    for g, z in zip(ds.to_reference(), zs):
        assert np.array_equal(g.x.cpu().numpy(), z["x_out"])
        assert np.array_equal(g.node_distances.cpu().numpy(), z["node_distances"])
        assert np.array_equal(g.normalization_matrix.cpu().numpy(), z["normalization_matrix"])
    ref_graphs = [SimpleNamespace(x=torch.tensor(z["x_out"]), node_distances=torch.tensor(z["node_distances"]),
                                  normalization_matrix=torch.tensor(z["normalization_matrix"]), y=torch.tensor([i % 2]))
                  for i, z in enumerate(zs)]
    back = PackedDataset.from_reference(ref_graphs, device=DEV)
    for k in ("x", "node_off", "hop", "hop_off", "level_counts", "y"):
        assert torch.equal(getattr(back, k), getattr(ds, k)), k
    path = tmp_path / "ds.gnan_b200.pt"
    ds.save(path)
    again = PackedDataset.load(path, device=DEV)
    for k in ("x", "node_off", "hop", "hop_off", "level_counts", "y"):
        assert torch.equal(getattr(again, k), getattr(ds, k)), k
    fp32_bytes = sum(2 * 4 * z["node_distances"].size for z in zs)          # what processed_data/{name}.pt stores per pair
    assert ds.hop.numel() * 8 == fp32_bytes


def test_packed_loader_batches_equal_per_graph_forward_and_train(tmp_path):
    from gnan_b200 import trainer
    from gnan_b200.models import TensorGNAN
    from gnan_b200.packed import PackedDataset
    from gnan_b200.preprocess import pre_process
    rng = np.random.default_rng(4)
    graphs = []
    for i in range(9):
        n = int(rng.integers(3, 40))
        graphs.append(SimpleNamespace(x=torch.tensor(rng.normal(size=(n, 4))).float(), y=torch.tensor([float(i % 2)]),
                                      edge_index=torch.tensor(random_graph(rng, n, 2.2, False, n_isolated=1 if n > 8 else 0))))
    pre_process(graphs, True, "toy", processed_data_dir=str(tmp_path), device=DEV)          # reference call shape; writes the file
    ds = PackedDataset.load(tmp_path / "toy.gnan_b200.pt", device=DEV)
    assert len(ds) == 9 and ds.x.shape[1] == 5
    torch.manual_seed(0)
    m = TensorGNAN(5, 1, 3, 64, is_graph_task=True, readout_n_layers=0).to(DEV)
    m.fs.xavier_normal_(1.0); m.rho.xavier_normal_(1.0)
    per_graph = torch.cat([m.forward(SimpleNamespace(x=g.x.to(DEV), hop_data=g.hop_data)).T for g in graphs])   # [9,1]
    ids = [7, 2, 5, 0]
    out = m(ds.batch(ids))
    assert G.rel_err(out.detach().cpu().numpy(), per_graph[ids].detach().cpu().numpy()) < TOL
    seen = torch.cat([m(pk).detach() for pk in ds.loader(4)])
    assert G.rel_err(seen.cpu().numpy(), per_graph.detach().cpu().numpy()) < TOL
    # an epoch of mini-batch training through the drop-in trainer == the same steps written out by hand
    loss_fn = torch.nn.BCEWithLogitsLoss()
    sd0 = {k: v.clone() for k, v in m.state_dict().items()}
    opt = torch.optim.Adam(m.parameters(), lr=1e-2)
    l1, a1, _ = trainer.train_epoch(m, ds.loader(4), loss_fn, opt, DEV, is_graph_task=True)
    w1 = m.fs.wh.detach().clone()
    m.load_state_dict(sd0)
    opt = torch.optim.Adam(m.parameters(), lr=1e-2)
    tot = 0.0
    for pk in ds.loader(4):
        opt.zero_grad()
        l = loss_fn(m(pk).flatten(), pk.y.float()); l.backward(); opt.step(); tot += float(l.detach())
    assert abs(l1 - tot / 3) < 1e-6 * max(1.0, abs(l1)) and 0.0 <= a1 <= 1.0
    assert torch.allclose(w1, m.fs.wh.detach(), rtol=0, atol=1e-7)


def test_node_dataset_file_roundtrip(tmp_path):
    from gnan_b200.packed import load_node
    from gnan_b200.preprocess import pre_process
    z = G.load("preprocess_node_task")
    d = SimpleNamespace(x=torch.tensor(z["x"]), edge_index=torch.tensor(z["edge_index"].reshape(2, -1)),
                        y=torch.arange(z["x"].shape[0]) % 3, train_mask=torch.arange(z["x"].shape[0]) % 2 == 0)
    pre_process(d, False, "node", processed_data_dir=str(tmp_path), device=DEV)
    back = load_node(tmp_path / "node.gnan_b200.pt", device=DEV)
    n = back.hop_data.num_nodes
    assert torch.equal(back.hop_data.hop[:, :n], d.hop_data.hop[:, :n]) and torch.equal(back.hop_data.level_counts, d.hop_data.level_counts)
    assert torch.equal(back.x.cpu(), d.x) and torch.equal(back.y.cpu(), d.y) and torch.equal(back.train_mask.cpu(), d.train_mask)
    nd, nm = back.hop_data.reference_format()
    assert np.array_equal(nd.cpu().numpy(), z["node_distances"]) and np.array_equal(nm.cpu().numpy(), z["normalization_matrix"])


# ---- interpretability export (SURVEY §8f-3) ------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["gnanpy_tensor_graph", "gnanpy_tensor_node", "gnanpy_tensor_node_l1", "gnanpy_tensor_node_l4",
                                  "models_tensor_graph_readout", "batched_graph"])
def test_interpretability_tables_match_reference_modules(name):
    """What the notebook computes point by point with model.fs[i].forward / model.m.forward (cells 4, 6, 9), in bulk from
    the kernels, against the port's scalar MLP on the golden weights."""
    from gnan_b200 import interpret
    z = G.load(name)
    m = build_module(z, DEV).eval()
    fs = gnan_port.to_torch(z["fs"]); rho = gnan_port.to_torch(z["rho"])
    grid = torch.linspace(-1.5, 2.0, 23)
    got = interpret.shape_function_table(m, grid).cpu()
    want = torch.stack([gnan_port.scalar_mlp(fs, k, grid.view(-1, 1)) for k in range(z["K"])], dim=1)
    assert tuple(got.shape) == (23, z["K"], want.shape[-1])
    assert G.rel_err(got.numpy(), want.numpy()) < TOL
    D = 9
    d = torch.arange(D + 1).float()
    u = d if z["variant"] == "batched" else 1.0 / (1.0 + d)
    want_r = gnan_port.scalar_mlp(rho, 0, u.view(-1, 1))
    got_r = interpret.distance_function_table(m, D).cpu()
    assert G.rel_err(got_r.numpy(), want_r.numpy()) < TOL
    hm = interpret.heatmap(m, D).cpu()
    f1 = torch.stack([gnan_port.scalar_mlp(fs, k, torch.ones(1, 1))[0, 0] for k in range(z["K"])])
    assert G.rel_err(hm.numpy(), torch.outer(f1, want_r[:, 0]).numpy()) < TOL


def test_mlp_per_group_chunked_with_gradients():
    """K*C > 64 forces several kernel calls; values and weight gradients against autograd of the port."""
    from gnan_b200 import ops
    gen = torch.Generator().manual_seed(5)
    R, K, C, H, L = 70, 30, 7, 64, 3
    p = dict(w1=torch.randn(K, H, generator=gen), b1=torch.randn(K, H, generator=gen),
             wh=torch.randn(1, K, H, H, generator=gen) / 8, bh=torch.randn(1, K, H, generator=gen) * 0.1,
             wo=torch.randn(K, C, H, generator=gen) / 8, bo=torch.randn(K, C, generator=gen))
    u = torch.randn(R, K, generator=gen)
    w = torch.randn(R, K, C, generator=gen)
    q = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    want = gnan_port.shape_functions(q, u)
    (want * w).sum().backward()
    d = {k: v.to(DEV).requires_grad_(True) for k, v in p.items()}
    got = ops.mlp_per_group(u.to(DEV), d["w1"], d["b1"], d["wh"], d["bh"], d["wo"], d["bo"], L)
    (got * w.to(DEV)).sum().backward()
    assert tuple(got.shape) == (R, K, C)
    assert G.rel_err(got.detach().cpu().numpy(), want.detach().numpy()) < TOL
    for k in p:
        assert G.rel_err(d[k].grad.cpu().numpy(), q[k].grad.numpy()) < TOL, k


# ---- compressed features: shared shape-function evaluations (SURVEY §8d value dedup) --------------------------------------
def _compressible_x(rng, N, K, kind):
    x = np.zeros((N, K), np.float32)
    if kind == "bow":                                            # Cora-like: ~1.3 % non-zeros, rows normalised, constant column
        m = rng.random((N, K - 1)) < 0.013
        x[:, :-1] = m / np.maximum(m.sum(1, keepdims=True), 1)
        x[:, -1] = 1.0
    elif kind == "onehot":                                       # Mutagenicity-like
        x[np.arange(N), rng.integers(0, K - 1, N)] = 1.0
        x[:, -1] = 1.0
    else:                                                        # mixed: a dense-ish column, a two-valued one, an empty one
        x[:, 0] = np.where(rng.random(N) < 0.2, rng.normal(size=N), 0.0)
        x[:, 1] = np.where(rng.random(N) < 0.5, 2.0, -1.0)
        x[rng.integers(0, N, 5), 3] = 7.0
    return torch.tensor(x)


@pytest.mark.parametrize("kind,N,K,H,C,L", [("bow", 700, 300, 64, 7, 3), ("onehot", 5000, 15, 64, 1, 3), ("mixed", 333, 5, 16, 3, 4),
                                            ("onehot", 129, 6, 32, 2, 2)])
def test_compressed_feature_sums_equal_dense_kernels(kind, N, K, H, C, L):
    """sparse.feature_sums (one evaluation per distinct (feature, value) pair + row gather) against the dense fp32 kernels
    and the float64 oracle on the same x: outputs and every weight gradient."""
    from gnan_b200 import ops, sparse
    rng = np.random.default_rng(N + K)
    x = _compressible_x(rng, N, K, kind)
    gen = torch.Generator().manual_seed(K)
    nh = L - 2
    p = dict(w1=torch.randn(K, H, generator=gen), b1=torch.randn(K, H, generator=gen) * 0.5,
             wh=torch.randn(nh, K, H, H, generator=gen) / H ** 0.5, bh=torch.randn(nh, K, H, generator=gen) * 0.1,
             wo=torch.randn(K, C, H, generator=gen) / H ** 0.5, bo=torch.randn(K, C, generator=gen))
    w = torch.randn(N, C, generator=gen)
    cx = sparse.compress_features(x.to(DEV))
    assert cx is not None and torch.equal(cx.to_dense().cpu(), x)
    res = {}
    for mode in ("dense", "sparse"):
        d = {k: v.to(DEV).requires_grad_(True) for k, v in p.items()}
        args = (d["w1"], d["b1"], d["wh"], d["bh"], d["wo"], d["bo"], L)
        S = ops.mlp(x.to(DEV), *args) if mode == "dense" else sparse.feature_sums(cx, *args)
        (S * w.to(DEV)).sum().backward()
        res[mode] = (S.detach().cpu().numpy(), {k: v.grad.cpu().numpy() for k, v in d.items()})
    q = {k: v.double().requires_grad_(True) for k, v in p.items()}
    want = gnan_port.shape_functions(q, x.double()).sum(dim=1)
    (want * w.double()).sum().backward()
    for mode in ("dense", "sparse"):
        assert G.rel_err(res[mode][0], want.detach().numpy()) < TOL, mode
        for k in p:
            if p[k].numel():
                assert G.rel_err(res[mode][1][k], q[k].grad.numpy()) < TOL, (mode, k)
    if H == 64 and L == 3 and C <= 8:
        # backward on the tcgen05 kernel in entries mode against the same kernel on the dense matrix: a row's activations (and
        # ReLU masks) do not depend on which tile it sits in, so the two differ only by fp32 summation order
        tc = {}
        for mode in ("dense", "sparse"):
            d = {k: v.to(DEV).requires_grad_(True) for k, v in p.items()}
            args = (d["w1"], d["b1"], d["wh"], d["bh"], d["wo"], d["bo"], L)
            S = ops.mlp(x.to(DEV), *args, precision="tf32x3") if mode == "dense" else sparse.feature_sums(cx, *args, precision="tf32x3")
            (S * w.to(DEV)).sum().backward()
            tc[mode] = {k: v.grad.cpu().numpy() for k, v in d.items()}
        for k in p:
            assert G.rel_err(tc["sparse"][k], tc["dense"][k]) < TOL, ("tcgen05 entries", k)
            assert G.rel_err(tc["sparse"][k], q[k].grad.numpy()) < 1e-3, ("tcgen05 entries vs oracle (no kink filtering)", k)


@pytest.mark.parametrize("name", ["gnanpy_tensor_graph", "models_tensor_graph", "gnanpy_tensor_graph_nonorm_disconnected",
                                  "gnanpy_tensor_node", "gnanpy_tensor_node_directed_nobias"])
def test_modules_dedup_on_and_off_match_reference_golden(name):
    """Golden cases through the compressed-feature path (explicit `x_compressed`: these graphs are far below the size where
    the modules build it on their own) and through the dense kernels; both must reproduce the reference."""
    from gnan_b200.sparse import compress_features
    z = G.load(name)
    outs = {}
    for dedup in (True, False):
        m = build_module(z, DEV).eval()
        m.dedup = dedup
        x = torch.tensor(z["x"])
        data = SimpleNamespace(x=x, edge_index=torch.tensor(z["edge_index"]), node_distances=torch.tensor(z["node_distances"]),
                               normalization_matrix=torch.tensor(z["normalization_matrix"]),
                               x_compressed=compress_features(x.to(DEV), max_density=None))
        out = m.forward(data)
        (out * torch.tensor(z["out_weight"], device=DEV)).sum().backward()
        assert G.rel_err(out.detach().cpu().numpy(), z["out"]) < TOL
        check_grads(z, grads_of(m.fs), z["grad_fs"], "fs")
        check_grads(z, grads_of(m.rho), z["grad_rho"], "rho")
        outs[dedup] = out.detach()
    assert G.rel_err(outs[True].cpu().numpy(), outs[False].cpu().numpy()) < 1e-6


def test_dropout_training_uses_the_dense_kernels(monkeypatch):
    """Per-row dropout masks make rows with equal inputs differ: with dropout active the compressed path must not be used.
    Also: the modules compress a large enough persistent input on their own, and never a small one."""
    from gnan_b200 import sparse
    from gnan_b200.GNAN import TensorGNAN
    from gnan_b200.preprocess import apsp
    calls = []
    real = sparse.feature_sums
    monkeypatch.setattr(sparse, "feature_sums", lambda *a, **k: (calls.append(1), real(*a, **k))[1])
    rng = np.random.default_rng(2)
    n, K = 6000, 12                                                       # 72 000 (row, feature) pairs: above the auto threshold
    x = _compressible_x(rng, n, K, "onehot")
    data = SimpleNamespace(x=x, hop_data=apsp(torch.tensor(random_graph(rng, n, 2.5)), n, device=DEV))
    torch.manual_seed(0)
    m = TensorGNAN(K, 3, 3, 64, dropout=0.5).to(DEV)
    m.fs.xavier_normal_(1.0); m.rho.xavier_normal_(1.0)
    m.train()
    a = m.forward(data)
    assert not calls and getattr(data, "_gnan_b200_cx_cache", None) is None   # dropout active: dense kernels, nothing compressed
    m.eval()
    b = m.forward(data)
    assert len(calls) == 1 and data._gnan_b200_cx_cache[1] is not None    # eval: built once, shared evaluations
    m.forward(data)
    assert len(calls) == 2
    m.dedup = False
    c = m.forward(data)
    assert len(calls) == 2
    assert G.rel_err(b.detach().cpu().numpy(), c.detach().cpu().numpy()) < 1e-6
    assert G.rel_err(a.detach().cpu().numpy(), c.detach().cpu().numpy()) > 1e-3   # dropout really was active
    small = SimpleNamespace(x=x[:100], hop_data=apsp(torch.tensor(random_graph(rng, 100, 2.5)), 100, device=DEV))
    m.dedup = True
    m.forward(small)
    assert len(calls) == 2 and getattr(small, "_gnan_b200_cx_cache", None) is None   # too small to be worth analysing


def test_compressed_features_edge_cases():
    """No exceptions at all (every column constant), a single row, and a column whose mode is not zero."""
    from gnan_b200 import ops, sparse
    gen = torch.Generator().manual_seed(3)
    K, H, C, L = 4, 32, 2, 3
    p = dict(w1=torch.randn(K, H, generator=gen), b1=torch.randn(K, H, generator=gen), wh=torch.randn(1, K, H, H, generator=gen) / 6,
             bh=torch.randn(1, K, H, generator=gen) * 0.1, wo=torch.randn(K, C, H, generator=gen) / 6, bo=torch.randn(K, C, generator=gen))
    cases = {"all_constant": torch.tensor([[1.0, 0.0, -2.0, 0.5]]).repeat(50, 1),
             "single_row": torch.tensor([[0.3, 0.0, 1.0, 0.0]]),
             "nonzero_mode": torch.cat([torch.full((40, K), 3.0), torch.zeros(3, K)])}
    for name, x in cases.items():
        cx = sparse.compress_features(x.to(DEV), max_density=None)
        assert torch.equal(cx.to_dense().cpu(), x), name
        if name == "all_constant":
            assert cx.num_entries == K and cx.csr_eid.numel() == 0
        res = {}
        for mode in ("dense", "sparse"):
            d = {k: v.to(DEV).requires_grad_(True) for k, v in p.items()}
            args = (d["w1"], d["b1"], d["wh"], d["bh"], d["wo"], d["bo"], L)
            S = ops.mlp(x.to(DEV), *args) if mode == "dense" else sparse.feature_sums(cx, *args)
            S.square().sum().backward()
            res[mode] = (S.detach().cpu().numpy(), {k: v.grad.cpu().numpy() for k, v in d.items()})
        assert G.rel_err(res["sparse"][0], res["dense"][0]) < TOL, name
        for k in p:
            assert G.rel_err(res["sparse"][1][k], res["dense"][1][k]) < TOL, (name, k)


def test_device_seed_word_is_xored_into_the_dropout_seed():
    """gnan_mlp_fwd/bwd(seed, seed_dev) == gnan_mlp_fwd/bwd(seed ^ *seed_dev): same masks, same gradients, both kernel paths."""
    from gnan_b200 import ops
    gen = torch.Generator().manual_seed(9)
    R, K, H, C, L = 260, 5, 64, 3, 3
    p = dict(w1=torch.randn(K, H, generator=gen), b1=torch.randn(K, H, generator=gen), wh=torch.randn(1, K, H, H, generator=gen) / 8,
             bh=torch.randn(1, K, H, generator=gen) * 0.1, wo=torch.randn(K, C, H, generator=gen) / 8, bo=torch.randn(K, C, generator=gen))
    u = torch.randn(R, K, generator=gen).to(DEV)
    w = torch.randn(R, C, generator=gen).to(DEV)
    s, word = 0x1234ABCD5678, 0x0F0F00FF1234567
    for prec in ("fp32", "tf32x3"):
        res = []
        for seed, sd in ((s, torch.tensor([word], dtype=torch.int64, device=DEV)), (s ^ word, None)):
            d = {k: v.to(DEV).requires_grad_(True) for k, v in p.items()}
            out = ops.mlp(u, d["w1"], d["b1"], d["wh"], d["bh"], d["wo"], d["bo"], L, dropout_p=0.4, seed=seed, precision=prec, seed_dev=sd)
            (out * w).sum().backward()
            res.append((out.detach(), d["wh"].grad.clone(), d["w1"].grad.clone()))
        for a, b in zip(*res):
            assert torch.equal(a, b), prec
        plain = ops.mlp(u, *[p[k].to(DEV) for k in ("w1", "b1", "wh", "bh", "wo", "bo")], L, dropout_p=0.4, seed=s, precision=prec)
        assert not torch.equal(plain, res[0][0])                     # the word really changes the masks


def test_captured_step_with_dropout_draws_fresh_masks():
    """A captured training step replays by-value kernel arguments; the device-side seed word advances per replay, so two replays
    from identical weights give different dropout masks (different losses), like two eager steps do."""
    from gnan_b200 import trainer
    from gnan_b200.GNAN import TensorGNAN
    from gnan_b200.preprocess import apsp
    rng = np.random.default_rng(12)
    n, K, C = 400, 8, 3
    x = torch.tensor(rng.normal(size=(n, K))).float().to(DEV)
    y = torch.tensor(rng.integers(0, C, size=n)).to(DEV)
    data = SimpleNamespace(x=x, hop_data=apsp(torch.tensor(random_graph(rng, n, 2.5)), n, device=DEV))
    torch.manual_seed(0)
    m = TensorGNAN(K, C, 3, 64, dropout=0.5).to(DEV)
    m.fs.xavier_normal_(1.0); m.rho.xavier_normal_(1.0)
    m.train()
    opt = torch.optim.SGD(m.parameters(), lr=0.0)                    # lr 0: the weights stay put, only the masks change
    step = trainer.CapturedStep(lambda: torch.nn.functional.cross_entropy(m.forward(data), y), opt, warmup=1)
    losses = [float(step()) for _ in range(4)]
    assert len(set(losses)) == 4, losses
    g1 = m.fs.wh.grad.clone()
    step()
    assert not torch.equal(g1, m.fs.wh.grad)


def test_size_bucketed_captured_steps_follow_the_eager_trajectory():
    """train_epoch(capture_steps=True): per-graph steps replayed from one CUDA graph per graph size give the same epoch
    results and weights as the eager per-graph steps (plain, non-capturable Adam as the reference builds it, main.py:141)."""
    from gnan_b200 import trainer
    from gnan_b200.models import TensorGNAN
    z = dict(np.load(f"{G.GOLDEN_DIR}/trainer_graph_bce.npz"))
    graph_task, n_items, K, C, H, epochs, _, _ = [int(t) for t in z["meta"]]
    lr, wd = [float(t) for t in z["hyper"]]
    hist, weights = {}, {}
    for capture in (False, True):
        m = TensorGNAN(K, C, 3, H, is_graph_task=True, readout_n_layers=0)
        m.load_state_dict({k[4:]: torch.tensor(v) for k, v in z.items() if k.startswith("sd0.")}, strict=True)
        m = m.to(DEV)
        items = _trainer_items(z, True, n_items)
        loss_fn = torch.nn.BCEWithLogitsLoss()
        opt = torch.optim.Adam(params=m.parameters(), lr=lr, weight_decay=wd)
        h = []
        for ep in range(4):
            if ep == 2:
                for g in opt.param_groups:
                    g["lr"] = lr * 0.5                                  # what an LR scheduler does between epochs
            h.append(trainer.train_epoch(m, items, loss_fn, opt, DEV, classify=True, is_graph_task=True, capture_steps=capture))
        hist[capture] = np.array(h, dtype=np.float64)
        weights[capture] = {k: v.detach().cpu().numpy() for k, v in m.state_dict().items()}
        if capture:
            cache = next(iter(m._gnan_b200_step_cache.values()))
            assert cache.usable and 1 <= len(cache.entries) <= n_items
    # capturable Adam evaluates its bias corrections in fp32 on the device (the eager one in Python floats) and Adam's
    # g / sqrt(v) amplifies that in the first steps: measured 6e-6..3e-5 on the epoch losses
    assert np.allclose(hist[True][:, 0], hist[False][:, 0], rtol=2e-4), (hist[True], hist[False])
    assert np.allclose(hist[True][:, 1], hist[False][:, 1], atol=1e-9)
    for k in weights[True]:
        assert G.rel_err(weights[True][k], weights[False][k]) < 2e-3, k


def test_size_bucketed_captured_steps_with_dropout_run_and_vary():
    from gnan_b200 import trainer
    from gnan_b200.models import TensorGNAN
    from gnan_b200.preprocess import apsp
    rng = np.random.default_rng(31)
    items = []
    for i in range(12):
        n = int(rng.integers(5, 9))
        ei = torch.tensor(random_graph(rng, n, 2.0))
        items.append(SimpleNamespace(x=torch.tensor(rng.normal(size=(n, 4))).float().to(DEV), hop_data=apsp(ei, n, device=DEV),
                                     y=torch.tensor([float(i % 2)])))
    torch.manual_seed(0)
    m = TensorGNAN(4, 1, 3, 64, dropout=0.5, is_graph_task=True, readout_n_layers=0).to(DEV)
    m.fs.xavier_normal_(1.0); m.rho.xavier_normal_(1.0)
    m.train()
    opt = torch.optim.Adam(m.parameters(), lr=0.0)                      # lr 0: epochs differ only through the dropout masks
    l1 = trainer.train_epoch(m, items, torch.nn.BCEWithLogitsLoss(), opt, DEV, is_graph_task=True, capture_steps=True)[0]
    l2 = trainer.train_epoch(m, items, torch.nn.BCEWithLogitsLoss(), opt, DEV, is_graph_task=True, capture_steps=True)[0]
    assert np.isfinite(l1) and np.isfinite(l2) and l1 != l2
