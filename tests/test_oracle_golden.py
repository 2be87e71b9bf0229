"""CPU: pin the oracle (oracle/gnan_port.py, oracle/gnan_lut.py, oracle/apsp_oracle.c) against the golden
vectors produced by the unmodified reference (oracle/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import apsp as oapsp
from oracle import gnan_lut, gnan_port
from tests import _golden as G

TOL_PORT = 2e-6   # fp32 port vs fp32 reference (same op order; measured ~1e-7)
TOL_LUT = 5e-6    # fp64 re-ordered restatement vs fp32 reference


def run_port(z, dtype):
    fs = gnan_port.to_torch(z["fs"], dtype, True)
    rho = gnan_port.to_torch(z["rho"], dtype, True)
    x = torch.tensor(z["x"]).to(dtype)
    extra = {}
    if z["variant"] == "batched":
        out = gnan_port.tensor_gnan_batched(fs, rho, x, torch.tensor(z["dist_batch"]).to(dtype),
                                            torch.tensor(z["batch_vector"]), z["is_graph_task"])
    else:
        nd = torch.tensor(z["node_distances"]).to(dtype)
        nm = torch.tensor(z["normalization_matrix"]).to(dtype)
        if z["variant"] == "gnanpy_tensor":
            out = gnan_port.tensor_gnan_gnanpy(fs, rho, x, nd, nm, z["normalize_rho"], z["is_graph_task"])
        elif z["variant"] == "models_tensor":
            ro = gnan_port.to_torch(z["readout"], dtype, True) if "readout" in z else None
            extra["readout"] = ro
            out = gnan_port.tensor_gnan_models(fs, rho, x, nd, nm, z["normalize_rho"], z["is_graph_task"], ro)
        else:
            ids = z["node_ids"].tolist() if "node_ids" in z else None
            out = gnan_port.gnan_rowloop(fs, rho, x, nd, nm, z["normalize_rho"], ids)
    (out * torch.tensor(z["out_weight"]).to(dtype)).sum().backward()
    return out, fs, rho, extra


def check_grads(z, got, key, tol):
    want = z[key]
    has_bias = z["rho_has_bias"] if key == "grad_rho" else z["bias"]
    for k in ("w1", "b1", "wh", "bh", "wo", "bo"):
        if want[k] is None or want[k].size == 0:
            continue
        if k.startswith("b") and not has_bias:      # the reference has no such parameter (GNAN.py:36-37)
            continue
        g = got[k].grad
        g = np.zeros_like(want[k]) if g is None else g.numpy()
        if np.linalg.norm(want[k]) == 0:
            assert np.abs(g).max() < 1e-6, (key, k)
        else:
            assert G.rel_err(g, want[k]) < tol, (z["name"], key, k, G.rel_err(g, want[k]))


@pytest.mark.parametrize("name", G.MODEL_CASES + G.BATCHED_CASES)
def test_port_matches_reference(name):
    z = G.load(name)
    out, fs, rho, extra = run_port(z, torch.float32)
    assert out.shape == z["out"].shape
    assert G.rel_err(out.detach().numpy(), z["out"]) < TOL_PORT
    check_grads(z, fs, "grad_fs", 2e-5)
    check_grads(z, rho, "grad_rho", 2e-5)
    if extra.get("readout") is not None:
        check_grads(z, extra["readout"], "grad_readout", 2e-5)


def lut_mode(z):
    if z["variant"] == "batched":
        return "raw"
    if not z["normalize_rho"]:
        return "none"
    return "input" if z["variant"] == "gnanpy_tensor" else "output"


def run_lut(z):
    """float64 table restatement (oracle/gnan_lut.py) of a loaded case -> (out, fs, rho) after backward of sum(out * out_weight)"""
    dt = torch.float64
    fs = gnan_port.to_torch(z["fs"], dt, True)
    rho = gnan_port.to_torch(z["rho"], dt, True)
    x = torch.tensor(z["x"]).to(dt)
    if z["variant"] == "batched":
        hop = torch.tensor(z["dist_batch"]).long()           # -1 marks cross-graph / unreachable
        cnt = None
    else:
        hop = gnan_lut.hops_from_reference(torch.tensor(z["node_distances"]))
        cnt = gnan_lut.counts_from_hops(hop)
        # the reference's normalisation matrix is exactly the gathered level sizes
        idx = torch.where(hop < 0, torch.full_like(hop, cnt.shape[1] - 1), hop)
        assert torch.equal(torch.gather(cnt, 1, idx).float(), torch.tensor(z["normalization_matrix"]))
    if z["variant"] == "gnan_loop" and "node_ids" in z:
        ids = torch.tensor(z["node_ids"])
        hop, cnt = hop[ids], cnt[ids]
    out = gnan_lut.forward_rows(fs, rho, x, hop, cnt, lut_mode(z))
    if z["variant"] == "batched":
        if z["is_graph_task"]:
            B = int(z["batch_vector"].max()) + 1
            out = torch.zeros(B, out.shape[1], dtype=dt).index_add(0, torch.tensor(z["batch_vector"]), out)
    elif z["is_graph_task"]:
        out = out.sum(0).view(-1, 1)
    (out * torch.tensor(z["out_weight"]).to(dt)).sum().backward()
    return out, fs, rho


@pytest.mark.parametrize("name", [n for n in G.MODEL_CASES if "readout" not in n] + G.BATCHED_CASES)
def test_lut_restatement_matches_reference(name):
    z = G.load(name)
    out, fs, rho = run_lut(z)
    assert out.shape == z["out"].shape
    assert G.rel_err(out.detach().numpy(), z["out"]) < TOL_LUT
    check_grads(z, fs, "grad_fs", 2e-5)
    check_grads(z, rho, "grad_rho", 2e-5)


@pytest.mark.parametrize("name", G.PREPROCESS_CASES)
def test_apsp_oracle_bit_exact(name):
    z = G.load(name)
    n = int(z["meta"][0])
    node_task = bool(z["meta"][2])
    ei = z["edge_index"].reshape(2, -1)
    hop = oapsp.apsp(ei, n)
    cnt = oapsp.level_counts(hop)
    nd, nm = oapsp.reference_format(hop, cnt)
    assert np.array_equal(nd, z["node_distances"])            # bit-exact float32
    assert np.array_equal(nm, z["normalization_matrix"])
    assert np.array_equal(z["x_out"][:, :-1], z["x"]) and np.all(z["x_out"][:, -1] == 1.0)   # :108 / :127
    assert cnt.sum(axis=1).tolist() == [n] * n
    del node_task


@pytest.mark.parametrize("seed", range(12))
def test_apsp_oracle_matches_scipy_dijkstra_on_random_graphs(seed):
    """The C oracle against the library call the reference makes (scipy.sparse.csgraph.dijkstra on the unit-weight directed adjacency,
    pre_process_datasets.py:109-110,128-129) and a numpy restatement of its normaliser (:112-121), on random directed / undirected
    graphs with isolated nodes, self loops and several components: hops, level counts and both fp32 matrices bit for bit."""
    import scipy.sparse
    from scipy.sparse.csgraph import dijkstra
    rng = np.random.default_rng(100 + seed)
    n = int(rng.integers(2, 70))
    m = int(rng.integers(0, 3 * n))
    src, dst = rng.integers(0, n, size=m), rng.integers(0, n, size=m)
    if seed % 2 == 0:                                                     # undirected: both directions
        src, dst = np.concatenate([src, dst]), np.concatenate([dst, src])
    ei = np.unique(np.stack([src, dst]), axis=1).astype(np.int64)         # simple (no repeated pairs); self loops stay
    adj = scipy.sparse.coo_matrix((np.ones(ei.shape[1]), (ei[0], ei[1])), shape=(n, n))
    d = dijkstra(scipy.sparse.lil_matrix(adj))
    want_hop = np.where(np.isinf(d), -1, d).astype(np.int64)
    hop = oapsp.apsp(ei, n)
    assert np.array_equal(np.asarray(hop, dtype=np.int64), want_hop)
    cnt = oapsp.level_counts(hop)
    D = int(want_hop.max())
    assert cnt.shape == (n, D + 2) and cnt.sum(axis=1).tolist() == [n] * n
    for lvl in range(D + 1):
        assert np.array_equal(cnt[:, lvl], (want_hop == lvl).sum(axis=1))
    assert np.array_equal(cnt[:, -1], (want_hop < 0).sum(axis=1))
    nd, nm = oapsp.reference_format(hop, cnt)
    want_nd = (1.0 / (torch.nan_to_num(torch.from_numpy(d).float(), posinf=np.inf) + 1)).numpy()      # :112-115
    assert nd.dtype == np.float32 and np.array_equal(nd, want_nd)
    want_nm = np.stack([(want_nd[i][None, :] == want_nd[i][:, None]).sum(axis=1) for i in range(n)]).astype(np.float32)   # :117-121
    assert np.array_equal(nm, want_nm)
    rows = min(n, 5)
    assert np.array_equal(oapsp.apsp_rows(ei, n, rows), np.asarray(hop)[:rows])


def _random_weights(model, seed):
    """The golden generator's re-draw (oracle/make_golden.reinit), applied through the module's reference-format state_dict."""
    g = torch.Generator().manual_seed(seed)
    sd = {k: torch.randn(v.shape, generator=g) * ((1.2 / max(v.shape[1], 1) ** 0.5) if k.endswith("weight") else 0.3)
          for k, v in model.state_dict().items()}
    model.load_state_dict(sd, strict=True)
    return {f"sd.{k}": v.numpy() for k, v in model.state_dict().items()}


def _random_model_case(out_dir, name, cls, variant, rng, *, N, K_raw, C, H, L, is_graph_task, normalize_rho, rho_per_feature=False,
                       n_isolated=0, node_ids=None, directed=False, layers_kw="n_layers", bias=True):
    """oracle/make_golden.model_case with the same random draws, minus the reference: the weights are written by the gnan_b200 module
    of that configuration (the reference's state_dict layout) and the inputs by the C BFS in the reference's fp32 format (bit-exact
    to its pre_process: test_apsp_oracle_bit_exact, test_apsp_oracle_matches_scipy_dijkstra_on_random_graphs)."""
    import oracle.make_golden as mg
    ei = mg.random_graph(rng, N, n_isolated=n_isolated, directed=directed)
    x = ((rng.random((N, K_raw)) < 0.5) * rng.normal(size=(N, K_raw))).astype(np.float32)
    hop = oapsp.apsp(ei, N)
    nd, nm = oapsp.reference_format(hop, oapsp.level_counts(hop))
    x = np.concatenate([x, np.ones((N, 1), np.float32)], 1)                 # pre_process_datasets.py:108
    K = K_raw + 1
    kw = dict(in_channels=K, out_channels=C, hidden_channels=H, bias=bias, dropout=0.0, normalize_rho=normalize_rho,
              rho_per_feature=rho_per_feature, **{layers_kw: L})
    if variant != "gnan_loop":
        kw["is_graph_task"] = is_graph_task
    if variant == "models_tensor":
        kw["readout_n_layers"] = 0
    sd = _random_weights(cls(**kw), int(rng.integers(0, 2 ** 31)))
    rho_has_bias = bias if variant == "gnan_loop" else (not is_graph_task)
    meta = np.array([N, K, C, H, L, int(is_graph_task), int(normalize_rho), int(rho_per_feature), 0, int(rho_has_bias), int(bias)])
    extra = {} if node_ids is None else {"node_ids": np.array(node_ids, dtype=np.int64)}
    np.savez(os.path.join(out_dir, name + ".npz"), x=x, edge_index=ei, node_distances=nd, normalization_matrix=nm, meta=meta, **extra, **sd)


def _random_batched_case(out_dir, name, rng, *, B, K, C, H, is_graph_task):
    """oracle/make_golden.batched_case with the same random draws: per-graph hop matrices from the C BFS (-1 unreachable, as the
    networkx BFS of batched_pyg_main.py:39-44), weights written by gnan_b200's batched module."""
    import oracle.make_golden as mg
    from gnan_b200 import batched
    xs, dists, bv = [], [], []
    for g_ in range(B):
        n = int(rng.integers(3, 12))
        ei = mg.random_graph(rng, n, n_isolated=1 if g_ % 3 == 0 and n > 4 else 0)
        dists.append(np.asarray(oapsp.apsp(ei, n), dtype=np.float32))
        xs.append(rng.normal(size=(n, K)).astype(np.float32)); bv += [g_] * n
    tot = len(bv)
    dist_batch = np.full((tot, tot), -1, dtype=np.float32)
    o = 0
    for dm in dists:
        dist_batch[o:o + dm.shape[0], o:o + dm.shape[0]] = dm; o += dm.shape[0]
    model = batched.TensorGNAN(in_channels=K, out_channels=C, n_layers=2, hidden_channels=H, is_graph_task=is_graph_task)
    sd = _random_weights(model, int(rng.integers(0, 2 ** 31)))
    np.savez(os.path.join(out_dir, name + ".npz"), x=np.concatenate(xs), dist_batch=dist_batch, batch_vector=np.array(bv, dtype=np.int64),
             meta=np.array([tot, K, C, H, 2, int(is_graph_task)]), **sd)


@pytest.mark.parametrize("seed", [1, 2, 3, 4, 5, 6, 7, 8, 14, 33])     # 14 and 33: ill-conditioned draws (see below)
def test_table_restatement_matches_the_port_on_fresh_random_cases(tmp_path, monkeypatch, seed):
    """Beyond the committed fixtures: NEW random configurations (sizes, widths, depths 1-4, directed graphs, isolated nodes, bias and
    normalisation switches, row subsets, all four variants), drawn from the seed as oracle/make_golden.py draws them. Both restatements
    must agree on outputs and all parameter gradients: the float64 table form (gnan_lut) and the fp32 port's op order carried in float64
    (gnan_port). The port itself is pinned to the reference's outputs by test_port_matches_reference."""
    from gnan_b200 import GNAN as gnan_py, models as models_py
    rng = np.random.default_rng(9000 + seed)
    monkeypatch.setattr(G, "GOLDEN_DIR", str(tmp_path))
    pick = lambda *v: v[int(rng.integers(0, len(v)))]
    names = []
    for variant, cls, kw in (("gnanpy_tensor", gnan_py.TensorGNAN, {}), ("models_tensor", models_py.TensorGNAN, {}),
                             ("gnan_loop", pick(gnan_py.GNAN, models_py.GNAN), {})):
        graph = bool(rng.integers(0, 2)) and variant != "gnan_loop"
        name = f"{variant}_live{seed}"
        if variant == "gnan_loop":
            kw = dict(layers_kw="n_layers" if cls is gnan_py.GNAN else "num_layers", rho_per_feature=bool(rng.integers(0, 2)),
                      node_ids=pick(None, [2, 0, 5]))
        elif variant == "models_tensor":
            kw = dict(rho_per_feature=bool(rng.integers(0, 2)) and not graph)
        _random_model_case(str(tmp_path), name, cls, variant, rng, N=int(rng.integers(8, 30)), K_raw=int(rng.integers(2, 7)),
                           C=1 if graph else int(rng.integers(1, 6)), H=pick(8, 16, 32, 64), L=pick(1, 2, 3, 4) if variant == "gnanpy_tensor" else pick(2, 3),
                           is_graph_task=graph, normalize_rho=bool(rng.integers(0, 2)), n_isolated=int(rng.integers(0, 3)),
                           directed=bool(rng.integers(0, 2)), bias=bool(rng.integers(0, 4)), **kw)
        names.append(name)
    _random_batched_case(str(tmp_path), f"batched_live{seed}", rng, B=int(rng.integers(2, 6)), K=int(rng.integers(2, 6)), C=int(rng.integers(1, 5)),
                         H=pick(8, 16), is_graph_task=bool(rng.integers(0, 2)))
    names.append(f"batched_live{seed}")
    for i, name in enumerate(names):
        z = G.load(name)
        z["out_weight"] = np.float64(1.0)
        shape = run_port(z, torch.float64)[0].shape
        z["out_weight"] = torch.randn(shape, generator=torch.Generator().manual_seed(seed * 10 + i), dtype=torch.float64).numpy()
        # a random case may be ill-conditioned (outputs that are small differences of O(1) terms), where fp32 rounding exceeds any fixed
        # bound against float64; the algebra is checked where rounding does not enter (left: the fp32 rounding of the 1/(1+d) inputs
        # the port is fed, 6e-8, which such a case amplifies: hence 1e-6 on outputs and 2e-5 on gradients)
        out_l, fs_l, rho_l = run_lut(z)
        out_p, fs_p, rho_p, _ = run_port(z, torch.float64)
        assert out_l.shape == out_p.shape and G.rel_err(out_l.detach().numpy(), out_p.detach().numpy()) < 1e-6, name
        for got, want in ((fs_l, fs_p), (rho_l, rho_p)):
            for k in ("w1", "b1", "wh", "bh", "wo", "bo"):
                if want[k] is None or want[k].grad is None or got[k].grad is None or float(want[k].grad.norm()) == 0:
                    continue
                assert G.rel_err(got[k].grad.numpy(), want[k].grad.numpy()) < 2e-5, (name, k)
