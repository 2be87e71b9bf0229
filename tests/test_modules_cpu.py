"""CPU: host-side logic of the drop-in modules — reference state_dict keys, fs[k]/rho accessors, ctor signatures,
and that nothing silently computes on the CPU."""
import inspect

import numpy as np
import pytest
import torch

from oracle import gnan_port
from tests import _golden as G
from tests._build import build_module


@pytest.mark.parametrize("name", G.MODEL_CASES + G.BATCHED_CASES)
def test_loads_reference_state_dict(name):
    z = G.load(name)
    m = build_module(z)                      # strict load of the reference's own keys
    sd = m.state_dict()
    ref = z["sd"]                            # every key, incl. the never-used `rhos.{k}.*` of GNAN(rho_per_feature=True)
    assert sorted(sd) == sorted(ref)
    for k, v in ref.items():
        assert np.array_equal(sd[k].numpy(), v), k
    n_ref = sum(v.size for k, v in ref.items() if not k.startswith("rhos."))     # rhos[K-1] shares rho's tensors upstream
    assert sum(p.numel() for p in m.parameters()) == n_ref


@pytest.mark.parametrize("name", ["gnanpy_tensor_node", "gnanpy_tensor_node_l1", "gnanpy_tensor_node_l4", "batched_graph"])
def test_shape_function_accessors_match_oracle(name):
    z = G.load(name)
    m = build_module(z).eval()
    t = torch.linspace(-2, 2, 9).view(-1, 1)
    fs = gnan_port.to_torch(z["fs"]); rho = gnan_port.to_torch(z["rho"])
    for k in (0, z["K"] - 1):
        assert torch.allclose(m.fs[k](t), gnan_port.scalar_mlp(fs, k, t), atol=1e-6)
        assert torch.allclose(m.fs[k].forward(t), gnan_port.scalar_mlp(fs, k, t), atol=1e-6)
    assert torch.allclose(m.rho(t), gnan_port.scalar_mlp(rho, 0, t), atol=1e-6)
    assert len(m.fs) == z["K"]
    names = [n for n, _ in m.rho.reference_named_parameters()]
    assert names[0] == "0.weight"
    # nn.Module semantics are intact: leaf Parameters an optimizer can take (ADVICE round 1)
    assert all(isinstance(p, torch.nn.Parameter) and p.is_leaf for p in m.rho.parameters())
    torch.optim.Adam(m.rho.parameters(), lr=1e-3)


def test_constructor_signatures_match_reference():
    from gnan_b200 import GNAN as g, batched as b, models as mo
    want = ["in_channels", "out_channels", "n_layers", "hidden_channels", "bias", "dropout", "device", "rho_per_feature",
            "normalize_rho", "is_graph_task", "readout_n_layers"]
    assert list(inspect.signature(g.TensorGNAN.__init__).parameters)[1:] == want      # GNAN.py:10-11
    assert list(inspect.signature(mo.TensorGNAN.__init__).parameters)[1:] == want     # models.py:304-305
    assert list(inspect.signature(mo.GNAN.__init__).parameters)[1:4] == ["in_channels", "out_channels", "num_layers"]
    assert list(inspect.signature(g.GNAN.__init__).parameters)[1:10] == [
        "in_channels", "out_channels", "n_layers", "hidden_channels", "bias", "dropout", "device", "normalize_rho",
        "rho_per_feature"]                                                               # GNAN.py:83-84
    assert list(inspect.signature(b.TensorGNAN.__init__).parameters)[1:] == [
        "in_channels", "out_channels", "n_layers", "hidden_channels", "device", "bias", "dropout", "is_graph_task"]
    assert list(inspect.signature(g.GNAN.forward).parameters)[1:] == ["inputs", "node_ids"]


def test_reference_init_statistics():
    from gnan_b200.GNAN import GNAN, TensorGNAN
    torch.manual_seed(0)
    m = TensorGNAN(40, 7, 3, 64)
    assert float(m.fs.b1.abs().max()) == 0.0                       # GNAN.py:52-53
    assert abs(float(m.fs.wh.std()) - 0.01 * (2 / 128) ** 0.5) < 2e-5   # xavier_normal_(gain=0.01), GNAN.py:51
    g = GNAN(40, 7, 3, 64)
    assert abs(float(g.fs.wh.abs().max()) - 1 / 8) < 1e-3          # nn.Linear default: U(-1/sqrt(64), 1/sqrt(64))
    assert not hasattr(m.rho, "nonexistent")
    assert TensorGNAN(4, 1, 3, 8, is_graph_task=True).rho.has_bias is False     # GNAN.py:36-37


def test_no_cpu_fallback():
    """Forward on CPU tensors must fail loudly, never compute."""
    from types import SimpleNamespace
    from gnan_b200._lib import GnanError
    z = G.load("gnanpy_tensor_node")
    m = build_module(z)
    data = SimpleNamespace(x=torch.tensor(z["x"]), node_distances=torch.tensor(z["node_distances"]),
                           normalization_matrix=torch.tensor(z["normalization_matrix"]))
    with pytest.raises((GnanError, RuntimeError)):
        m.forward(data)


def test_trainer_auc_matches_sklearn_and_signatures_match_reference():
    import inspect
    from sklearn.metrics import roc_auc_score
    from gnan_b200 import trainer
    rng = np.random.default_rng(0)
    for n in (7, 200):
        y = rng.integers(0, 2, size=n); y[0], y[1] = 0, 1
        s = np.round(rng.random(n), 1 if n > 50 else 3)            # the coarse rounding creates ties
        assert abs(trainer.roc_auc(torch.tensor(y), torch.tensor(s)) - roc_auc_score(y, s)) < 1e-12
    assert list(inspect.signature(trainer.train_epoch).parameters) == [
        "model", "dloader", "loss_fn", "optimizer", "device", "classify", "label_index", "compute_auc", "is_graph_task",
        "capture_steps"]                                                  # the reference's nine (trainer.py:23) + one opt-in extension
    assert list(inspect.signature(trainer.test_epoch).parameters) == [
        "model", "dloader", "loss_fn", "device", "classify", "label_index", "compute_auc", "val_mask", "is_graph_task"]


def test_trainer_label_handling_follows_reference():
    from types import SimpleNamespace
    from gnan_b200 import trainer
    bce, ce = torch.nn.BCEWithLogitsLoss(), torch.nn.CrossEntropyLoss()
    d = SimpleNamespace(y=torch.tensor([[-1.0, 1.0], [1.0, -1.0]]))
    assert trainer._labels_of(d, bce, 0).tolist() == [0.0, 1.0]          # trainer.py:33-39 ({-1,1} -> {0,1}, column pick)
    assert trainer._labels_of(d, bce, 1).tolist() == [1.0, 0.0]
    d = SimpleNamespace(y=torch.tensor([2, 0, 1]))
    lab = trainer._labels_of(d, ce, 0)
    assert lab.dtype == torch.long and lab.tolist() == [2, 0, 1]
    out = torch.tensor([[0.3], [-0.2], [2.0]])
    assert trainer.get_accuracy(out, torch.tensor([1.0, 0.0, 0.0])) == 2  # trainer.py:5-12
    assert int(trainer.get_accuracy(torch.tensor([[0.1, 0.9], [0.8, 0.2]]), torch.tensor([1, 1]))) == 1


def _toy_packed():
    from gnan_b200.packed import PackedDataset
    sizes = [2, 3, 1]
    hops = [torch.tensor([[0, 1], [1, 0]]), torch.tensor([[0, 1, 255], [1, 0, 255], [255, 255, 0]]), torch.tensor([[0]])]
    node_off = torch.tensor([0, 2, 5, 6], dtype=torch.int32)
    hop_off = torch.tensor([0, 4, 13, 14], dtype=torch.int64)
    hop = torch.cat([h.reshape(-1) for h in hops]).to(torch.uint8)
    cnt = torch.tensor([[1, 1, 0], [1, 1, 0], [1, 1, 1], [1, 1, 1], [1, 0, 2], [1, 0, 0]], dtype=torch.int32)
    x = torch.arange(12, dtype=torch.float32).view(6, 2)
    return PackedDataset(x, node_off, hop, hop_off, cnt, torch.tensor([1, 0, 1])), hops


def test_packed_dataset_batch_gather_save_load_and_reference_view(tmp_path):
    """Host logic of the packed format (pure tensor indexing: runs on any device)."""
    from gnan_b200.packed import PackedDataset
    ds, hops = _toy_packed()
    assert len(ds) == 3 and ds.nbins == 3 and ds.max_nodes == 3
    b = ds.batch([2, 0])
    assert b.node_off.tolist() == [0, 1, 3] and b.hop_off.tolist() == [0, 1, 5]
    assert b.hop.tolist() == [0, 0, 1, 1, 0] and b.x.tolist() == [[10.0, 11.0], [0.0, 1.0], [2.0, 3.0]]
    assert b.level_counts.tolist() == [[1, 0, 0], [1, 1, 0], [1, 1, 0]] and b.y.tolist() == [1, 1] and b.max_nodes == 2
    seen = []
    for pk in ds.loader(2, shuffle=True, generator=torch.Generator().manual_seed(0)):
        seen += pk.y.tolist()
        assert pk.hop.numel() == int(pk.hop_off[-1])
    assert sorted(seen) == [0, 1, 1]
    path = tmp_path / "toy.gnan_b200.pt"
    ds.save(path)
    back = PackedDataset.load(path, device=None)
    for k in ("x", "node_off", "hop", "hop_off", "level_counts", "y"):
        assert torch.equal(getattr(back, k), getattr(ds, k)), k
    with pytest.raises(ValueError):
        torch.save({"format": "something else"}, tmp_path / "bad.pt")
        PackedDataset.load(tmp_path / "bad.pt", device=None)
    ref = ds.to_reference()
    g = ref[1]                                                           # pre_process_datasets.py:112-121 on the 3-node graph
    assert torch.equal(g.node_distances, torch.tensor([[1.0, 0.5, 0.0], [0.5, 1.0, 0.0], [0.0, 0.0, 1.0]]))
    assert torch.equal(g.normalization_matrix, torch.tensor([[1.0, 1.0, 1.0], [1.0, 1.0, 1.0], [2.0, 2.0, 1.0]]))


def test_compress_features_structure_and_roundtrip():
    """Host logic of gnan_b200.sparse.compress_features (pure tensor ops): baseline = column mode, exceptions in CSC order,
    CSR view, work items; exact reconstruction; density cut-off."""
    from gnan_b200.sparse import TILE, compress_features
    rng = np.random.default_rng(0)
    N, K = 300, 7
    x = np.zeros((N, K), np.float32)
    x[:, 0] = 1.0                                                # constant column (pre_process_datasets.py:108)
    x[rng.integers(0, N, 40), 1] = rng.normal(size=40)           # sparse column
    x[:, 2] = rng.integers(0, 2, N)                              # binary column: baseline = the more frequent of {0,1}
    x[np.arange(N), 3 + rng.integers(0, 3, N)] = 1.0             # one-hot over columns 3..5
    x[:200, 6] = 2.5                                             # 200 x 2.5, the rest zeros -> baseline 2.5
    xt = torch.tensor(x)
    cx = compress_features(xt, max_density=0.5)
    assert cx is not None and cx.num_rows == N and cx.num_features == K
    assert torch.equal(cx.to_dense(), xt)
    assert cx.base[0] == 1.0 and cx.base[6] == 2.5 and cx.base[1] == 0.0
    gp = cx.grp_ptr.tolist()
    assert gp[1] - gp[0] == 1                                    # constant column: the baseline only
    assert gp[7] - gp[6] == 1 + 100
    for k in range(K):
        assert cx.ent_row[gp[k]] == -1 and float(cx.val[gp[k]]) == float(cx.base[k])
        rows = cx.ent_row[gp[k] + 1:gp[k + 1]]
        assert bool((rows[1:] > rows[:-1]).all())               # exceptions sorted by row inside a group
        assert bool((cx.ent_grp[gp[k]:gp[k + 1]] == k).all())
    # CSR view lists exactly the exceptions of each row
    cp = cx.csr_ptr.tolist()
    assert cp[-1] == cx.num_entries - K
    for r in (0, 17, N - 1):
        eids = cx.csr_eid[cp[r]:cp[r + 1]]
        assert bool((cx.ent_row[eids] == r).all())
        assert sorted(cx.ent_grp[eids].tolist()) == sorted(np.nonzero(x[r] != cx.base.numpy())[0].tolist())
    # work items: every (group, tile) exactly once
    want = [(k, t) for k in range(K) for t in range((gp[k + 1] - gp[k] + TILE - 1) // TILE)]
    assert [tuple(i) for i in cx.items.tolist()] == want and cx.max_group == max(gp[k + 1] - gp[k] for k in range(K))
    # compact host copy (narrow index arrays for the PCIe transfer, per-entry values dropped when values are shared): same
    # content, fewer bytes
    ch = cx.compact_host()
    assert ch.ent_row.dtype == torch.int32 and ch.csr_eid.dtype == torch.int32 and ch.ent_grp.dtype == torch.uint8
    assert cx.shared is not None and ch.val.numel() == 0 and ch.shared.inv.dtype in (torch.uint8, torch.int16)
    assert ch.nbytes() < 0.6 * cx.nbytes()
    assert all(torch.equal(a.long(), b.long()) for a, b in zip(ch._tensors(), cx._tensors()) if a.numel() == b.numel() and not a.dtype.is_floating_point)
    assert torch.equal(ch.shared.val, cx.shared.val) and torch.equal(ch.base, cx.base)
    assert torch.equal(ch.to_dense(), xt)
    plain = compress_features(xt, max_density=0.5, share_values=False).compact_host()      # no sharing: the values travel
    assert plain.val.numel() == plain.ent_row.numel() and torch.equal(plain.to_dense(), xt)
    assert compress_features(torch.tensor(rng.normal(size=(50, 4)).astype(np.float32))) is None      # dense data: not worth it
    assert compress_features(torch.tensor(rng.normal(size=(50, 4)).astype(np.float32)), max_density=None) is not None


def test_local_edges_host_form():
    """preprocess.LocalEdges.from_edge_index: uint8 endpoints inside the graph + per-graph edge offsets; unsorted edge lists are
    grouped by graph (stable); cross-graph edges and graphs of more than 256 nodes raise."""
    from gnan_b200.preprocess import LocalEdges
    node_off = np.array([0, 3, 3, 8, 264])
    ei = torch.tensor([[4, 0, 263, 1, 7, 8], [5, 2, 8, 0, 3, 263]])
    le = LocalEdges.from_edge_index(ei, node_off)
    assert le.src.dtype == torch.uint8 and le.edge_off.dtype == torch.int32 and le.nbytes() == 12 + 20
    assert le.edge_off.tolist() == [0, 2, 2, 4, 6]
    assert le.src.tolist() == [0, 1, 1, 4, 255, 0] and le.dst.tolist() == [2, 0, 2, 0, 0, 255]
    with pytest.raises(ValueError):
        LocalEdges.from_edge_index(torch.tensor([[0], [3]]), node_off)                 # leaves its graph
    with pytest.raises(ValueError):
        LocalEdges.from_edge_index(torch.tensor([[0], [1]]), np.array([0, 300]))       # too large for uint8 indices


def test_host_bundle_views_roundtrip():
    """packed.HostBundle: tensors of mixed dtypes / shapes (empty ones included) in one byte buffer, typed views give them back"""
    from gnan_b200.packed import HostBundle
    ts = [torch.arange(7, dtype=torch.uint8), torch.randn(3, 5), torch.zeros(0, dtype=torch.int64), torch.arange(-3, 9, dtype=torch.int16),
          torch.arange(6, dtype=torch.int64).reshape(2, 3), torch.tensor([1.5])]
    hb = HostBundle(ts, pin=False)
    assert hb.payload_bytes == sum(t.numel() * t.element_size() for t in ts) and hb.host.numel() % HostBundle.ALIGN == 0
    other = torch.zeros_like(hb.host)
    hb.copy_to(other)
    for t, v in zip(ts, hb.views(other)):
        assert v.dtype == t.dtype and v.shape == t.shape and torch.equal(v, t)
    with pytest.raises(TypeError):
        hb.views(torch.zeros(3, dtype=torch.uint8))


def test_feature_compression_policy():
    """_inputs.compressed_of: explicit x_compressed is always honoured; implicit building only for persistent, large inputs."""
    from types import SimpleNamespace
    from gnan_b200 import _inputs
    from gnan_b200.preprocess import PackedBatch
    from gnan_b200.sparse import CompressedFeatures, compress_features
    big = torch.zeros(_inputs.AUTO_DEDUP_MIN_EVALUATIONS // 8, 8)
    big[::7, 3] = 1.0
    small = big[:50]
    holder = SimpleNamespace(x=big)
    cx = _inputs.compressed_of(holder, big, "cpu")
    assert isinstance(cx, CompressedFeatures) and holder._gnan_b200_cx_cache[1] is cx
    assert _inputs.compressed_of(holder, big, "cpu") is cx                              # cached on the object
    big[0, 0] = 5.0                                                                      # in-place edit bumps the version: rebuilt
    assert _inputs.compressed_of(holder, big, "cpu") is not cx
    assert _inputs.compressed_of(SimpleNamespace(x=small), small, "cpu") is None        # too small to be worth analysing
    assert _inputs.compressed_of(holder, big, "cpu", enabled=False) is None             # dropout active / model.dedup = False
    dense = torch.randn(big.shape)
    h2 = SimpleNamespace(x=dense)
    assert _inputs.compressed_of(h2, dense, "cpu") is None and h2._gnan_b200_cx_cache[1] is None   # analysed once, verdict cached
    pk = PackedBatch(big, None, None, torch.tensor([0, big.shape[0]], dtype=torch.int32), None)
    assert _inputs.compressed_of(pk, big, "cpu") is None                                # a per-step batch object is never analysed
    pk._gnan_b200_persistent = True
    assert _inputs.compressed_of(pk, big, "cpu") is not None
    explicit = compress_features(small, max_density=None)
    assert _inputs.compressed_of(SimpleNamespace(x=None, x_compressed=explicit), None, "cpu") is explicit


def test_value_sharing_of_compressed_features_cpu():
    """gnan_b200.sparse: entries of a feature with equal values collapse to one evaluation (one-hot columns, row-normalised
    bags of words); the mapping reproduces the entries exactly and is skipped when nothing coincides."""
    from gnan_b200.sparse import compress_features
    g = torch.Generator().manual_seed(0)
    n = 500
    onehot = torch.zeros(n, 6)
    onehot[torch.arange(n), torch.randint(0, 5, (n,), generator=g)] = 1.0
    onehot[:, 5] = 1.0
    cx = compress_features(onehot)
    assert torch.equal(cx.to_dense(), onehot)
    assert cx.shared is not None and cx.num_evaluations == 5 * 2 + 1 and cx.num_entries == n + 6
    sh = cx.shared
    assert torch.equal(sh.val[sh.inv], cx.val)
    grp_of = torch.repeat_interleave(torch.arange(6), sh.grp_ptr[1:] - sh.grp_ptr[:-1])
    assert torch.equal(grp_of[sh.inv].int(), cx.ent_grp)
    assert torch.equal(torch.sort(sh.inv, stable=True).indices, sh.order)
    assert int(sh.seg_ptr[-1]) == cx.num_entries and sh.seg_ptr.numel() == cx.num_evaluations + 1
    cont = torch.rand(200, 4, generator=g) * (torch.rand(200, 4, generator=g) < 0.2)
    c2 = compress_features(cont)
    assert c2.shared is None and c2.num_evaluations == c2.num_entries
    assert compress_features(onehot, share_values=False).shared is None
    moved = cx.clone_tensors()
    moved.copy_tensors_(cx)
    assert torch.equal(moved.shared.inv, sh.inv) and moved.nbytes() == cx.nbytes()


def test_round2_host_logic_without_a_gpu():
    """PackedBatch carrying only the fused normaliser; the optimizer and the fused losses refuse CPU tensors (no fallback)."""
    import pytest
    from gnan_b200 import _lib
    from gnan_b200.optim import Adam
    from gnan_b200.preprocess import PackedBatch
    pk = PackedBatch(None, torch.zeros(4, dtype=torch.uint8), torch.tensor([0, 4]), torch.tensor([0, 2], dtype=torch.int32), None,
                     level_rscale=torch.ones(2, 48))
    assert pk.nbins == 48 and pk.num_graphs == 1 and pk.to("cpu").level_rscale.shape == (2, 48)
    p = torch.nn.Parameter(torch.zeros(3))
    p.grad = torch.ones(3)
    with pytest.raises((TypeError, _lib.GnanError)):
        Adam([p], lr=1e-3).step()
    with pytest.raises(ValueError):
        Adam([p], lr=-1.0)
    from gnan_b200 import ops
    with pytest.raises(_lib.GnanError):
        ops.bce_with_logits(torch.zeros(3, requires_grad=True), torch.zeros(3))


@pytest.mark.parametrize("wide", [False, True])
def test_node_file_roundtrip_keeps_hop_dtype_and_padding(tmp_path, wide):
    """packed.save_node / load_node on host tensors: the uint8 form (255 = unreachable) and the int16 form of deep graphs
    (-1 = unreachable) both come back with their dtype, their unreachable marker in the padding columns and a 16-element row stride."""
    from types import SimpleNamespace

    from gnan_b200.ops import hop_ld
    from gnan_b200.packed import load_node, save_node
    from gnan_b200.preprocess import HopData
    N, R = 21, 5
    g = torch.Generator().manual_seed(3)
    if wide:
        hop = torch.randint(0, 400, (R, hop_ld(N)), generator=g).to(torch.int16)
        hop[1, 3] = -1
    else:
        hop = torch.randint(0, 9, (R, hop_ld(N)), generator=g).to(torch.uint8)
        hop[1, 3] = 255
    cnt = torch.randint(0, 5, (R, 11), generator=g).to(torch.int32)
    data = SimpleNamespace(x=torch.randn(R, 4, generator=g), hop_data=HopData(hop, cnt, N, row_begin=16), y=torch.arange(R),
                           train_mask=torch.tensor([True, False, True, False, True]))
    path = tmp_path / "node.gnan_b200.pt"
    save_node(data, path)
    back = load_node(path, device="cpu")
    hd = back.hop_data
    assert hd.hop.dtype == hop.dtype and hd.wide == wide and hd.hop.shape == (R, hop_ld(N))
    assert torch.equal(hd.hop[:, :N], hop[:, :N]) and bool((hd.hop[:, N:] == (-1 if wide else 255)).all())
    assert torch.equal(hd.level_counts, cnt) and hd.num_nodes == N and hd.row_begin == 16
    assert torch.equal(back.x, data.x) and torch.equal(back.y, data.y) and torch.equal(back.train_mask, data.train_mask)
    assert not hasattr(back, "val_mask")
    torch.save({"format": "gnan_b200.node", "version": 1, "x": data.x, "hop": hop[:, :N].float(), "level_counts": cnt,
                "num_nodes": N, "row_begin": 0}, tmp_path / "bad.pt")
    with pytest.raises(ValueError):
        load_node(tmp_path / "bad.pt", device="cpu")


def test_reference_format_inputs_are_converted_once_and_again_after_an_in_place_refresh(monkeypatch):
    """_inputs.resolve caches the compact hop data of a reference-style Data object (fp32 node_distances / normalization_matrix) on
    the object; the cache key carries both tensors' version counters, so `copy_` into either matrix triggers a new conversion, and
    inference tensors (no version counter) are accepted."""
    from types import SimpleNamespace

    from gnan_b200 import _inputs
    from gnan_b200.preprocess import HopData
    calls = []

    def fake_convert(nd, nm):
        calls.append((nd.clone(), None if nm is None else nm.clone()))
        return HopData(torch.zeros(nd.shape[0], 16, dtype=torch.uint8), torch.zeros(nd.shape[0], 3, dtype=torch.int32), nd.shape[1])
    monkeypatch.setattr(_inputs, "from_reference_format", fake_convert)
    nd, nm = torch.rand(4, 4), torch.ones(4, 4)
    data = SimpleNamespace(x=torch.rand(4, 2), node_distances=nd, normalization_matrix=nm)
    _, hd1 = _inputs.resolve(data, "cpu")
    _, hd2 = _inputs.resolve(data, "cpu")
    assert hd1 is hd2 and len(calls) == 1
    nd.copy_(torch.rand(4, 4))
    _, hd3 = _inputs.resolve(data, "cpu")
    assert hd3 is not hd1 and len(calls) == 2 and torch.equal(calls[1][0], nd)
    nm.mul_(2.0)
    _inputs.resolve(data, "cpu")
    assert len(calls) == 3 and torch.equal(calls[2][1], nm)
    _inputs.resolve(data, "cpu")
    assert len(calls) == 3
    with torch.inference_mode():
        frozen = SimpleNamespace(x=torch.rand(4, 2), node_distances=torch.rand(4, 4), normalization_matrix=None)
    _inputs.resolve(frozen, "cpu"); _inputs.resolve(frozen, "cpu")
    assert len(calls) == 4
    with pytest.raises(AttributeError):
        _inputs.resolve(SimpleNamespace(x=torch.rand(4, 2)), "cpu")


@pytest.mark.parametrize("name", G.MODEL_CASES + G.BATCHED_CASES)
def test_checkpoints_keep_the_reference_layout_in_both_directions(name):
    """The gnan_b200 -> reference direction of test_loads_reference_state_dict: a FRESH module of a golden case's configuration (no
    reference weights loaded) writes exactly the keys, shapes and dtypes the reference module wrote for that case (the sd.* arrays), so
    its checkpoint loads strictly into the reference class. After the strict load of the reference's checkpoint, the per-feature
    accessors `fs[k]` / `rho` evaluate the reference's Sequential (oracle/gnan_port.scalar_mlp, float64) on the stored weights."""
    from gnan_b200 import GNAN as g
    z = G.load(name)
    ref = {k: torch.from_numpy(v) for k, v in z["sd"].items()}
    fresh = [build_module(z, load=False)]
    if z["variant"] == "gnan_loop":                      # both copies of the reference's GNAN class write the same layout
        fresh.append(g.GNAN(z["K"], z["C"], n_layers=z["L"], hidden_channels=z["H"], bias=z["bias"], normalize_rho=z["normalize_rho"],
                            rho_per_feature=z["rho_per_feature"]))
    for m in fresh:
        sd = m.state_dict()
        assert sorted(sd) == sorted(ref), (type(m).__module__, sorted(set(sd) ^ set(ref)))
        for k, v in sd.items():
            assert v.shape == ref[k].shape and v.dtype == ref[k].dtype, k
    m = build_module(z).eval()
    t = torch.linspace(-1.5, 1.5, 7).view(-1, 1)
    fs, rho = gnan_port.to_torch(z["fs"], torch.float64), gnan_port.to_torch(z["rho"], torch.float64)
    for k in range(z["K"]):
        assert torch.allclose(m.fs[k](t).double(), gnan_port.scalar_mlp(fs, k, t.double()), rtol=1e-5, atol=1e-5), k
    assert torch.allclose(m.rho(t).double(), gnan_port.scalar_mlp(rho, 0, t.double()), rtol=1e-5, atol=1e-5)


def test_product_package_never_imports_the_oracle_or_the_tests():
    """The oracle is test infrastructure: nothing under the package directory (nor the import alias) may import `oracle`, `tests`, `baseline`
    or the reference's module names; bench.py may, and only inside its reference / cpu_baseline functions."""
    import ast
    import glob
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    files = glob.glob(os.path.join(root, "graph-neural-additive-networks---gnan_b200", "*.py")) + glob.glob(os.path.join(root, "gnan_b200", "*.py"))
    assert len(files) >= 15
    banned = {"oracle", "tests", "baseline", "pre_process_datasets", "batched_pyg_main", "scipy", "networkx"}
    for f in files:
        for node in ast.walk(ast.parse(open(f).read())):
            mods = []
            if isinstance(node, ast.Import):
                mods = [a.name for a in node.names]
            elif isinstance(node, ast.ImportFrom) and node.level == 0 and node.module:
                mods = [node.module]
            for mname in mods:
                assert mname.split(".")[0] not in banned, (os.path.basename(f), mname)
    bench = ast.parse(open(os.path.join(root, "bench.py")).read())
    allowed = {"reference_step_fn", "reference_apsp_record"}
    for fn in [n for n in ast.walk(bench) if isinstance(n, ast.FunctionDef)]:
        for node in ast.walk(fn):
            if isinstance(node, ast.ImportFrom) and node.module and node.module.split(".")[0] == "oracle":
                assert fn.name in allowed, fn.name
    assert not [n for n in bench.body if isinstance(n, (ast.Import, ast.ImportFrom)) and "oracle" in ast.dump(n)]
