"""Drop-in for the reference's GNAN.py: `TensorGNAN` (GNAN.py:9-79) and `GNAN` (GNAN.py:82-176) with the same
constructor and forward signatures, computing on sm_100a kernels.

    from gnan_b200.GNAN import GNAN, TensorGNAN      # instead of `from GNAN import GNAN, TensorGNAN`

Semantics kept from the reference:
  * TensorGNAN: rho has `out_channels` outputs; `normalize_rho` divides rho's INPUT (GNAN.py:65-67); rho has no bias
    for graph tasks (:36-37); graph tasks return [C,1] (:76-79); init xavier_normal_(gain=0.01), zero biases (:49-53).
  * GNAN: rho has 1 output unless `rho_per_feature`; `normalize_rho` divides rho's OUTPUT (:163-168); default
    nn.Linear init; `forward(inputs, node_ids)` evaluates a row subset (:146-149).
What differs: x and the distance data must end up on a CUDA device (no CPU path); dropout masks come from a
counter-based generator (they cannot match torch's CPU stream; parity tests use p=0 / eval()).
"""
import torch
import torch.nn as nn

from . import ops
from ._inputs import _version, capturing, compressed_of, resolve
from ._stacked import StackedMLP
from .preprocess import PackedBatch


class _Base(nn.Module):
    precision = "fp32"      # "fp32" | "tf32x3" | "tf32": how the HxH hidden layers are contracted (see gnan_b200.h)
    dedup = True            # share shape-function evaluations between rows with equal feature values (gnan_b200.sparse) when
                            # dropout is off and the input is compressible (bag-of-words, one-hot, constant columns)

    def _device(self):
        return self.fs.wo.device

    def _seed(self):
        self._calls = getattr(self, "_calls", 0) + 1
        # _seed_salt: the first global row of a row shard (dist.row_sharded_forward): the kernels key a mask on the LOCAL row
        # index, so shards that share torch's seed would otherwise drop the same (local row, unit) pairs
        salt = int(getattr(self, "_seed_salt", 0))
        return (torch.initial_seed() * 0x9E3779B97F4A7C15 + self._calls * 0xD1B54A32D192ED03 + salt * 0xC2B2AE3D27D4EB4F) & (2 ** 63 - 1)

    def _seed_word(self):
        """Device-side half of the dropout seed: a counter advanced ON THE DEVICE by every dropout forward and snapshotted for
        that call's backward. The by-value seed above is frozen when a step is captured into a CUDA graph; this word keeps
        advancing with every replay, so captured training steps draw fresh masks."""
        dev = self._device()
        st = getattr(self, "_seed_state", None)
        if st is None or st.device != dev:
            st = torch.zeros(1, dtype=torch.int64, device=dev)
            self._seed_state = st
        st.add_(-0x61C8864680B583EB)               # += 0x9E3779B97F4A7C15 (mod 2^64)
        return st.clone()

    def _dedup_ok(self):
        return bool(self.dedup) and self.fs.n_layers >= 2 and not (self.training and self.fs.dropout > 0)

    def _features(self, holder):
        """(x on the device or None, CompressedFeatures or None) of an input object (reference Data-like or PackedBatch)."""
        dev = self._device()
        x = holder.x
        cx = compressed_of(holder, x, dev, self._dedup_ok())
        if cx is None:
            if x is None:
                raise ValueError("inputs.x is None and its compressed form cannot be used (dropout active or dedup disabled)")
            x = x.to(device=dev, dtype=torch.float32, non_blocking=True).contiguous()
        return (None if cx is not None else x), cx

    def _feature_sums(self, x, cx=None):
        if cx is not None:
            from . import sparse
            return sparse.feature_sums(cx, *self.fs.kernel_args(), precision=self.precision)
        if x.shape[1] != self.fs.groups:
            raise ValueError(f"x has {x.shape[1]} features, model was built for {self.fs.groups}")
        p = self.fs.dropout if self.training else 0.0
        return ops.mlp(x, *self.fs.kernel_args(), dropout_p=p, seed=self._seed() if p > 0 else 0, precision=self.precision,
                       seed_dev=self._seed_word() if p > 0 else None)

    def _table(self, u):
        """rho on a flat vector of scalar inputs -> [len(u), Cr]"""
        return ops.mlp(u.reshape(-1, 1), *self.rho.kernel_args(), precision=self.precision)

    def _row_tables(self, holder, u, cnt=None):
        """rho on the per-row inputs u [R,nbins] (GNAN.py:65-67: node_distances / normalization_matrix) -> [R*nbins, Cr].
        1/((1+d) * cnt) takes few distinct values (small integers): rho runs once per distinct value, rows gather."""
        if not self.dedup:
            return self._table(u)
        if capturing() and not getattr(holder, "static_level_counts", False):
            # a captured step would bake the value -> row mapping of THIS call's level counts into the graph; an in-place
            # refresh of the counts between replays would then silently gather the wrong table rows. Only objects that
            # declare their level counts immutable (holder.static_level_counts = True) keep the shared evaluation.
            return self._table(u)
        uq, inv, order, seg_ptr = _unique_inputs(holder, u, cnt)
        if uq.numel() * 2 > u.numel():
            return self._table(u)
        return ops.gather_rows(self._table(uq), inv, order, seg_ptr)

    def print_rho_params(self):
        for name, param in self.rho[0].named_parameters():     # reference key names ("0.weight", ...), GNAN.py:174-176
            print(name, param)


def _unique_inputs(holder, u, cnt=None):
    """(unique values, inverse, sort order, segment offsets) of the per-row rho inputs u [R,nbins]; they depend only on the
    BFS level sizes, so they are computed once per hop-data object and cached on it."""
    # keyed on the level-count tensor's identity AND version: an in-place refresh of the counts invalidates the mapping
    key = (tuple(u.shape), str(u.device)) + ((cnt.data_ptr(), _version(cnt)) if cnt is not None else ())
    cache = getattr(holder, "_gnan_b200_rho_unique", None)
    if cache is not None and cache[0] == key:
        return cache[1]
    uq, inv = torch.unique(u.reshape(-1), return_inverse=True)
    order = torch.sort(inv, stable=True).indices
    seg_ptr = torch.zeros(uq.numel() + 1, dtype=torch.int64, device=u.device)
    seg_ptr[1:] = torch.cumsum(torch.bincount(inv, minlength=uq.numel()), 0)
    out = (uq.contiguous(), inv.contiguous(), order.contiguous(), seg_ptr)
    try:
        holder._gnan_b200_rho_unique = (key, out)
    except Exception:
        pass
    return out


def _emit_rhos(module, state_dict, prefix, local_metadata):
    """state_dict hook of GNAN(rho_per_feature=True): `rhos.{k}.{i}.weight/bias` as the reference saves them. Entry K-1 IS
    rho (shared tensors upstream); the others are what a loaded checkpoint held, else copies of rho."""
    rho, K = module.rho, module.fs.groups
    for k in range(K):
        for i, (w, b) in zip(rho.linear_indices(), rho.layer_tensors(0)):
            for nme, t in (("weight", w), ("bias", b)):
                if t is None:
                    continue
                key = f"rhos.{k}.{i}.{nme}"
                kept = module._rhos_extra.get(key) if k < K - 1 else None
                state_dict[prefix + key] = kept if kept is not None else t.detach()
    return state_dict


def _absorb_rhos(module, state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs):
    pre = prefix + "rhos."
    for key in [k for k in state_dict if k.startswith(pre)]:
        module._rhos_extra[key[len(prefix):]] = state_dict.pop(key).detach().clone()


class TensorGNAN(_Base):
    def __init__(self, in_channels, out_channels, n_layers, hidden_channels=None, bias=True, dropout=0.0,
                 device='cpu', rho_per_feature=False, normalize_rho=True, is_graph_task=False, readout_n_layers=1):
        super().__init__()
        self.device = device
        self.out_channels = out_channels
        self.hidden_channels = hidden_channels
        self.n_layers = n_layers
        self.bias = bias
        self.dropout = dropout
        self.rho_per_feature = rho_per_feature
        self.normalize_rho = normalize_rho
        self.is_graph_task = is_graph_task
        self.fs = StackedMLP(in_channels, out_channels, n_layers, hidden_channels, bias, 3, dropout)
        self.rho = StackedMLP(1, out_channels, n_layers, hidden_channels, not is_graph_task, 2, single=True)
        self.fs.xavier_normal_(0.01)
        self.rho.xavier_normal_(0.01)

    def _aggregation(self, src, S):
        """ops.Aggregation of a resolved HopData or a PackedBatch `src`, for feature sums shaped like S"""
        dev = self._device()
        packed = isinstance(src, PackedBatch)
        kw = dict(hop_off=src.hop_off, node_off=src.node_off, reduce_graph=self.is_graph_task) if packed else {}
        if self.normalize_rho:                                                       # GNAN.py:65-67: rho(nd / norm)
            u = ops.rho_table_inputs(src.nbins, dev, cnt=src.level_counts)           # [R,nbins]
            T = self._row_tables(src, u, src.level_counts).view(S.shape[0] if packed else src.rows, src.nbins, self.out_channels)
            return ops.Aggregation(T, src.hop, per_row=True, **kw)
        T = self._table(ops.rho_table_inputs(src.nbins, dev))                        # [nbins,C]
        return ops.Aggregation(T, src.hop, **kw)

    def forward(self, inputs):
        if isinstance(inputs, PackedBatch):
            return self.forward_packed(inputs)
        dev = self._device()
        _, hd = resolve(inputs, dev, need_x=False)
        S = self._feature_sums(*self._features(inputs))                              # [N,C]   GNAN.py:57-62 (+ :73 by linearity)
        out = self._aggregation(hd, S)(S)
        if self.is_graph_task:
            out = out.sum(dim=0).view(1, -1).T                                        # [C,1]  GNAN.py:76-79
        return out


    def forward_packed(self, pk):
        """Many graphs in one call (extension; the reference trains with batch_size=1, datasets.py:339-341): `pk` is a
        preprocess.PackedBatch; returns [B,C] for graph tasks (row b == the reference's out.T for graph b) or [sumN,C]."""
        dev = self._device()
        if pk.hop.device != dev:
            pk = pk.to(dev)
        S = self._feature_sums(*self._features(pk))
        return self._aggregation(pk, S)(S)


class GNAN(_Base):
    def __init__(self, in_channels, out_channels, n_layers=None, hidden_channels=None, bias=True, dropout=0.0,
                 device='cpu', normalize_rho=True, rho_per_feature=False, num_layers=None):
        super().__init__()
        if n_layers is None:
            n_layers = num_layers                      # models.py:388 spells it num_layers (what main.py:79-83 passes)
        if n_layers is None:
            raise TypeError("n_layers (or num_layers) is required")
        self.device = device
        self.out_channels = out_channels
        self.hidden_channels = hidden_channels
        self.num_layers = n_layers
        self.bias = bias
        self.dropout = dropout
        self.rho_per_feature = rho_per_feature
        self.normalize_rho = normalize_rho
        self.fs = StackedMLP(in_channels, out_channels, n_layers, hidden_channels, bias, 3, dropout)
        self.rho = StackedMLP(1, out_channels if rho_per_feature else 1, n_layers, hidden_channels, bias, 2, single=True)
        if rho_per_feature:
            # the reference also registers `rhos`, K never-used copies of the distance MLP, the last one sharing its
            # tensors with `rho` (GNAN.py:108-124,141): carried through state_dict so that checkpoints round-trip
            self._rhos_extra = {}
            self._register_state_dict_hook(_emit_rhos)
            self.register_load_state_dict_pre_hook(_absorb_rhos)

    def _aggregation(self, hd, S=None, node_ids=None):
        """ops.Aggregation of the rows `node_ids` (all rows when None) of a resolved HopData"""
        dev = self._device()
        T = self._table(ops.rho_table_inputs(hd.nbins, dev))                         # [nbins,Cr]  rho(1/(1+d))
        hop, cnt = hd.hop, hd.level_counts
        if node_ids is not None:                                                     # row subset, GNAN.py:146-149
            ids = torch.as_tensor(node_ids, device=dev, dtype=torch.long)
            hop, cnt = hop.index_select(0, ids), cnt.index_select(0, ids)
        rs = ops.level_rscale(cnt) if self.normalize_rho else None                   # GNAN.py:163-168: rho(.) / norm
        return ops.Aggregation(T, hop, rscale=rs)

    def forward(self, inputs, node_ids=None):
        dev = self._device()
        _, hd = resolve(inputs, dev, need_x=False)
        S = self._feature_sums(*self._features(inputs))                              # f_sums, GNAN.py:150-157
        return self._aggregation(hd, S, node_ids)(S)                                 # [len(node_ids), C]
