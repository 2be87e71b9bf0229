"""Drop-in for the GNAN classes of the reference's models.py (what main.py imports, main.py:2,77-90):
`TensorGNAN` (models.py:303-384), `GNAN` (models.py:387-481, identical math to GNAN.py's, kw `num_layers`).

Differences from GNAN.py's TensorGNAN that are honoured here (models.py:320-321,366-370):
  * rho has ONE output unless `rho_per_feature` (then out_channels);
  * `normalize_rho` divides rho's OUTPUT by the normalisation matrix;
  * graph task with `readout_n_layers > 0`: shape functions and rho have ONE output, the aggregated value is kept per
    feature (hidden[k] = sum_i sum_j W_ij f_k(x_jk), :374-379) and a `NAM` (:258-300) over those K values produces the
    graph output (:380-381). The per-feature form runs on the same kernels: f's output layer is expanded to a
    block-diagonal [K,K,H] weight so that "channel" k of the kernel's feature sum is f_k alone (K <= 64).
"""
import torch

from . import ops
from ._inputs import resolve
from ._stacked import StackedMLP
from .GNAN import GNAN as _GNAN, _Base
from .preprocess import PackedBatch


class NAM(_Base):
    """models.py:258-300: out[r,:] = sum_k g_k(x[r,k]) on the grouped-MLP kernel."""

    def __init__(self, in_channels, out_channels, num_layers, hidden_channels=None, bias=True, dropout=0.0, device='cpu'):
        super().__init__()
        self.device = device
        self.out_channels = out_channels
        self.hidden_channels = hidden_channels
        self.num_layers = num_layers
        self.bias = bias
        self.dropout = dropout
        self.fs = StackedMLP(in_channels, out_channels, num_layers, hidden_channels, bias, 3, dropout)

    def forward(self, x):
        return self._feature_sums(x.to(self._device()).float().contiguous())


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
        self.readout_n_layers = readout_n_layers
        self._readout = bool(is_graph_task and readout_n_layers > 0)
        self.actual_output_dim_f = 1 if self._readout else out_channels                       # models.py:320-321
        self.actual_output_dim_rho = 1 if (not rho_per_feature or self._readout) else out_channels
        self.fs = StackedMLP(in_channels, self.actual_output_dim_f, n_layers, hidden_channels, bias, 3, dropout)
        self.rho = StackedMLP(1, self.actual_output_dim_rho, n_layers, hidden_channels, not is_graph_task, 2, single=True)
        if self._readout:
            self.readout_nam = NAM(in_channels, out_channels, readout_n_layers, hidden_channels, bias, dropout, device)
            self.readout_nam.fs.xavier_normal_(0.01)                                 # models.py:352-356 covers it too
        self.fs.xavier_normal_(0.01)
        self.rho.xavier_normal_(0.01)

    def _per_feature(self, x):
        """Y[j,k] = f_k(x_jk) (one output per shape function): the kernel sums over features per channel, so give feature
        k its own channel through a block-diagonal output layer (ops.mlp_per_group)."""
        if x.shape[1] != self.fs.groups:
            raise ValueError(f"x has {x.shape[1]} features, model was built for {self.fs.groups}")
        p = self.fs.dropout if self.training else 0.0
        return ops.mlp_per_group(x, *self.fs.kernel_args(), dropout_p=p, seed=self._seed() if p > 0 else 0,
                                 precision=self.precision, seed_dev=self._seed_word() if p > 0 else None).squeeze(-1)   # [N,K,1] -> [N,K]

    def _aggregation(self, src, S):
        """ops.Aggregation of a resolved HopData or a PackedBatch `src`, for feature sums shaped like S"""
        dev = self._device()
        T = self._table(ops.rho_table_inputs(src.nbins, dev))                        # [nbins,Cr]
        if not isinstance(src, PackedBatch):
            rs = ops.level_rscale(src.level_counts) if self.normalize_rho else None  # models.py:368-370
            return ops.Aggregation(T, src.hop, rscale=rs)
        if (src.deferred and self.normalize_rho and self.is_graph_task and T.dim() == 2 and ops.BLOCKDIAG_GRAPH_KERNEL
                and ops.load().gnan_aggregate_blockdiag_graph_supported(T.shape[0], T.shape[1], S.shape[1])):
            # distances not computed yet (preprocess.apsp_batched on a LocalEdges batch): the BFS and this readout run as one
            # kernel, neither the hop bytes nor the normaliser table are ever written (models.py:366-384)
            return ops.Aggregation(T, node_off=src.node_off, reduce_graph=True, fused=(src.edges, src.max_nodes, src.status))
        rs = None
        if self.normalize_rho:       # models.py:368-370; a batch straight from apsp_batched(..., rscale=True) carries it already
            rs = src.level_rscale if getattr(src, "level_rscale", None) is not None else ops.level_rscale(src.level_counts)
        return ops.Aggregation(T, src.hop, rscale=rs, hop_off=src.hop_off, node_off=src.node_off, reduce_graph=self.is_graph_task)

    def forward(self, inputs):
        if isinstance(inputs, PackedBatch):
            return self.forward_packed(inputs)
        dev = self._device()
        if self._readout:
            x, hd = resolve(inputs, dev)
            S = self._per_feature(x)
        else:
            _, hd = resolve(inputs, dev, need_x=False)
            S = self._feature_sums(*self._features(inputs))
        out = self._aggregation(hd, S)(S)
        if self._readout:
            hidden = out.sum(dim=0).view(1, -1)                                      # [1,K]  models.py:379
            return self.readout_nam(hidden).T                                        # [C,1]  models.py:380-384
        if self.is_graph_task:
            out = out.sum(dim=0).view(1, -1).T
        return out


    def forward_packed(self, pk):
        """Many graphs in one call (extension; see gnan_b200.GNAN.TensorGNAN.forward_packed): [B,C] for graph tasks."""
        dev = self._device()
        if pk.node_off.device != dev:
            pk = pk.to(dev)
        S = self._per_feature(pk.x.float().contiguous()) if self._readout else self._feature_sums(*self._features(pk))
        out = self._aggregation(pk, S)(S)
        return self.readout_nam(out) if self._readout else out                       # [B,K] -> [B,C]


class GNAN(_GNAN):
    def __init__(self, in_channels, out_channels, num_layers, hidden_channels=None, bias=True, dropout=0.0,
                 device='cpu', normalize_rho=True, rho_per_feature=False):
        super().__init__(in_channels, out_channels, n_layers=num_layers, hidden_channels=hidden_channels, bias=bias,
                         dropout=dropout, device=device, normalize_rho=normalize_rho, rho_per_feature=rho_per_feature)
