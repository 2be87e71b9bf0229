"""Drop-in for the batched block-diagonal model of batched_pyg_main.py:98-184, plus the packed-batch form.

    model = TensorGNAN(in_channels, out_channels, n_layers, hidden_channels=16, ...)
    out = model(x_batch, dist_batch, batch_vector)        # reference call: dense [sumN,sumN] fp32, -1 off-block (:133)
    out = model(packed)                                   # gnan_b200.preprocess.PackedBatch: no (sum N)^2 tensor at all

Kept from the reference: 2-layer MLPs whatever `n_layers` says (:116-131), rho has bias and a Dropout slot (key indices
0,3), rho is fed RAW hop counts (:154), pairs with dist < 0 contribute zero AFTER rho (:158-159), graph readout is a
sum per graph (:176-181), default nn.Linear init.
"""
import torch
import torch.nn as nn

from . import ops
from ._lib import HOP_UNREACHABLE
from ._stacked import StackedMLP
from .GNAN import _Base
from .preprocess import PackedBatch


def pack_dense(x_batch, dist_batch, batch_vector):
    """dense reference batch (batched_pyg_main.py:54-91) -> PackedBatch, on the device of dist_batch."""
    dev = dist_batch.device
    bv = batch_vector.to(dev)
    B = int(bv.max().item()) + 1 if bv.numel() else 0
    sizes = torch.bincount(bv, minlength=B)
    node_off = torch.zeros(B + 1, dtype=torch.int64, device=dev)
    node_off[1:] = torch.cumsum(sizes, 0)
    hop_off = torch.zeros(B + 1, dtype=torch.int64, device=dev)
    hop_off[1:] = torch.cumsum(sizes * sizes, 0)
    # gather each node's row restricted to its own graph's columns
    n_i = sizes[bv]                                                     # [sumN] size of the node's graph
    start_i = node_off[:-1][bv]                                         # first node of the node's graph
    row_off = hop_off[:-1][bv] + (torch.arange(bv.numel(), device=dev) - start_i) * n_i
    total = int(hop_off[-1].item())
    flat_row = torch.repeat_interleave(torch.arange(bv.numel(), device=dev), n_i)
    pos = torch.arange(total, device=dev) - torch.repeat_interleave(row_off, n_i)
    d = dist_batch[flat_row, torch.repeat_interleave(start_i, n_i) + pos]
    if d.numel() and float(d.max().item()) > 254:
        raise NotImplementedError("hop distance > 254 does not fit the uint8 hop matrix")
    hop = torch.where(d < 0, torch.full_like(d, HOP_UNREACHABLE), d).round().to(torch.uint8)
    dmax = int(d.max().item()) if d.numel() else 0
    nbins = max(dmax, 0) + 2
    cnt = torch.zeros(bv.numel(), nbins, dtype=torch.int32, device=dev)   # not used by this model (no normaliser)
    return PackedBatch(x_batch.to(dev).float().contiguous(), hop.contiguous(), hop_off, node_off.to(torch.int32), cnt,
                       None, int(sizes.max().item()) if B else 1)


class TensorGNAN(_Base):
    def __init__(self, in_channels, out_channels, n_layers, hidden_channels=16, device='cpu', bias=True, dropout=0.0,
                 is_graph_task=True):
        super().__init__()
        self.device = device
        self.out_channels = out_channels
        self.is_graph_task = is_graph_task
        self.fs = StackedMLP(in_channels, out_channels, 2, hidden_channels, bias, 3, dropout)
        # the reference rho has a Dropout too (:125-131); it is only live in train mode with dropout > 0
        self.rho = StackedMLP(1, out_channels, 2, hidden_channels, bias, 3, dropout, single=True)

    def forward(self, x_batch, dist_batch=None, batch_vector=None):
        if isinstance(x_batch, PackedBatch):
            pk = x_batch
        else:
            dev = self._device()
            pk = pack_dense(x_batch.to(dev), dist_batch.to(dev), batch_vector.to(dev))
        dev = self._device()
        if pk.hop.device != dev:
            pk = pk.to(dev)
        S = self._feature_sums(*self._features(pk))
        return self._aggregation(pk, S)(S)

    def _aggregation(self, pk, S):
        """ops.Aggregation of a PackedBatch `pk` on the device, for feature sums shaped like S"""
        dev = self._device()
        nb = pk.nbins
        p = self.rho.dropout if self.training else 0.0
        keep = torch.ones(nb, 1, device=dev)
        keep[-1] = 0.0                                                                    # masked pairs: :158-159
        u = ops.rho_table_inputs(nb, dev, raw=True)                                       # d = 0..nbins-2
        kw = dict(hop_off=pk.hop_off, node_off=pk.node_off, reduce_graph=self.is_graph_task)
        if p > 0:
            # The reference runs rho (with its Dropout) on every pair (:125-131,154): an independent mask per pair. A single
            # [nbins] table would share ONE mask between all pairs at the same distance; here every ROW gets its own table
            # (independent masks per (row, distance)), so pairs of different rows are independent and only a row's pairs at
            # equal distance share a mask. Exact per-pair masks would need sum n_b^2 rho evaluations.
            n_rows = S.shape[0]
            T = ops.mlp(u.repeat(n_rows).reshape(-1, 1), *self.rho.kernel_args(), dropout_p=p, seed=self._seed(),
                        precision=self.precision, seed_dev=self._seed_word())
            T = (T.view(n_rows, nb, -1) * keep).contiguous()
            return ops.Aggregation(T, pk.hop, per_row=True, **kw)
        T = ops.mlp(u.reshape(-1, 1), *self.rho.kernel_args(), precision=self.precision) * keep
        return ops.Aggregation(T, pk.hop, **kw)
