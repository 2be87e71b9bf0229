"""Interpretability export: the curves the reference's notebook plots (mutagenicity_visualizations.ipynb cells 4-9,
README.md:29-31), evaluated in bulk on the GPU from the stacked parameters instead of one `model.fs[i].forward(t)` /
`model.m.forward(val)` call per point.

    f   = shape_function_table(model, grid)            # [len(grid), K, C]   f_k(t)            (cell 6 uses t = 1.0)
    rho = distance_function_table(model, max_distance) # [D+1, C_rho]        rho(1/(1+d))      (cell 4)
    z   = heatmap(model, max_distance)                 # [K, D+1]            f_k(1) * rho(d)   (cell 9: np.outer)

and the per-prediction decomposition the model exists to give (GNAN.py:68-70 forms it as mf before summing over features):

    e = explain(model, inputs, node_ids=None)
    e.out       # [R,C]        the eval-mode fp32 output these contributions decompose
    e.features  # [R,K,C]      contribution of shape function k to output row r; sums over k to e.out
    e.nodes     # [sum N,C]    graph tasks: contribution of each node to its graph's output (None for the NAM readout / node tasks)
"""
from typing import NamedTuple, Optional

import torch
from torch import Tensor

from . import ops


def shape_function_table(model, grid):
    """f_k(t) for every feature k and every t in `grid` (1-D tensor / list) -> [len(grid), K, C]."""
    st = model.fs
    dev = st.wo.device
    t = torch.as_tensor(grid, dtype=torch.float32, device=dev).reshape(-1)
    u = t.view(-1, 1).expand(-1, st.groups).contiguous()
    with torch.no_grad():
        return ops.mlp_per_group(u, *st.kernel_args(), precision="fp32")


def distance_function_table(model, max_distance, raw=None):
    """rho at the hop distances d = 0..max_distance -> [max_distance+1, C_rho]. The distance models feed rho 1/(1+d)
    (GNAN.py:65-67, notebook cell 4); the batched variant feeds the raw hop count d (batched_pyg_main.py:154), which is
    selected automatically for gnan_b200.batched.TensorGNAN or with raw=True."""
    st = model.rho
    dev = st.wo.device
    if raw is None:
        raw = model.__class__.__module__.endswith(".batched")
    u = ops.rho_table_inputs(int(max_distance) + 2, dev, raw=bool(raw))[: int(max_distance) + 1]      # drop the unreachable bin
    with torch.no_grad():
        return ops.mlp(u.reshape(-1, 1).contiguous(), *st.kernel_args(), precision="fp32")


def heatmap(model, max_distance, x_value=1.0, channel=0):
    """z[k,d] = f_k(x_value)[channel] * rho(d)[channel or 0]: the feature x distance contribution map of notebook cell 9."""
    f = shape_function_table(model, [x_value])[0, :, channel]                    # [K]
    r = distance_function_table(model, max_distance)
    r = r[:, channel if r.shape[1] > 1 else 0]                                   # [D+1]
    return torch.outer(f, r)


class Explanation(NamedTuple):
    out: Tensor
    features: Tensor
    nodes: Optional[Tensor]


def explain(model, inputs, node_ids=None) -> Explanation:
    """Exact additive attributions of the eval-mode model with fp32 shape-function kernels.

    model: GNAN.TensorGNAN / GNAN.GNAN / models.TensorGNAN / models.GNAN / batched.TensorGNAN; inputs: whatever its forward takes (a
    reference-style Data with node_distances / normalization_matrix or hop_data, a preprocess.PackedBatch, deferred or not, or for
    batched.TensorGNAN the (x_batch, dist_batch, batch_vector) tuple). Rows R: node tasks the rows `node_ids` (default all,
    duplicates allowed); a graph task on one graph 1; a packed graph task B; packed node-level output sum N.

    With W[i,j,c'] the aggregation weight of the module (DESIGN.md §2):
      node rows   features[i,k,c] = sum_j W[i,j,c'] f_k(x_jk)[c]
      graph rows  features[b,k,c] = sum_{i in b} features[i,k,c],  nodes[j,c] = sum_{i in graph(j)} W[i,j,c'] * S[j,c]
      NAM readout features[b,k,c] = g_k(hidden[b,k])[c]  (models.py:374-381), nodes None
    so that sum_k features[r] = out[r] and, for graph rows, sum_{j in b} nodes[j] = out[b] (to fp32 rounding)."""
    training, precision = model.training, model.precision
    model.eval()
    model.precision = "fp32"
    try:
        with torch.no_grad():
            return _explain(model, inputs, node_ids)
    finally:
        model.train(training)
        model.precision = precision


def _explain(model, inputs, node_ids):
    from . import batched, sparse
    from ._inputs import compressed_of, resolve
    from .GNAN import GNAN as RowGNAN
    from .preprocess import PackedBatch
    dev = model._device()
    dense_batch = isinstance(model, batched.TensorGNAN) and not isinstance(inputs, PackedBatch)
    if dense_batch:
        x_batch, dist_batch, batch_vector = inputs
        src = holder = batched.pack_dense(x_batch.to(dev), dist_batch.to(dev), batch_vector.to(dev))
    elif isinstance(inputs, PackedBatch):
        src = holder = inputs if inputs.node_off.device == dev else inputs.to(dev)
    else:
        _, src = resolve(inputs, dev, need_x=False)
        holder = inputs
        if src.wide:
            raise NotImplementedError("explain: int16 hop matrices (hop distances > 254) are not covered")
    packed = isinstance(src, PackedBatch)
    graph = bool(getattr(model, "is_graph_task", False))
    if graph and node_ids is not None:
        raise ValueError("node_ids selects rows of a node task; a graph task explains its graphs")
    if node_ids is not None:
        # the rows kernel takes them as hop-row / table indices on the device: out-of-range ids are refused here
        ids = torch.as_tensor(node_ids, dtype=torch.long)
        limit = int(src.node_off[-1]) if packed else src.rows
        if ids.numel() and (int(ids.min()) < 0 or int(ids.max()) >= limit):
            raise IndexError(f"node_ids must lie in [0, {limit})")
    if dense_batch:
        out = model(x_batch, dist_batch, batch_vector)
    else:
        out = model(inputs, node_ids) if isinstance(model, RowGNAN) else model(inputs)
    if graph and not packed:
        out = out.T                                                                  # [C,1] -> [1,C]
    elif node_ids is not None and not isinstance(model, RowGNAN):
        out = out[torch.as_tensor(node_ids, device=out.device, dtype=torch.long)]

    cx = compressed_of(holder, holder.x, dev)
    if cx is None:
        cx = sparse.compress_features(holder.x.to(dev), max_density=None)
    Y = sparse.entry_values(cx, *model.fs.kernel_args())                            # [E,Cf]: f_k of every entry
    S = sparse.entries_to_rows(Y, cx.grp_ptr, cx.csr_ptr, cx.csr_eid, cx.ent_grp, cx.ent_row)     # [N,Cf]
    N = S.shape[0]
    node_off = src.node_off if packed else torch.tensor([0, N], dtype=torch.int32, device=dev)
    seg = ops.explain_segments(cx.grp_ptr, cx.ent_row, node_off)
    agg = model._aggregation(src, S)
    if graph:
        # colw[j,c] = sum_{i in graph(j)} W[i,j,c']: the aggregation's backward for a unit output gradient (it is channel-wise)
        unit = torch.ones_like(S).requires_grad_()
        with torch.enable_grad():
            colw = torch.autograd.grad(agg(unit).sum(), unit)[0].contiguous()
        colw_sum = ops.gather_segment_sum(colw, None, node_off.long())
        F = ops.explain_graph_features(Y, cx.grp_ptr, cx.ent_row, seg, colw, colw_sum)
        if getattr(model, "_readout", False):
            nam = model.readout_nam.fs
            return Explanation(out, ops.mlp_per_group(F[:, :, 0].contiguous(), *nam.kernel_args(), precision="fp32"), None)
        return Explanation(out, F, colw * S)
    rows = None if node_ids is None else torch.as_tensor(node_ids, device=dev, dtype=torch.long)
    n_rows = (N if packed else src.rows) if rows is None else rows.numel()
    ncols = src.num_nodes if not packed else (src.max_nodes or int((node_off[1:] - node_off[:-1]).max()) if N else 0)
    F = ops.explain_rows_features(agg.hop, agg.hop_off, node_off, ncols, rows, n_rows, agg.T,
                                  agg.per_row, agg.rscale, Y, cx.grp_ptr, cx.ent_row, seg)
    return Explanation(out, F, None)
