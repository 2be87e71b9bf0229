"""Compressed feature matrix: evaluate every shape function once per DISTINCT work item instead of once per (node, feature).

When dropout is off, all rows that carry the same value in feature column k see the same f_k output and (by linearity of
the backward in dS) can share one backward evaluation fed the SUM of their dS rows. The reference's inputs are made for
this: Cora / PubMed bag-of-words rows are ~99 % / ~90 % zeros (datasets.py:94), Mutagenicity atoms are one-hot, and
pre_process() appends a constant column (pre_process_datasets.py:108,127). SURVEY.md §8d allows the shortcut as long as
achieved FLOPs are counted on the evaluations actually executed (bench.py does).

Representation (built once per dataset, cached next to the hop data): per feature k a baseline value base[k] (the
column's most frequent value) plus the list of exceptions (row, value) that differ from it, in CSC order:

    val      fp32  [E]    entries grouped by feature; group k = [base[k], exceptions of k sorted by row]
    grp_ptr  int64 [K+1]
    ent_row  int64 [E]    row of an exception, -1 for a baseline
    ent_grp  int32 [E]    feature of an entry
    csr_ptr  int64 [N+1], csr_eid int64 [n_exc]   the exception entries of each row (for the row gather)
    items    int32 [n_items,2]                    (feature, 128-entry tile) work list of the forward kernel

    S[r,:] = sum_k Y[base_k,:] + sum_{e in exceptions(r)} (Y[e,:] - Y[base_k(e),:]),     Y[e,:] = f_k(e)(val[e])

The C ABI side is gnan_mlp_entries_fwd_ex/bwd + gnan_entries_to_rows / gnan_rows_to_entries (include/gnan_b200.h); all fp32
kernels, deterministic. With dropout active the modules fall back to the dense kernels (per-row masks break the sharing).
"""
from typing import Optional

import torch
from torch import Tensor

from . import ops
from ._lib import MlpGrads, check, load, ptr, stream_handle

TILE = 128                  # entries per forward work item (rows per CTA tile of the MLP kernels)
MAX_DENSITY = 0.25          # build a compressed form only if exceptions / (N*K) is below this


class ValueSharing:
    """Second level of sharing: entries of a feature that carry the SAME value (every `1` of a one-hot column, the few
    distinct 1/len values of a row-normalised bag of words) are one evaluation. uq_* describe the distinct (feature, value)
    pairs like val / grp_ptr / items describe the entries; Y_entry = Y_distinct[inv], and the backward of that gather is a
    fixed-order segment sum over `order` / `seg_ptr` (ops.gather_rows: deterministic)."""
    _FIELDS = ("val", "grp_ptr", "items", "inv", "order", "seg_ptr")

    def __init__(self, val, grp_ptr, items, inv, order, seg_ptr, max_group):
        self.val, self.grp_ptr, self.items, self.inv, self.order, self.seg_ptr = val, grp_ptr, items, inv, order, seg_ptr
        self.max_group = int(max_group)

    _I64 = ("grp_ptr", "inv", "order", "seg_ptr")        # kernel-side dtype of the index fields (a compact host copy may hold int32)

    def map(self, fn):
        return ValueSharing(*[fn(getattr(self, f)) for f in self._FIELDS], self.max_group)

    def map_named(self, fn):
        return ValueSharing(*[fn(f, getattr(self, f)) for f in self._FIELDS], self.max_group)


class CompressedFeatures:
    _FIELDS = ("base", "val", "grp_ptr", "ent_row", "ent_grp", "csr_ptr", "csr_eid", "items")

    def __init__(self, num_rows, base, val, grp_ptr, ent_row, ent_grp, csr_ptr, csr_eid, items, max_group, shared=None):
        self.num_rows = int(num_rows)
        self.base, self.val, self.grp_ptr, self.ent_row, self.ent_grp = base, val, grp_ptr, ent_row, ent_grp
        self.csr_ptr, self.csr_eid, self.items = csr_ptr, csr_eid, items
        self.max_group = int(max_group)
        self.shared = shared            # ValueSharing or None

    _I64 = ("grp_ptr", "ent_row", "csr_ptr", "csr_eid")

    def _map(self, fn):
        return CompressedFeatures(self.num_rows, *[fn(getattr(self, f)) for f in self._FIELDS], self.max_group,
                                  None if self.shared is None else self.shared.map(fn))

    def _map_named(self, fn):
        return CompressedFeatures(self.num_rows, *[fn(f, getattr(self, f)) for f in self._FIELDS], self.max_group,
                                  None if self.shared is None else self.shared.map_named(fn))

    def compact_host(self):
        """Host-side copy for transfers, every index array in the narrowest integer type that holds its values (int64 -> int32,
        feature ids and value ids -> uint8 / int16 when they fit); with shared values the per-entry `val` array is dropped (it is
        shared.val[shared.inv]: the kernels never read it then). `.to(device)` / `copy_tensors_` widen again on the device.
        One-hot molecule batch: 14 bytes per entry + 4 per row cross PCIe instead of 28 + 4."""
        def shrink(t, narrow):
            if t.dtype in (torch.int64, torch.int32) and t.numel():
                lo, hi = int(t.min()), int(t.max())
                for dt, a, b in ((torch.uint8, 0, 255), (torch.int16, -2 ** 15, 2 ** 15 - 1), (torch.int32, -2 ** 31, 2 ** 31 - 1)):
                    if (narrow or dt == torch.int32) and lo >= a and hi <= b:
                        return t.to(dt)
            return t

        def f(name, t):
            t = t.cpu()
            if name == "val" and self.shared is not None and t.numel() == self.ent_row.numel():
                return t.new_empty(0)
            return shrink(t, name in ("ent_grp", "inv"))
        sh = None if self.shared is None else self.shared.map_named(lambda n, t: shrink(t.cpu(), n == "inv"))
        return CompressedFeatures(self.num_rows, *[f(n, getattr(self, n)) for n in self._FIELDS], self.max_group, sh)

    @property
    def num_evaluations(self):
        """shape-function evaluations per pass: distinct (feature, value) pairs when values are shared, else the entries"""
        return self.shared.val.numel() if self.shared is not None else self.val.numel()

    @property
    def num_features(self):
        return self.base.numel()

    @property
    def num_entries(self):
        return self.val.numel()

    @property
    def device(self):
        return self.val.device

    def density(self):
        return (self.num_entries - self.num_features) / max(1, self.num_rows * self.num_features)

    def _tensors(self):
        out = [getattr(self, f) for f in self._FIELDS]
        if self.shared is not None:
            out += [getattr(self.shared, f) for f in ValueSharing._FIELDS]
        return out

    def nbytes(self):
        return sum(t.numel() * t.element_size() for t in self._tensors())

    @staticmethod
    def _kernel_dtype(own, name, t):
        """dtype the kernels read a field in (a compact host copy may hold something narrower)"""
        if not t.dtype.is_floating_point:
            return torch.int64 if name in own._I64 else torch.int32
        return t.dtype

    def to(self, device, raw=False):
        """raw=True keeps a compact copy's narrow dtypes on the device (to be widened by copy_tensors_ into preallocated tensors)"""
        on_gpu = torch.device(device).type == "cuda"

        def move(own):
            def f(name, t):
                t = t.to(device, non_blocking=True)
                if on_gpu and not raw:                                          # a compact host copy: widen on the device
                    t = t.to(self._kernel_dtype(own, name, t))
                return t
            return f
        sh = None if self.shared is None else self.shared.map_named(move(ValueSharing))
        out = CompressedFeatures(self.num_rows, *[move(CompressedFeatures)(f, getattr(self, f)) for f in self._FIELDS], self.max_group, sh)
        if on_gpu and not raw and sh is not None and out.val.numel() == 0 and out.ent_row.numel():
            out.val = sh.val[sh.inv]
        return out

    def pin_memory(self):
        return self._map(lambda t: t.pin_memory())

    def clone_tensors(self):
        return self._map(lambda t: t.clone())

    def copy_tensors_(self, other):
        """In-place refresh from another compressed form of the SAME structure sizes (static inputs of a CUDA graph)."""
        for dst, src in zip(self._tensors(), other._tensors()):
            if src.numel() == dst.numel():                  # copy_ widens a compact copy's narrow index types
                dst.copy_(src, non_blocking=True)
        if other.val.numel() != self.val.numel():           # compact copy with shared values: the per-entry values are derived
            torch.index_select(self.shared.val, 0, self.shared.inv, out=self.val)
        return self

    def to_dense(self):
        """x [N,K] back (exactly)."""
        x = self.base.unsqueeze(0).repeat(self.num_rows, 1)
        exc = self.ent_row >= 0
        val = self.val if self.val.numel() == self.ent_row.numel() else self.shared.val[self.shared.inv.long()]   # compact copy
        x[self.ent_row[exc].long(), self.ent_grp[exc].long()] = val[exc]
        return x


MAX_SHARED_FRACTION = 0.5   # share equal values only if the distinct (feature, value) pairs are at most this fraction of the entries


def _tiles_of(sizes, K, dev):
    tiles = (sizes + TILE - 1) // TILE
    n_items = int(tiles.sum().item())
    item_grp = torch.repeat_interleave(torch.arange(K, device=dev), tiles, output_size=n_items)
    item_tile = torch.arange(n_items, device=dev) - (torch.cumsum(tiles, 0) - tiles)[item_grp]
    return torch.stack([item_grp, item_tile], dim=1).to(torch.int32).contiguous()


def _share_values(val, ent_grp, K):
    """ValueSharing of the entries (val [E], ent_grp [E]) or None when too few entries coincide."""
    dev = val.device
    E = val.numel()
    key = (ent_grp.long() << 32) | (val.view(torch.int32).long() & 0xFFFFFFFF)      # sorted by feature, then by value bits
    uq, inv = torch.unique(key, sorted=True, return_inverse=True)
    if uq.numel() > MAX_SHARED_FRACTION * E:
        return None
    uq_grp = uq >> 32
    uq_val = (uq & 0xFFFFFFFF).to(torch.int32).view(torch.float32)
    sizes = torch.bincount(uq_grp, minlength=K)
    grp_ptr = torch.zeros(K + 1, dtype=torch.int64, device=dev)
    grp_ptr[1:] = torch.cumsum(sizes, 0)
    order = torch.sort(inv, stable=True).indices
    seg_ptr = torch.zeros(uq.numel() + 1, dtype=torch.int64, device=dev)
    seg_ptr[1:] = torch.cumsum(torch.bincount(inv, minlength=uq.numel()), 0)
    return ValueSharing(uq_val.contiguous(), grp_ptr, _tiles_of(sizes, K, dev), inv.contiguous(), order.contiguous(), seg_ptr,
                        int(sizes.max().item()))


def compress_features(x: Tensor, max_density: Optional[float] = MAX_DENSITY, share_values: bool = True) -> Optional[CompressedFeatures]:
    """x [N,K] (any device) -> CompressedFeatures on x's device, or None when more than `max_density` of the entries differ
    from their column's most frequent value (the dense kernels are the better choice then). One-off cost: a column-wise
    mode and a few sorts; synchronises."""
    if x.dim() != 2:
        raise ValueError("x must be [N,K]")
    x = x.detach().float()
    N, K = x.shape
    dev = x.device
    if N == 0 or K == 0:
        return None
    base = torch.mode(x, dim=0).values.contiguous()                           # most frequent value of each column
    mask = x != base.unsqueeze(0)
    n_exc = int(mask.sum().item())
    if max_density is not None and n_exc > max_density * N * K:
        return None
    cols, rows = mask.t().nonzero(as_tuple=True)                              # CSC order: by feature, then by row
    counts = torch.bincount(cols, minlength=K)
    sizes = counts + 1                                                        # + the baseline entry
    grp_ptr = torch.zeros(K + 1, dtype=torch.int64, device=dev)
    grp_ptr[1:] = torch.cumsum(sizes, 0)
    E = K + n_exc
    exc_start = torch.cumsum(counts, 0) - counts                              # first exception of each column in the CSC list
    eid = grp_ptr[:-1][cols] + 1 + (torch.arange(n_exc, device=dev) - exc_start[cols])
    val = torch.empty(E, dtype=torch.float32, device=dev)
    val[grp_ptr[:-1]] = base
    val[eid] = x[rows, cols]
    ent_row = torch.full((E,), -1, dtype=torch.int64, device=dev)
    ent_row[eid] = rows
    ent_grp = torch.repeat_interleave(torch.arange(K, device=dev, dtype=torch.int32), sizes, output_size=E)
    order = torch.sort(rows, stable=True).indices                             # CSR view of the same exceptions
    csr_eid = eid[order].contiguous()
    csr_ptr = torch.zeros(N + 1, dtype=torch.int64, device=dev)
    csr_ptr[1:] = torch.cumsum(torch.bincount(rows, minlength=N), 0)
    items = _tiles_of(sizes, K, dev)
    shared = _share_values(val, ent_grp, K) if share_values else None
    return CompressedFeatures(N, base, val, grp_ptr, ent_row, ent_grp, csr_ptr, csr_eid, items, int(sizes.max().item()), shared)


# ---------------------------------------------------------------------------------------------------------------------
# ops
# ---------------------------------------------------------------------------------------------------------------------
@torch.library.custom_op("gnan_b200::mlp_entries_fwd", mutates_args=())
def mlp_entries_fwd(val: Tensor, grp_ptr: Tensor, items: Tensor, w1: Tensor, b1: Tensor, wh: Tensor, bh: Tensor, wo: Tensor,
                    bo: Tensor, n_layers: int, max_group: int, precision: int) -> Tensor:
    lib = load()
    val, w1, b1, wh, bh, wo, bo = (ops._f32(t, n) for t, n in zip((val, w1, b1, wh, bh, wo, bo), "val w1 b1 wh bh wo bo".split()))
    if grp_ptr.dtype != torch.int64 or items.dtype != torch.int32 or grp_ptr.numel() != wo.shape[0] + 1:
        raise TypeError("grp_ptr must be int64 [G+1], items int32 [n,2]")
    p, G, H, C = ops._mlp_params(w1, b1, wh, bh, wo, bo, n_layers)
    E = val.numel()
    Y = torch.empty(E, C, dtype=torch.float32, device=val.device)
    with ops._timed("mlp_entries_fwd"):
        check(lib.gnan_mlp_entries_fwd_ex(ptr(val), ptr(grp_ptr), E, ptr(items.contiguous()), items.shape[0], p, precision, ptr(Y),
                                          stream_handle()), "gnan_mlp_entries_fwd_ex")
    return Y


@mlp_entries_fwd.register_fake
def _(val, grp_ptr, items, w1, b1, wh, bh, wo, bo, n_layers, max_group, precision):
    return val.new_empty(val.numel(), wo.shape[1])


@torch.library.custom_op("gnan_b200::mlp_entries_bwd", mutates_args=())
def mlp_entries_bwd(val: Tensor, grp_ptr: Tensor, w1: Tensor, b1: Tensor, wh: Tensor, bh: Tensor, wo: Tensor, bo: Tensor,
                    n_layers: int, max_group: int, precision: int, dY: Tensor) -> tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    lib = load()
    val, w1, b1, wh, bh, wo, bo, dY = (ops._f32(t, n) for t, n in zip((val, w1, b1, wh, bh, wo, bo, dY), "val w1 b1 wh bh wo bo dY".split()))
    p, G, H, C = ops._mlp_params(w1, b1, wh, bh, wo, bo, n_layers)
    outs = [torch.empty_like(t) for t in (w1, b1, wh, bh, wo, bo)]
    g = MlpGrads(*[ptr(t) for t in outs], None)
    ws = ops._ws(lib.gnan_mlp_entries_workspace_bytes(max_group, p, 1, precision), val.device)
    with ops._timed("mlp_entries_bwd"):
        check(lib.gnan_mlp_entries_bwd(ptr(val), ptr(grp_ptr), val.numel(), max_group, p, precision, ptr(dY), g, ptr(ws), ws.numel(),
                                       stream_handle()), "gnan_mlp_entries_bwd")
    return tuple(outs)


@mlp_entries_bwd.register_fake
def _(val, grp_ptr, w1, b1, wh, bh, wo, bo, n_layers, max_group, precision, dY):
    return tuple(torch.empty_like(t) for t in (w1, b1, wh, bh, wo, bo))


def _entries_setup(ctx, inputs, output):
    val, grp_ptr, items, w1, b1, wh, bh, wo, bo, n_layers, max_group, precision = inputs
    ctx.save_for_backward(val, grp_ptr, w1, b1, wh, bh, wo, bo)
    ctx.cfg = (n_layers, max_group, precision)


def _entries_backward(ctx, dY):
    val, grp_ptr, w1, b1, wh, bh, wo, bo = ctx.saved_tensors
    g = mlp_entries_bwd(val, grp_ptr, w1, b1, wh, bh, wo, bo, ctx.cfg[0], ctx.cfg[1], ctx.cfg[2], dY.contiguous())
    return (None, None, None) + tuple(g) + (None, None, None)


mlp_entries_fwd.register_autograd(_entries_backward, setup_context=_entries_setup)


@torch.library.custom_op("gnan_b200::entries_to_rows", mutates_args=())
def entries_to_rows(Y: Tensor, grp_ptr: Tensor, csr_ptr: Tensor, csr_eid: Tensor, ent_grp: Tensor, ent_row: Tensor) -> Tensor:
    lib = load()
    Y = ops._f32(Y, "Y")
    N, G, C = csr_ptr.numel() - 1, grp_ptr.numel() - 1, Y.shape[1]
    S = torch.empty(N, C, dtype=torch.float32, device=Y.device)
    S0 = torch.empty(C, dtype=torch.float32, device=Y.device)
    with ops._timed("entries_to_rows"):
        check(lib.gnan_entries_to_rows(ptr(Y), N, G, C, ptr(grp_ptr), ptr(csr_ptr), ptr(csr_eid), ptr(ent_grp), ptr(S0), ptr(S),
                                       stream_handle()), "gnan_entries_to_rows")
    return S


@entries_to_rows.register_fake
def _(Y, grp_ptr, csr_ptr, csr_eid, ent_grp, ent_row):
    return Y.new_empty(csr_ptr.numel() - 1, Y.shape[1])


@torch.library.custom_op("gnan_b200::rows_to_entries", mutates_args=())
def rows_to_entries(dS: Tensor, grp_ptr: Tensor, ent_row: Tensor) -> Tensor:
    lib = load()
    dS = ops._f32(dS, "dS")
    N, C = dS.shape
    G, E = grp_ptr.numel() - 1, ent_row.numel()
    dY = torch.empty(E, C, dtype=torch.float32, device=dS.device)
    tot = torch.empty(lib.gnan_rows_to_entries_scratch_floats(G, C, E), dtype=torch.float32, device=dS.device)
    with ops._timed("rows_to_entries"):
        check(lib.gnan_rows_to_entries(ptr(dS), N, G, C, ptr(grp_ptr), E, ptr(ent_row), ptr(tot), ptr(dY), stream_handle()),
              "gnan_rows_to_entries")
    return dY


@rows_to_entries.register_fake
def _(dS, grp_ptr, ent_row):
    return dS.new_empty(ent_row.numel(), dS.shape[1])


def _e2r_setup(ctx, inputs, output):
    Y, grp_ptr, csr_ptr, csr_eid, ent_grp, ent_row = inputs
    ctx.save_for_backward(grp_ptr, ent_row)


def _e2r_backward(ctx, dS):
    grp_ptr, ent_row = ctx.saved_tensors
    return rows_to_entries(dS.contiguous(), grp_ptr, ent_row), None, None, None, None, None


entries_to_rows.register_autograd(_e2r_backward, setup_context=_e2r_setup)


def entry_values(cx: CompressedFeatures, w1, b1, wh, bh, wo, bo, n_layers, precision="fp32") -> Tensor:
    """Y [E,C] = f_k(val[e]) for every entry e of the compressed form (k = ent_grp[e]); differentiable w.r.t. the weights.
    `precision` selects the kernels (fp32 FFMA, or the tcgen05 3xTF32 kernels for H = 64, 3 layers, C <= 8), forward and
    backward. A single Linear(1,C) (n_layers = 1, which the entries kernels do not take) is an affine map per feature."""
    if wo.shape[0] != cx.num_features:
        raise ValueError(f"compressed x has {cx.num_features} features, the model {wo.shape[0]}")
    if int(n_layers) == 1:
        g = cx.ent_grp.long()
        return cx.val[:, None] * wo[g, :, 0] + bo[g]
    from ._lib import PRECISIONS
    sh = cx.shared
    if sh is not None:      # one evaluation per distinct (feature, value); entries gather it (backward: fixed-order segment sums)
        Yq = mlp_entries_fwd(sh.val, sh.grp_ptr, sh.items, w1, b1, wh, bh, wo, bo, int(n_layers), sh.max_group, PRECISIONS[precision])
        return ops.gather_rows(Yq, sh.inv, sh.order, sh.seg_ptr)
    return mlp_entries_fwd(cx.val, cx.grp_ptr, cx.items, w1, b1, wh, bh, wo, bo, int(n_layers), cx.max_group, PRECISIONS[precision])


def feature_sums(cx: CompressedFeatures, w1, b1, wh, bh, wo, bo, n_layers, precision="fp32") -> Tensor:
    """S [N,C] = sum_k f_k(x[:,k]) from the compressed form (entry_values, then the baseline + exceptions sum of each row)."""
    Y = entry_values(cx, w1, b1, wh, bh, wo, bo, n_layers, precision)
    return entries_to_rows(Y, cx.grp_ptr, cx.csr_ptr, cx.csr_eid, cx.ent_grp, cx.ent_row)
