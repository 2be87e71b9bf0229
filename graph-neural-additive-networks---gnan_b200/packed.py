"""Packed in-memory / on-disk format of a preprocessed graph-level dataset, and its batch loader.

Replaces (SURVEY.md §8f-2):
  * `processed_data/{name}.pt`: a pickled list of PyG `Data` objects each carrying two fp32 [n,n] matrices
    (pre_process_datasets.py:144-148, read back at datasets.py:124-129) = 8 bytes per node pair;
  * `batch_size=1` loaders (datasets.py:339-341: the [n,n] attributes cannot be collated) and the dense (sum n)^2
    block-diagonal collate of batched_pyg_main.py:54-91.

Here a dataset is six tensors: x [sumN,K] fp32 (constant column already appended), node_off int32 [B+1], hop uint8
[sum n_b^2] (graph b's n_b x n_b block at hop_off[b]; 255 = unreachable) = 1 byte per node pair, hop_off int64 [B+1],
level_counts int32 [sumN, nbins] (BFS level sizes, last column = unreachable) and y. It lives on the GPU; a mini-batch is
a gather of blocks (`batch(ids)` -> preprocess.PackedBatch, what the models' forward_packed takes), nothing is collated on
the host. `to_reference()` / `from_reference()` convert to and from the reference's per-graph fp32 tensors bit-exactly.
"""
from types import SimpleNamespace
from typing import Iterator, Optional, Sequence

import torch

from .preprocess import PackedBatch, apsp_batched, from_reference_format

FORMAT = "gnan_b200.packed"
VERSION = 1


class HostBundle:
    """All host tensors of one batch in ONE pinned byte buffer: a batch then crosses PCIe as a single copy (one
    cudaMemcpyAsync instead of one per tensor; twenty small copies cost more host time than a 0.2 ms training step), and the
    device side sees typed views of the staging buffer it was copied into. Offsets are 256-byte aligned."""
    ALIGN = 256

    def __init__(self, tensors: Sequence[torch.Tensor], pin: bool = True):
        self.meta, off = [], 0
        for t in tensors:
            if t.is_cuda:
                raise TypeError("HostBundle takes host tensors")
            nb = t.numel() * t.element_size()
            self.meta.append((off, nb, t.dtype, tuple(t.shape)))
            off = (off + nb + self.ALIGN - 1) // self.ALIGN * self.ALIGN
        self.payload_bytes = sum(m[1] for m in self.meta)
        self.host = torch.empty(max(off, 1), dtype=torch.uint8)
        if pin:
            self.host = self.host.pin_memory()
        for t, v in zip(tensors, self.views(self.host)):
            v.copy_(t)

    def views(self, buf: torch.Tensor):
        """typed views of `buf` (the pinned buffer itself or a device buffer of the same size), in constructor order"""
        if buf.dtype != torch.uint8 or buf.numel() != self.host.numel():
            raise TypeError("HostBundle.views: need a uint8 buffer of the bundle's size")
        return [buf[o:o + nb].view(dt).view(sh) for o, nb, dt, sh in self.meta]

    def device_buffer(self, device):
        return torch.empty(self.host.numel(), dtype=torch.uint8, device=device)

    def copy_to(self, buf: torch.Tensor):
        """the one host -> device copy (asynchronous on the current stream when the bundle is pinned)"""
        buf.copy_(self.host, non_blocking=True)
        return buf


def _ranges(starts, sizes):
    """concat_b arange(starts[b], starts[b] + sizes[b]) on the device, without a host loop."""
    total = int(sizes.sum().item())
    if total == 0:
        return torch.zeros(0, dtype=torch.int64, device=sizes.device)
    out_off = torch.cumsum(sizes, 0) - sizes
    rep = torch.repeat_interleave(torch.arange(sizes.numel(), device=sizes.device), sizes, output_size=total)
    return starts[rep] + (torch.arange(total, device=sizes.device) - out_off[rep])


class PackedDataset:
    def __init__(self, x, node_off, hop, hop_off, level_counts, y=None, max_nodes=None):
        self.x, self.node_off, self.hop, self.hop_off, self.level_counts, self.y = x, node_off, hop, hop_off, level_counts, y
        sizes = (node_off[1:] - node_off[:-1])
        self.max_nodes = int(max_nodes) if max_nodes is not None else (int(sizes.max().item()) if sizes.numel() else 1)

    # ---- construction -----------------------------------------------------------------------------------------------
    @classmethod
    def from_graphs(cls, graphs: Sequence, device="cuda", add_constant_column=True):
        """Graphs with `.x [n,K]`, `.edge_index [2,E]` (local ids) and optionally `.y`: ONE batched GPU BFS for the whole
        dataset (pre_process_datasets.py:106-122 without the per-graph Python loop) for graphs of up to
        preprocess._lib.APSP_BATCHED_MAX_NODES (1024) nodes, which covers the TU graph-classification sets (Mutagenicity, PROTEINS).
        A dataset with a larger graph, or with duplicate edges, is preprocessed graph by graph instead (same result, slower)."""
        sizes = torch.tensor([int(g.x.shape[0]) for g in graphs], dtype=torch.int64)
        node_off = torch.zeros(len(graphs) + 1, dtype=torch.int64)
        node_off[1:] = torch.cumsum(sizes, 0)
        ei = [torch.as_tensor(g.edge_index).reshape(2, -1).long() + int(node_off[i]) for i, g in enumerate(graphs)]
        ei = torch.cat(ei, dim=1) if ei else torch.zeros(2, 0, dtype=torch.int64)
        x = torch.cat([torch.as_tensor(g.x).float() for g in graphs]) if len(graphs) else torch.zeros(0, 1)
        if add_constant_column:                                              # pre_process_datasets.py:108
            x = torch.cat((x, torch.ones(x.shape[0], 1)), dim=-1)
        ys = [getattr(g, "y", None) for g in graphs]
        y = None if any(t is None for t in ys) or not ys else torch.cat([torch.as_tensor(t).reshape(1, -1) for t in ys]).squeeze(-1)
        pk = apsp_batched(ei, node_off, device=device, x=x.to(device), y=None if y is None else y.to(device))
        return cls(pk.x, pk.node_off, pk.hop, pk.hop_off, pk.level_counts, pk.y, pk.max_nodes)

    @classmethod
    def from_reference(cls, graphs: Sequence, device="cuda"):
        """Graphs already preprocessed by the reference (`.x` with the constant column, fp32 `.node_distances`,
        `.normalization_matrix`), e.g. a loaded processed_data/{name}.pt."""
        hops, cnts, sizes = [], [], []
        for g in graphs:
            hd = from_reference_format(g.node_distances.to(device), g.normalization_matrix.to(device))
            n = hd.num_nodes
            hops.append(hd.hop[:, :n].reshape(-1))
            cnts.append(hd.level_counts)
            sizes.append(n)
        nb = max(c.shape[1] for c in cnts)
        lc = torch.zeros(sum(sizes), nb, dtype=torch.int32, device=device)
        r = 0
        for c, n in zip(cnts, sizes):                                        # widen every graph to the common level range
            lc[r:r + n, :c.shape[1] - 1] = c[:, :-1]
            lc[r:r + n, -1] = c[:, -1]
            r += n
        sz = torch.tensor(sizes, dtype=torch.int64, device=device)
        node_off = torch.zeros(len(sizes) + 1, dtype=torch.int64, device=device)
        node_off[1:] = torch.cumsum(sz, 0)
        hop_off = torch.zeros(len(sizes) + 1, dtype=torch.int64, device=device)
        hop_off[1:] = torch.cumsum(sz * sz, 0)
        ys = [getattr(g, "y", None) for g in graphs]
        y = None if any(t is None for t in ys) else torch.cat([torch.as_tensor(t).reshape(1, -1) for t in ys]).squeeze(-1).to(device)
        x = torch.cat([g.x.float() for g in graphs]).to(device)
        return cls(x, node_off.to(torch.int32), torch.cat(hops).contiguous(), hop_off, lc, y, max(sizes))

    # ---- views ------------------------------------------------------------------------------------------------------
    def __len__(self):
        return self.node_off.numel() - 1

    @property
    def device(self):
        return self.hop.device

    @property
    def nbins(self):
        return self.level_counts.shape[1]

    @property
    def sizes(self):
        return (self.node_off[1:] - self.node_off[:-1]).long()

    def nbytes(self):
        ts = (self.x, self.node_off, self.hop, self.hop_off, self.level_counts) + (() if self.y is None else (self.y,))
        return sum(t.numel() * t.element_size() for t in ts)

    def to(self, device):
        mv = lambda t: None if t is None else t.to(device, non_blocking=True)
        return PackedDataset(mv(self.x), mv(self.node_off), mv(self.hop), mv(self.hop_off), mv(self.level_counts), mv(self.y),
                             self.max_nodes)

    def as_batch(self) -> PackedBatch:
        """The whole dataset as one batch (no copy; the same object every time, so per-input caches stick to it)."""
        if getattr(self, "_whole", None) is None:
            self._whole = PackedBatch(self.x, self.hop, self.hop_off, self.node_off, self.level_counts, self.y, self.max_nodes)
            self._whole._gnan_b200_persistent = True     # lives as long as the dataset: feature compression is cached on it
        return self._whole

    def batch(self, ids) -> PackedBatch:
        """Mini-batch of the graphs `ids` (any order, repeats allowed): a device gather of their blocks."""
        dev = self.device
        ids = torch.as_tensor(ids, device=dev, dtype=torch.int64).reshape(-1)
        n = self.sizes[ids]
        node_off = torch.zeros(ids.numel() + 1, dtype=torch.int64, device=dev)
        node_off[1:] = torch.cumsum(n, 0)
        hop_off = torch.zeros(ids.numel() + 1, dtype=torch.int64, device=dev)
        hop_off[1:] = torch.cumsum(n * n, 0)
        rows = _ranges(self.node_off[:-1].long()[ids], n)
        cells = _ranges(self.hop_off[:-1][ids], n * n)
        hop = self.hop[cells] if cells.numel() else torch.zeros(1, dtype=torch.uint8, device=dev)
        y = None if self.y is None else self.y[ids]
        return PackedBatch(self.x[rows], hop, hop_off, node_off.to(torch.int32), self.level_counts[rows], y,
                           int(n.max().item()) if ids.numel() else 1)

    def loader(self, batch_size: int, shuffle: bool = False, generator: Optional[torch.Generator] = None,
               drop_last: bool = False) -> Iterator[PackedBatch]:
        """Iterate once over the dataset in mini-batches (what `DataLoader(dataset, batch_size, shuffle, collate_fn=
        distance_collate_fn)` does at batched_pyg_main.py:193, minus the host collate)."""
        B = len(self)
        order = torch.randperm(B, generator=generator) if shuffle else torch.arange(B)
        if batch_size >= B and not shuffle:
            yield self.as_batch()
            return
        for s in range(0, B, batch_size):
            ids = order[s:s + batch_size]
            if drop_last and ids.numel() < batch_size:
                break
            yield self.batch(ids)

    # ---- converters -------------------------------------------------------------------------------------------------
    def to_reference(self, ids=None):
        """Per-graph objects with the reference's attributes: x, node_distances = 1/(1+hop) (0 if unreachable),
        normalization_matrix = level_counts gathered by hop (pre_process_datasets.py:112-121), y. fp32, bit-identical to
        what pre_process() attaches."""
        ids = range(len(self)) if ids is None else ids
        node_off, hop_off = self.node_off.tolist(), self.hop_off.tolist()
        nb = self.nbins
        out = []
        for b in ids:
            r0, r1 = node_off[b], node_off[b + 1]
            n = r1 - r0
            h = self.hop[hop_off[b]:hop_off[b + 1]].view(n, n).long()
            unreach = h == 255
            nd = torch.where(unreach, torch.zeros((), device=h.device), 1.0 / (h.float() + 1.0))
            cnt = self.level_counts[r0:r1].float()
            nm = torch.gather(cnt, 1, torch.where(unreach, torch.full_like(h, nb - 1), h))
            out.append(SimpleNamespace(x=self.x[r0:r1], node_distances=nd, normalization_matrix=nm,
                                       y=None if self.y is None else self.y[b:b + 1]))
        return out

    # ---- disk -------------------------------------------------------------------------------------------------------
    def save(self, path):
        cpu = lambda t: None if t is None else t.cpu()
        torch.save({"format": FORMAT, "version": VERSION, "x": cpu(self.x), "node_off": cpu(self.node_off), "hop": cpu(self.hop),
                    "hop_off": cpu(self.hop_off), "level_counts": cpu(self.level_counts), "y": cpu(self.y),
                    "max_nodes": self.max_nodes}, path)

    @classmethod
    def load(cls, path, device="cuda"):
        d = torch.load(path, map_location="cpu", weights_only=True)
        if not isinstance(d, dict) or d.get("format") != FORMAT:
            raise ValueError(f"{path} is not a {FORMAT} file")
        if d.get("version") != VERSION:
            raise ValueError(f"{path}: format version {d.get('version')} (this build reads {VERSION})")
        ds = cls(d["x"], d["node_off"], d["hop"], d["hop_off"], d["level_counts"], d["y"], d["max_nodes"])
        return ds.to(device) if device is not None else ds


# ---- node-level datasets: one graph ------------------------------------------------------------------------------------
NODE_FORMAT = "gnan_b200.node"
_NODE_EXTRAS = ("y", "train_mask", "val_mask", "test_mask", "edge_index")


def save_node(data, path):
    """One preprocessed node-task graph (`.x` with the constant column, `.hop_data`, optional y / masks / edge_index):
    N^2 bytes of hops instead of the reference's two fp32 [N,N] matrices (PubMed: 0.39 GB instead of 3.1 GB)."""
    hd = data.hop_data
    d = {"format": NODE_FORMAT, "version": VERSION, "x": data.x.cpu(), "hop": hd.hop[:, :hd.num_nodes].cpu().contiguous(),
         "level_counts": hd.level_counts.cpu(), "num_nodes": hd.num_nodes, "row_begin": hd.row_begin}
    for k in _NODE_EXTRAS:
        v = getattr(data, k, None)
        if v is not None:
            d[k] = torch.as_tensor(v).cpu()
    torch.save(d, path)


def load_node(path, device="cuda"):
    """-> SimpleNamespace(x, hop_data, y, masks...) ready for model.forward / trainer.train_epoch."""
    from .ops import hop_ld
    from .preprocess import HopData
    d = torch.load(path, map_location="cpu", weights_only=True)
    if not isinstance(d, dict) or d.get("format") != NODE_FORMAT:
        raise ValueError(f"{path} is not a {NODE_FORMAT} file")
    if d.get("version") != VERSION:
        raise ValueError(f"{path}: format version {d.get('version')} (this build reads {VERSION})")
    N = int(d["num_nodes"])
    wide = d["hop"].dtype == torch.int16                                             # deep graphs: int16 hops, -1 = unreachable
    if d["hop"].dtype not in (torch.uint8, torch.int16):
        raise ValueError(f"{path}: hop matrix of dtype {d['hop'].dtype}")
    hop = torch.full((d["hop"].shape[0], hop_ld(N)), -1 if wide else 255, dtype=d["hop"].dtype)   # row stride padded for 16-byte loads
    hop[:, :N] = d["hop"]
    out = SimpleNamespace(x=d["x"].to(device), hop_data=HopData(hop.to(device), d["level_counts"].to(device), N, int(d["row_begin"])))
    for k in _NODE_EXTRAS:
        if k in d:
            setattr(out, k, d[k].to(device))
    return out
