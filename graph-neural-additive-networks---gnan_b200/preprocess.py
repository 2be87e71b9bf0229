"""GPU all-pairs hop-distance preprocessing with the reference's `pre_process` call shape.

Reference: pre_process_datasets.py:104-148 (append a constant-1 feature column, all-pairs Dijkstra on unit weights,
node_distances = 1/(1+d) with inf -> 0, normalization_matrix[i,j] = #{j': d(i,j') = d(i,j)}), and the per-node
networkx BFS of batched_pyg_main.py:36-44. Here the distances stay integers: a uint8 hop matrix (255 = unreachable)
plus int32 BFS level sizes; the reference's two fp32 [N,N] matrices are derived views (HopData.reference_format()).

Duplicate edges: the reference's COO->LIL conversion sums a (src,dst) pair listed k times into ONE edge of weight k
(pre_process_datasets.py:109,129), and its Dijkstra then returns weighted distances. The CSR builder detects duplicates and
`apsp` / `apsp_batched` emulate that behaviour exactly by subdividing such an edge into a chain of k unit edges through
k-1 virtual nodes (dropped from the result): distances stay integers, bit-exact with the reference (tested against scipy).
"""
from typing import List, Optional, Sequence

import torch

from . import _lib
from ._lib import check, load, ptr, stream_handle
from .ops import hop_ld


class HopData:
    """Compact distance data of one graph (or a row shard [row_begin, row_begin+R) of it).

    hop          uint8 [R, ld]  hop count, 255 = unreachable; columns >= N are padding
                 (deep graphs, a hop distance > 254: int16 [R, ld], -1 = unreachable; see csrc/wide.cu and `wide`)
    level_counts int32 [R, nbins]  cnt[i,d] = #{j : hop[i,j] = d}, last column = #unreachable; nbins = D+2
    """

    def __init__(self, hop, level_counts, num_nodes, row_begin=0):
        self.hop = hop
        self.level_counts = level_counts
        self.num_nodes = int(num_nodes)
        self.row_begin = int(row_begin)

    @property
    def nbins(self):
        return self.level_counts.shape[1]

    @property
    def rows(self):
        return self.hop.shape[0]

    @property
    def wide(self):
        """True for the int16 form (hop distances beyond 254)"""
        return self.hop.dtype == torch.int16

    def to(self, device):
        return HopData(self.hop.to(device, non_blocking=True), self.level_counts.to(device, non_blocking=True),
                       self.num_nodes, self.row_begin)

    def reference_format(self):
        """(node_distances, normalization_matrix) as fp32 [R,N], bit-identical to pre_process_datasets.py:112-121."""
        lib = load()
        R, N = self.rows, self.num_nodes
        if self.wide:                                     # deep graphs: same arithmetic (fp32 division) with device tensor ops
            h = self.hop[:, :N].long()
            nd = torch.where(h < 0, torch.zeros((), device=h.device), 1.0 / (h.float() + 1.0))
            b = torch.where(h < 0, torch.full_like(h, self.nbins - 1), h.clamp(max=self.nbins - 1))
            return nd, torch.gather(self.level_counts, 1, b).float()
        nd = torch.empty(R, N, dtype=torch.float32, device=self.hop.device)
        nm = torch.empty(R, N, dtype=torch.float32, device=self.hop.device)
        check(lib.gnan_hops_to_reference(ptr(self.hop), R, N, self.hop.shape[1], ptr(self.level_counts), self.nbins,
                                         ptr(nd), ptr(nm), stream_handle()), "gnan_hops_to_reference")
        return nd, nm


def from_reference_format(node_distances, normalization_matrix=None):
    """fp32 [R,N] reference tensors (on the GPU) -> HopData. One device sync to size the level table."""
    lib = load()
    nd = node_distances.contiguous()
    if nd.dtype != torch.float32:
        raise TypeError("node_distances must be float32")
    R, N = nd.shape
    dev = nd.device
    pos = nd[nd > 0]
    dmax = int(torch.round(1.0 / pos.min() - 1.0).item()) if pos.numel() else 0
    if dmax > 254:
        return _from_reference_wide(nd, normalization_matrix, dmax)
    nbins = dmax + 2
    hop = torch.empty(R, hop_ld(N), dtype=torch.uint8, device=dev)
    cnt = torch.zeros(R, nbins, dtype=torch.int32, device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    nm = None if normalization_matrix is None else normalization_matrix.contiguous().float()
    check(lib.gnan_hops_from_reference(ptr(nd), ptr(nm), R, N, ptr(hop), hop.shape[1], ptr(cnt), nbins, ptr(flag),
                                       stream_handle()), "gnan_hops_from_reference")
    return HopData(hop, cnt, N)


WIDE_MAX_LEVEL = 32766      # deepest level of the int16 hop matrix


def _from_reference_wide(nd, normalization_matrix, dmax):
    """from_reference_format for hop distances beyond 254: int16 hops (-1 = unreachable)"""
    if dmax > WIDE_MAX_LEVEL:
        raise NotImplementedError(f"hop distance {dmax} > {WIDE_MAX_LEVEL} does not fit the int16 hop matrix")
    lib = load()
    R, N = nd.shape
    nbins = dmax + 2
    hop = torch.full((R, hop_ld(N)), -1, dtype=torch.int16, device=nd.device)
    h = torch.where(nd > 0, torch.round(1.0 / nd - 1.0), torch.full_like(nd, -1.0))
    hop[:, :N] = h.to(torch.int16)
    cnt = torch.zeros(R, nbins, dtype=torch.int32, device=nd.device)
    if normalization_matrix is None:
        check(lib.gnan_level_counts16(ptr(hop), R, N, hop.shape[1], ptr(cnt), nbins, stream_handle()), "gnan_level_counts16")
    else:                                                  # the counts are whatever the caller's normaliser says (as the uint8 converter)
        b = torch.where(h < 0, torch.full_like(h, float(nbins - 1)), h).long()
        cnt.scatter_(1, b, torch.round(normalization_matrix.float()).to(torch.int32))
    return HopData(hop, cnt, N)


def _apsp_wide(rowptr, col, N, row_begin, row_end, device):
    """Rows [row_begin,row_end) of the hop matrix of a graph whose diameter exceeds 254: int16 hops by a warp-per-source BFS,
    then the level histogram sized by the deepest level found (one device sync)."""
    lib = load()
    R = row_end - row_begin
    hop = torch.empty(R, hop_ld(N), dtype=torch.int16, device=device)
    st = torch.zeros(2, dtype=torch.int32, device=device)              # [overflow, deepest level]
    ws = torch.empty(max(lib.gnan_apsp_bfs16_workspace_bytes(N, R), 1), dtype=torch.uint8, device=device)
    with _timed("apsp_bfs"):
        check(lib.gnan_apsp_bfs16(ptr(rowptr), ptr(col), N, row_begin, row_end, ptr(hop), hop.shape[1], st.data_ptr(), st.data_ptr() + 4,
                                  ptr(ws), ws.numel(), stream_handle()), "gnan_apsp_bfs16")
    over, D = (int(v) for v in st.tolist())
    if over:
        raise NotImplementedError(f"a hop distance > {WIDE_MAX_LEVEL} does not fit the int16 hop matrix")
    cnt = torch.empty(R, D + 2, dtype=torch.int32, device=device)
    check(lib.gnan_level_counts16(ptr(hop), R, N, hop.shape[1], ptr(cnt), D + 2, stream_handle()), "gnan_level_counts16")
    return HopData(hop, cnt, N, row_begin)


def build_csr(edge_index, num_nodes, device, status=None):
    """Directed CSR (rowptr int32 [N+1], col int32 [E]) of edges followed source -> target, built on the device by a counting
    sort (csrc/csr.cu: no comparison sort, no host synchronisation). Returns (rowptr, col, status): status is a device int32
    word, bit 0 = endpoint out of range, bit 1 = duplicate edges present (see _expand_multi_edges); the caller reads it together
    with its own flags."""
    lib = load()
    ei = torch.as_tensor(edge_index).to(device=device, dtype=torch.int64, non_blocking=True).contiguous()
    if ei.dim() != 2 or ei.shape[0] != 2:
        raise ValueError("edge_index must be [2,E]")
    E = ei.shape[1]
    rowptr = torch.empty(num_nodes + 1, dtype=torch.int32, device=device)
    col = torch.empty(max(E, 1), dtype=torch.int32, device=device)
    if status is None:
        status = torch.zeros(1, dtype=torch.int32, device=device)
    ws = torch.empty(max(lib.gnan_build_csr_workspace_bytes(num_nodes, E), 1), dtype=torch.uint8, device=device)
    with _timed("build_csr"):
        check(lib.gnan_build_csr(ptr(ei[0]), ptr(ei[1]), E, num_nodes, ptr(rowptr), ptr(col), status.data_ptr(), ptr(ws), ws.numel(),
                                 stream_handle()), "gnan_build_csr")
    return rowptr, col, status


def _timed(name):
    from . import ops
    return ops._timed(name)


def _check_status(st):
    if st & 1:
        raise ValueError("edge_index out of range")


def _expand_multi_edges(edge_index, num_nodes, device):
    """(edge_index', N') with every (src,dst) pair listed k > 1 times replaced by a chain of k unit edges through k-1 virtual
    nodes N, N+1, ...: unit-weight BFS on the result reproduces the reference's Dijkstra on the summed weights
    (pre_process_datasets.py:109-110). Slow path (sort-based), only taken when the CSR builder reports duplicates."""
    ei = torch.as_tensor(edge_index).to(device=device, dtype=torch.int64)
    key, cnt = torch.unique(ei[0] * num_nodes + ei[1], return_counts=True)
    s, d = key // num_nodes, key % num_nodes
    single = cnt == 1
    ms, md, mk = s[~single], d[~single], cnt[~single]
    nv = mk - 1                                                         # virtual nodes per multi-edge
    first = num_nodes + torch.cumsum(nv, 0) - nv                        # id of the first virtual node of each chain
    eid = torch.repeat_interleave(torch.arange(ms.numel(), device=device), mk)    # one entry per unit edge of a chain
    pos = torch.arange(eid.numel(), device=device) - torch.repeat_interleave(torch.cumsum(mk, 0) - mk, mk)
    a = torch.where(pos == 0, ms[eid], first[eid] + pos - 1)
    b = torch.where(pos == mk[eid] - 1, md[eid], first[eid] + pos)
    out = torch.stack([torch.cat([s[single], a]), torch.cat([d[single], b])])
    return out, num_nodes + int(nv.sum().item())


def _recount_levels(hop, n_cols):
    """[R,256] level histogram of the first n_cols columns (torch ops; multi-edge slow path only)"""
    R = hop.shape[0]
    cnt = torch.zeros(R, 256, dtype=torch.int32, device=hop.device)
    for r0 in range(0, R, 2048):
        blk = hop[r0:r0 + 2048, :n_cols].long()
        cnt[r0:r0 + 2048].scatter_add_(1, blk, torch.ones_like(blk, dtype=torch.int32))
    return cnt


def _trim_counts(cnt256):
    """[R,256] level histogram -> [R, D+2] (levels 0..D, then the unreachable bin). One device sync."""
    finite = cnt256[:, :255]
    nz = (finite.sum(0) > 0).nonzero()
    D = int(nz.max().item()) if nz.numel() else 0
    return torch.cat([finite[:, :D + 1], cnt256[:, 255:256]], dim=1).contiguous()


MSBFS_MIN_NODES = 4096      # graphs at least this large use the bit-parallel multi-source BFS


def apsp(edge_index, num_nodes, device="cuda", row_begin=0, row_end=None, method="auto", _expanded=False):
    """All-pairs (or rows [row_begin,row_end) of the) hop distances of one graph on the GPU -> HopData.

    method: "auto" | "warp" (one warp per source: small graphs, few rows) | "msbfs" (bit-parallel multi-source BFS over
    1024 columns at a time: large graphs; the cost does not depend on the number of rows kept)."""
    lib = load()
    N = int(num_nodes)
    row_end = N if row_end is None else int(row_end)
    R = row_end - row_begin
    st = torch.zeros(2, dtype=torch.int32, device=device)              # [csr status, hop overflow]
    rowptr, col, _ = build_csr(edge_index, N, device, status=st[0:1])
    hop = torch.empty(R, hop_ld(N), dtype=torch.uint8, device=device)
    cnt = torch.empty(R, 256, dtype=torch.int32, device=device)
    flag = st[1:2]
    if method == "auto":
        method = "msbfs" if N >= MSBFS_MIN_NODES and R * 8 >= N else "warp"
    if method == "msbfs":
        ws = torch.empty(max(lib.gnan_apsp_msbfs_workspace_bytes(N), 1), dtype=torch.uint8, device=device)
        with _timed("apsp_msbfs"):
            check(lib.gnan_apsp_msbfs(ptr(rowptr), ptr(col), N, row_begin, row_end, ptr(hop), hop.shape[1], ptr(cnt), 256, flag.data_ptr(),
                                      ptr(ws), ws.numel(), stream_handle()), "gnan_apsp_msbfs")
    else:
        ws = torch.empty(max(lib.gnan_apsp_bfs_workspace_bytes(N, R), 1), dtype=torch.uint8, device=device)
        with _timed("apsp_bfs"):
            check(lib.gnan_apsp_bfs(ptr(rowptr), ptr(col), N, row_begin, row_end, ptr(hop), hop.shape[1], ptr(cnt), 256, flag.data_ptr(),
                                    ptr(ws), ws.numel(), stream_handle()), "gnan_apsp_bfs")
    status, over = (int(v) for v in st.tolist())
    _check_status(status)
    if status & 2 and not _expanded:                                   # duplicate edges: weight-k emulation, then drop the virtual nodes
        ei2, n2 = _expand_multi_edges(edge_index, N, device)
        big = apsp(ei2, n2, device=device, row_begin=row_begin, row_end=row_end, method=method, _expanded=True)
        if big.wide:
            raise NotImplementedError("duplicate edges in a graph with hop distances > 254 are not supported")
        hop = torch.full((R, hop_ld(N)), _lib.HOP_UNREACHABLE, dtype=torch.uint8, device=device)
        hop[:, :N] = big.hop[:, :N]
        return HopData(hop, _trim_counts(_recount_levels(hop, N)) if R else cnt[:, :2], N, row_begin)
    if R and over:                                         # a level beyond 254: once more with int16 hops (csrc/wide.cu)
        return _apsp_wide(rowptr, col, N, row_begin, row_end, device)
    return HopData(hop, _trim_counts(cnt) if R else cnt[:, :2], N, row_begin)


class PackedBatch:
    """A batch of small graphs in packed block-diagonal form (replaces the dense (sum N)^2 collate of
    batched_pyg_main.py:54-91).

    x [sumN,K] fp32, hop uint8 [sum n_b^2] (graph b's n_b x n_b block at hop_off[b]), node_off int32 [B+1],
    hop_off int64 [B+1], level_counts int32 [sumN,nbins], batch_vector int64 [sumN] (kept for API parity), y.
    """

    def __init__(self, x, hop, hop_off, node_off, level_counts, y=None, max_nodes=None, level_rscale=None):
        self.x, self.hop, self.hop_off, self.node_off, self.level_counts, self.y = x, hop, hop_off, node_off, level_counts, y
        self.max_nodes = max_nodes
        # optional fp32 [sumN,nbins] 1/level_counts (0 for empty levels), written by the batched BFS itself
        # (apsp_batched(..., rscale=True)); level_counts may then be None
        self.level_rscale = level_rscale

    deferred = False    # see _DeferredBatch

    @property
    def num_graphs(self):
        return self.node_off.numel() - 1

    @property
    def nbins(self):
        for t in (self.level_counts, self.level_rscale):
            if t is not None:
                return t.shape[1]
        raise ValueError("PackedBatch without a level table")

    @property
    def batch_vector(self):
        sizes = (self.node_off[1:] - self.node_off[:-1]).long()
        return torch.repeat_interleave(torch.arange(self.num_graphs, device=sizes.device), sizes)

    def to(self, device):
        mv = lambda t: None if t is None else t.to(device, non_blocking=True)
        return PackedBatch(mv(self.x), mv(self.hop), mv(self.hop_off), mv(self.node_off), mv(self.level_counts), mv(self.y),
                           self.max_nodes, mv(self.level_rscale))

    def pin_memory(self):
        pm = lambda t: None if t is None else t.pin_memory()
        return PackedBatch(pm(self.x), pm(self.hop), pm(self.hop_off), pm(self.node_off), pm(self.level_counts), pm(self.y),
                           self.max_nodes, pm(self.level_rscale))


class _DeferredBatch(PackedBatch):
    """What apsp_batched returns for the configuration of a training step that preprocesses its own batch (LocalEdges, nbins,
    rscale=True, graphs of at most 128 nodes): the batched BFS has not run yet. models.TensorGNAN's output-normalised graph readout
    consumes the edge segments `edges` directly (ops.bfs_graph_readout: the BFS and the readout in one kernel, neither hop bytes
    nor a normaliser table in memory). The first read of `hop` or `level_rscale` runs the batched BFS once, exactly as
    apsp_batched runs it otherwise, and keeps the result; `deferred` is False from then on."""

    def __init__(self, x, hop_off, node_off, y, max_nodes, nbins, edges, materialise):
        self._materialise, self._nbins, self.edges = materialise, nbins, edges
        super().__init__(x, None, hop_off, node_off, None, y, max_nodes)

    @property
    def deferred(self):
        return self._materialise is not None

    def _distances(self):
        if self._materialise is not None:
            self._hop, self._level_rscale = self._materialise()
            self._materialise = None

    @property
    def hop(self):
        self._distances()
        return self._hop

    @hop.setter
    def hop(self, v):
        self._hop = v

    @property
    def level_rscale(self):
        self._distances()
        return self._level_rscale

    @level_rscale.setter
    def level_rscale(self, v):
        self._level_rscale = v

    @property
    def nbins(self):
        return self._nbins


class LocalEdges:
    """The edge list of a batch of small graphs as it should cross PCIe: src / dst uint8 [E] = node indices INSIDE the edge's
    graph, edge_off int32 [B+1] = first edge of every graph (edges grouped by graph). 2 bytes per directed edge instead of the
    16 of PyG's int64 [2,E] (batched_pyg_main.py:54-91 hands the model the latter). `expand` rebuilds the global int64
    edge_index on the device (gnan_edges_from_local), bit-identical up to the order of the graphs' edge groups."""

    def __init__(self, src, dst, edge_off):
        self.src, self.dst, self.edge_off = src, dst, edge_off

    @classmethod
    def from_edge_index(cls, edge_index, node_off):
        """Host-side, once per batch / dataset. edge_index int64 [2,E] with global ids, node_off [B+1]. Edges are grouped by the
        graph of their source (stable: the order inside a graph is kept); an edge across graphs or a graph of more than 256
        nodes raises."""
        import numpy as np
        ei = torch.as_tensor(edge_index).cpu().numpy().astype(np.int64)
        no = np.asarray(torch.as_tensor(node_off).cpu().numpy(), dtype=np.int64)
        B = no.shape[0] - 1
        if B > 0 and int((no[1:] - no[:-1]).max()) > 256:
            raise ValueError("LocalEdges: graphs of more than 256 nodes")
        g = np.searchsorted(no, ei[0], side="right") - 1
        if ei.shape[1] and (ei.min() < 0 or ei.max() >= no[-1] or np.any(np.searchsorted(no, ei[1], side="right") - 1 != g)):
            raise ValueError("LocalEdges: an edge leaves its graph or the node range")
        if np.any(g[1:] < g[:-1]):
            perm = np.argsort(g, kind="stable")
            ei, g = ei[:, perm], g[perm]
        edge_off = np.zeros(B + 1, dtype=np.int64)
        np.cumsum(np.bincount(g, minlength=B), out=edge_off[1:])
        base = no[g]
        return cls(torch.from_numpy((ei[0] - base).astype(np.uint8)), torch.from_numpy((ei[1] - base).astype(np.uint8)),
                   torch.from_numpy(edge_off.astype(np.int32)))

    @property
    def num_edges(self):
        return self.src.numel()

    def nbytes(self):
        return self.src.numel() + self.dst.numel() + 4 * self.edge_off.numel()

    def to(self, device):
        return LocalEdges(*[t.to(device, non_blocking=True) for t in (self.src, self.dst, self.edge_off)])

    def pin_memory(self):
        return LocalEdges(self.src.pin_memory(), self.dst.pin_memory(), self.edge_off.pin_memory())

    def expand(self, node_off, out=None):
        """int64 [2,E] global edge_index on the device (node_off: int32 device tensor [B+1]); `out` = a preallocated result
        (the static input of a captured step)"""
        lib = load()
        E, B = self.num_edges, self.edge_off.numel() - 1
        if not self.src.is_cuda or node_off.dtype != torch.int32 or node_off.numel() != B + 1:
            raise TypeError("LocalEdges.expand: tensors must be on the GPU, node_off int32 [B+1]")
        if out is None:
            out = torch.empty(2, E, dtype=torch.int64, device=self.src.device)
        elif out.shape != (2, E) or out.dtype != torch.int64 or not out.is_contiguous():
            raise TypeError("LocalEdges.expand: out must be contiguous int64 [2,E]")
        check(lib.gnan_edges_from_local(ptr(self.src), ptr(self.dst), ptr(self.edge_off), ptr(node_off.contiguous()), B, E, ptr(out),
                                        stream_handle()), "gnan_edges_from_local")
        return out


def check_batched_status(status):
    """Raise for a status word returned by apsp_batched(..., nbins=...) (one device read; call it once per epoch or when a
    result looks wrong, not once per step). The status of a deferred batch (see apsp_batched) is filled by whichever kernel
    consumes its edges first: the fused BFS + readout of the model's forward, or the BFS run by the first read of `hop` /
    `level_rscale`; read it after that."""
    st, over, _ = (int(v) for v in status.tolist())
    _check_status(st)
    if st & 2:
        raise ValueError("duplicate edges in the batch: call apsp_batched without nbins (multi-edge emulation path)")
    if over:
        raise ValueError("a hop distance does not fit the fixed-width level table: pass a larger nbins")


def apsp_batched(edge_index, node_off, device="cuda", x=None, y=None, node_off_device=None, _level_table_width=48, nbins=None,
                 hop_off_device=None, rscale=False, pair_stats=False):
    """Hop blocks of B graphs in one launch. edge_index uses GLOBAL node ids of the
    concatenated node set; node_off [B+1] are the graph boundaries. Graphs of up to _lib.APSP_BATCHED_MAX_NODES (1024) nodes run
    in the batched BFS, each by its own size: up to 128 nodes on groups of 4 warps, more on one CTA each. A batch with a larger
    graph goes through per-graph `apsp` calls in the free mode (slow, one synchronisation per graph) and raises ValueError in the
    fixed-width mode (nbins=...), before any launch. edge_index may also be a `LocalEdges` (the batch's edge list
    in its transfer form): batches of graphs with at most 128 nodes then skip the CSR builder altogether — every 4-warp group of
    the BFS kernel builds its graph's adjacency bit matrix in shared memory from the graph's own edge segment
    (gnan_apsp_bfs_batched_local); other batches expand it to the int64 list first.

    nbins: fixed level-table width (levels 0..nbins-2, last column = unreachable). The call then never synchronises with the
    host (it can be captured in a CUDA graph with the rest of a training step); empty levels carry a zero count and
    contribute nothing. The returned batch has `.status` (device int32 [3]: CSR status, overflow flag, largest hop) to be
    checked lazily with check_batched_status. hop_off_device: optional int64 device copy of the block offsets
    (cumsum of n_b^2, B+1 entries; with node_off_device it removes every host -> device copy from the call).
    rscale=True (fixed-width mode, graphs of at most 128 nodes): the BFS writes the output normaliser 1/level_counts
    (`PackedBatch.level_rscale`, fp32) INSTEAD of the int32 level counts, which the output-normalised models
    (models.TensorGNAN, normalize_rho=True) consume directly: one table written, none converted.
    With a `LocalEdges` input the distances are DEFERRED: the call launches nothing and returns a batch
    that holds the edge segments (`deferred` is True). models.TensorGNAN's output-normalised graph readout then runs the BFS and
    the readout as one kernel (ops.bfs_graph_readout) and never materialises hop bytes or the normaliser table; the first read of
    `hop` or `level_rscale` runs this BFS once and caches both. `status` is the same device word either way, filled by the
    first kernel that consumes the edges (check it after the forward).
    pair_stats=True (`LocalEdges` input only) returns the same deferred batch as rscale=True: the pair statistics of the graph
    readout are formed only inside the fused BFS + readout kernel.

    Pass node_off as a HOST tensor / array (what a data loader has): block sizes and offsets are then computed on the host
    and the call synchronises exactly once, at the end (overflow flag + largest hop, which sizes the level table).
    node_off_device: optional int32 device copy of node_off (skips its upload).
    The level table is first allocated 48 columns wide (hop distances inside small graphs rarely exceed that: the table is
    sumN x width int32, zero-filled); a deeper batch is detected by the kernel and redone once with max_n + 1 columns."""
    import numpy as np
    lib = load()
    if torch.is_tensor(node_off) and node_off.is_cuda:
        node_off_device = node_off.to(torch.int32) if node_off_device is None else node_off_device
        no_h = node_off.cpu().numpy().astype(np.int64)                 # device-resident offsets cost one extra synchronisation
    else:
        no_h = np.asarray(node_off, dtype=np.int64)
    B = no_h.shape[0] - 1
    sumN = int(no_h[-1]) if B >= 0 and no_h.size else 0
    sizes = no_h[1:] - no_h[:-1]
    max_n = int(sizes.max()) if B > 0 else 1
    hop_off_h = np.zeros(B + 1, dtype=np.int64)
    np.cumsum(sizes * sizes, out=hop_off_h[1:])
    total = int(hop_off_h[-1])
    if max_n > _lib.APSP_BATCHED_MAX_NODES:
        if nbins is not None:
            raise ValueError(f"apsp_batched: a graph of {max_n} nodes; the fixed-width mode (nbins=...) takes graphs of at most "
                             f"{_lib.APSP_BATCHED_MAX_NODES} nodes (call it without nbins: per-graph path)")
        return _apsp_batched_per_graph(edge_index, no_h, device, x, y)       # (a LocalEdges list cannot address such a graph)
    if node_off_device is None:
        node_off_device = torch.from_numpy(no_h.astype(np.int32)).to(device, non_blocking=True)
    node_off_d = node_off_device
    hop_off = hop_off_device if hop_off_device is not None else torch.from_numpy(hop_off_h).to(device, non_blocking=True)
    st = torch.zeros(3, dtype=torch.int32, device=device)              # [csr status, overflow, largest finite hop]
    local = None
    if isinstance(edge_index, LocalEdges):
        if not edge_index.src.is_cuda:
            edge_index = edge_index.to(device)
        if max_n <= 128 and sumN > 0 and B > 0:
            local = edge_index
        else:
            edge_index = edge_index.expand(node_off_d)
    if local is None:
        rowptr, col, _ = build_csr(edge_index, sumN, device, status=st[0:1])

    def bfs(hop, cnt_t, rs_t):
        # scratch of the size classes the BFS groups the graphs by (a fifth class above 128 nodes)
        order_ws = torch.empty(5 * B + 5 if max_n > 128 else 4 * B + 4, dtype=torch.int32, device=device)
        if local is not None:
            check(lib.gnan_apsp_bfs_batched_local(ptr(local.src), ptr(local.dst), ptr(local.edge_off), ptr(node_off_d), ptr(hop_off), B, max_n,
                                                  ptr(hop), ptr(cnt_t), ptr(rs_t), nb, st.data_ptr(), st.data_ptr() + 4, st.data_ptr() + 8,
                                                  ptr(order_ws), stream_handle()), "gnan_apsp_bfs_batched_local")
        else:
            check(lib.gnan_apsp_bfs_batched_ex(ptr(rowptr), ptr(col), ptr(node_off_d), ptr(hop_off), B, max_n, ptr(hop), ptr(cnt_t),
                                               ptr(rs_t), nb, st.data_ptr() + 4, st.data_ptr() + 8, ptr(order_ws), stream_handle()),
                  "gnan_apsp_bfs_batched_ex")
    nb_full = min(256, max_n + 1)                # a finite hop inside a graph is at most max_n - 1; last column = unreachable
    nb = min(nb_full, _level_table_width) if _level_table_width else nb_full
    if nbins is not None:
        nb = int(nbins)
    if pair_stats and (local is None or nbins is None):
        raise ValueError("pair_stats=True needs a LocalEdges edge list, graphs of at most 128 nodes and the fixed-width mode (nbins=...)")
    if rscale or pair_stats:
        if nbins is None or max_n > 128 or sumN == 0:
            raise ValueError("rscale=True needs the fixed-width mode (nbins=...) and graphs of at most 128 nodes")
        if local is not None:
            def materialise():
                hop = torch.empty(max(total, 1), dtype=torch.uint8, device=device)
                rs = torch.empty(sumN, nb, dtype=torch.float32, device=device)
                with _timed("apsp_bfs_batched"):
                    bfs(hop, None, rs)
                return hop, rs
            pk = _DeferredBatch(x, hop_off, node_off_d, y, max_n, nb, local, materialise)
            pk.status = st
            return pk
        hop = torch.empty(max(total, 1), dtype=torch.uint8, device=device)
        rs = torch.empty(sumN, nb, dtype=torch.float32, device=device)
        with _timed("apsp_bfs_batched"):
            bfs(hop, None, rs)
        pk = PackedBatch(x, hop, hop_off, node_off_d, None, y, max_n, level_rscale=rs)
        pk.status = st
        return pk
    hop = torch.empty(max(total, 1), dtype=torch.uint8, device=device)
    cnt = torch.empty(sumN, nb, dtype=torch.int32, device=device)
    with _timed("apsp_bfs_batched"):
        bfs(hop, cnt, None)
    if nbins is not None:
        pk = PackedBatch(x, hop, hop_off, node_off_d, cnt, y, max_n)
        pk.status = st
        return pk
    status, over, D = (int(v) for v in st.tolist()) if B > 0 else (0, 0, 0)
    _check_status(status)
    if status & 2:
        if isinstance(edge_index, LocalEdges):
            edge_index = edge_index.expand(node_off_d)
        return _apsp_batched_per_graph(edge_index, no_h, device, x, y)
    if over and nb < nb_full:                    # deeper than the narrow level table: once more with the full width
        return apsp_batched(edge_index, node_off, device, x, y, node_off_device, _level_table_width=0, hop_off_device=hop_off_device)
    if over:
        raise NotImplementedError("a hop distance > 254 does not fit the uint8 hop matrix")
    if sumN == 0:
        return PackedBatch(x, hop, hop_off, node_off_d, cnt[:, :2], y, max_n)
    lc = torch.cat([cnt[:, :D + 1], cnt[:, nb - 1:nb]], dim=1).contiguous()
    return PackedBatch(x, hop, hop_off, node_off_d, lc, y, max_n)


def _apsp_batched_per_graph(edge_index, no_h, device, x, y):
    """Slow path of apsp_batched for batches with duplicate edges (per-graph `apsp` emulates the reference's summed weights) or
    with a graph of more than _lib.APSP_BATCHED_MAX_NODES nodes: one `apsp` call per graph (any size), assembled into the
    packed form."""
    import numpy as np
    ei = torch.as_tensor(edge_index).to(device=device, dtype=torch.int64)
    B = no_h.shape[0] - 1
    hops, cnts, D = [], [], 0
    for b in range(B):
        lo, hi = int(no_h[b]), int(no_h[b + 1])
        sel = (ei[0] >= lo) & (ei[0] < hi)
        hd = apsp(ei[:, sel] - lo, hi - lo, device=device, method="warp")
        if hd.wide:
            raise NotImplementedError("a hop distance > 254 does not fit the uint8 hop matrix")
        hops.append(hd.hop[:, :hi - lo].reshape(-1))
        cnts.append(hd.level_counts)
        D = max(D, hd.nbins - 2)
    lc = torch.zeros(int(no_h[-1]), D + 2, dtype=torch.int32, device=device)
    for b, c in enumerate(cnts):
        lc[int(no_h[b]):int(no_h[b + 1]), :c.shape[1] - 1] = c[:, :-1]
        lc[int(no_h[b]):int(no_h[b + 1]), -1] = c[:, -1]
    sizes = no_h[1:] - no_h[:-1]
    hop_off = torch.from_numpy(np.concatenate([[0], np.cumsum(sizes * sizes)]).astype(np.int64)).to(device)
    return PackedBatch(x, torch.cat(hops) if hops else torch.empty(1, dtype=torch.uint8, device=device), hop_off,
                       torch.from_numpy(no_h.astype(np.int32)).to(device), lc, y, int(sizes.max()) if B else 1)


def pre_process(data, is_graph_task, data_name=None, processed_data_dir=None, device="cuda", reference_format=False):
    """Drop-in for pre_process_datasets.pre_process (:104-148): same call shape, same mutation of the inputs.

    Appends the constant-1 column to x (:108/:127) and attaches `.hop_data` (HopData, on `device`). With
    reference_format=True also attaches fp32 `.node_distances` / `.normalization_matrix` like the reference.
    Graph task: `data` is a list of graphs; node task: one graph (num_nodes inferred from edge_index like :128).
    With `processed_data_dir` (and `data_name`) the result is written once, like :144-148, but in the packed format of
    gnan_b200.packed ({dir}/{name}.gnan_b200.pt: 1 byte per node pair instead of 8); read it back with
    packed.PackedDataset.load (graph task) or packed.load_node (node task). The graph-task file is built by one batched BFS
    (packed.PackedDataset.from_graphs) for graphs of up to _lib.APSP_BATCHED_MAX_NODES (1024) nodes, per graph beyond.
    """
    import os
    graphs = list(data) if is_graph_task else [data]
    for g in graphs:
        g.x = torch.cat((g.x, torch.ones(g.x.size(0), 1, dtype=g.x.dtype, device=g.x.device)), dim=-1)
        ei = torch.as_tensor(g.edge_index)
        n = g.x.size(0) if is_graph_task else (int(ei.max().item()) + 1 if ei.numel() else g.x.size(0))
        hd = apsp(ei, n, device=device)
        g.hop_data = hd
        if reference_format:
            g.node_distances, g.normalization_matrix = hd.reference_format()
    if processed_data_dir is not None and data_name is not None:
        path = os.path.join(processed_data_dir, f"{data_name}.gnan_b200.pt")
        if not os.path.exists(path):
            os.makedirs(processed_data_dir, exist_ok=True)
            from . import packed
            if is_graph_task:
                packed.PackedDataset.from_graphs(graphs, device=device, add_constant_column=False).save(path)
            else:
                packed.save_node(data, path)
    return data
