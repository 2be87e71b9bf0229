"""torch.library ops over the C ABI (include/gnan_b200.h). Each op is a thin ctypes call on raw device pointers and the
current stream; autograd is wired with register_autograd so the nn.Modules (GNAN.py, models.py, batched.py) compose them like any torch op.

Nothing here computes on the CPU: non-CUDA inputs raise (see _lib.ptr)."""
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _lib
from ._lib import MlpGrads, MlpParams, check, load, ptr, stream_handle

__all__ = ["mlp", "aggregate_rows", "aggregate_blockdiag", "rho_table_inputs", "level_rscale", "alloc_hop", "hop_ld",
           "cross_entropy_rows", "bce_with_logits"]


# ---- optional per-call CUDA-event timing (bench.py): events are recorded on the launching stream ----------------------
_TIMING = None


def enable_timing(on: bool):
    global _TIMING
    _TIMING = {} if on else None


def timing_results():
    """{op: (calls, total_ms)}; synchronises."""
    torch.cuda.synchronize()
    return {k: (len(v), sum(a.elapsed_time(b) for a, b in v)) for k, v in (_TIMING or {}).items()}


class _timed:
    def __init__(self, name):
        self.name = name

    def __enter__(self):
        if _TIMING is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.a.record()

    def __exit__(self, *exc):
        if _TIMING is not None:
            self.b.record()
            _TIMING.setdefault(self.name, []).append((self.a, self.b))


def hop_ld(n: int) -> int:
    """leading dimension (bytes per row) of a hop block with n columns: rows are 16-byte aligned for 128-bit loads"""
    return max(16, (int(n) + 15) // 16 * 16)


def alloc_hop(rows: int, n: int, device) -> Tensor:
    return torch.full((rows, hop_ld(n)), _lib.HOP_UNREACHABLE, dtype=torch.uint8, device=device)


def _ws(nbytes: int, device) -> Optional[Tensor]:
    return torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=device)


def _f32(t: Tensor, name: str) -> Tensor:
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32, got {t.dtype}")
    return t.contiguous()


MLP_EXT_MAX_BYTES = 24 << 30      # dh + a1 buffers of the one-pass backward for C > 8 (beyond this the channel-slice passes run)


class _matmul_tf32:
    """torch.matmul with TF32 tensor cores forced on / off for the GEMMs around gnan_mlp_bwd_ext, whatever the caller set globally"""

    def __init__(self, allow: bool):
        self._allow = allow

    def __enter__(self):
        self._was = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = self._allow

    def __exit__(self, *exc):
        torch.backends.cuda.matmul.allow_tf32 = self._was


def _split_tf32(t: Tensor):
    """t = hi + lo with hi rounded to TF32 (10 mantissa bits, round half away) and lo = t - hi exact in fp32"""
    hi = ((t.contiguous().view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)
    return hi, t - hi


def _matmul_3xtf32(a: Tensor, b: Tensor) -> Tensor:
    """a @ b at fp32-level accuracy on the TF32 tensor cores: the three split terms a_hi b_hi + a_lo b_hi + a_hi b_lo as ONE GEMM
    over a K dimension concatenated three times (fp32 accumulation; the result is written once). For a short K (the class
    dimension) and a large result: the plain-fp32 SIMT GEMM is compute bound there, this one is bound by writing the result."""
    ah, al = _split_tf32(a)
    bh, bl = _split_tf32(b)
    with _matmul_tf32(True):
        return torch.matmul(torch.cat([ah, al, ah], dim=1), torch.cat([bh, bh, bl], dim=0))


def _mlp_params(w1, b1, wh, bh, wo, bo, n_layers):
    G, C = wo.shape[0], wo.shape[1]
    H = wo.shape[2] if n_layers >= 2 else 0
    p = MlpParams(G, H, C, n_layers, ptr(w1), ptr(b1), ptr(wh), ptr(bh), ptr(wo), ptr(bo))
    return p, G, H, C


# ---------------------------------------------------------------------------------------------------------------------
# grouped scalar-input MLP:  S[r,:] = sum_g f_g(u[r,g])
# ---------------------------------------------------------------------------------------------------------------------
@torch.library.custom_op("gnan_b200::mlp_fwd", mutates_args=())
def mlp_fwd(u: Tensor, w1: Tensor, b1: Tensor, wh: Tensor, bh: Tensor, wo: Tensor, bo: Tensor, n_layers: int,
            dropout_p: float, seed: int, precision: int, seed_dev: Optional[Tensor] = None) -> Tensor:
    lib = load()
    u, w1, b1, wh, bh, wo, bo = (_f32(t, n) for t, n in zip((u, w1, b1, wh, bh, wo, bo), "u w1 b1 wh bh wo bo".split()))
    if u.dim() != 2 or u.shape[1] != wo.shape[0]:
        raise ValueError(f"u must be [R,G] with G={wo.shape[0]}, got {tuple(u.shape)}")
    p, G, H, C = _mlp_params(w1, b1, wh, bh, wo, bo, n_layers)
    R = u.shape[0]
    S = torch.empty(R, C, dtype=torch.float32, device=u.device)
    ws = _ws(lib.gnan_mlp_workspace_bytes(R, p, 0, precision), u.device)
    with _timed("mlp_fwd"):
        check(lib.gnan_mlp_fwd(ptr(u), R, u.shape[1], p, float(dropout_p), int(seed) & (2 ** 64 - 1), ptr(seed_dev), precision, ptr(S),
                               ptr(ws), ws.numel(), stream_handle()), "gnan_mlp_fwd")
    return S


@mlp_fwd.register_fake
def _(u, w1, b1, wh, bh, wo, bo, n_layers, dropout_p, seed, precision, seed_dev=None):
    return u.new_empty(u.shape[0], wo.shape[1])


@torch.library.custom_op("gnan_b200::mlp_bwd", mutates_args=())
def mlp_bwd(u: Tensor, w1: Tensor, b1: Tensor, wh: Tensor, bh: Tensor, wo: Tensor, bo: Tensor, n_layers: int,
            dropout_p: float, seed: int, precision: int, dS: Tensor,
            need_du: bool, seed_dev: Optional[Tensor] = None) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    lib = load()
    u, w1, b1, wh, bh, wo, bo, dS = (_f32(t, n) for t, n in zip((u, w1, b1, wh, bh, wo, bo, dS), "u w1 b1 wh bh wo bo dS".split()))
    p, G, H, C = _mlp_params(w1, b1, wh, bh, wo, bo, n_layers)
    R = u.shape[0]
    outs = [torch.empty_like(t) for t in (w1, b1, wh, bh, wo, bo)]
    outs.append(torch.empty((R, G) if need_du else (0,), dtype=torch.float32, device=u.device))
    ws = _ws(lib.gnan_mlp_workspace_bytes(R, p, 1, precision), u.device)
    if (not need_du and R > 0 and lib.gnan_mlp_bwd_ext_supported(p, precision) and 2 * R * G * H * 4 <= MLP_EXT_MAX_BYTES):
        # more than 8 output channels on the tensor-core path: the output layer runs as two plain GEMMs around ONE pass of the
        # kernel (dh = dS Wo in, a1 out, dWo = dS^T a1) instead of ceil(C/8) passes that each repeat the recompute
        with _timed("mlp_bwd"), _matmul_tf32(False):
            dh = _matmul_3xtf32(dS, wo.permute(1, 0, 2).reshape(C, G * H))                      # [R, G*H]
            a1 = torch.empty(R, G * H, dtype=torch.float32, device=u.device)
            g = MlpGrads(ptr(outs[0]), ptr(outs[1]), ptr(outs[2]), ptr(outs[3]), None, ptr(outs[5]), None)
            check(lib.gnan_mlp_bwd_ext(ptr(u), R, u.shape[1], p, float(dropout_p), int(seed) & (2 ** 64 - 1), ptr(seed_dev), precision,
                                       ptr(dS), ptr(dh), ptr(a1), g, ptr(ws), ws.numel(), stream_handle()), "gnan_mlp_bwd_ext")
            outs[4].copy_(torch.matmul(dS.t(), a1).view(C, G, H).permute(1, 0, 2))             # dWo[g,c,:] = sum_r dS[r,c] a1[r,g,:]
        return tuple(outs)
    g = MlpGrads(*[ptr(t) for t in outs[:6]], ptr(outs[6]) if need_du else None)
    with _timed("mlp_bwd"):
        check(lib.gnan_mlp_bwd(ptr(u), R, u.shape[1], p, float(dropout_p), int(seed) & (2 ** 64 - 1), ptr(seed_dev), precision, ptr(dS),
                               g, ptr(ws), ws.numel(), stream_handle()), "gnan_mlp_bwd")
    return tuple(outs)


@mlp_bwd.register_fake
def _(u, w1, b1, wh, bh, wo, bo, n_layers, dropout_p, seed, precision, dS, need_du, seed_dev=None):
    return tuple(torch.empty_like(t) for t in (w1, b1, wh, bh, wo, bo)) + (u.new_empty(u.shape if need_du else (0,)),)


def _mlp_setup(ctx, inputs, output):
    u, w1, b1, wh, bh, wo, bo, n_layers, dropout_p, seed, precision, seed_dev = inputs
    ctx.save_for_backward(u, w1, b1, wh, bh, wo, bo)
    ctx.seed_dev = seed_dev
    ctx.cfg = (n_layers, dropout_p, seed, precision)


def _mlp_backward(ctx, dS):
    u, w1, b1, wh, bh, wo, bo = ctx.saved_tensors
    n_layers, dropout_p, seed, precision = ctx.cfg
    need_du = bool(ctx.needs_input_grad[0])
    g = mlp_bwd(u, w1, b1, wh, bh, wo, bo, n_layers, dropout_p, seed, precision, dS.contiguous(), need_du, ctx.seed_dev)
    return (g[6] if need_du else None,) + tuple(g[:6]) + (None, None, None, None, None)


mlp_fwd.register_autograd(_mlp_backward, setup_context=_mlp_setup)


def mlp(u, w1, b1, wh, bh, wo, bo, n_layers, dropout_p=0.0, seed=0, precision="fp32", seed_dev=None):
    """S[r,:] = sum_g f_g(u[r,g]); differentiable w.r.t. the weights, and w.r.t. u when u requires grad (only the NAM
    readout feeds computed values in; x itself is data, GNAN.py:56). seed_dev: optional 1-element int64 CUDA tensor XORed
    into the dropout seed on the device (fresh masks for every replay of a captured step)."""
    if seed_dev is not None and (seed_dev.dtype != torch.int64 or seed_dev.numel() != 1):
        raise TypeError("seed_dev must be a 1-element int64 CUDA tensor")
    return mlp_fwd(u, w1, b1, wh, bh, wo, bo, int(n_layers), float(dropout_p), int(seed), _lib.PRECISIONS[precision],
                   seed_dev if dropout_p > 0 else None)


MAX_KERNEL_CHANNELS = 64      # gnan_mlp_* limit on C


def mlp_per_group(u, w1, b1, wh, bh, wo, bo, n_layers, dropout_p=0.0, seed=0, precision="fp32", seed_dev=None):
    """Y[r,g,:] = f_g(u[r,g]) WITHOUT the sum over groups -> [R,G,C] (the reference's `fx`, GNAN.py:57-62, which the NAM
    readout, models.py:374-381, and the interpretability plots need per feature).

    Same kernels: the output layer of a chunk of groups is expanded to a block-diagonal [Gc, Gc*C, H] weight, so group g
    owns channels [g*C, (g+1)*C) of the kernel's feature sum and every other group contributes exactly 0 there. Differentiable
    like `mlp`. Chunks keep Gc*C <= 64."""
    R, G = u.shape
    C = wo.shape[1]
    if C > MAX_KERNEL_CHANNELS:
        raise ValueError(f"out_channels {C} > {MAX_KERNEL_CHANNELS}")
    gc_max = max(1, MAX_KERNEL_CHANNELS // C)
    outs = []
    for g0 in range(0, G, gc_max):
        g1 = min(G, g0 + gc_max)
        gc = g1 - g0
        idx = torch.arange(gc, device=wo.device)
        wo_x = wo.new_zeros(gc, gc, C, wo.shape[2])
        wo_x[idx, idx] = wo[g0:g1]
        bo_x = bo.new_zeros(gc, gc, C)
        bo_x[idx, idx] = bo[g0:g1]
        hid = n_layers >= 2
        y = mlp(u[:, g0:g1].contiguous(), w1[g0:g1] if hid else w1, b1[g0:g1] if hid else b1,
                wh[:, g0:g1].contiguous() if hid else wh, bh[:, g0:g1].contiguous() if hid else bh,
                wo_x.view(gc, gc * C, -1), bo_x.view(gc, gc * C), n_layers, dropout_p=dropout_p,
                seed=(seed + g0) if dropout_p > 0 else 0, precision=precision, seed_dev=seed_dev if dropout_p > 0 else None)
        outs.append(y.view(R, gc, C))
    return outs[0] if len(outs) == 1 else torch.cat(outs, dim=1)


# ---------------------------------------------------------------------------------------------------------------------
# dense row-block aggregation
# ---------------------------------------------------------------------------------------------------------------------
def _agg_dims(hop, T, S, per_row):
    if hop.dtype not in (torch.uint8, torch.int16) or hop.dim() != 2:
        raise TypeError("hop must be a uint8 (or, for deep graphs, int16) [R, ld] matrix")
    R, ld = hop.shape
    N, C = S.shape
    nbins, Cr = T.shape[-2], T.shape[-1]
    if per_row and (T.dim() != 3 or T.shape[0] != R):
        raise ValueError(f"per-row table must be [R,nbins,Cr], got {tuple(T.shape)}")
    if not per_row and T.dim() != 2:
        raise ValueError(f"global table must be [nbins,Cr], got {tuple(T.shape)}")
    return R, ld, N, C, nbins, Cr


@torch.library.custom_op("gnan_b200::agg_rows_fwd", mutates_args=())
def agg_rows_fwd(hop: Tensor, T: Tensor, rscale: Optional[Tensor], S: Tensor, per_row: bool, save: bool,
                 algo: int = 0) -> Tuple[Tensor, Tensor]:
    lib = load()
    T, S = _f32(T, "T"), _f32(S, "S")
    rscale = None if rscale is None else _f32(rscale, "rscale")
    R, ld, N, C, nbins, Cr = _agg_dims(hop, T, S, per_row)
    out = torch.empty(R, C, dtype=torch.float32, device=S.device)
    bsum = torch.empty((R, nbins, C) if save else (0,), dtype=torch.float32, device=S.device)
    nws = 0 if algo == _lib.AGG_CUDA_CORES else lib.gnan_aggregate_rows_fwd_workspace_bytes(R, N, ld, nbins, C)
    ws = _ws(nws, S.device)
    with _timed("aggregate_rows_fwd_save"):
        check(lib.gnan_aggregate_rows_fwd_ws(ptr(hop), R, N, ld, ptr(T), int(per_row), nbins, Cr, ptr(rscale), ptr(S), C,
                                             ptr(out), ptr(bsum), int(algo), ptr(ws) if nws else None, nws, stream_handle()),
              "gnan_aggregate_rows_fwd_ws")
    return out, bsum


@agg_rows_fwd.register_fake
def _(hop, T, rscale, S, per_row, save, algo=0):
    R, C, nbins = hop.shape[0], S.shape[1], T.shape[-2]
    return S.new_empty(R, C), S.new_empty((R, nbins, C) if save else (0,))


@torch.library.custom_op("gnan_b200::agg_rows_bwd", mutates_args=())
def agg_rows_bwd(hop: Tensor, T: Tensor, rscale: Optional[Tensor], S: Tensor, per_row: bool, g: Tensor,
                 bsum: Tensor, algo: int = 0) -> Tuple[Tensor, Tensor]:
    lib = load()
    T, S, g = _f32(T, "T"), _f32(S, "S"), _f32(g, "g")
    rscale = None if rscale is None else _f32(rscale, "rscale")
    R, ld, N, C, nbins, Cr = _agg_dims(hop, T, S, per_row)
    dS = torch.empty_like(S)
    dT = torch.empty_like(T)
    if not bsum.numel():
        algo = _lib.AGG_CUDA_CORES          # nothing saved: the CUDA-core path rebuilds the bin sums with one extra pass
    ws = _ws(lib.gnan_aggregate_rows_bwd_ws_bytes(R, N, ld, nbins, Cr, C, int(algo)), S.device)
    with _timed("aggregate_rows_bwd_saved"):
        check(lib.gnan_aggregate_rows_bwd_ws(ptr(hop), R, N, ld, ptr(T), int(per_row), nbins, Cr, ptr(rscale), ptr(S), C,
                                             ptr(g), ptr(bsum) if bsum.numel() else None, ptr(dS), ptr(dT), int(algo), ptr(ws),
                                             ws.numel(), stream_handle()), "gnan_aggregate_rows_bwd_ws")
    return dS, dT


@agg_rows_bwd.register_fake
def _(hop, T, rscale, S, per_row, g, bsum, algo=0):
    return torch.empty_like(S), torch.empty_like(T)


def _agg_setup(ctx, inputs, output):
    hop, T, rscale, S, per_row, save, algo = inputs
    ctx.save_for_backward(hop, T, rscale, S, output[1])
    ctx.per_row = per_row
    ctx.algo = algo


def _agg_backward(ctx, g, _g_bsum):
    hop, T, rscale, S, bsum = ctx.saved_tensors
    dS, dT = agg_rows_bwd(hop, T, rscale, S, ctx.per_row, g.contiguous(), bsum, ctx.algo)
    return None, dT, None, dS, None, None, None


agg_rows_fwd.register_autograd(_agg_backward, setup_context=_agg_setup)


AGG_ALGO = "auto"      # "auto" | "cuda" | "tc": kernel family of aggregate_rows (gnan_b200.h: GNAN_AGG_*); tests force each


# deep graphs: int16 hops (-1 = unreachable), direct kernels of csrc/wide.cu
@torch.library.custom_op("gnan_b200::agg_rows16_fwd", mutates_args=())
def agg_rows16_fwd(hop: Tensor, T: Tensor, rscale: Optional[Tensor], S: Tensor, per_row: bool) -> Tensor:
    lib = load()
    T, S = _f32(T, "T"), _f32(S, "S")
    rscale = None if rscale is None else _f32(rscale, "rscale")
    R, ld, N, C, nbins, Cr = _agg_dims(hop, T, S, per_row)
    out = torch.empty(R, C, dtype=torch.float32, device=S.device)
    with _timed("aggregate_rows_fwd_save"):
        check(lib.gnan_aggregate_rows16_fwd(ptr(hop), R, N, ld, ptr(T), int(per_row), nbins, Cr, ptr(rscale), ptr(S), C, ptr(out),
                                            stream_handle()), "gnan_aggregate_rows16_fwd")
    return out


@agg_rows16_fwd.register_fake
def _(hop, T, rscale, S, per_row):
    return S.new_empty(hop.shape[0], S.shape[1])


@torch.library.custom_op("gnan_b200::agg_rows16_bwd", mutates_args=())
def agg_rows16_bwd(hop: Tensor, T: Tensor, rscale: Optional[Tensor], S: Tensor, per_row: bool, g: Tensor) -> Tuple[Tensor, Tensor]:
    lib = load()
    T, S, g = _f32(T, "T"), _f32(S, "S"), _f32(g, "g")
    rscale = None if rscale is None else _f32(rscale, "rscale")
    R, ld, N, C, nbins, Cr = _agg_dims(hop, T, S, per_row)
    dS, dT = torch.empty_like(S), torch.empty_like(T)
    flags = torch.empty(max(R, 1), dtype=torch.uint8, device=S.device)
    with _timed("aggregate_rows_bwd_saved"):
        check(lib.gnan_aggregate_rows16_bwd(ptr(hop), R, N, ld, ptr(T), int(per_row), nbins, Cr, ptr(rscale), ptr(S), C, ptr(g), ptr(dS),
                                            ptr(dT), ptr(flags), stream_handle()), "gnan_aggregate_rows16_bwd")
    return dS, dT


@agg_rows16_bwd.register_fake
def _(hop, T, rscale, S, per_row, g):
    return torch.empty_like(S), torch.empty_like(T)


def _agg16_setup(ctx, inputs, output):
    hop, T, rscale, S, per_row = inputs
    ctx.save_for_backward(hop, T, rscale, S)
    ctx.per_row = per_row


def _agg16_backward(ctx, g):
    hop, T, rscale, S = ctx.saved_tensors
    dS, dT = agg_rows16_bwd(hop, T, rscale, S, ctx.per_row, g.contiguous())
    return None, dT, None, dS, None


agg_rows16_fwd.register_autograd(_agg16_backward, setup_context=_agg16_setup)


def aggregate_rows(hop, T, S, rscale=None, per_row=False, algo=None):
    """out[i,c] = sum_j T[(i,) b(hop[i,j]), c'] * rscale[i,b] * S[j,c] over a [R, ld] uint8 hop block; see gnan_b200.h.
    An int16 hop block (deep graphs, preprocess.apsp's fallback for hop distances > 254) takes the direct kernels of csrc/wide.cu."""
    if hop.dtype == torch.int16:
        return agg_rows16_fwd(hop, T, rscale, S, bool(per_row))
    save = torch.is_grad_enabled() and (T.requires_grad or S.requires_grad)
    return agg_rows_fwd(hop, T, rscale, S, bool(per_row), bool(save), _lib.AGG_ALGOS[algo or AGG_ALGO])[0]


# ---------------------------------------------------------------------------------------------------------------------
# block-diagonal (batched graphs) aggregation
# ---------------------------------------------------------------------------------------------------------------------
@torch.library.custom_op("gnan_b200::agg_blockdiag_fwd", mutates_args=())
def agg_blockdiag_fwd(hop: Tensor, hop_off: Tensor, node_off: Tensor, T: Tensor, rscale: Optional[Tensor], S: Tensor,
                      per_row: bool, reduce_graph: bool) -> Tensor:
    lib = load()
    T, S = _f32(T, "T"), _f32(S, "S")
    rscale = None if rscale is None else _f32(rscale, "rscale")
    if hop.dtype != torch.uint8 or hop_off.dtype != torch.int64 or node_off.dtype != torch.int32:
        raise TypeError("hop uint8, hop_off int64, node_off int32 expected")
    B = node_off.numel() - 1
    N, C = S.shape
    nbins, Cr = T.shape[-2], T.shape[-1]
    out = torch.empty(B if reduce_graph else N, C, dtype=torch.float32, device=S.device)
    with _timed("aggregate_blockdiag_fwd"):
        check(lib.gnan_aggregate_blockdiag_fwd(ptr(hop), ptr(hop_off), ptr(node_off), B, ptr(T), int(per_row), nbins, Cr,
                                               ptr(rscale), ptr(S), C, int(reduce_graph), ptr(out), stream_handle()),
              "gnan_aggregate_blockdiag_fwd")
    return out


@agg_blockdiag_fwd.register_fake
def _(hop, hop_off, node_off, T, rscale, S, per_row, reduce_graph):
    return S.new_empty(node_off.numel() - 1 if reduce_graph else S.shape[0], S.shape[1])


@torch.library.custom_op("gnan_b200::agg_blockdiag_bwd", mutates_args=())
def agg_blockdiag_bwd(hop: Tensor, hop_off: Tensor, node_off: Tensor, T: Tensor, rscale: Optional[Tensor], S: Tensor,
                      per_row: bool, reduce_graph: bool, g: Tensor) -> Tuple[Tensor, Tensor]:
    lib = load()
    T, S, g = _f32(T, "T"), _f32(S, "S"), _f32(g, "g")
    rscale = None if rscale is None else _f32(rscale, "rscale")
    B = node_off.numel() - 1
    N, C = S.shape
    nbins, Cr = T.shape[-2], T.shape[-1]
    dS = torch.zeros_like(S)
    dT = torch.zeros_like(T)
    with _timed("aggregate_blockdiag_bwd"):
        check(lib.gnan_aggregate_blockdiag_bwd(ptr(hop), ptr(hop_off), ptr(node_off), B, ptr(T), int(per_row), nbins, Cr,
                                               ptr(rscale), ptr(S), C, int(reduce_graph), ptr(g), ptr(dS), ptr(dT),
                                               stream_handle()), "gnan_aggregate_blockdiag_bwd")
    return dS, dT


@agg_blockdiag_bwd.register_fake
def _(hop, hop_off, node_off, T, rscale, S, per_row, reduce_graph, g):
    return torch.empty_like(S), torch.empty_like(T)


def _bd_setup(ctx, inputs, output):
    hop, hop_off, node_off, T, rscale, S, per_row, reduce_graph = inputs
    ctx.save_for_backward(hop, hop_off, node_off, T, rscale, S)
    ctx.flags = (per_row, reduce_graph)


def _bd_backward(ctx, g):
    hop, hop_off, node_off, T, rscale, S = ctx.saved_tensors
    dS, dT = agg_blockdiag_bwd(hop, hop_off, node_off, T, rscale, S, ctx.flags[0], ctx.flags[1], g.contiguous())
    return None, None, None, dT, None, dS, None, None


agg_blockdiag_fwd.register_autograd(_bd_backward, setup_context=_bd_setup)


# graph-level readout with a global table: one pass over the hop bytes for forward AND backward (csrc/agg_bd.cu)
@torch.library.custom_op("gnan_b200::agg_bd_graph_fwd", mutates_args=())
def agg_bd_graph_fwd(hop: Tensor, hop_off: Tensor, node_off: Tensor, T: Tensor, rscale: Optional[Tensor],
                     S: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    lib = load()
    T, S = _f32(T, "T"), _f32(S, "S")
    rscale = None if rscale is None else _f32(rscale, "rscale")
    if hop.dtype != torch.uint8 or hop_off.dtype != torch.int64 or node_off.dtype != torch.int32:
        raise TypeError("hop uint8, hop_off int64, node_off int32 expected")
    B = node_off.numel() - 1
    N, C = S.shape
    nbins, Cr = T.shape
    if rscale is not None and tuple(rscale.shape) != (N, nbins):
        raise ValueError(f"rscale must be [{N},{nbins}], got {tuple(rscale.shape)}")
    out = torch.empty(B, C, dtype=torch.float32, device=S.device)
    colw = torch.empty(N, Cr, dtype=torch.float32, device=S.device)
    Q = torch.empty(B, nbins, C, dtype=torch.float32, device=S.device)
    counter = torch.empty(1, dtype=torch.int32, device=S.device)
    with _timed("aggregate_blockdiag_fwd"):
        check(lib.gnan_aggregate_blockdiag_graph_fwd(ptr(hop), ptr(hop_off), ptr(node_off), B, ptr(T), nbins, Cr, ptr(rscale), ptr(S), C,
                                                     ptr(out), ptr(colw), ptr(Q), ptr(counter), stream_handle()),
              "gnan_aggregate_blockdiag_graph_fwd")
    return out, colw, Q


@agg_bd_graph_fwd.register_fake
def _(hop, hop_off, node_off, T, rscale, S):
    B = node_off.numel() - 1
    return S.new_empty(B, S.shape[1]), S.new_empty(S.shape[0], T.shape[1]), S.new_empty(B, T.shape[0], S.shape[1])


@torch.library.custom_op("gnan_b200::agg_bd_graph_bwd", mutates_args=())
def agg_bd_graph_bwd(node_off: Tensor, g: Tensor, colw: Tensor, Q: Tensor) -> Tuple[Tensor, Tensor]:
    lib = load()
    g = _f32(g, "g")
    B, nbins, C = Q.shape
    N, Cr = colw.shape
    dS = torch.empty(N, C, dtype=torch.float32, device=g.device)
    dT = torch.empty(nbins, Cr, dtype=torch.float32, device=g.device)
    ws = _ws(lib.gnan_aggregate_blockdiag_graph_bwd_workspace_bytes(nbins, C), g.device)
    with _timed("aggregate_blockdiag_bwd"):
        check(lib.gnan_aggregate_blockdiag_graph_bwd(ptr(node_off), B, nbins, Cr, C, ptr(g), ptr(colw), ptr(Q), ptr(dS), ptr(dT), ptr(ws),
                                                     ws.numel(), stream_handle()), "gnan_aggregate_blockdiag_graph_bwd")
    return dS, dT


@agg_bd_graph_bwd.register_fake
def _(node_off, g, colw, Q):
    return g.new_empty(colw.shape[0], Q.shape[2]), g.new_empty(Q.shape[1], colw.shape[1])


def _bdg_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[2], output[1], output[2])


def _bdg_backward(ctx, g, _g_colw, _g_q):
    node_off, colw, Q = ctx.saved_tensors
    dS, dT = agg_bd_graph_bwd(node_off, g.contiguous(), colw, Q)
    return None, None, None, dT, None, dS


agg_bd_graph_fwd.register_autograd(_bdg_backward, setup_context=_bdg_setup)


def bfs_graph_readout_fwd(edges, node_off: Tensor, max_n: int, T: Tensor, S: Tensor, status: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    """The batched BFS of a LocalEdges batch fused with the output-normalised graph readout (gnan_bfs_graph_readout_fwd): the
    (out, colw, Q) of agg_bd_graph_fwd on the batch's hop bytes and normaliser table, without writing either. status: the batch's
    device int32 [3] (edge status bits, overflow flag, largest hop), filled as apsp_batched's BFS fills it."""
    lib = load()
    T, S = _f32(T, "T"), _f32(S, "S")
    if node_off.dtype != torch.int32 or status.dtype != torch.int32 or status.numel() != 3:
        raise TypeError("node_off int32 [B+1] and status int32 [3] expected")
    B = node_off.numel() - 1
    N, C = S.shape
    nbins, Cr = T.shape
    out = torch.empty(B, C, dtype=torch.float32, device=S.device)
    colw = torch.empty(N, Cr, dtype=torch.float32, device=S.device)
    Q = torch.empty(B, nbins, C, dtype=torch.float32, device=S.device)
    order_ws = torch.empty(4 * B + 4, dtype=torch.int32, device=S.device)
    with _timed("bfs_graph_readout_fwd"):
        check(lib.gnan_bfs_graph_readout_fwd(ptr(edges.src), ptr(edges.dst), ptr(edges.edge_off), ptr(node_off), B, int(max_n), nbins, ptr(T),
                                             Cr, ptr(S), C, ptr(out), ptr(colw), ptr(Q), status.data_ptr(), status.data_ptr() + 4,
                                             status.data_ptr() + 8, ptr(order_ws), stream_handle()), "gnan_bfs_graph_readout_fwd")
    return out, colw, Q


class _BfsGraphReadout(torch.autograd.Function):
    """out = the graph readout of a LocalEdges batch whose distances were never materialised; backward = agg_bd_graph_bwd."""

    @staticmethod
    def forward(ctx, T, S, edges, node_off, max_n, status):
        out, colw, Q = bfs_graph_readout_fwd(edges, node_off, max_n, T, S, status)
        ctx.save_for_backward(node_off, colw, Q)
        return out

    @staticmethod
    def backward(ctx, g):
        node_off, colw, Q = ctx.saved_tensors
        dS, dT = agg_bd_graph_bwd(node_off, g.contiguous(), colw, Q)
        return dT, dS, None, None, None, None


def bfs_graph_readout(edges, node_off, max_n, T, S, status):
    """[B,C] output-normalised graph readout straight from the batch's edge list (preprocess.apsp_batched's deferred batches)"""
    if T.dim() != 2 or not load().gnan_aggregate_blockdiag_graph_supported(T.shape[0], T.shape[1], S.shape[1]):
        raise NotImplementedError("the fused BFS readout covers a global table with nbins <= 64 and C <= 4")
    return _BfsGraphReadout.apply(T, S, edges, node_off, max_n, status)


BLOCKDIAG_GRAPH_KERNEL = True     # tests switch it off to compare the two kernel families


def aggregate_blockdiag(hop, hop_off, node_off, T, S, rscale=None, per_row=False, reduce_graph=True):
    """Block-diagonal aggregation of a packed batch; see gnan_b200.h. A per-graph readout with a global table takes the one-pass
    kernels of csrc/agg_bd.cu (forward statistics reused by the backward), everything else the general kernels."""
    if (BLOCKDIAG_GRAPH_KERNEL and reduce_graph and not per_row and T.dim() == 2
            and load().gnan_aggregate_blockdiag_graph_supported(T.shape[0], T.shape[1], S.shape[1])):
        return agg_bd_graph_fwd(hop, hop_off, node_off, T, rscale, S)[0]
    return agg_blockdiag_fwd(hop, hop_off, node_off, T, rscale, S, bool(per_row), bool(reduce_graph))


# ---------------------------------------------------------------------------------------------------------------------
# row gather with a deterministic backward
# ---------------------------------------------------------------------------------------------------------------------
@torch.library.custom_op("gnan_b200::gather_segment_sum", mutates_args=())
def gather_segment_sum(src: Tensor, order: Optional[Tensor], seg_ptr: Tensor) -> Tensor:
    lib = load()
    src = _f32(src, "src")
    nseg, C = seg_ptr.numel() - 1, src.shape[1]
    out = torch.empty(nseg, C, dtype=torch.float32, device=src.device)
    check(lib.gnan_gather_segment_sum(ptr(src), ptr(order), ptr(seg_ptr), nseg, C, ptr(out), stream_handle()), "gnan_gather_segment_sum")
    return out


@gather_segment_sum.register_fake
def _(src, order, seg_ptr):
    return src.new_empty(seg_ptr.numel() - 1, src.shape[1])


class _GatherRows(torch.autograd.Function):
    """T = Tq[inv]; backward = fixed-order segment sums over a precomputed sort of inv (no atomics)."""

    @staticmethod
    def forward(ctx, tq, inv, order, seg_ptr):
        ctx.save_for_backward(order, seg_ptr)
        return tq.index_select(0, inv)

    @staticmethod
    def backward(ctx, dT):
        order, seg_ptr = ctx.saved_tensors
        return gather_segment_sum(dT.index_select(0, order), None, seg_ptr), None, None, None    # coalesced copy, then contiguous segments


def gather_rows(tq, inv, order, seg_ptr):
    return _GatherRows.apply(tq, inv, order, seg_ptr)


# ---------------------------------------------------------------------------------------------------------------------
# table inputs (no autograd: functions of the integer level counts only)
# ---------------------------------------------------------------------------------------------------------------------
def rho_table_inputs(nbins: int, device, cnt: Optional[Tensor] = None, raw: bool = False) -> Tensor:
    """u[d] (global, [nbins]) or u[i,d] ([rows,nbins], divided by cnt): the scalar inputs rho is evaluated on."""
    lib = load()
    rows = 0 if cnt is None else cnt.shape[0]
    if cnt is not None and (cnt.dtype != torch.int32 or cnt.shape[1] != nbins):
        raise TypeError("cnt must be int32 [rows,nbins]")
    u = torch.empty((max(rows, 1), nbins) if cnt is not None else (nbins,), dtype=torch.float32, device=device)
    if cnt is not None and rows == 0:
        return u[:0]
    check(lib.gnan_rho_table_inputs(ptr(cnt.contiguous()) if cnt is not None else None, rows, nbins, int(raw), ptr(u),
                                    stream_handle()), "gnan_rho_table_inputs")
    return u


def level_rscale(cnt: Tensor) -> Tensor:
    lib = load()
    if cnt.dtype != torch.int32 or cnt.dim() != 2:
        raise TypeError("cnt must be int32 [rows,nbins]")
    rs = torch.empty(cnt.shape, dtype=torch.float32, device=cnt.device)
    check(lib.gnan_level_rscale(ptr(cnt.contiguous()), cnt.shape[0], cnt.shape[1], ptr(rs), stream_handle()), "gnan_level_rscale")
    return rs


# ---------------------------------------------------------------------------------------------------------------------
# losses of the training step: value and gradient in one pass (csrc/train.cu; trainer.py:52-67)
# ---------------------------------------------------------------------------------------------------------------------
@torch.library.custom_op("gnan_b200::ce_rows", mutates_args=())
def _ce_rows(logits: Tensor, rows: Optional[Tensor], labels: Tensor, scale: float, want_grad: bool) -> Tuple[Tensor, Tensor, Tensor]:
    lib = load()
    logits = _f32(logits, "logits")
    if labels.dtype != torch.int64 or (rows is not None and rows.dtype != torch.int64):
        raise TypeError("labels / rows must be int64")
    N, C = logits.shape
    M = labels.numel()
    if rows is not None and rows.numel() != M:
        raise ValueError("rows and labels must have the same length")
    if rows is None and M != N:
        raise ValueError("labels must have one entry per row of logits")
    loss = torch.empty((), dtype=torch.float32, device=logits.device)
    d = torch.empty_like(logits) if want_grad else torch.empty(0, device=logits.device)
    bad = torch.zeros(1, dtype=torch.int32, device=logits.device)
    ws = _ws(lib.gnan_loss_workspace_bytes(), logits.device)
    with _timed("loss"):
        check(lib.gnan_cross_entropy_rows(ptr(logits), N, C, ptr(rows), ptr(labels.contiguous()), M, float(scale), ptr(loss),
                                          ptr(d) if want_grad else None, ptr(bad), ptr(ws), ws.numel(), stream_handle()),
              "gnan_cross_entropy_rows")
    return loss, d, bad


@_ce_rows.register_fake
def _(logits, rows, labels, scale, want_grad):
    return logits.new_empty(()), torch.empty_like(logits) if want_grad else logits.new_empty(0), logits.new_empty(1, dtype=torch.int32)


def _ce_setup(ctx, inputs, output):
    ctx.save_for_backward(output[1])


def _ce_backward(ctx, g, _gd, _gb):
    (d,) = ctx.saved_tensors
    return d * g, None, None, None, None


_ce_rows.register_autograd(_ce_backward, setup_context=_ce_setup)


def cross_entropy_rows(logits, labels, rows=None, reduction="mean", return_flag=False, scale=None):
    """CrossEntropyLoss of logits[rows] (all rows when rows is None) against int64 labels: the loss AND its gradient w.r.t. the
    whole [N,C] logits come out of one kernel (rows without a loss get a zero gradient). `rows` must not repeat an index.
    return_flag: also return the device int32 flag that is set by an out-of-range row / label (checked lazily by the caller)."""
    M = labels.numel()
    if scale is None:                # explicit scale: e.g. 1 / (global number of training rows) on a row shard
        scale = 1.0 / max(M, 1) if reduction == "mean" else 1.0
    loss, _, bad = _ce_rows(logits, None if rows is None else rows.contiguous(), labels, scale, bool(torch.is_grad_enabled() and logits.requires_grad))
    return (loss, bad) if return_flag else loss


@torch.library.custom_op("gnan_b200::bce_logits", mutates_args=())
def _bce_logits(logits: Tensor, targets: Tensor, scale: float, want_grad: bool) -> Tuple[Tensor, Tensor]:
    lib = load()
    logits, targets = _f32(logits, "logits"), _f32(targets, "targets")
    if logits.shape != targets.shape:
        raise ValueError("logits and targets must have the same shape")
    loss = torch.empty((), dtype=torch.float32, device=logits.device)
    d = torch.empty_like(logits) if want_grad else torch.empty(0, device=logits.device)
    ws = _ws(lib.gnan_loss_workspace_bytes(), logits.device)
    with _timed("loss"):
        check(lib.gnan_bce_with_logits(ptr(logits), ptr(targets), logits.numel(), float(scale), ptr(loss), ptr(d) if want_grad else None,
                                       ptr(ws), ws.numel(), stream_handle()), "gnan_bce_with_logits")
    return loss, d


@_bce_logits.register_fake
def _(logits, targets, scale, want_grad):
    return logits.new_empty(()), torch.empty_like(logits) if want_grad else logits.new_empty(0)


def _bce_setup(ctx, inputs, output):
    ctx.save_for_backward(output[1])


def _bce_backward(ctx, g, _gd):
    (d,) = ctx.saved_tensors
    return d * g, None, None, None


_bce_logits.register_autograd(_bce_backward, setup_context=_bce_setup)


def bce_with_logits(logits, targets, reduction="mean"):
    """BCEWithLogitsLoss (value + gradient in one kernel); logits and targets of equal shape, any rank."""
    scale = 1.0 / max(logits.numel(), 1) if reduction == "mean" else 1.0
    return _bce_logits(logits.contiguous(), targets.contiguous(), scale, bool(torch.is_grad_enabled() and logits.requires_grad))[0]
