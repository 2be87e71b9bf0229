"""ctypes binding of libgnan_b200.so (include/gnan_b200.h). No torch types cross this boundary: only raw device
pointers, sizes and the current CUDA stream handle. There is NO CPU fallback: if the library is missing the import
of any compute entry point raises, and every call on a non-CUDA tensor raises."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgnan_b200.so")

c_void_p, c_int, c_int32, c_int64, c_size_t, c_float, c_uint64 = (
    ctypes.c_void_p, ctypes.c_int, ctypes.c_int32, ctypes.c_int64, ctypes.c_size_t, ctypes.c_float, ctypes.c_uint64)

PREC_FP32, PREC_TF32X3, PREC_TF32 = 0, 1, 2
PRECISIONS = {"fp32": PREC_FP32, "tf32x3": PREC_TF32X3, "tf32": PREC_TF32}
HOP_UNREACHABLE = 255
APSP_BATCHED_MAX_NODES = 1024    # GNAN_APSP_BATCHED_MAX_NODES: largest graph of the batched BFS (gnan_apsp_bfs_batched_ex)
AGG_AUTO, AGG_CUDA_CORES, AGG_TENSOR_CORES = 0, 1, 2
AGG_ALGOS = {"auto": AGG_AUTO, "cuda": AGG_CUDA_CORES, "tc": AGG_TENSOR_CORES}


class MlpParams(ctypes.Structure):
    _fields_ = [("G", c_int32), ("H", c_int32), ("C", c_int32), ("n_layers", c_int32),
                ("w1", c_void_p), ("b1", c_void_p), ("wh", c_void_p), ("bh", c_void_p), ("wo", c_void_p), ("bo", c_void_p)]


class MlpGrads(ctypes.Structure):
    _fields_ = [("w1", c_void_p), ("b1", c_void_p), ("wh", c_void_p), ("bh", c_void_p), ("wo", c_void_p), ("bo", c_void_p),
                ("du", c_void_p)]


# name -> (restype, argtypes); must list every symbol include/gnan_b200.h declares (tests/test_cabi.py checks it)
SIGNATURES = {
    "gnan_version": (c_int, []),
    "gnan_last_error": (ctypes.c_char_p, []),
    "gnan_launch_count": (c_uint64, []),
    "gnan_mlp_workspace_bytes": (c_size_t, [c_int64, ctypes.POINTER(MlpParams), c_int, c_int]),
    "gnan_mlp_fwd": (c_int, [c_void_p, c_int64, c_int64, ctypes.POINTER(MlpParams), c_float, c_uint64, c_void_p, c_int, c_void_p,
                             c_void_p, c_size_t, c_void_p]),
    "gnan_mlp_bwd": (c_int, [c_void_p, c_int64, c_int64, ctypes.POINTER(MlpParams), c_float, c_uint64, c_void_p, c_int, c_void_p,
                             ctypes.POINTER(MlpGrads), c_void_p, c_size_t, c_void_p]),
    "gnan_mlp_bwd_ext_supported": (c_int, [ctypes.POINTER(MlpParams), c_int]),
    "gnan_mlp_bwd_ext": (c_int, [c_void_p, c_int64, c_int64, ctypes.POINTER(MlpParams), c_float, c_uint64, c_void_p, c_int, c_void_p,
                                 c_void_p, c_void_p, ctypes.POINTER(MlpGrads), c_void_p, c_size_t, c_void_p]),
    "gnan_mlp_entries_workspace_bytes": (c_size_t, [c_int64, ctypes.POINTER(MlpParams), c_int, c_int]),
    "gnan_mlp_entries_fwd_ex": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, ctypes.POINTER(MlpParams), c_int, c_void_p, c_void_p]),
    "gnan_mlp_entries_bwd": (c_int, [c_void_p, c_void_p, c_int64, c_int64, ctypes.POINTER(MlpParams), c_int, c_void_p,
                                     ctypes.POINTER(MlpGrads), c_void_p, c_size_t, c_void_p]),
    "gnan_entries_to_rows": (c_int, [c_void_p, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p]),
    "gnan_rows_to_entries_scratch_floats": (c_size_t, [c_int32, c_int32, c_int64]),
    "gnan_rows_to_entries": (c_int, [c_void_p, c_int64, c_int32, c_int32, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "gnan_gather_segment_sum": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p]),
    "gnan_rho_table_inputs": (c_int, [c_void_p, c_int64, c_int32, c_int, c_void_p, c_void_p]),
    "gnan_level_rscale": (c_int, [c_void_p, c_int64, c_int32, c_void_p, c_void_p]),
    "gnan_aggregate_rows_fwd_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int32, c_int32]),
    "gnan_aggregate_rows_fwd_ws": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int, c_int32, c_int32, c_void_p,
                                           c_void_p, c_int32, c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "gnan_aggregate_rows_bwd_ws_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int32, c_int32, c_int32, c_int]),
    "gnan_aggregate_rows_bwd_ws": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int, c_int32, c_int32, c_void_p,
                                           c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_size_t,
                                           c_void_p]),
    "gnan_aggregate_blockdiag_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_int, c_int32, c_int32,
                                             c_void_p, c_void_p, c_int32, c_int, c_void_p, c_void_p]),
    "gnan_aggregate_blockdiag_graph_supported": (c_int, [c_int32, c_int32, c_int32]),
    "gnan_aggregate_blockdiag_graph_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_int32, c_int32, c_void_p, c_void_p,
                                                   c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "gnan_aggregate_blockdiag_graph_bwd_workspace_bytes": (c_size_t, [c_int32, c_int32]),
    "gnan_aggregate_blockdiag_graph_bwd": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p,
                                                   c_void_p, c_void_p, c_size_t, c_void_p]),
    "gnan_aggregate_blockdiag_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_int, c_int32, c_int32,
                                             c_void_p, c_void_p, c_int32, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "gnan_apsp_bfs_batched_local": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                            c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "gnan_bfs_graph_readout_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_int32, c_void_p,
                                           c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "gnan_edges_from_local": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int64, c_void_p, c_void_p]),
    "gnan_build_csr_workspace_bytes": (c_size_t, [c_int32, c_int64]),
    "gnan_build_csr": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "gnan_apsp_bfs_workspace_bytes": (c_size_t, [c_int32, c_int32]),
    "gnan_apsp_bfs": (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_int64, c_void_p, c_int32, c_void_p,
                              c_void_p, c_size_t, c_void_p]),
    "gnan_apsp_msbfs_workspace_bytes": (c_size_t, [c_int32]),
    "gnan_apsp_msbfs": (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_int64, c_void_p, c_int32, c_void_p,
                                c_void_p, c_size_t, c_void_p]),
    "gnan_apsp_bfs_batched_ex": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_int32,
                                         c_void_p, c_void_p, c_void_p, c_void_p]),
    "gnan_loss_workspace_bytes": (c_size_t, []),
    "gnan_cross_entropy_rows": (c_int, [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_int64, c_float, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_size_t, c_void_p]),
    "gnan_bce_with_logits": (c_int, [c_void_p, c_void_p, c_int64, c_float, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "gnan_adam_step": (c_int, [c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_float, c_float, c_float,
                               c_float, c_void_p]),
    "gnan_apsp_bfs16_workspace_bytes": (c_size_t, [c_int32, c_int32]),
    "gnan_apsp_bfs16": (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_size_t,
                                c_void_p]),
    "gnan_level_counts16": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int32, c_void_p]),
    "gnan_aggregate_rows16_fwd": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int, c_int32, c_int32, c_void_p, c_void_p,
                                          c_int32, c_void_p, c_void_p]),
    "gnan_aggregate_rows16_bwd": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int, c_int32, c_int32, c_void_p, c_void_p,
                                          c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "gnan_hops_to_reference": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int32, c_void_p, c_void_p, c_void_p]),
    "gnan_hops_from_reference": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_int32, c_void_p,
                                         c_void_p]),
}

_lib = None


class GnanError(RuntimeError):
    pass


def load():
    """Load the library (once). Raises if it has not been built: there is no fallback path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise GnanError(f"{LIB_PATH} not found: build it with `python {os.path.join(_HERE, 'build.py')}` "
                            "(gnan_b200 has no CPU or eager fallback)")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc, what):
    if rc != 0:
        msg = load().gnan_last_error().decode("utf-8", "replace")
        kind = {1: ValueError, 2: NotImplementedError}.get(rc, GnanError)
        raise kind(f"{what}: {msg} (gnan_b200 error {rc})")


def ptr(t):
    """Raw device pointer of a tensor (None -> NULL). Refuses anything that is not a contiguous CUDA tensor."""
    if t is None:
        return None
    if not t.is_cuda:
        raise GnanError("gnan_b200 kernels need CUDA tensors (no CPU fallback)")
    if not t.is_contiguous():
        raise ValueError("gnan_b200 kernels need contiguous tensors")
    return t.data_ptr() if t.numel() > 0 else None


def stream_handle():
    import torch
    return torch.cuda.current_stream().cuda_stream
