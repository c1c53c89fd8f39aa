"""ctypes binding of libpcc.so (include/pcc.h).  No CPU fallback: if the shared library
is missing or the tensors are not CUDA tensors the call raises."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PCC_LIB", os.path.normpath(os.path.join(_HERE, "..", "lib", "libpcc.so")))

ACT = {"none": 0, "relu": 1, "gelu": 2, "silu": 3, "tanh": 4}
POOL = {"sum": 0, "mean": 1, "max": 2, "add": 3}

_vp, _i64, _i32, _f32 = C.c_void_p, C.c_int64, C.c_int, C.c_float

MAX_PHI_LAYERS = 6


class PhiDesc(C.Structure):
    """mirror of pcc_phi_desc (include/pcc.h)"""
    _fields_ = [("n_layers", C.c_int32), ("input_dim", C.c_int32), ("hidden", C.c_int32), ("act", C.c_int32),
                ("pooling", C.c_int32), ("residual_mask", C.c_int32),
                ("w", _vp * MAX_PHI_LAYERS), ("b", _vp * MAX_PHI_LAYERS)]


class HeadDesc(C.Structure):
    """mirror of pcc_head_desc (include/pcc.h)"""
    _fields_ = [("n_layers", C.c_int32), ("dims", C.c_int32 * 5), ("act", C.c_int32), ("w", _vp * 4), ("b", _vp * 4)]


# name -> argtypes (every entry returns int unless listed in _RESTYPES)
_SIGS = {
    "pcc_version": [],
    "pcc_check_device": [_i32],
    "pcc_segment_offsets": [_vp, _i64, _i64, _vp, _i32, _vp],
    "pcc_index_max": [_vp, _i64, _vp, _i32, _vp],
    "pcc_segment_pool_fwd": [_vp, _vp, _i64, _i64, _i64, _i32, _vp, _vp, _i32, _vp],
    "pcc_segment_pool_bwd": [_vp, _vp, _vp, _i64, _i64, _i64, _i32, _vp, _i32, _vp],
    "pcc_set_dense_precision": [_i32],
    "pcc_linear_fwd": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _i32, _i32, _i32, _vp],
    "pcc_linear_bwd_data": [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i32, _vp],
    "pcc_linear_bwd_weight": [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i32, _i32, _vp],
    "pcc_act_bwd": [_vp, _vp, _vp, _i64, _i32, _i32, _vp],
    "pcc_layernorm_fwd": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _f32, _i32, _vp],
    "pcc_layernorm_bwd": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _i32, _vp],
    "pcc_batchnorm_fwd_train": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _f32, _f32, _i32, _vp],
    "pcc_batchnorm_fwd_eval": [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _f32, _i32, _vp],
    "pcc_batchnorm_bwd": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _vp],
    "pcc_csr_workspace_bytes": [_i64, _i64],
    "pcc_csr_build": [_vp, _i64, _i64, _vp, _vp, _vp, _i32, _vp],
    "pcc_csr_transpose": [_vp, _vp, _i64, _i64, _i32, _vp, _vp, _vp, _i32, _vp],
    "pcc_csr_transpose_blocks": [_vp, _i32, _vp, _i64, _i64, _vp, _vp, _i32, _vp],
    "pcc_csr_transpose_pos": [_vp, _i32, _i64, _vp, _vp, _vp, _i32, _vp],
    "pcc_graph_aggregate_fwd": [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _vp, _vp, _i32, _vp],
    "pcc_graph_aggregate_bwd": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _vp, _i32, _vp],
    "pcc_knn": [_vp, _i64, _vp, _i64, _i64, _i32, _vp, _vp, _vp, _i32, _vp],
    "pcc_knn_edges": [_vp, _i64, _i32, _vp, _i32, _vp],
    "pcc_expand_segments": [_vp, _i64, _i64, _vp, _i32, _vp],
    "pcc_offset_edges": [_vp, _i64, _vp, _vp, _i64, _vp, _i32, _vp],
    "pcc_edge_weights_workspace_bytes": [_i64, _i64],
    "pcc_edge_weights": [_vp, _i64, _vp, _i64, _vp, _i64, _f32, _vp, _vp, _vp, _i32, _vp],
    "pcc_mlp_head_supported": [C.POINTER(HeadDesc)],
    "pcc_mlp_head_fwd": [C.POINTER(HeadDesc), _vp, _vp, _vp, _i64, _i32, _vp],
    "pcc_mlp_head_workspace_bytes": [C.POINTER(HeadDesc), _i64],
    "pcc_mlp_head_bwd": [C.POINTER(HeadDesc), _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp],
    "pcc_adam_step": [_vp, _i32, _i64, _vp, _vp, _vp, _f32, _f32, _f32, _f32, _f32, _i32, _i32, _vp],
    "pcc_peer_alloc": [_i64, C.POINTER(C.c_void_p), _vp, _i32],
    "pcc_peer_open": [_vp, C.POINTER(C.c_void_p), _i32],
    "pcc_peer_close": [_vp, _i32],
    "pcc_peer_free": [_vp, _i32],
    "pcc_peer_allreduce": [_vp, _i64, _vp, _i64, _i32, _i32, _f32, _vp, _i32, _vp],
    "pcc_bce_logits": [_vp, _vp, _i64, _vp, _vp, _i32, _vp],
    "pcc_gather_rows": [_vp, _vp, _i64, _i32, _i64, _vp, _vp, _vp, _i32, _vp],
    "pcc_gnn_packed_bytes": [],
    "pcc_gnn_max_blocks": [],
    "pcc_gnn_pack_weights": [_vp, _vp, _vp, _vp, _i32, _vp],
    "pcc_gnn_conv1_fwd": [_vp, _i32, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp, C.POINTER(C.c_int), _i32, _vp],
    "pcc_gnn_bn_finalize": [_vp, _i32, _i32, _i64, _vp, _vp, _f32, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp],
    "pcc_gnn_bn_eval": [_vp, _vp, _vp, _vp, _f32, _i32, _vp, _vp, _i32, _vp],
    "pcc_gnn_bn_apply": [_vp, _vp, _vp, _i64, _i32, _vp, _i32, _vp],
    "pcc_gnn_conv_fwd": [_vp, _vp, _vp, _vp, _i32, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _i64, _vp, C.POINTER(C.c_int), _i32, _vp],
    "pcc_gnn_fc1_pool_fwd": [_vp, _vp, _vp, _vp, _i64, _i64, _i32, _vp, _vp, C.POINTER(C.c_int), _i32, _vp],
    "pcc_gnn_pool_affine": [_vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _i32, _vp],
    "pcc_gnn_pool_bwd_prep": [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _i32, _vp],
    "pcc_gnn_bn_bwd_finalize": [_vp, _i32, _i32, _i64, _vp, _vp, _vp, _vp, _i32, _vp],
    "pcc_gnn_reduce": [_vp, _i32, _i64, _vp, _i32, _vp],
    "pcc_gnn_fc1_bwd": [_vp] * 12 + [_i64, _i32, _vp, _vp, _vp, _vp, C.POINTER(C.c_int), _i32, _vp],
    "pcc_gnn_conv_bwd": [_vp] * 12 + [_i64, _i32, _vp, _vp, _vp, _vp, C.POINTER(C.c_int), _i32, _vp],
    "pcc_gnn_agg_bwd": [_vp, _vp, _vp, _vp, _i32] + [_vp] * 6 + [_i64, _i32, _vp, C.POINTER(C.c_int), _i32, _vp],
    "pcc_gnn_conv1_bwd": [_vp] * 9 + [_i32, _i64, _i32, _vp, C.POINTER(C.c_int), _i32, _vp],
    "pcc_launch_count": [_i32],
    "pcc_prof_enable": [_i32],
    "pcc_prof_read": [_i32, C.POINTER(C.c_double), C.POINTER(C.c_int64)],
    "pcc_debug_set_trace": [_vp],
    "pcc_debug_set_fwd_pair": [_i32],
    "pcc_debug_set_bwd_pipe": [_i32],
    "pcc_debug_set_pdl": [_i32],
    "pcc_selftest_umma": [_i32, _vp, _i32, _vp],
    "pcc_selftest_fp32_peak": [_vp, _i32, _i32, _i32, _vp],
    "pcc_phi_fused_supported": [C.POINTER(PhiDesc)],
    "pcc_phi_fused_workspace_bytes": [C.POINTER(PhiDesc), _i64, _i64],
    "pcc_phi_packed_bytes": [C.POINTER(PhiDesc)],
    "pcc_deepsets_phi_pool_fwd": [C.POINTER(PhiDesc), _vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _i32, _vp],
    "pcc_deepsets_phi_pool_bwd": [C.POINTER(PhiDesc), _vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp],
}
_RESTYPES = {"pcc_gnn_packed_bytes": _i64, "pcc_gnn_max_blocks": C.c_int, "pcc_csr_workspace_bytes": _i64, "pcc_phi_fused_workspace_bytes": _i64, "pcc_launch_count": _i64,
             "pcc_phi_packed_bytes": _i64, "pcc_mlp_head_workspace_bytes": _i64,
             "pcc_edge_weights_workspace_bytes": _i64}
EXPORTS = tuple(_SIGS) + ("pcc_last_error",)

_lib = None


def load() -> C.CDLL:
    """Load libpcc.so or raise — there is no pure-Python / CPU path behind it."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"libpcc.so not found at {LIB_PATH}; build it with `python -c 'import __graft_entry__ as g; "
                           f"g.build()'` (nvcc, sm_100a).  There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    lib.pcc_last_error.restype = C.c_char_p
    lib.pcc_last_error.argtypes = []
    for name, args in _SIGS.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library disagree
        fn.argtypes = args
        fn.restype = _RESTYPES.get(name, C.c_int)
    _lib = lib
    return lib


def last_error() -> str:
    return load().pcc_last_error().decode("utf-8", "replace")


def call(name: str, *args):
    lib = load()
    rc = getattr(lib, name)(*args)
    if name in _RESTYPES:
        return rc
    if rc != 0:
        raise RuntimeError(f"{name} failed: {last_error()}")
    return rc


def ptr(t: Optional[torch.Tensor]):
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def require_cuda(*tensors: Optional[torch.Tensor]) -> int:
    """All tensors must live on one CUDA device; returns its index."""
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("pcc_b200 runs on CUDA tensors only (sm_100a kernels, no CPU fallback); "
                               f"got a tensor on {t.device}")
        if dev is None:
            dev = t.device.index
        elif t.device.index != dev:
            raise RuntimeError("tensors live on different CUDA devices")
    if dev is None:
        raise RuntimeError("no tensor given")
    return dev


def stream_ptr(device: int):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def f32c(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


def i64c(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.int64:
        t = t.long()
    return t if t.is_contiguous() else t.contiguous()
