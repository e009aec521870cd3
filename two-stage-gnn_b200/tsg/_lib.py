"""ctypes binding of libtsg.so (the C ABI declared in /include/tsg.h).

There is deliberately NO fallback: if the shared library is missing or an entry point fails,
importing / calling raises.  Tensors cross the boundary as raw device pointers.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int64, c_size_t, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "libtsg.so")

P, I64, SZ, I, F32 = c_void_p, c_int64, c_size_t, c_int, c_float

# name -> (restype, argtypes); mirrors include/tsg.h line by line
_PROTOTYPES = {
    "tsg_abi_version": (I, []),
    "tsg_last_error": (c_char_p, []),
    "tsg_check_device": (I, []),
    "tsg_init_device": (I, []),
    "tsg_pack_batch": (I, [P, P, P, I64, P, P, P, P, P, P, I64, P, P, P, P]),
    "tsg_pack_batch_compact": (I, [P, P, P, I64, P, P, P, P, P, P, P, P, P]),
    "tsg_pack_dense_batch": (I, [P, P, P, I64, I64, I64, P, P, P, P, P, I64, I64, P, P, P, P, P, P, P, P, P]),
    "tsg_pack_eigen_batch": (I, [P, P, P, P, P, I64, I64, I64, I64, I64, P, P, P, P, P, I64, P, P, P, P, I64, I64, P, P, P, P, I64, I64, I64, P, P, P, P, P, P, P, P, P, P, P, P, P, P, P, P, P, P, P, P, P]),
    "tsg_csr_build_workspace_bytes": (SZ, [I64, I64]),
    "tsg_csr_build": (I, [P, P, P, I64, P, I64, I, P, P, P, P, P, P, P, P, P, SZ, P]),
    "tsg_edge_ptr": (I, [P, I64, P, P, I64, P, P]),
    "tsg_csr_build_graphs_workspace_bytes": (SZ, [I64, I64]),
    "tsg_csr_build_graphs": (I, [P, P, P, P, I64, I64, I64, I64, P, P, P, P, P, P, P, P, P, SZ, P]),
    "tsg_csr_build_graphs_local": (I, [P, P, P, P, I64, I64, I64, I64, P, P, P, P, P, P, P, P, P, SZ, P]),
    "tsg_csr_build_graphs_sym_local": (I, [P, P, P, P, I64, I64, I64, I64, P, P, P, P, P]),
    "tsg_inv_perm": (I, [P, I64, I64, P, P]),
    "tsg_csr_filter_workspace_bytes": (SZ, [I64]),
    "tsg_csr_filter": (I, [P, P, P, P, P, P, I64, P, P, P, P, P, P, P, SZ, P]),
    "tsg_spmm": (I, [P, P, P, P, P, P, I64, I64, I, P]),
    "tsg_spmm_tma": (I, [P, P, P, P, P, P, P, I64, I64, I64, I, P, P]),
    "tsg_spmm_tiled": (I, [P, P, P, P, P, P, P, I64, I64, I64, I, P]),
    "tsg_colsum_workspace_bytes": (SZ, [I64, I64]),
    "tsg_relu_bwd_colsum": (I, [P, P, P, P, I64, I64, P, SZ, P]),
    "tsg_relu_bwd_colsum_rank1": (I, [P, P, P, P, P, P, I64, I64, P, SZ, P]),
    "tsg_linear_fwd": (I, [P, P, P, P, I64, I64, I64, I, I, P]),
    "tsg_dense_epilogue_bwd": (I, [P, P, P, P, P, I64, I64, I64, I, P]),
    "tsg_softmax_bwd": (I, [P, P, P, I64, I64, P]),
    "tsg_linear_bwd_weight_workspace_bytes": (SZ, [I64, I64]),
    "tsg_linear_bwd_weight": (I, [P, P, P, P, I64, I64, I64, P, SZ, P]),
    "tsg_sag_boundary_bwd": (I, [P, P, P, P, I64, P, P, I64, I64, I64, P, P, P, SZ, P]),
    "tsg_dense_to_coo_workspace_bytes": (SZ, [I64, I64]),
    "tsg_dense_to_coo": (I, [P, I64, I64, I64, P, P, P, P, P, P, P, I64, P, P, SZ, P]),
    "tsg_nodebn_fwd": (I, [P, P, P, P, I64, I64, I64, P]),
    "tsg_nodebn_bwd": (I, [P, P, P, P, I64, I64, I64, P]),
    "tsg_gat_fwd": (I, [P, P, P, P, P, P, P, I64, I64, I64, F32, P, P, P, P]),
    "tsg_gat_bwd_workspace_bytes": (SZ, [I64, I64]),
    "tsg_gat_bwd": (I, [P, P, P, P, P, P, P, P, P, P, P, I64, I64, I64, I64, F32, P, P, P, P, SZ, P]),
    "tsg_seg_contract": (I, [P, P, P, I64, I64, I64, P, I, P, P]),
    "tsg_seg_linear": (I, [P, P, P, I64, I64, I64, I, P, P]),
    "tsg_seg_linear_tc": (I, [P, P, P, I64, I64, I64, I, P, P, P]),
    "tsg_linear_tc": (I, [P, P, P, I64, I64, I64, I, I, P, P, P]),
    "tsg_topk_workspace_bytes": (SZ, [I64, I64]),
    "tsg_topk_sizes": (I, [P, I64, F32, P, P, SZ, P]),
    "tsg_topk": (I, [P, P, P, I64, I64, P, P, SZ, P]),
    "tsg_topk_bounded": (I, [P, P, P, I64, I64, I64, P, P, SZ, P]),
    "tsg_batch_to_ptr": (I, [P, I64, I64, P, P]),
    "tsg_filter_adj_workspace_bytes": (SZ, [I64]),
    "tsg_filter_adj": (I, [P, P, I64, P, P, I64, I64, P, P, P, P, P, SZ, P]),
    "tsg_gate_gather_fwd": (I, [P, P, P, P, P, P, I64, I64, P]),
    "tsg_gate_gather_bwd": (I, [P, P, P, P, P, P, I64, I64, P]),
    "tsg_readout_fwd": (I, [P, P, I64, I64, I, P, I64, P, P]),
    "tsg_readout_bwd": (I, [P, I64, P, P, I64, I64, I64, I, P, P]),
    "tsg_triplet_workspace_bytes": (SZ, [I64, I64, I64]),
    "tsg_triplet_fwd": (I, [P, P, I64, I64, I64, F32, F32, P, P, P, P, SZ, P]),
    "tsg_triplet_bwd": (I, [P, P, I64, I64, I64, F32, F32, P, P, P, P, P, SZ, P]),
    "tsg_pairdist_matrix": (I, [P, I64, I64, F32, P, P]),
    "tsg_eigpool_build": (I, [P, P, P, P, P, P, I64, I64, I, P, P, P, P, P]),
    "tsg_coarsen_edges_workspace_bytes": (SZ, [I64]),
    "tsg_coarsen_edges": (I, [P, P, P, I64, P, P, P, P, P, P, SZ, P]),
    "tsg_eigen_bfs_clusters": (I, [P, P, P, P, I64, I64, I64, I64, I64, I64, P, P, P, P, P, P, P, P, P]),
    "tsg_eigen_group_clusters": (I, [P, P, P, P, I64, I64, I64, I64, I64, P, P, P, P, P, P, P, P, P]),
    "tsg_eigen_coarse": (I, [P, I64, I64, P, P, P, P, P, P, P, P, P, P, P, P, P]),
    "tsg_eigen_final": (I, [P, P, P, P, I64, I64, I64, I64, I64, P, I64, P]),
    "tsg_linkpred_workspace_bytes": (SZ, [I64]),
    "tsg_linkpred_loss_fwd": (I, [P, P, P, P, I64, I64, ctypes.c_double, F32, P, P, SZ, P]),
    "tsg_linkpred_loss_bwd": (I, [P, P, P, P, I64, I64, ctypes.c_double, F32, P, P, P]),
    "tsg_pred_ce_workspace_bytes": (SZ, [P, I64]),
    "tsg_pred_ce_fwd": (I, [P, P, P, I64, P, P, P, P, SZ, P]),
    "tsg_pred_ce_bwd": (I, [P, P, P, I64, P, P, P, P, P, SZ, P]),
    "tsg_pred_classify_workspace_bytes": (SZ, [P, I64]),
    "tsg_pred_classify": (I, [P, P, P, I64, P, P, P, P, P, P, SZ, P]),
    "tsg_knn_predict": (I, [P, P, P, I64, I64, I64, I, I, P, P]),
    "tsg_knn_classify": (I, [P, P, P, P, I64, I64, I64, I, I, P, P, P, P]),
    "tsg_mlp1_predict": (I, [P, P, I64, I64, I64, I64, I64, P, F32, P, P, P, P, P]),
    "tsg_mlp1_train": (I, [P, P, I64, I64, I64, I64, I64, P, P, P, I64, F32, F32, F32, F32, F32, P, P]),
    "tsg_tu_load": (I, [c_char_p, I, I64, P]),
    "tsg_tu_sizes": (I, [P, P]),
    "tsg_tu_fill": (I, [P, P, P, P, P, P, P, P]),
    "tsg_tu_free": (None, [P]),
    "tsg_sag_arena_bytes": (SZ, [P]),
    "tsg_sag_arena_locate": (I, [P, I, I, P, P]),
    "tsg_sag_set_fused": (I, [I]),
    "tsg_sag_triplet_step_workspace_bytes": (SZ, [P, P]),
    "tsg_sag_triplet_step_compact": (I, [P, P, P, P, P, P, P, P, P, P, P, P, P, P, SZ, P, SZ, P]),
    "tsg_sag_step_fwd_compact": (I, [P, P, P, P, P, P, P, P, P, P, P, SZ, P, SZ, P]),
    "tsg_sag_step_bwd_compact": (I, [P, P, P, P, P, P, P, P, P, SZ, P, SZ, P]),
    "tsg_sag_nll_step_workspace_bytes": (SZ, [P, P]),
    "tsg_sag_nll_step_compact": (I, [P, P, P, P, P, P, P, P, P, P, P, P, P, P, SZ, P, SZ, P]),
    "tsg_sag_classify_workspace_bytes": (SZ, [P, P]),
    "tsg_sag_classify_compact": (I, [P, P, P, P, P, P, P, P, P, P, P, P, P, P, SZ, P, SZ, P]),
    "tsg_sag_encoder_fwd": (I, [P, P, P, P, P, P, P, P, SZ, P]),
    "tsg_sag_encoder_bwd": (I, [P, P, P, P, P, P, P, SZ, P]),
    "tsg_sag_encoder_fwd_compact": (I, [P, P, P, P, P, P, P, P, P, SZ, P]),
    "tsg_sag_encoder_bwd_compact": (I, [P, P, P, P, P, P, P, SZ, P]),
    "tsg_sag_encoder_embed_compact": (I, [P, P, P, P, P, P, P, P, P, SZ, P]),
    "tsg_gate_score_bwd_workspace_bytes": (SZ, []),
    "tsg_gate_score_bwd": (I, [P, P, P, P, I64, I64, I64, P, P, P, SZ, P]),
    "tsg_gate_readout_fwd": (I, [P, P, P, P, I64, I64, P, P, I64, P, P]),
    "tsg_gate_readout_linear_fwd": (I, [P, P, P, P, I64, I64, I64, P, P, I64, P, P, P, P]),
    "tsg_spmm_label_dot": (I, [P, P, P, P, P, I64, P, P, P, P, I64, I64, I, P]),
    "tsg_spmm_dot": (I, [P, P, P, P, P, P, P, P, I64, I64, I, P]),
    "tsg_sag_conv_bwd_fused": (I, [P, P, P, P, P, P, P, P, P, I64, I64, P, SZ, P]),
    "tsg_embed_fwd": (I, [P, P, P, I64, I64, I64, P]),
    "tsg_embed_bwd_weight_workspace_bytes": (SZ, [I64, I64]),
    "tsg_embed_bwd_weight": (I, [P, P, P, I64, I64, I64, P, SZ, P]),
}


class SagShape(ctypes.Structure):
    """tsg_sag_shape (include/tsg.h)."""
    _fields_ = [("num_graphs", c_int64), ("in_feat", c_int64), ("hidden", c_int64), ("num_edges", c_int64),
                ("n", c_int64 * 4), ("max_graph_nodes", c_int64 * 3), ("max_graph_edges", c_int64), ("pooling_ratio", ctypes.c_double), ("flags", c_int64), ("status", c_void_p)]

class SagHead(ctypes.Structure):
    """tsg_sag_head (include/tsg.h)."""
    _fields_ = [("num_classes", c_int64), ("num_triplets", c_int64), ("margin", c_float), ("eps", c_float),
                ("dropout_p", c_float), ("seed", ctypes.c_uint64)]

class PredHead(ctypes.Structure):
    """tsg_pred_head (include/tsg.h)."""
    _fields_ = [("num_layers", c_int64), ("in_dim", c_int64), ("out_dim", c_int64 * 8), ("relu_mask", c_int64),
                ("softmax_first", c_int64), ("weight", c_void_p * 8), ("bias", c_void_p * 8)]



EXPORTS = tuple(_PROTOTYPES)

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(or `make -C two-stage-gnn_b200/csrc`). tsg has no CPU or eager fallback.")

lib = ctypes.CDLL(LIB_PATH)
for _name, (_res, _args) in _PROTOTYPES.items():
    _fn = getattr(lib, _name)          # AttributeError here = header/library mismatch
    _fn.restype = _res
    _fn.argtypes = _args

if lib.tsg_abi_version() != 1:
    raise ImportError(f"libtsg ABI version {lib.tsg_abi_version()} != 1")

# kernels each entry point enqueues (memsets not counted); bench.py reports the sum as gpu_launches
# kernels one call enqueues at the bench shape (counted from profiles/r01c_launches_{dense,compact}_step.csv:
# 90 / 88 of ours per step = 26 outside the executor + 38 / 36 forward + 26 backward)
KERNELS_PER_CALL = {
    "tsg_pack_batch": 1, "tsg_csr_build": 12, "tsg_edge_ptr": 1, "tsg_csr_build_graphs": 5, "tsg_csr_build_graphs_local": 5, "tsg_embed_fwd": 1, "tsg_embed_bwd_weight": 2, "tsg_spmm": 1, "tsg_spmm_tiled": 1, "tsg_relu_bwd_colsum": 1, "tsg_topk_sizes": 3, "tsg_topk": 2,
    "tsg_batch_to_ptr": 1, "tsg_filter_adj": 7, "tsg_gate_gather_fwd": 1, "tsg_gate_gather_bwd": 1,
    "tsg_readout_fwd": 1, "tsg_readout_bwd": 1, "tsg_triplet_fwd": 2, "tsg_triplet_bwd": 9,
    "tsg_pairdist_matrix": 1, "tsg_linear_fwd": 1, "tsg_dense_epilogue_bwd": 1, "tsg_linear_bwd_weight": 2, "tsg_sag_boundary_bwd": 2,
    "tsg_eigpool_build": 1, "tsg_coarsen_edges": 6, "tsg_eigen_bfs_clusters": 1, "tsg_eigen_group_clusters": 1, "tsg_eigen_coarse": 1, "tsg_eigen_final": 1, "tsg_inv_perm": 1, "tsg_csr_filter": 5, "tsg_sag_encoder_fwd": 38, "tsg_sag_encoder_bwd": 22, "tsg_sag_encoder_fwd_compact": 36, "tsg_sag_encoder_embed_compact": 3, "tsg_sag_triplet_step_compact": 72, "tsg_sag_step_fwd_compact": 37, "tsg_sag_step_bwd_compact": 25, "tsg_sag_nll_step_compact": 64, "tsg_sag_classify_compact": 6, "tsg_linkpred_loss_fwd": 3, "tsg_linkpred_loss_bwd": 1, "tsg_spmm_label_dot": 1, "tsg_gate_readout_fwd": 1, "tsg_gate_readout_linear_fwd": 2, "tsg_sag_encoder_bwd_compact": 22, "tsg_relu_bwd_colsum_rank1": 1, "tsg_sag_conv_bwd_fused": 1, "tsg_gate_score_bwd": 1, "tsg_spmm_dot": 1, "tsg_pack_batch_compact": 1, "tsg_pack_dense_batch": 1, "tsg_pack_eigen_batch": 1, "tsg_seg_contract": 1, "tsg_seg_linear": 1, "tsg_seg_linear_tc": 1, "tsg_linear_tc": 2, "tsg_gat_fwd": 2, "tsg_gat_bwd": 2, "tsg_dense_to_coo": 6, "tsg_nodebn_fwd": 1, "tsg_nodebn_bwd": 1,
    "tsg_pred_ce_fwd": 2, "tsg_pred_ce_bwd": 1, "tsg_pred_classify": 2,
}
launch_calls = 0        # libtsg entry points called since import
kernel_launches = 0     # kernels enqueued by them
profile = None          # set to {} to record (start, end) CUDA events per entry point


def last_error() -> str:
    return lib.tsg_last_error().decode()


def ptr(t):
    """Device pointer of a tensor (None -> NULL). Refuses CPU tensors: no fallback."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("tsg: expected a CUDA tensor (there is no CPU path)")
    if not t.is_contiguous():
        raise RuntimeError("tsg: expected a contiguous tensor")
    return t.data_ptr()


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


_inited_devices = set()


def init_device() -> None:
    """tsg_init_device() for the current device, once (the only allocating entry point: keeps every compute entry
    allocation free and stream-capture safe)."""
    d = torch.cuda.current_device()
    if d not in _inited_devices:
        if lib.tsg_init_device() != 0:
            raise RuntimeError(f"tsg_init_device failed: {last_error()}")
        _inited_devices.add(d)


def call(name: str, *args) -> None:
    global launch_calls, kernel_launches
    if not _inited_devices or torch.cuda.current_device() not in _inited_devices:
        init_device()
    if profile is not None:
        s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
        s.record()
        rc = getattr(lib, name)(*args)
        e.record()
        profile.setdefault(name, []).append((s, e))
    else:
        rc = getattr(lib, name)(*args)
    launch_calls += 1
    kernel_launches += KERNELS_PER_CALL.get(name, 1)
    if rc != 0:
        raise RuntimeError(f"{name} failed ({rc}): {last_error()}")


def workspace(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
