"""Modules mirroring the reference's operator/plugin surface for the SAGPool path.

* `GCNConv`   -- same constructor, parameter names/shapes/initialisers and forward signature as
  PyG 1.6.3's GCNConv as used in Code/sag/network.py:19-23 and Code/sag/layers.py:12, so the
  reference's `state_dict` keys (`conv1.weight` [in,out], `pool1.score_layer.bias`, ...) round-trip.
* `PackedSAGNet` -- Code/sag/network.py:9-53 `Net` with the `batch` vector the reference's
  commented-out line (network.py:31) would have passed: one forward over a block-diagonal packed
  batch of many graphs instead of one graph per call.  Same parameters, same arithmetic per graph.
"""
from __future__ import annotations

import ctypes
import math
import os
from typing import Optional

import numpy as np
import torch
import torch.nn.functional as F

from . import ops
from .ops import CSR, EdgeList


USE_EXECUTOR = os.environ.get("TSG_SAG_EXECUTOR", "1") != "0"   # K10 native step executor for PackedSAGNet
USE_NATIVE_STEP = os.environ.get("TSG_NATIVE_STEP", "1") != "0"  # K14: forward + loss + backward in one C-ABI call


def _glorot_(t: torch.Tensor) -> None:
    a = math.sqrt(6.0 / (t.size(-2) + t.size(-1)))
    with torch.no_grad():
        t.uniform_(-a, a)


class _CsrCache:
    """conv_k and pool_k.score_layer receive the SAME edge_index tensor (Code/sag/network.py:34-35,
    layers.py:18): build K1's CSR once per pooling level and reuse it.  Keyed on the tensor object
    (held alive so its storage cannot be recycled) plus its version counter."""

    def __init__(self, slots: int = 4):
        self.slots, self.items = slots, []

    def get(self, edge_index: torch.Tensor, num_nodes: int) -> CSR:
        for ei, ver, n, csr in self.items:
            if ei is edge_index and ver == edge_index._version and n == num_nodes:
                return csr
        csr = ops.build_csr(EdgeList.from_edge_index(edge_index), num_nodes)
        self.items.append((edge_index, edge_index._version, num_nodes, csr))
        if len(self.items) > self.slots:
            self.items.pop(0)
        return csr


_GLOBAL_CSR_CACHE = _CsrCache()


class GCNConv(torch.nn.Module):
    """Drop-in for torch_geometric.nn.GCNConv (defaults improved=False, cached=False,
    add_self_loops=True, normalize=True, bias=True)."""

    def __init__(self, in_channels: int, out_channels: int, improved: bool = False,
                 cached: bool = False, add_self_loops: bool = True, normalize: bool = True,
                 bias: bool = True, **kwargs):
        super().__init__()
        if improved or not add_self_loops or not normalize:
            raise NotImplementedError("tsg.GCNConv implements the configuration the reference uses: "
                                      "improved=False, add_self_loops=True, normalize=True")
        self.in_channels, self.out_channels = in_channels, out_channels
        self.weight = torch.nn.Parameter(torch.empty(in_channels, out_channels))
        self.bias = torch.nn.Parameter(torch.empty(out_channels)) if bias else None
        self.reset_parameters()

    def reset_parameters(self) -> None:
        _glorot_(self.weight)
        if self.bias is not None:
            torch.nn.init.zeros_(self.bias)

    def forward(self, x: torch.Tensor, edge_index, edge_weight: Optional[torch.Tensor] = None,
                relu: bool = False) -> torch.Tensor:
        if isinstance(edge_index, CSR):
            csr = edge_index
        elif edge_weight is not None:
            csr = ops.build_csr(EdgeList.from_edge_index(edge_index), x.size(0), edge_weight=edge_weight)
        else:
            csr = _GLOBAL_CSR_CACHE.get(edge_index, x.size(0))
        return ops.gcn_conv(x, csr, self.weight, self.bias, relu=relu)

    def __repr__(self):
        return f"{self.__class__.__name__}({self.in_channels}, {self.out_channels})"


class _ScoreLayerHolder(torch.nn.Module):
    """Keeps the reference's module path `poolK.score_layer.{weight,bias}` (Code/sag/layers.py:12)."""

    def __init__(self, in_channels: int):
        super().__init__()
        self.score_layer = GCNConv(in_channels, 1)


def host_level_ptrs(node_ptr: np.ndarray, ratio: float, levels: int = 3) -> np.ndarray:
    """Node offsets of every pooling level, computed on the host from the graph sizes exactly as
    PyG's topk does on the device: k = ceil(float32(ratio) * float32(n)).  int64 [levels+1, G+1]."""
    n = np.diff(node_ptr).astype(np.int64)
    out = np.zeros((levels + 1, n.shape[0] + 1), np.int64)
    out[0, 1:] = np.cumsum(n)
    for l in range(1, levels + 1):
        n = np.ceil(np.float32(ratio) * n.astype(np.float32)).astype(np.int64)
        out[l, 1:] = np.cumsum(n)
    return out


KEEP_ARENA = False        # tests: keep (shape, arena) of the last executor forward in LAST_ARENA
LAST_ARENA = None
_STATUS = {}              # device index -> persistent int32 word the verifying kernels (K1d, K13) OR their bits into
_STATUS_DIRTY = set()     # devices whose word may have been written since the last check


def _status_word(dev: torch.device) -> torch.Tensor:
    i = dev.index if dev.index is not None else torch.cuda.current_device()
    w = _STATUS.get(i)
    if w is None:
        w = _STATUS[i] = torch.zeros(1, dtype=torch.int32, device=dev)
    _STATUS_DIRTY.add(i)
    return w
SAG_FIELDS = {"status": (8, torch.int32), "perm": (0, torch.int64), "score": (1, torch.float32), "h": (2, torch.float32), "xg": (3, torch.float32),
              "rowptr": (4, torch.int32), "colidx": (5, torch.int32), "val": (6, torch.float32), "inv": (7, torch.int32)}


def sag_arena_view(shape, arena: torch.Tensor, level: int, field: str) -> torch.Tensor:
    """A saved tensor of the executor's forward, viewed in place inside the arena (tsg_sag_arena_locate): what
    SAGPool.forward returns besides x (Code/sag/layers.py:26: perm) and the level's CSR, for callers / parity tests."""
    from . import _lib
    code, dt = SAG_FIELDS[field]
    off, nb = ctypes.c_size_t(), ctypes.c_size_t()
    rc = _lib.lib.tsg_sag_arena_locate(ctypes.byref(shape), int(level), code, ctypes.byref(off), ctypes.byref(nb))
    if rc != 0:
        raise RuntimeError(f"tsg_sag_arena_locate failed: {_lib.last_error()}")
    return arena[off.value:off.value + nb.value].view(dt)


LABEL_RANGE = 8           # TSG_SAG_LABEL_RANGE (include/tsg.h)
EIGEN_OPERANDS = 16       # K0e tsg_pack_eigen_batch: the EigenPooling operands of a graph are not what it relies on


def check_fused_status(already_read: Optional[dict] = None) -> None:
    """Look at the status word the verifying kernels (K1d, K13, K0d / K0e, and the label checks of the supervised step, the
    classification forward and the stage-2 heads) OR-ed their bits into since the last call -- ONE device
    read per device, so callers do it where they synchronise anyway (loss read-back, end of a feeder loop, tests).  A non-zero word means a graph's
    edge list was not what those kernels require (endpoints in range, no self loops, sorted by (row, col), symmetric:
    the TUDataset / TU-loader form); its embedding was zeroed.  There is no silent fallback: this raises.
    `already_read` {device index: word}: words the caller copied back together with its own results (no second read)."""
    if not _STATUS_DIRTY:
        return
    bits = 0
    for i in list(_STATUS_DIRTY):
        bits |= int(already_read[i]) if already_read and i in already_read else int(_STATUS[i].item())
        _STATUS[i].zero_()
    _STATUS_DIRTY.clear()
    if bits & LABEL_RANGE:
        raise RuntimeError("tsg: a graph label lies outside [0, num_classes) (status bit 8, set by the supervised step, "
                           "the classification forward or a stage-2 head); it was clamped, so the loss and the accuracy "
                           "are invalid")
    if bits & EIGEN_OPERANDS:
        raise RuntimeError("tsg: a graph's EigenPooling operands are invalid (status bit 16, set by pack_eigen): a cluster "
                           "id outside [0, clusters of the graph), more clusters than max_nodes, or a coarsened "
                           "adjacency list that is out of range, unsorted, has a self loop or is not symmetric in "
                           "position and weight" + (f"; adjacency bits {bits & 7} are set too" if bits & 7 else "") +
                           ".  Build them with tsg.eigen_synth.operands_from_clusters.")
    if bits:
        names = [n for b, n in ((1, "edge endpoint out of range / self loop"), (2, "edge list not sorted by (row, col)"),
                                (4, "edge list not symmetric")) if bits & b]
        raise RuntimeError("tsg: a graph's edge list is not in the coalesced, symmetric form the caller promised (" +
                           "; ".join(names) + "); its results are invalid.  Coalesce the edge lists (TUDataset form), or "
                           "drop CompactBatch.coalesced and run with TSG_SAG_FUSED=0: the general kernels take any list.")


class _SagEncoderFn(torch.autograd.Function):
    """The three conv/pool/readout levels through the native executor (K10): two C-ABI calls per step
    instead of ~110.  Same kernels in the same order as the op-by-op path below."""

    @staticmethod
    def forward(ctx, x, row, col, ptrs, shape, *params):
        from . import _lib
        dev = x.device
        x = x.contiguous()
        params = [p.contiguous() for p in params]
        arena_bytes = _lib.lib.tsg_sag_arena_bytes(ctypes.byref(shape))
        if arena_bytes == 0:
            raise RuntimeError("tsg: bad SAG encoder shape")
        arena = torch.empty(arena_bytes, dtype=torch.uint8, device=dev)
        z = torch.empty(shape.num_graphs, 2 * shape.hidden, dtype=torch.float32, device=dev)
        parr = (ctypes.c_void_p * 12)(*[p.data_ptr() for p in params])
        _lib.call("tsg_sag_encoder_fwd", ctypes.byref(shape), _lib.ptr(x), _lib.ptr(row), _lib.ptr(col), _lib.ptr(ptrs),
                  parr, _lib.ptr(z), _lib.ptr(arena), arena_bytes, _lib.stream_ptr())
        ctx.shape, ctx.arena, ctx.arena_bytes = shape, arena, arena_bytes
        ctx.save_for_backward(x, ptrs, *params)
        if KEEP_ARENA:
            global LAST_ARENA
            LAST_ARENA = (shape, arena)
        return z

    @staticmethod
    def backward(ctx, dz):
        from . import _lib
        x, ptrs, *params = ctx.saved_tensors
        dz = dz.contiguous()
        grads = [torch.empty_like(p) for p in params]
        parr = (ctypes.c_void_p * 12)(*[p.data_ptr() for p in params])
        garr = (ctypes.c_void_p * 12)(*[g.data_ptr() for g in grads])
        _lib.call("tsg_sag_encoder_bwd", ctypes.byref(ctx.shape), _lib.ptr(x), _lib.ptr(ptrs), parr, _lib.ptr(dz), garr,
                  _lib.ptr(ctx.arena), ctx.arena_bytes, _lib.stream_ptr())
        ctx.arena = None
        return (None, None, None, None, None, *grads)


class _SagEncoderCompactFn(torch.autograd.Function):
    """K10 on the compact level-0 input (ops.CompactBatch): labels instead of the one-hot x, local int32 endpoints
    instead of the int64 edge_index.  Same arena, same kernels below level 0."""

    @staticmethod
    def forward(ctx, cb, ptrs, shape, *params):
        from . import _lib
        dev = cb.label.device
        params = [p.contiguous() for p in params]
        arena_bytes = _lib.lib.tsg_sag_arena_bytes(ctypes.byref(shape))
        if arena_bytes == 0:
            raise RuntimeError("tsg: bad SAG encoder shape")
        arena = torch.empty(arena_bytes, dtype=torch.uint8, device=dev)
        z = torch.empty(shape.num_graphs, 2 * shape.hidden, dtype=torch.float32, device=dev)
        parr = (ctypes.c_void_p * 12)(*[p.data_ptr() for p in params])
        _lib.call("tsg_sag_encoder_fwd_compact", ctypes.byref(shape), _lib.ptr(cb.label), _lib.ptr(cb.row), _lib.ptr(cb.col),
                  _lib.ptr(cb.edge_ptr), _lib.ptr(ptrs), parr, _lib.ptr(z), _lib.ptr(arena), arena_bytes, _lib.stream_ptr())
        ctx.shape, ctx.arena, ctx.arena_bytes, ctx.label = shape, arena, arena_bytes, cb.label
        ctx.save_for_backward(ptrs, *params)
        if KEEP_ARENA:
            global LAST_ARENA
            LAST_ARENA = (shape, arena)
        return z

    @staticmethod
    def backward(ctx, dz):
        from . import _lib
        ptrs, *params = ctx.saved_tensors
        dz = dz.contiguous()
        grads = [torch.empty_like(p) for p in params]
        parr = (ctypes.c_void_p * 12)(*[p.data_ptr() for p in params])
        garr = (ctypes.c_void_p * 12)(*[g.data_ptr() for g in grads])
        _lib.call("tsg_sag_encoder_bwd_compact", ctypes.byref(ctx.shape), _lib.ptr(ctx.label), _lib.ptr(ptrs), parr,
                  _lib.ptr(dz), garr, _lib.ptr(ctx.arena), ctx.arena_bytes, _lib.stream_ptr())
        ctx.arena = None
        return (None, None, None, *grads)


def _sag_embed_compact(cb, ptrs, shape, params):
    """Forward-only encoder (torch.no_grad(): the evaluation loops of the reference scripts embed every graph and never
    call backward): tsg_sag_encoder_embed_compact = the graph-resident kernels (K13) where the shape allows them."""
    from . import _lib
    dev = cb.label.device
    params = [p.contiguous() for p in params]
    arena_bytes = _lib.lib.tsg_sag_arena_bytes(ctypes.byref(shape))
    if arena_bytes == 0:
        raise RuntimeError("tsg: bad SAG encoder shape")
    arena = torch.empty(arena_bytes, dtype=torch.uint8, device=dev)
    z = torch.empty(shape.num_graphs, 2 * shape.hidden, dtype=torch.float32, device=dev)
    parr = (ctypes.c_void_p * 12)(*[p.data_ptr() for p in params])
    _lib.call("tsg_sag_encoder_embed_compact", ctypes.byref(shape), _lib.ptr(cb.label), _lib.ptr(cb.row), _lib.ptr(cb.col),
              _lib.ptr(cb.edge_ptr), _lib.ptr(ptrs), parr, _lib.ptr(z), _lib.ptr(arena), arena_bytes, _lib.stream_ptr())
    if KEEP_ARENA:
        global LAST_ARENA
        LAST_ARENA = (shape, arena)
    return z


class PackedSAGNet(torch.nn.Module):
    """Code/sag/network.py `Net` over a packed batch.  Three levels of
    GCNConv -> ReLU -> SAGPool(score GCNConv, top-k, gate, filter_adj) -> [gmp || gap],
    summed, then lin1/ReLU/dropout/lin2/ReLU/lin3/log_softmax."""

    accepts_compact = True       # forward(x=ops.CompactBatch, edge_index=None, node_ptr_host)

    def __init__(self, num_features: int, nhid: int, num_classes: int, pooling_ratio: float,
                 dropout_ratio: float):
        super().__init__()
        self.num_features, self.nhid, self.num_classes = num_features, nhid, num_classes
        self.pooling_ratio, self.dropout_ratio = pooling_ratio, dropout_ratio
        self.conv1 = GCNConv(num_features, nhid); self.pool1 = _ScoreLayerHolder(nhid)
        self.conv2 = GCNConv(nhid, nhid); self.pool2 = _ScoreLayerHolder(nhid)
        self.conv3 = GCNConv(nhid, nhid); self.pool3 = _ScoreLayerHolder(nhid)
        self.lin1 = torch.nn.Linear(nhid * 2, nhid)
        self.lin2 = torch.nn.Linear(nhid, nhid // 2)
        self.lin3 = torch.nn.Linear(nhid // 2, num_classes)

    def forward(self, x: torch.Tensor, edge_index, node_ptr_host: np.ndarray,
                return_aux: bool = False):
        """x [sum n, F] f32, edge_index int64 [2, sum E] (or an EdgeList), node_ptr_host int64 [G+1]
        on the HOST (graph sizes are known where the batch was packed, so every level's sizes are
        computed without a device round trip)."""
        compact = x if isinstance(x, ops.CompactBatch) else None
        dev = compact.label.device if compact is not None else x.device
        plan, ptrs = self._level_plan(node_ptr_host, dev)
        if compact is not None:
            # labels + local endpoints straight into the executor; anything it does not cover expands first (K0)
            z = self._encode_compact(compact, plan, ptrs) if (USE_EXECUTOR and not return_aux) else None
            if z is not None:
                return self.head(z)
            x, edge_index = compact.expand()
        edges = edge_index if isinstance(edge_index, EdgeList) else EdgeList.from_edge_index(edge_index)
        # K2 shared-memory tiles: runs of whole graphs per pooling level (block-diagonal => self-contained)
        tiles = ([torch.from_numpy(ops.make_tiles(plan[l])).pin_memory().to(dev, non_blocking=True)
                  for l in range(3)] if ops.USE_TILED_SPMM else [None] * 3)
        if USE_EXECUTOR and not return_aux and edges.count is None and x.dim() == 2:
            shape = self._sag_shape(plan, x.size(1), edges.cap)
            if shape is not None:
                params = self._encoder_params()
                z = _SagEncoderFn.apply(x, edges.row, edges.col, ptrs, shape, *params)
                return self.head(z)
        aux = {"perm": [], "edges": [], "score": []}
        outs = []
        for lvl, (conv, pool) in enumerate(((self.conv1, self.pool1), (self.conv2, self.pool2),
                                            (self.conv3, self.pool3))):
            n_l, k_l = int(plan[lvl, -1]), int(plan[lvl + 1, -1])
            if ops.USE_GRAPH_CSR and n_l > 0:
                csr = ops.build_csr_graphs(edges, ptrs[lvl], n_l, int(np.diff(plan[lvl]).max()))
            else:
                csr = ops.build_csr(edges, n_l)
            csr.tile_ptr = tiles[lvl]
            h = conv(x, csr, relu=True)                                   # network.py:34
            score = pool.score_layer(h, csr).view(-1)                     # layers.py:18
            perm = ops.topk(score, ptrs[lvl], ptrs[lvl + 1], k_l)         # layers.py:20
            edges, inv = ops.filter_adj(edges, perm, n_l)                 # layers.py:23
            x = ops.gate_gather(h, score, perm, inv)                      # layers.py:21
            outs.append(ops.readout(x, ptrs[lvl + 1]))                    # network.py:36
            if return_aux:
                aux["perm"].append(perm); aux["edges"].append(edges); aux["score"].append(score)
        z = self.head(outs[0] + outs[1] + outs[2])                        # network.py:46
        return (z, aux) if return_aux else z

    def _sag_shape(self, plan, in_feat, num_edges):
        from . import _lib
        shape = _lib.SagShape(plan.shape[1] - 1, in_feat, self.nhid, num_edges)
        for l in range(4):
            shape.n[l] = int(plan[l, -1])
        for l in range(3):
            shape.max_graph_nodes[l] = max(int(np.diff(plan[l]).max()), 1)
        ok = min(shape.n) > 0 and max(shape.max_graph_nodes) <= ops.GRAPH_CSR_MAX_NODES
        return shape if ok else None

    def _encoder_params(self):
        params = []
        for conv, pool in ((self.conv1, self.pool1), (self.conv2, self.pool2), (self.conv3, self.pool3)):
            params += [conv.weight, conv.bias, pool.score_layer.weight, pool.score_layer.bias]
        return params

    def _encode_compact(self, cb, plan, ptrs):
        from . import _lib
        if cb.num_labels != self.num_features:
            raise ValueError(f"tsg: batch has {cb.num_labels} node labels, conv1 expects {self.num_features} input columns")
        if _lib.lib.tsg_embed_bwd_weight_workspace_bytes(cb.num_labels, self.nhid) == 0:
            return None
        shape = self._sag_shape(plan, cb.num_labels, int(cb.row.shape[0]))
        if shape is None:
            return None
        shape.max_graph_edges = int(cb.max_graph_edges)
        shape.pooling_ratio = float(self.pooling_ratio)
        shape.flags = 1 if cb.coalesced else 0
        if cb.coalesced or cb.max_graph_edges > 0:      # K1d / K13 verify the edge lists on the device: persistent status word
            shape.status = _status_word(cb.label.device).data_ptr()
        if not torch.is_grad_enabled():
            return _sag_embed_compact(cb, ptrs, shape, [p.detach() for p in self._encoder_params()])
        return _SagEncoderCompactFn.apply(cb, ptrs, shape, *self._encoder_params())

    # ------------------------------------------------------------------------------------------------------------
    # K14: the whole training step (forward, MarginRankingLoss, backward) behind one C-ABI call
    # ------------------------------------------------------------------------------------------------------------
    def _step_params(self):
        return self._encoder_params() + [self.lin1.weight, self.lin1.bias, self.lin2.weight, self.lin2.bias,
                                         self.lin3.weight, self.lin3.bias]

    def _flat_grads(self):
        """One flat fp32 buffer [all 18 gradients | loss | weight]; every parameter's .grad is a VIEW into it, so the
        data-parallel all-reduce is one collective on one tensor with no gather / scatter copies around it."""
        params = self._step_params()
        fg, views = self.__dict__.get("_flat_grad"), self.__dict__.get("_grad_views")
        stale = fg is None or fg.device != params[0].device or any(p.grad is not v for p, v in zip(params, views))
        if stale:
            n = sum(p.numel() for p in params)
            fg = torch.zeros(n + 2, dtype=torch.float32, device=params[0].device)
            views, off = [], 0
            for p in params:
                v = fg[off:off + p.numel()].view_as(p); off += p.numel()
                p.grad = v
                views.append(v)
            self.__dict__["_flat_grad"], self.__dict__["_grad_views"] = fg, views
        return fg, views

    def _head_fits(self) -> bool:
        """The head's shape is one the native steps run (the workspace query is 0 otherwise): a pure host query, cached."""
        from . import _lib
        key = (self.nhid, self.num_classes)
        hit = self.__dict__.get("_head_fits_cache")
        if hit is None or hit[0] != key:
            shape = _lib.SagShape(1, self.num_features, self.nhid, 0)
            head = _lib.SagHead(self.num_classes, 1, 0.0, 0.0, 0.0, 0)
            hit = self.__dict__["_head_fits_cache"] = (
                key, _lib.lib.tsg_sag_triplet_step_workspace_bytes(ctypes.byref(shape), ctypes.byref(head)) != 0)
        return hit[1]

    def native_step_supported(self, cb, node_ptr_host=None) -> bool:
        """Can K14 take this batch?  (Compact input, even hidden width, a head the native steps run, label table within
        the kernels' range, float32 CUDA parameters, and -- when the offsets are given -- every graph within the executor's per-graph limits;
        otherwise the caller uses the autograd path, which handles anything.)"""
        from . import _lib
        if not (USE_EXECUTOR and USE_NATIVE_STEP and isinstance(cb, ops.CompactBatch)) or self.nhid % 2:
            return False
        if cb.num_labels != self.num_features or _lib.lib.tsg_embed_bwd_weight_workspace_bytes(cb.num_labels, self.nhid) == 0:
            return False
        if not self._head_fits():
            return False
        if node_ptr_host is not None:
            plan, _ = self._level_plan(node_ptr_host, cb.label.device)
            if self._sag_shape(plan, cb.num_labels, int(cb.row.shape[0])) is None:
                return False
        return all(p.is_cuda and p.dtype == torch.float32 and p.is_contiguous() for p in self._step_params())

    _WS_QUERY = {"triplet": "tsg_sag_triplet_step_workspace_bytes", "nll": "tsg_sag_nll_step_workspace_bytes",
                 "classify": "tsg_sag_classify_workspace_bytes"}

    def _native_setup(self, cb, node_ptr_host, num_triplets, margin, eps, dropout_mask, entry="triplet"):
        from . import _lib
        dev = cb.label.device
        plan, ptrs = self._level_plan(node_ptr_host, dev)
        shape = self._sag_shape(plan, cb.num_labels, int(cb.row.shape[0]))
        if shape is None:
            raise RuntimeError("tsg: batch shape outside the executor's range (empty level or a graph beyond the per-graph CSR builder)")
        shape.max_graph_edges = int(cb.max_graph_edges)
        shape.pooling_ratio = float(self.pooling_ratio)
        shape.flags = 1 if cb.coalesced else 0
        if cb.coalesced or entry != "triplet":      # the label checks report through the persistent word as well
            shape.status = _status_word(dev).data_ptr()
        if entry == "classify":                     # evaluation: dropout off, and no draw from the step counter
            count, p_drop = 0, 0.0
        else:
            count = self.__dict__["_native_steps"] = self.__dict__.get("_native_steps", 0) + 1
            p_drop = float(self.dropout_ratio) if (self.training and dropout_mask is None) else 0.0
        head = _lib.SagHead(self.num_classes, max(int(num_triplets), 1), float(margin), float(eps), p_drop,
                            (torch.initial_seed() * 0x9E3779B1 + count) & 0xFFFFFFFFFFFFFFFF)
        arena_bytes = _lib.lib.tsg_sag_arena_bytes(ctypes.byref(shape))
        ws_bytes = getattr(_lib.lib, self._WS_QUERY[entry])(ctypes.byref(shape), ctypes.byref(head))
        if arena_bytes == 0 or ws_bytes == 0:
            raise RuntimeError("tsg: bad shape for the native training step")
        arena = torch.empty(arena_bytes, dtype=torch.uint8, device=dev)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        params = self._step_params()
        parr = (ctypes.c_void_p * 18)(*[p.data_ptr() for p in params])
        return shape, head, ptrs, arena, arena_bytes, ws, ws_bytes, parr

    def native_step(self, cb, node_ptr_host, triplets: torch.Tensor, margin: float = 1.5, eps: float = 1e-6,
                    dropout_mask: Optional[torch.Tensor] = None, return_emb: bool = False):
        """Forward + triplet margin loss + backward of the whole model on a CompactBatch through
        tsg_sag_triplet_step_compact.  Returns the loss (device scalar, a view into the flat gradient buffer) and leaves
        every parameter's gradient in .grad (written, not accumulated).  Dropout follows self.training; `dropout_mask`
        [G, nhid] injects the keep multipliers (parity tests)."""
        from . import _lib
        dev = cb.label.device
        shape, head, ptrs, arena, arena_bytes, ws, ws_bytes, parr = self._native_setup(
            cb, node_ptr_host, triplets.shape[0], margin, eps, dropout_mask)
        flat, views = self._flat_grads()
        emb = torch.empty(shape.num_graphs, self.num_classes, dtype=torch.float32, device=dev) if return_emb else None
        garr = (ctypes.c_void_p * 18)(*[v.data_ptr() for v in views])
        loss = flat[-2:-1]
        _lib.call("tsg_sag_triplet_step_compact", ctypes.byref(shape), ctypes.byref(head), _lib.ptr(cb.label), _lib.ptr(cb.row),
                  _lib.ptr(cb.col), _lib.ptr(cb.edge_ptr), _lib.ptr(ptrs), parr, _lib.ptr(triplets.contiguous()),
                  _lib.ptr(dropout_mask.contiguous()) if dropout_mask is not None else None, garr, loss.data_ptr(),
                  _lib.ptr(emb), _lib.ptr(arena), arena_bytes, _lib.ptr(ws), ws_bytes, _lib.stream_ptr())
        if KEEP_ARENA:
            global LAST_ARENA
            LAST_ARENA = (shape, arena)
        return (loss.view(()), emb) if return_emb else loss.view(())

    def native_nll_step(self, cb, node_ptr_host, y: torch.Tensor, dropout_mask: Optional[torch.Tensor] = None,
                        return_emb: bool = False):
        """The supervised step of Code/sag/train.py:194 -- forward, F.nll_loss(out, y) (mean over the batch's graphs) and
        backward -- through tsg_sag_nll_step_compact.  `y` int64 [G] graph labels on the device.  Same contract as
        native_step: returns the loss (device scalar, a view into the flat gradient buffer) and WRITES every parameter's
        .grad; dropout follows self.training, `dropout_mask` [G, nhid] injects the keep multipliers.  A label outside
        [0, num_classes) raises at the next check_fused_status()."""
        from . import _lib
        dev = cb.label.device
        G = int(np.asarray(node_ptr_host).shape[0]) - 1
        if tuple(y.shape) != (G,):
            raise ValueError(f"tsg: y has shape {tuple(y.shape)}, the batch has {G} graphs")
        shape, head, ptrs, arena, arena_bytes, ws, ws_bytes, parr = self._native_setup(
            cb, node_ptr_host, 1, 0.0, 0.0, dropout_mask, entry="nll")
        flat, views = self._flat_grads()
        emb = torch.empty(G, self.num_classes, dtype=torch.float32, device=dev) if return_emb else None
        garr = (ctypes.c_void_p * 18)(*[v.data_ptr() for v in views])
        loss = flat[-2:-1]
        _lib.call("tsg_sag_nll_step_compact", ctypes.byref(shape), ctypes.byref(head), _lib.ptr(cb.label), _lib.ptr(cb.row),
                  _lib.ptr(cb.col), _lib.ptr(cb.edge_ptr), _lib.ptr(ptrs), parr, _lib.ptr(y.to(torch.int64).contiguous()),
                  _lib.ptr(dropout_mask.contiguous()) if dropout_mask is not None else None, garr, loss.data_ptr(),
                  _lib.ptr(emb), _lib.ptr(arena), arena_bytes, _lib.ptr(ws), ws_bytes, _lib.stream_ptr())
        if KEEP_ARENA:
            global LAST_ARENA
            LAST_ARENA = (shape, arena)
        return (loss.view(()), emb) if return_emb else loss.view(())

    def native_classify(self, cb, node_ptr_host, y: Optional[torch.Tensor] = None):
        """`test()` of Code/sag/train.py:19-29 on one packed batch through tsg_sag_classify_compact: the model.eval()
        forward (dropout off whatever self.training says), pred = out.max(dim=1)[1] and, with labels `y` (int64 [G] on
        the device), the batch's correct count and summed NLL, reduced on the device.  Returns
        (pred int64 [G], log-probabilities [G, C], correct int64 [1] or None, nll_sum float32 [1] or None)."""
        from . import _lib
        dev = cb.label.device
        G = int(np.asarray(node_ptr_host).shape[0]) - 1
        if y is not None and tuple(y.shape) != (G,):
            raise ValueError(f"tsg: y has shape {tuple(y.shape)}, the batch has {G} graphs")
        shape, head, ptrs, arena, arena_bytes, ws, ws_bytes, parr = self._native_setup(
            cb, node_ptr_host, 1, 0.0, 0.0, None, entry="classify")
        pred = torch.empty(G, dtype=torch.int64, device=dev)
        logp = torch.empty(G, self.num_classes, dtype=torch.float32, device=dev)
        correct = nll_sum = None
        if y is not None:
            y = y.to(torch.int64).contiguous()
            correct = torch.empty(1, dtype=torch.int64, device=dev)
            nll_sum = torch.empty(1, dtype=torch.float32, device=dev)
        _lib.call("tsg_sag_classify_compact", ctypes.byref(shape), ctypes.byref(head), _lib.ptr(cb.label), _lib.ptr(cb.row),
                  _lib.ptr(cb.col), _lib.ptr(cb.edge_ptr), _lib.ptr(ptrs), parr, _lib.ptr(y), _lib.ptr(pred), _lib.ptr(logp),
                  _lib.ptr(correct), _lib.ptr(nll_sum), _lib.ptr(arena), arena_bytes, _lib.ptr(ws), ws_bytes,
                  _lib.stream_ptr())
        if KEEP_ARENA:
            global LAST_ARENA
            LAST_ARENA = (shape, arena)
        return pred, logp, correct, nll_sum

    def native_forward(self, cb, node_ptr_host, dropout_mask: Optional[torch.Tensor] = None):
        """First half of the native step: embeddings [G, C] (no autograd graph) + the context native_backward needs."""
        from . import _lib
        dev = cb.label.device
        shape, head, ptrs, arena, arena_bytes, ws, ws_bytes, parr = self._native_setup(cb, node_ptr_host, 1, 0.0, 1e-6, dropout_mask)
        emb = torch.empty(shape.num_graphs, self.num_classes, dtype=torch.float32, device=dev)
        _lib.call("tsg_sag_step_fwd_compact", ctypes.byref(shape), ctypes.byref(head), _lib.ptr(cb.label), _lib.ptr(cb.row),
                  _lib.ptr(cb.col), _lib.ptr(cb.edge_ptr), _lib.ptr(ptrs), parr,
                  _lib.ptr(dropout_mask.contiguous()) if dropout_mask is not None else None, _lib.ptr(emb), _lib.ptr(arena),
                  arena_bytes, _lib.ptr(ws), ws_bytes, _lib.stream_ptr())
        return emb, (shape, head, ptrs, arena, arena_bytes, ws, ws_bytes, parr, cb.label, emb)

    def native_backward(self, ctx, demb: torch.Tensor) -> None:
        """Second half: d(loss)/d(emb) [G, C] -> every parameter's .grad (views of the flat buffer, written)."""
        from . import _lib
        shape, head, ptrs, arena, arena_bytes, ws, ws_bytes, parr, label, emb = ctx
        flat, views = self._flat_grads()
        garr = (ctypes.c_void_p * 18)(*[v.data_ptr() for v in views])
        _lib.call("tsg_sag_step_bwd_compact", ctypes.byref(shape), ctypes.byref(head), _lib.ptr(label), _lib.ptr(ptrs), parr,
                  _lib.ptr(emb), _lib.ptr(demb.contiguous()), garr, _lib.ptr(arena), arena_bytes, _lib.ptr(ws), ws_bytes,
                  _lib.stream_ptr())

    def _level_plan(self, node_ptr_host, dev):
        """(host plan int64 [4, G+1], the same on the device).  Batches that come round again (an epoch over a fixed
        set of packed batches) reuse their device copy.  Keyed on the CONTENT of the offsets (hash of the bytes, then an
        exact comparison with the stored copy): object identity is not a key -- feeders create a short-lived array per
        step and CPython reuses ids."""
        arr = np.ascontiguousarray(np.asarray(node_ptr_host, dtype=np.int64))
        key = (hash(arr.tobytes()), arr.shape[0], str(dev), self.pooling_ratio)
        cache = self.__dict__.setdefault("_plan_cache", {})
        hit = cache.get(key)
        if hit is not None and np.array_equal(hit[0][0], arr):
            return hit
        plan = host_level_ptrs(arr, self.pooling_ratio)
        ptrs = torch.from_numpy(plan).pin_memory().to(dev, non_blocking=True)
        if len(cache) >= 16:
            cache.pop(next(iter(cache)))
        cache[key] = (plan, ptrs)
        return plan, ptrs

    def head(self, z: torch.Tensor) -> torch.Tensor:
        """network.py:48-52: lin1 / ReLU / dropout / lin2 / ReLU / lin3 / log_softmax."""
        # the three Linear layers run on the tall-skinny K3 kernels ([G, 64] operands: cuBLAS picks split-K SIMT
        # GEMMs that cost 250 us per step here); parameters stay nn.Linear so the state_dict keys are the reference's
        lin = lambda layer, t: ops.linear(t, layer.weight.t().contiguous(), layer.bias)
        z = F.relu(lin(self.lin1, z))
        z = F.dropout(z, p=self.dropout_ratio, training=self.training)
        z = F.relu(lin(self.lin2, z))
        return F.log_softmax(lin(self.lin3, z), dim=-1)


class PackedTripletNet(torch.nn.Module):
    """Code/sag/tripletnet.py over packed batches: ONE forward over all graphs of the step, then
    K9 on index triplets.  Returns (loss, dist_p, dist_n, embeddings)."""

    def __init__(self, model: torch.nn.Module, margin: float = 1.5):
        super().__init__()
        self.model, self.margin = model, margin

    def forward(self, x, edge_index, node_ptr_host, triplets: torch.Tensor):
        emb = self.model(x, edge_index, node_ptr_host)
        loss, dp, dn = ops.triplet_loss(emb, triplets, self.margin)
        return loss, dp, dn, emb
