"""Host-side operator layer over libtsg.so: torch.autograd.Function wrappers whose forward and
backward are hand-written sm_100a kernels reached through the C ABI (include/tsg.h).

PyTorch is plumbing here (device memory, streams, autograd graph bookkeeping, the dense
Linear/GEMM pieces); every message-passing / pooling / readout / triplet kernel is ours.
There is no CPU path: CPU tensors raise.
"""
from __future__ import annotations

import ctypes
import os
from dataclasses import dataclass
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import call, ptr, stream_ptr, workspace, lib

CSR_GCN, CSR_RAW = 0, 1
USE_TILED_SPMM = False   # shared-memory-staged K2 (tsg_spmm_tiled); measured slower than the L1-blocked kernel
USE_TCGEN05 = True      # tcgen05 (3xTF32, TMEM) kernel for the K7 contraction / GEMM-shaped dW; False = fp32 SIMT kernels
SPMM_RELU = 1
SPMM_EXACT = 2
SPMM_EXACT_DEFAULT = False   # True: separately rounded products everywhere (6 % slower K2)
READOUT_MAX, READOUT_MEAN, READOUT_SUM = 1, 2, 4
LIN_NORMALIZE, LIN_RELU, LIN_NODEBN, LIN_SOFTMAX = 1, 2, 4, 8


# --------------------------------------------------------------------------------------------
# containers
# --------------------------------------------------------------------------------------------
@dataclass
class EdgeList:
    """COO edge list; `count` (device int64 scalar) overrides `cap` when the number of valid
    edges is data dependent (after filter_adj) so no host sync is needed."""
    row: torch.Tensor
    col: torch.Tensor
    cap: int
    count: Optional[torch.Tensor] = None

    @staticmethod
    def from_edge_index(edge_index: torch.Tensor) -> "EdgeList":
        if edge_index.dtype != torch.int64 or edge_index.dim() != 2 or edge_index.size(0) != 2:
            raise RuntimeError("edge_index must be int64 [2, E]")
        ei = edge_index.contiguous()
        return EdgeList(ei[0], ei[1], int(ei.size(1)))

    def edge_index(self) -> torch.Tensor:
        """Exact-shape PyG edge_index [2, E'] (synchronises once if the count is on the device)."""
        e = self.cap if self.count is None else int(self.count.item())
        return torch.stack([self.row[:e], self.col[:e]])


@dataclass
class CompactBatch:
    """A packed batch as the dataset stores it (SURVEY 8f n1 feeder): one categorical label per node -- the
    reference's one-hot `data.x` (Code/sag/train.py:34; load_data.py:74-87) is onehot(label) -- and graph-LOCAL
    int32 edge endpoints.  All tensors live on the device; `node_ptr` / `edge_ptr` are int64 [G+1] offsets.
    PackedSAGNet consumes it directly (K10 compact entries: no fp32 one-hot matrix, no int64 edge_index);
    `expand()` materialises the PyG wire format with K0 for every other consumer."""
    label: torch.Tensor
    row: torch.Tensor
    col: torch.Tensor
    node_ptr: torch.Tensor
    edge_ptr: torch.Tensor
    num_labels: int
    max_graph_edges: int = 0      # host-side max of diff(edge_ptr) (0 = unknown: the graph-resident kernels are not used)
    coalesced: bool = False       # promise: every graph's list is sorted by (row, col), loop free and symmetric (the
                                  # TUDataset / TU loader / tsg.synth form) -> one CSR orientation per level (K1d).  Verified
                                  # on the device; a violation raises at the next tsg.nn.check_fused_status()

    def expand(self) -> Tuple[torch.Tensor, torch.Tensor]:
        """(x [N, num_labels] fp32 one-hot, edge_index [2, E] int64 with batch-global ids) via tsg_pack_batch."""
        dev = self.label.device
        G, N, E = self.node_ptr.shape[0] - 1, int(self.label.shape[0]), int(self.row.shape[0])
        ids = torch.arange(G, dtype=torch.int64, device=dev)
        x = torch.empty(N, self.num_labels, dtype=torch.float32, device=dev)
        ei = torch.empty(2, E, dtype=torch.int64, device=dev)
        call("tsg_pack_batch", ptr(ids), ptr(self.node_ptr), ptr(self.edge_ptr), G, ptr(self.node_ptr), ptr(self.edge_ptr),
             ptr(self.row), ptr(self.col), ptr(self.label), None, self.num_labels, ptr(x), ptr(ei[0]), ptr(ei[1]), stream_ptr())
        return x, ei


@dataclass
class CSR:
    rowptr: torch.Tensor
    colidx: torch.Tensor
    val: torch.Tensor
    eid: Optional[torch.Tensor]
    t_rowptr: Optional[torch.Tensor]
    t_colidx: Optional[torch.Tensor]
    t_val: Optional[torch.Tensor]
    t_eid: Optional[torch.Tensor]
    num_nodes: int
    tile_ptr: Optional[torch.Tensor] = None     # int64 [T+1]: self-contained row runs (whole graphs)
    tma_ok: bool = False                        # arrays have the 16-byte slack the TMA-staged K2 needs


def build_csr(edges: EdgeList, num_nodes: int, mode: int = CSR_GCN, transposed: bool = True,
              edge_weight: Optional[torch.Tensor] = None, want_eid: bool = False) -> CSR:
    """K1: stable counting sort of the (self-loop augmented) COO list into dst-major (+ src-major)
    CSR with GCN normalisation.  Reference: PyG gcn_norm via Code/sag/network.py:34."""
    dev = edges.row.device
    E, N = edges.cap, int(num_nodes)
    cap = E + (N if mode == CSR_GCN else 0)
    i32 = dict(dtype=torch.int32, device=dev)
    rowptr = torch.empty(N + 1, **i32)
    colidx = torch.empty(cap, **i32)
    val = torch.empty(cap, dtype=torch.float32, device=dev)
    eid = torch.empty(cap, **i32) if want_eid else None
    if transposed:
        t_rowptr = torch.empty(N + 1, **i32)
        t_colidx = torch.empty(cap, **i32)
        t_val = torch.empty(cap, dtype=torch.float32, device=dev)
        t_eid = torch.empty(cap, **i32) if want_eid else None
    else:
        t_rowptr = t_colidx = t_val = t_eid = None
    wsb = lib.tsg_csr_build_workspace_bytes(E, N)
    ws = workspace(wsb, dev)
    call("tsg_csr_build", ptr(edges.row), ptr(edges.col), ptr(edge_weight), E, ptr(edges.count), N,
         mode, ptr(rowptr), ptr(colidx), ptr(val), ptr(eid), ptr(t_rowptr), ptr(t_colidx),
         ptr(t_val), ptr(t_eid), ptr(ws), wsb, stream_ptr())
    return CSR(rowptr, colidx, val, eid, t_rowptr, t_colidx, t_val, t_eid, N)


USE_GRAPH_CSR = os.environ.get("TSG_GRAPH_CSR", "1") != "0"     # K1b (one CTA per graph, shared memory) for packed batches; False = generic K1
GRAPH_CSR_MAX_NODES = 6000   # shared-memory budget of K1b (7 ints per node)


def build_csr_graphs(edges: EdgeList, node_ptr: torch.Tensor, num_nodes: int, max_graph_nodes: int,
                     transposed: bool = True, want_eid: bool = False) -> CSR:
    """K1b: same result as build_csr(mode=CSR_GCN) for a packed batch whose edges are grouped by graph
    (PyG Batch layout; preserved by filter_adj).  node_ptr int64 [G+1] on the device; max_graph_nodes is
    the host-side bound over the batch.  Falls back to K1 when a graph exceeds the smem budget."""
    if max_graph_nodes > GRAPH_CSR_MAX_NODES:
        return build_csr(edges, num_nodes, CSR_GCN, transposed, None, want_eid)
    dev = edges.row.device
    E, N, G = edges.cap, int(num_nodes), node_ptr.numel() - 1
    cap = E + N
    i32 = dict(dtype=torch.int32, device=dev)
    # 16 bytes of slack behind every array: the TMA-staged K2 rounds its bulk copies up to 16 bytes
    rowptr = torch.empty(N + 1 + 4, **i32)[:N + 1]
    colidx = torch.empty(cap + 4, **i32)[:cap]
    val = torch.empty(cap + 4, dtype=torch.float32, device=dev)[:cap]
    eid = torch.empty(cap, **i32) if want_eid else None
    if transposed:
        t_rowptr = torch.empty(N + 1 + 4, **i32)[:N + 1]
        t_colidx = torch.empty(cap + 4, **i32)[:cap]
        t_val = torch.empty(cap + 4, dtype=torch.float32, device=dev)[:cap]
        t_eid = torch.empty(cap, **i32) if want_eid else None
    else:
        t_rowptr = t_colidx = t_val = t_eid = None
    eptr = torch.empty(G + 1, dtype=torch.int64, device=dev)
    call("tsg_edge_ptr", ptr(edges.row), E, ptr(edges.count), ptr(node_ptr), G, ptr(eptr), stream_ptr())
    wsb = lib.tsg_csr_build_graphs_workspace_bytes(G, E)
    ws = workspace(wsb, dev)
    call("tsg_csr_build_graphs", ptr(edges.row), ptr(edges.col), ptr(eptr), ptr(node_ptr), G, N, E,
         int(max_graph_nodes), ptr(rowptr), ptr(colidx), ptr(val), ptr(eid), ptr(t_rowptr), ptr(t_colidx),
         ptr(t_val), ptr(t_eid), ptr(ws), wsb, stream_ptr())
    csr = CSR(rowptr, colidx, val, eid, t_rowptr, t_colidx, t_val, t_eid, N)
    csr.tile_ptr = node_ptr            # graph boundaries = self-contained tiles (K1b traps on a leaving edge)
    csr.tma_ok = True                  # arrays carry the 16-byte slack tsg_spmm_tma needs
    return csr


def build_csr_graphs_local(cb: "CompactBatch", num_nodes: int, max_graph_nodes: int) -> CSR:
    """K1b on a CompactBatch: graph-local int32 endpoints + per-graph edge offsets; same CSR (both orientations,
    GCN normalisation) as build_csr_graphs on the expanded batch."""
    if max_graph_nodes > GRAPH_CSR_MAX_NODES:
        raise RuntimeError(f"tsg: a graph of {max_graph_nodes} nodes exceeds the per-graph CSR builder "
                           f"({GRAPH_CSR_MAX_NODES}); expand() the batch and use build_csr")
    dev = cb.label.device
    E, N, G = int(cb.row.shape[0]), int(num_nodes), cb.node_ptr.numel() - 1
    cap = E + N
    i32 = dict(dtype=torch.int32, device=dev)
    arrs = [torch.empty(N + 1 + 4, **i32)[:N + 1], torch.empty(cap + 4, **i32)[:cap],
            torch.empty(cap + 4, dtype=torch.float32, device=dev)[:cap]]
    arrs += [torch.empty(N + 1 + 4, **i32)[:N + 1], torch.empty(cap + 4, **i32)[:cap],
             torch.empty(cap + 4, dtype=torch.float32, device=dev)[:cap]]
    wsb = lib.tsg_csr_build_graphs_workspace_bytes(G, E)
    ws = workspace(wsb, dev)
    call("tsg_csr_build_graphs_local", ptr(cb.row), ptr(cb.col), ptr(cb.edge_ptr), ptr(cb.node_ptr), G, N, E,
         int(max_graph_nodes), ptr(arrs[0]), ptr(arrs[1]), ptr(arrs[2]), None, ptr(arrs[3]), ptr(arrs[4]),
         ptr(arrs[5]), None, ptr(ws), wsb, stream_ptr())
    csr = CSR(arrs[0], arrs[1], arrs[2], None, arrs[3], arrs[4], arrs[5], None, N)
    csr.tile_ptr = cb.node_ptr
    csr.tma_ok = True
    return csr


def embed_fwd(weight: torch.Tensor, label: torch.Tensor) -> torch.Tensor:
    """K3c: onehot(label) @ weight without the one-hot matrix.  weight [K, M] f32, label int32 [N]."""
    weight = weight.contiguous()
    out = torch.empty(label.numel(), weight.size(1), dtype=torch.float32, device=weight.device)
    call("tsg_embed_fwd", ptr(weight), ptr(label), ptr(out), label.numel(), weight.size(0), weight.size(1), stream_ptr())
    return out


def embed_bwd_weight(label: torch.Tensor, dy: torch.Tensor, num_labels: int) -> torch.Tensor:
    """K3c: onehot(label)^T @ dy as a fixed-order segment sum.  dy [N, M] f32 -> [num_labels, M]."""
    dy = dy.contiguous()
    m = dy.size(1)
    wsb = lib.tsg_embed_bwd_weight_workspace_bytes(num_labels, m)
    if wsb == 0:
        raise RuntimeError(f"tsg: a {num_labels} x {m} label table does not fit shared memory")
    ws = workspace(wsb, dy.device)
    dw = torch.empty(num_labels, m, dtype=torch.float32, device=dy.device)
    call("tsg_embed_bwd_weight", ptr(label), ptr(dy), ptr(dw), label.numel(), num_labels, m, ptr(ws), wsb, stream_ptr())
    return dw


def spmm_raw(rowptr, colidx, val, H: torch.Tensor, bias=None, relu: bool = False,
             tile_ptr: Optional[torch.Tensor] = None, exact: Optional[bool] = None, tma: bool = False) -> torch.Tensor:
    """exact=True rounds every product before the add (bit-identical to index_add_ in COO order);
    the default (SPMM_EXACT_DEFAULT = False) fuses it (FFMA): same order, <= 1 ulp per term."""
    n = rowptr.numel() - 1
    H = H.contiguous()
    Y = torch.empty(n, H.size(1), dtype=torch.float32, device=H.device)
    flags = (SPMM_RELU if relu else 0) | (SPMM_EXACT if (SPMM_EXACT_DEFAULT if exact is None else exact) else 0)
    if tma and tile_ptr is not None and H.size(1) % 4 == 0 and H.size(1) <= 32:
        status = torch.zeros(1, dtype=torch.int32, device=H.device)
        call("tsg_spmm_tma", ptr(rowptr), ptr(colidx), ptr(val), ptr(H), ptr(bias), ptr(Y), ptr(tile_ptr),
             tile_ptr.numel() - 1, n, H.size(1), flags, ptr(status), stream_ptr())
        return Y
    if USE_TILED_SPMM and tile_ptr is not None and H.size(1) % 4 == 0:
        call("tsg_spmm_tiled", ptr(rowptr), ptr(colidx), ptr(val), ptr(H), ptr(bias), ptr(Y), ptr(tile_ptr),
             tile_ptr.numel() - 1, n, H.size(1), flags, stream_ptr())
    else:
        call("tsg_spmm", ptr(rowptr), ptr(colidx), ptr(val), ptr(H), ptr(bias), ptr(Y), n, H.size(1),
             flags, stream_ptr())
    return Y


def make_tiles(node_ptr_host, max_rows: int = 512):
    """Greedy host-side tiling of a packed level: consecutive whole graphs per tile while the tile stays
    <= max_rows rows (a larger graph is its own tile and takes the kernel's global-gather path).
    Returns int64 numpy offsets [T+1]."""
    import numpy as np
    ptr_ = np.asarray(node_ptr_host, dtype=np.int64)
    out = [0]
    start = 0
    for g in range(1, ptr_.shape[0]):
        if ptr_[g] - start > max_rows and ptr_[g - 1] > start:
            out.append(int(ptr_[g - 1])); start = int(ptr_[g - 1])
    if ptr_[-1] > out[-1] or len(out) == 1:
        out.append(int(ptr_[-1]))
    return np.asarray(out, dtype=np.int64)


def relu_bwd_colsum(dY: torch.Tensor, Y: Optional[torch.Tensor], want_masked: bool):
    """dYm = dY * (Y > 0) and dbias = column sums of dYm in one pass (deterministic)."""
    dY = dY.contiguous()
    n, f = dY.shape
    dYm = torch.empty_like(dY) if want_masked else None
    db = torch.empty(f, dtype=torch.float32, device=dY.device)
    wsb = lib.tsg_colsum_workspace_bytes(n, f)
    ws = workspace(wsb, dY.device)
    call("tsg_relu_bwd_colsum", ptr(dY), ptr(Y), ptr(dYm), ptr(db), n, f, ptr(ws), wsb, stream_ptr())
    return dYm, db


class _SpMM(torch.autograd.Function):
    """Y = A_hat H (+ bias) (ReLU);  dH = A_hat^T dY' via the src-major CSR (K2 both ways)."""

    @staticmethod
    def forward(ctx, H, bias, csr: CSR, relu: bool):
        Y = spmm_raw(csr.rowptr, csr.colidx, csr.val, H, bias, relu, csr.tile_ptr)
        ctx.csr, ctx.relu, ctx.has_bias = csr, relu, bias is not None
        ctx.save_for_backward(Y if relu else None)
        return Y

    @staticmethod
    def backward(ctx, dY):
        (Y,) = ctx.saved_tensors
        csr = ctx.csr
        if csr.t_rowptr is None:
            raise RuntimeError("tsg: CSR was built without the transposed orientation")
        dY = dY.contiguous()
        db = None
        if ctx.relu or ctx.has_bias:
            dYm, db = relu_bwd_colsum(dY, Y, want_masked=ctx.relu)
            if ctx.relu:
                dY = dYm
            if not ctx.has_bias:
                db = None
        dH = (spmm_raw(csr.t_rowptr, csr.t_colidx, csr.t_val, dY, tile_ptr=csr.tile_ptr)
              if ctx.needs_input_grad[0] else None)
        return dH, db, None, None


def spmm(csr: CSR, H: torch.Tensor, bias: Optional[torch.Tensor] = None, relu: bool = False):
    return _SpMM.apply(H, bias, csr, relu)


# --------------------------------------------------------------------------------------------
# K3 row-local dense products
# --------------------------------------------------------------------------------------------
def linear_raw(x: torch.Tensor, w: torch.Tensor, bias=None, transposed: bool = False, flags: int = 0):
    x = x.contiguous(); w = w.contiguous()
    n, k = x.shape
    m = w.size(0) if transposed else w.size(1)
    if (w.size(1) if transposed else w.size(0)) != k:
        raise RuntimeError(f"tsg.linear: shape mismatch x{tuple(x.shape)} w{tuple(w.shape)} T={transposed}")
    y = torch.empty(n, m, dtype=torch.float32, device=x.device)
    call("tsg_linear_fwd", ptr(x), ptr(w), ptr(bias), ptr(y), n, k, m, int(transposed), flags, stream_ptr())
    return y


DW_TC_MIN_WORK = 64 * 64        # K*M at which dW = X^T dY moves from the tall-skinny SIMT kernel to tcgen05
DW_TC_SEG_ROWS = 512            # tcgen05 accumulates fp32 with truncation: the error grows linearly with the rows per
                                # accumulator (measured 1.7e-6 @256, 7e-6 @1024, 2.8e-5 @4096), so segments stay short


def _linear_bwd_weight_tc(x: torch.Tensor, dy: torch.Tensor) -> torch.Tensor:
    """dW = X^T dY for GEMM-shaped K x M (DiffPool's Linear(164 -> 100) on ~10^6 rows) on the K7 tcgen05
    contraction: rows are cut into fixed pseudo-segments of DW_TC_SEG_ROWS, every segment's partial K x M product is
    one CTA's TMEM accumulator (3xTF32), partials are summed by one fixed-shape reduction (deterministic)."""
    n, k = x.shape; m = dy.size(1)
    segs = (n + DW_TC_SEG_ROWS - 1) // DW_TC_SEG_ROWS
    ptr_ = torch.arange(segs + 1, device=x.device, dtype=torch.int64) * DW_TC_SEG_ROWS
    ptr_[-1] = n
    out = torch.empty(k, m, dtype=torch.float32, device=x.device)
    for m0 in range(0, m, 256):
        dyc = dy if (m0 == 0 and m <= 256) else dy[:, m0:m0 + 256].contiguous()
        for k0 in range(0, k, 128):
            xc = x if (k0 == 0 and k <= 128) else x[:, k0:k0 + 128].contiguous()
            part = seg_contract_raw(xc, dyc, ptr_, tensor_cores=True)            # [segs, kx, my]
            out[k0:k0 + xc.size(1), m0:m0 + dyc.size(1)] = part.sum(dim=0)
    return out


def linear_bwd_weight(x: torch.Tensor, dy: torch.Tensor, want_bias: bool):
    x = x.contiguous(); dy = dy.contiguous()
    n, k = x.shape; m = dy.size(1)
    if USE_TCGEN05 and k * m >= DW_TC_MIN_WORK and n >= 16384 and k % 4 == 0 and m % 4 == 0:
        dw = _linear_bwd_weight_tc(x, dy)
        db = relu_bwd_colsum(dy, None, want_masked=False)[1] if want_bias else None
        return dw, db
    dw = torch.empty(k, m, dtype=torch.float32, device=x.device)
    db = torch.empty(m, dtype=torch.float32, device=x.device) if want_bias else None
    wsb = lib.tsg_linear_bwd_weight_workspace_bytes(k, m)
    ws = workspace(wsb, x.device)
    call("tsg_linear_bwd_weight", ptr(x), ptr(dy), ptr(dw), ptr(db), n, k, m, ptr(ws), wsb, stream_ptr())
    return dw, db


LINEAR_TC = os.environ.get("TSG_LINEAR_NOTC", "0") != "1"


def _linear_tc_ok(n: int, kin: int, m: int) -> bool:
    return n >= 16384 and kin % 4 == 0 and m % 4 == 0 and 32 <= m <= 256 and kin >= 32


def linear_tc_raw(x, w, bias, transposed: bool, softmax: bool):
    """tsg_linear_tc: y = x @ w (w [Kin, M]; transposed: w [M, Kin] used as w^T) on tcgen05, optional softmax(y + bias)."""
    x, w = x.contiguous(), w.contiguous()
    m = w.size(0) if transposed else w.size(1)
    y = torch.empty(x.size(0), m, dtype=torch.float32, device=x.device)
    status = torch.zeros(1, dtype=torch.int32, device=x.device)
    call("tsg_linear_tc", ptr(x), ptr(w), ptr(bias.contiguous()) if bias is not None else None, x.size(0), x.size(1), m,
         int(transposed), int(softmax), ptr(y), ptr(status), stream_ptr())
    return y


class _Linear(torch.autograd.Function):
    """Y = epilogue(X W + b).  flags = 0: plain product (PyG GCNConv's `x @ weight`);
    flags = NORMALIZE|RELU|NODEBN: the dense GraphConv epilogue (encoders.py:36-40,177,134-138)."""

    @staticmethod
    def forward(ctx, x, w, bias, flags: int):
        x, w = x.contiguous(), w.contiguous()
        # DiffPool's assignment Linear + softmax (encoders.py:366-369) at batch size is a tall GEMM: tcgen05 (3xTF32)
        ctx.tc = bool(flags == LIN_SOFTMAX and USE_TCGEN05 and LINEAR_TC and _linear_tc_ok(x.size(0), x.size(1), w.size(1)))
        y = linear_tc_raw(x, w, bias, False, True) if ctx.tc else linear_raw(x, w, bias, False, flags)
        ctx.flags = flags
        ctx.save_for_backward(x, w, bias, y if flags == LIN_SOFTMAX else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w, bias, y = ctx.saved_tensors
        dy = dy.contiguous()
        if ctx.flags == LIN_SOFTMAX:               # from the saved output: no recomputation of the product
            du = torch.empty_like(dy)
            call("tsg_softmax_bwd", ptr(y), ptr(dy), ptr(du), dy.size(0), dy.size(1), stream_ptr())
            dy = du
        elif ctx.flags:
            du = torch.empty_like(dy)
            n, k = x.shape
            call("tsg_dense_epilogue_bwd", ptr(x), ptr(w), ptr(bias), ptr(dy), ptr(du), n, k, dy.size(1),
                 ctx.flags, stream_ptr())
            dy = du
        dx = None
        if ctx.needs_input_grad[0]:
            tc = ctx.tc and _linear_tc_ok(dy.size(0), dy.size(1), w.size(0))
            dx = linear_tc_raw(dy, w, None, True, False) if tc else linear_raw(dy, w, None, True)
        dw = db = None
        if ctx.needs_input_grad[1] or (bias is not None and ctx.needs_input_grad[2]):
            dw, db = linear_bwd_weight(x, dy, bias is not None)
        return dx, dw, db, None


def linear(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, flags: int = 0):
    return _Linear.apply(x, w, bias, flags)


def gcn_conv(x: torch.Tensor, csr: CSR, weight: torch.Tensor, bias: Optional[torch.Tensor],
             relu: bool = False) -> torch.Tensor:
    """PyG GCNConv.forward (Code/sag/network.py:34): (A_hat (X W)) + b, CSR prebuilt by K1."""
    return spmm(csr, linear(x, weight), bias, relu)


# --------------------------------------------------------------------------------------------
# top-k / filter_adj / gate
# --------------------------------------------------------------------------------------------
def batch_to_ptr(batch: torch.Tensor, num_graphs: int) -> torch.Tensor:
    gptr = torch.empty(num_graphs + 1, dtype=torch.int64, device=batch.device)
    call("tsg_batch_to_ptr", ptr(batch.contiguous()), batch.numel(), num_graphs, ptr(gptr), stream_ptr())
    return gptr


def topk_sizes(graph_ptr: torch.Tensor, ratio: float) -> torch.Tensor:
    G = graph_ptr.numel() - 1
    kptr = torch.empty(G + 1, dtype=torch.int64, device=graph_ptr.device)
    wsb = lib.tsg_topk_workspace_bytes(0, G)
    ws = workspace(wsb, graph_ptr.device)
    call("tsg_topk_sizes", ptr(graph_ptr), G, float(ratio), ptr(kptr), ptr(ws), wsb, stream_ptr())
    return kptr


def topk(score: torch.Tensor, graph_ptr: torch.Tensor, k_ptr: torch.Tensor, num_selected: int
         ) -> torch.Tensor:
    """K5a. perm [num_selected] int64, graph-major, score-descending, ties -> lower id."""
    score = score.detach().contiguous()
    G, N = graph_ptr.numel() - 1, score.numel()
    perm = torch.empty(num_selected, dtype=torch.int64, device=score.device)
    wsb = lib.tsg_topk_workspace_bytes(N, G)
    ws = workspace(wsb, score.device)
    call("tsg_topk", ptr(score), ptr(graph_ptr), ptr(k_ptr), G, N, ptr(perm), ptr(ws), wsb, stream_ptr())
    return perm


def filter_adj(edges: EdgeList, perm: torch.Tensor, num_nodes: int) -> Tuple[EdgeList, torch.Tensor]:
    """K5b. Returns the relabelled surviving edges (capacity buffers + device count) and inv_perm."""
    dev = perm.device
    E = edges.cap
    inv = torch.empty(num_nodes, dtype=torch.int32, device=dev)
    out = torch.empty(2, max(E, 1), dtype=torch.int64, device=dev)
    cnt = torch.empty(1, dtype=torch.int64, device=dev)
    wsb = lib.tsg_filter_adj_workspace_bytes(E)
    ws = workspace(wsb, dev)
    call("tsg_filter_adj", ptr(edges.row), ptr(edges.col), E, ptr(edges.count), ptr(perm),
         perm.numel(), num_nodes, ptr(inv), ptr(out[0]), ptr(out[1]), ptr(cnt), ptr(ws), wsb,
         stream_ptr())
    return EdgeList(out[0], out[1], E, cnt), inv


class _GateGather(torch.autograd.Function):
    """xo = x[perm] * tanh(score[perm])  (Code/sag/layers.py:21)."""

    @staticmethod
    def forward(ctx, x, score, perm, inv_perm):
        x = x.contiguous(); score = score.contiguous()
        K, F = perm.numel(), x.size(1)
        xo = torch.empty(K, F, dtype=torch.float32, device=x.device)
        call("tsg_gate_gather_fwd", ptr(x), ptr(score), ptr(perm), None, ptr(xo), None, K, F, stream_ptr())
        ctx.save_for_backward(x, score, inv_perm)
        return xo

    @staticmethod
    def backward(ctx, dxo):
        x, score, inv = ctx.saved_tensors
        dxo = dxo.contiguous()
        dx = torch.empty_like(x)
        ds = torch.empty_like(score)
        call("tsg_gate_gather_bwd", ptr(dxo), ptr(x), ptr(score), ptr(inv), ptr(dx), ptr(ds),
             x.size(0), x.size(1), stream_ptr())
        return dx, ds, None, None


def gate_gather(x, score, perm, inv_perm):
    return _GateGather.apply(x, score, perm, inv_perm)


def gather_batch(batch: torch.Tensor, perm: torch.Tensor) -> torch.Tensor:
    return batch[perm]


# --------------------------------------------------------------------------------------------
# readout
# --------------------------------------------------------------------------------------------
class _Readout(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, graph_ptr, mode):
        x = x.contiguous()
        G, F = graph_ptr.numel() - 1, x.size(1)
        width = F * (bool(mode & READOUT_MAX) + bool(mode & (READOUT_MEAN | READOUT_SUM)))
        out = torch.empty(G, width, dtype=torch.float32, device=x.device)
        am = torch.empty(G, F, dtype=torch.int32, device=x.device) if mode & READOUT_MAX else None
        call("tsg_readout_fwd", ptr(x), ptr(graph_ptr), G, F, mode, ptr(out), width, ptr(am), stream_ptr())
        ctx.mode, ctx.n, ctx.f = mode, x.size(0), F
        ctx.save_for_backward(graph_ptr, am)
        return out

    @staticmethod
    def backward(ctx, dout):
        gptr, am = ctx.saved_tensors
        dout = dout.contiguous()
        # contract: graph_ptr covers every row (graph_ptr[G] == N), so the kernel writes all of dx
        dx = torch.empty(ctx.n, ctx.f, dtype=torch.float32, device=dout.device)
        call("tsg_readout_bwd", ptr(dout), dout.size(1), ptr(am), ptr(gptr), gptr.numel() - 1, ctx.n,
             ctx.f, ctx.mode, ptr(dx), stream_ptr())
        return dx, None, None


def readout(x: torch.Tensor, graph_ptr: torch.Tensor, mode: int = READOUT_MAX | READOUT_MEAN):
    """K6: [gmp || gap] per graph (Code/sag/network.py:36)."""
    return _Readout.apply(x, graph_ptr, mode)


class _BroadcastRows(torch.autograd.Function):
    """out[i,:] = v[g(i),:] for the rows i of graph g (the adjoint of the per-graph SUM readout): forward is
    K6's backward kernel in SUM mode, backward is K6's forward -- no index tensor, no sort-based
    index_put in the gradient."""

    @staticmethod
    def forward(ctx, v, graph_ptr, n):
        v = v.contiguous()
        G, F = v.shape
        out = torch.empty(n, F, dtype=torch.float32, device=v.device)
        call("tsg_readout_bwd", ptr(v), F, None, ptr(graph_ptr), G, n, F, READOUT_SUM, ptr(out), stream_ptr())
        ctx.save_for_backward(graph_ptr)
        ctx.g, ctx.f = G, F
        return out

    @staticmethod
    def backward(ctx, dout):
        (gptr,) = ctx.saved_tensors
        dout = dout.contiguous()
        dv = torch.empty(ctx.g, ctx.f, dtype=torch.float32, device=dout.device)
        call("tsg_readout_fwd", ptr(dout), ptr(gptr), ctx.g, ctx.f, READOUT_SUM, ptr(dv), ctx.f, None, stream_ptr())
        return dv, None, None


def broadcast_rows(v: torch.Tensor, graph_ptr: torch.Tensor, n: int) -> torch.Tensor:
    return _BroadcastRows.apply(v, graph_ptr, n)


# --------------------------------------------------------------------------------------------
# triplet loss
# --------------------------------------------------------------------------------------------
class _TripletLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, emb, triplets, margin, eps):
        emb = emb.contiguous(); triplets = triplets.contiguous()
        T, (M, D) = triplets.size(0), emb.shape
        dev = emb.device
        dp = torch.empty(T, dtype=torch.float32, device=dev)
        dn = torch.empty(T, dtype=torch.float32, device=dev)
        loss = torch.empty((), dtype=torch.float32, device=dev)
        wsb = lib.tsg_triplet_workspace_bytes(T, M, D)
        ws = workspace(wsb, dev)
        call("tsg_triplet_fwd", ptr(emb), ptr(triplets), T, M, D, float(margin), float(eps), ptr(dp),
             ptr(dn), ptr(loss), ptr(ws), wsb, stream_ptr())
        ctx.margin, ctx.eps = float(margin), float(eps)
        ctx.save_for_backward(emb, triplets, dp, dn)
        ctx.mark_non_differentiable(dp, dn)
        return loss, dp, dn

    @staticmethod
    def backward(ctx, dloss, _ddp, _ddn):
        emb, triplets, dp, dn = ctx.saved_tensors
        T, (M, D) = triplets.size(0), emb.shape
        demb = torch.empty_like(emb)
        wsb = lib.tsg_triplet_workspace_bytes(T, M, D)
        ws = workspace(wsb, emb.device)
        dloss = dloss.contiguous().view(1)
        call("tsg_triplet_bwd", ptr(emb), ptr(triplets), T, M, D, ctx.margin, ctx.eps, ptr(dp), ptr(dn),
             ptr(dloss), ptr(demb), ptr(ws), wsb, stream_ptr())
        return demb, None, None, None


def triplet_loss(emb: torch.Tensor, triplets: torch.Tensor, margin: float, eps: float = 1e-6):
    """K9: (loss, d_pos, d_neg) for index triplets [T,3] into emb [M,D]
    (Code/sag/tripletnet.py:21-22 + train_triplet.py:196,208-211)."""
    return _TripletLoss.apply(emb, triplets, margin, eps)


def pairdist_matrix(emb: torch.Tensor, eps: float = 1e-6) -> torch.Tensor:
    emb = emb.detach().contiguous()
    M, D = emb.shape
    out = torch.empty(M, M, dtype=torch.float32, device=emb.device)
    call("tsg_pairdist_matrix", ptr(emb), M, D, float(eps), ptr(out), stream_ptr())
    return out


# --------------------------------------------------------------------------------------------
# K7 per-graph dense contractions (DiffPool)
# --------------------------------------------------------------------------------------------


def seg_contract_raw(x: torch.Tensor, y: torch.Tensor, graph_ptr: torch.Tensor,
                     tensor_cores: Optional[bool] = None) -> torch.Tensor:
    """C[g] = sum_{r in g} x[r,:]^T y[r,:]  -> [G, Kx, Ky]."""
    x = x.contiguous(); y = y.contiguous()
    G, kx, ky = graph_ptr.numel() - 1, x.size(1), y.size(1)
    tc = USE_TCGEN05 if tensor_cores is None else tensor_cores
    tc = bool(tc) and kx <= 128 and ky <= 256
    c = torch.empty(G, kx, ky, dtype=torch.float32, device=x.device)
    status = torch.zeros(1, dtype=torch.int32, device=x.device) if tc else None
    call("tsg_seg_contract", ptr(x), ptr(y), ptr(graph_ptr), G, kx, ky, ptr(c), int(tc), ptr(status), stream_ptr())
    return c


SEG_LINEAR_TC = os.environ.get("TSG_SEG_LINEAR_NOTC", "0") != "1"


def seg_linear_raw(x: torch.Tensor, w: torch.Tensor, graph_ptr: torch.Tensor, transposed: bool = False,
                   tensor_cores: Optional[bool] = None):
    """y[r,:] = x[r,:] . w[g]  (w [G, Kin, M])  or  x[r,:] . w[g]^T  (w [G, M, Kin]) for r in graph g.
    tensor_cores (default ops.USE_TCGEN05): the tcgen05 3xTF32 kernel where the shape allows it, else fp32 SIMT."""
    x = x.contiguous(); w = w.contiguous()
    G, kin = graph_ptr.numel() - 1, x.size(1)
    m = w.size(1) if transposed else w.size(2)
    if (w.size(2) if transposed else w.size(1)) != kin or w.size(0) != G:
        raise RuntimeError(f"tsg.seg_linear: shape mismatch x{tuple(x.shape)} w{tuple(w.shape)} T={transposed}")
    y = torch.empty(x.size(0), m, dtype=torch.float32, device=x.device)
    tc = USE_TCGEN05 if tensor_cores is None else tensor_cores
    if tc and SEG_LINEAR_TC and kin % 4 == 0 and m % 4 == 0 and m <= 256 and kin >= 32:
        status = torch.zeros(1, dtype=torch.int32, device=x.device)
        call("tsg_seg_linear_tc", ptr(x), ptr(w), ptr(graph_ptr), G, kin, m, int(transposed), ptr(y), ptr(status), stream_ptr())
        return y
    call("tsg_seg_linear", ptr(x), ptr(w), ptr(graph_ptr), G, kin, m, int(transposed), ptr(y), stream_ptr())
    return y


class _SegContract(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, y, graph_ptr):
        ctx.save_for_backward(x, y, graph_ptr)
        return seg_contract_raw(x, y, graph_ptr)

    @staticmethod
    def backward(ctx, dc):
        x, y, gptr = ctx.saved_tensors
        dc = dc.contiguous()
        dx = seg_linear_raw(y, dc, gptr, transposed=True) if ctx.needs_input_grad[0] else None   # Y dC^T
        dy = seg_linear_raw(x, dc, gptr, transposed=False) if ctx.needs_input_grad[1] else None  # X dC
        return dx, dy, None


class _SegLinear(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, graph_ptr):
        ctx.save_for_backward(x, w, graph_ptr)
        return seg_linear_raw(x, w, graph_ptr, False)

    @staticmethod
    def backward(ctx, dy):
        x, w, gptr = ctx.saved_tensors
        dy = dy.contiguous()
        dx = seg_linear_raw(dy, w, gptr, transposed=True) if ctx.needs_input_grad[0] else None
        dw = seg_contract_raw(x, dy, gptr) if ctx.needs_input_grad[1] else None
        return dx, dw, None


def seg_contract(x, y, graph_ptr):
    return _SegContract.apply(x, y, graph_ptr)


def seg_linear(x, w, graph_ptr):
    return _SegLinear.apply(x, w, graph_ptr)


# --------------------------------------------------------------------------------------------
# K15 DiffPool link-prediction loss
# --------------------------------------------------------------------------------------------
class _LinkPredLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, s, graph_ptr, csr: CSR, num_entries: float, eps: float):
        s = s.contiguous()
        G, K = graph_ptr.numel() - 1, s.size(1)
        loss = torch.empty((), dtype=torch.float32, device=s.device)
        wsb = lib.tsg_linkpred_workspace_bytes(G)
        ws = workspace(wsb, s.device)
        call("tsg_linkpred_loss_fwd", ptr(s), ptr(graph_ptr), ptr(csr.rowptr), ptr(csr.colidx), G, K, float(num_entries),
             float(eps), ptr(loss), ptr(ws), wsb, stream_ptr())
        ctx.csr, ctx.num_entries, ctx.eps = csr, float(num_entries), float(eps)
        ctx.save_for_backward(s, graph_ptr)
        return loss

    @staticmethod
    def backward(ctx, dloss):
        s, gptr = ctx.saved_tensors
        ds = torch.empty_like(s)
        call("tsg_linkpred_loss_bwd", ptr(s), ptr(gptr), ptr(ctx.csr.rowptr), ptr(ctx.csr.colidx), gptr.numel() - 1, s.size(1),
             ctx.num_entries, ctx.eps, ptr(dloss.contiguous().view(1)), ptr(ds), stream_ptr())
        return ds, None, None, None, None


def linkpred_loss(s: torch.Tensor, graph_ptr: torch.Tensor, csr_raw: CSR, num_entries: float, eps: float = 1e-7):
    """K15: SoftPoolingGcnEncoder.loss's link-prediction term (Code/sage+gat+diffpool/encoders.py:416-440) on packed
    assignment rows s [sum n, K] and the RAW CSR of the 0/1 adjacency; num_entries = sum_g n_g^2 (host)."""
    return _LinkPredLoss.apply(s, graph_ptr, csr_raw, num_entries, eps)


# --------------------------------------------------------------------------------------------
# K16 prediction head + cross-entropy
# --------------------------------------------------------------------------------------------
PRED_MAX_LAYERS, PRED_MAX_WIDTH = 8, 256


def check_pred_head(in_dim: int, out_dims) -> None:
    """Raise ValueError unless a head over rows of width `in_dim` with layers of widths `out_dims` fits K16 (at most 8
    layers, every width in [1, 256]): there is no other path for such a head."""
    widths = [int(in_dim)] + [int(w) for w in out_dims]
    if len(widths) - 1 > PRED_MAX_LAYERS or min(widths) < 1 or max(widths) > PRED_MAX_WIDTH:
        raise ValueError(f"tsg: the prediction head ({len(widths) - 1} layers, widths {widths}) is beyond K16's limits: at "
                         f"most {PRED_MAX_LAYERS} Linear layers, every width in [1, {PRED_MAX_WIDTH}]")


def pred_head_desc(in_dim: int, layers, softmax_first: bool) -> "_lib.PredHead":
    """The tsg_pred_head of a chain of `layers` [(weight [out, in], bias [out] or None, relu_after), ...] over rows of
    width `in_dim` (check_pred_head first)."""
    check_pred_head(in_dim, [int(w.size(0)) for w, _, _ in layers])
    h = _lib.PredHead()
    h.num_layers, h.in_dim, h.softmax_first = len(layers), int(in_dim), int(bool(softmax_first))
    mask, inp = 0, int(in_dim)
    for l, (w, b, relu) in enumerate(layers):
        if w.dim() != 2 or w.size(1) != inp:
            raise ValueError(f"tsg: prediction-head layer {l} takes {tuple(w.shape)} weights after a width of {inp}")
        h.out_dim[l], h.weight[l], h.bias[l] = int(w.size(0)), ptr(w), ptr(b)
        mask |= (1 << l) if relu else 0
        inp = int(w.size(0))
    h.relu_mask = mask
    return h


class _PredCE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, r, y, softmax_first, relus, *params):
        from . import nn as tnn
        r = r.contiguous()
        layers = [(params[2 * l].contiguous(), None if params[2 * l + 1] is None else params[2 * l + 1].contiguous(), relus[l])
                  for l in range(len(relus))]
        desc = pred_head_desc(r.size(1), layers, softmax_first)
        G = r.size(0)
        wsb = lib.tsg_pred_ce_workspace_bytes(ctypes.byref(desc), G)
        ws = workspace(wsb, r.device)
        loss = torch.empty((), dtype=torch.float32, device=r.device)
        call("tsg_pred_ce_fwd", ctypes.byref(desc), ptr(r), ptr(y), G, ptr(loss), None, ptr(tnn._status_word(r.device)),
             ptr(ws), wsb, stream_ptr())
        ctx.desc, ctx.ws, ctx.wsb, ctx.layers = desc, ws, wsb, layers      # the layers keep desc's pointers alive
        ctx.save_for_backward(r, y)
        return loss

    @staticmethod
    def backward(ctx, dloss):
        r, y = ctx.saved_tensors
        L = len(ctx.layers)
        dr = torch.empty_like(r) if ctx.needs_input_grad[0] else None
        dws = [torch.empty_like(w) for w, _, _ in ctx.layers]
        dbs = [None if b is None else torch.empty_like(b) for _, b, _ in ctx.layers]
        arr = ctypes.c_void_p * max(L, 1)
        call("tsg_pred_ce_bwd", ctypes.byref(ctx.desc), ptr(r), ptr(y), r.size(0), ptr(dloss.contiguous().view(1)), ptr(dr),
             arr(*[ptr(t) for t in dws]), arr(*[ptr(t) for t in dbs]), ptr(ctx.ws), ctx.wsb, stream_ptr())
        grads = []
        for dw, db in zip(dws, dbs):
            grads += [dw, db]
        return (dr, None, None, None, *grads)


def pred_ce(r: torch.Tensor, layers, y: torch.Tensor, softmax_first: bool = False) -> torch.Tensor:
    """K16: mean cross-entropy of the head `layers` [(weight [out, in], bias or None, relu_after), ...] over the readout
    rows r [G, D0] against int64 labels y [G] (softmax_first: of softmax(logits), the reference's 2stg+ stage 2).  An
    autograd Function: backward reaches r (and the encoder below it) and every weight and bias.  A label outside
    [0, C) sets status bit 8 (tsg.nn.check_fused_status raises)."""
    flat = []
    for w, b, _ in layers:
        flat += [w, b]
    return _PredCE.apply(r, y.contiguous(), bool(softmax_first), tuple(bool(x) for _, _, x in layers), *flat)


def pred_classify(r: torch.Tensor, layers, y: Optional[torch.Tensor] = None, softmax_first: bool = False,
                  want_logits: bool = False):
    """K16's eval-mode forward: -> (pred int64 [G] (first-index argmax of the logits), logits [G, C] or None,
    correct int64 [1] or None, ce_sum float32 [1] or None); the last two need the labels y and are fixed-order totals
    (ce_sum includes the softmax_first loss)."""
    from . import nn as tnn
    r = r.contiguous()
    with torch.no_grad():
        layers = [(w.detach().contiguous(), None if b is None else b.detach().contiguous(), relu) for w, b, relu in layers]
        desc = pred_head_desc(r.size(1), layers, softmax_first)
        G, dev = r.size(0), r.device
        C = layers[-1][0].size(0) if layers else r.size(1)
        pred = torch.empty(G, dtype=torch.int64, device=dev)
        logits = torch.empty(G, C, dtype=torch.float32, device=dev) if want_logits else None
        correct = torch.empty(1, dtype=torch.int64, device=dev) if y is not None else None
        ce_sum = torch.empty(1, dtype=torch.float32, device=dev) if y is not None else None
        wsb = lib.tsg_pred_classify_workspace_bytes(ctypes.byref(desc), G)
        ws = workspace(wsb, dev)
        call("tsg_pred_classify", ctypes.byref(desc), ptr(r), ptr(None if y is None else y.contiguous()), G, ptr(pred),
             ptr(logits), ptr(correct), ptr(ce_sum), ptr(tnn._status_word(dev)), ptr(ws), wsb, stream_ptr())
    return pred, logits, correct, ce_sum
