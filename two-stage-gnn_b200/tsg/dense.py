"""Dense-directory operator surface on the packed CSR layout.

The reference's `Code/sage+gat+diffpool` and `Code/eigengcn` models take zero-padded dense tensors
(`x [B,N,F]`, `adj [B,N,N]`, `num_nodes [B]`; N = --max-nodes = 1000 by default) and multiply them
with `torch.matmul`.  Here the same arithmetic runs on the packed layout: real node rows only,
adjacency / pooling operators as CSR, every layer = K2 aggregation + K3 row-local epilogue.

Dense quirks reproduced exactly (SURVEY A.2):
  * raw 0/1 adjacency, no self loops, no normalisation; L2-normalise after the bias; ReLU; fresh
    BatchNorm1d(num_nodes) per call == per-node statistics over the features (batch of one graph);
  * `GcnEncoderGraph.forward` max-reads over ALL N rows, unmasked: every padded row equals the
    bias-derived "virtual node" epilogue(b_l) (its adjacency row is zero), so the readout of a graph
    with n < N is max(max over real rows, v_l).  `gcn_forward` paths (DiffPool / Wave) zero the padded
    rows instead, so their readout is max(max over real rows, 0).
Batch semantics: each packed graph is its own batch of one (what every shipped script runs:
triplet paths forward single graphs; `--batch-size` defaults to 1).
"""
from __future__ import annotations

from typing import List, Optional, Sequence

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops
from ._lib import call, lib, ptr, stream_ptr, workspace
from .ops import CSR, CSR_RAW, EdgeList, LIN_NODEBN, LIN_NORMALIZE, LIN_RELU, READOUT_MAX


# ---------------------------------------------------------------------------------------------
# adapters
# ---------------------------------------------------------------------------------------------
def dense_to_csr(mat: torch.Tensor, nrows: Sequence[int], ncols: Sequence[int], transpose: bool = False,
                 packed: bool = True, capacity: Optional[int] = None, want_eid: bool = False):
    """Zero-padded dense operators M[B,R,C] -> CSR of the block-diagonal packed operator.

    transpose=False: y[row_off+r] = sum_c M[r,c] x[col_off+c]      (adjacency: adj @ x)
    transpose=True : y[col_off+c] = sum_r M[r,c] x[row_off+r]      (eigen pooling: P^T @ x)
    Returns (csr, num_out_rows, num_in_rows).  One host sync (the non-zero count sizes the CSR)."""
    mat = mat.contiguous()
    B, R, C = mat.shape
    dev = mat.device
    nr = np.asarray(nrows, dtype=np.int64).reshape(B); nc = np.asarray(ncols, dtype=np.int64).reshape(B)
    if packed:
        roff = np.concatenate([[0], np.cumsum(nr)]).astype(np.int64)
        coff = np.concatenate([[0], np.cumsum(nc)]).astype(np.int64)
    else:
        roff = (np.arange(B + 1) * R).astype(np.int64); coff = (np.arange(B + 1) * C).astype(np.int64)
    meta = torch.from_numpy(np.stack([nr, nc, roff[:-1], coff[:-1]])).to(dev)
    cap = int(capacity) if capacity is not None else int((nr * nc).sum())
    cap = max(cap, 1)
    out_r = torch.empty(cap, dtype=torch.int64, device=dev)
    out_c = torch.empty(cap, dtype=torch.int64, device=dev)
    out_w = torch.empty(cap, dtype=torch.float32, device=dev)
    cnt = torch.empty(1, dtype=torch.int64, device=dev)
    wsb = lib.tsg_dense_to_coo_workspace_bytes(B, R)
    ws = workspace(wsb, dev)
    call("tsg_dense_to_coo", ptr(mat), B, R, C, ptr(meta[0]), ptr(meta[1]), ptr(meta[2]), ptr(meta[3]),
         ptr(out_r), ptr(out_c), ptr(out_w), cap, ptr(cnt), ptr(ws), wsb, stream_ptr())
    nnz = int(cnt.item())
    n_rows, n_cols = int(roff[-1]), int(coff[-1])
    if transpose:      # destination = matrix column, source = matrix row
        el = EdgeList(out_r[:nnz].contiguous(), out_c[:nnz].contiguous(), nnz)
        n_out, n_in = n_cols, n_rows
    else:              # destination = matrix row, source = matrix column
        el = EdgeList(out_c[:nnz].contiguous(), out_r[:nnz].contiguous(), nnz)
        n_out, n_in = n_rows, n_cols
    csr = build_rect_csr(el, out_w[:nnz].contiguous(), n_out, n_in, want_eid)
    return csr, n_out, n_in


def build_rect_csr(el: EdgeList, w: torch.Tensor, n_out: int, n_in: int, want_eid: bool = False) -> CSR:
    """K1 in RAW mode for a rectangular operator (n_out x n_in): the forward CSR has n_out rows, the
    transposed one n_in rows; built over max(n_out, n_in) rows and trimmed."""
    n = max(n_out, n_in)
    csr = ops.build_csr(el, n, mode=CSR_RAW, transposed=True, edge_weight=w, want_eid=want_eid)
    csr.rowptr = csr.rowptr[:n_out + 1]
    csr.t_rowptr = csr.t_rowptr[:n_in + 1]
    csr.num_nodes = n_out
    return csr


def pack_rows(x: torch.Tensor, num_nodes: Sequence[int]) -> torch.Tensor:
    """x [B,N,F] -> [sum n, F]: the real rows of every graph, graph-major."""
    B, N, Fd = x.shape
    nn_ = torch.as_tensor(np.asarray(num_nodes, dtype=np.int64), device=x.device)
    idx = torch.arange(N, device=x.device).view(1, N) < nn_.view(B, 1)
    return x[idx]


class _NodeBN(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        x = x.contiguous()
        B, N, Fd = x.shape
        y = torch.empty_like(x)
        mean = torch.empty(N, dtype=torch.float32, device=x.device)
        rstd = torch.empty(N, dtype=torch.float32, device=x.device)
        call("tsg_nodebn_fwd", ptr(x), ptr(y), ptr(mean), ptr(rstd), B, N, Fd, stream_ptr())
        ctx.save_for_backward(y, rstd)
        return y

    @staticmethod
    def backward(ctx, dy):
        y, rstd = ctx.saved_tensors
        dy = dy.contiguous()
        dx = torch.empty_like(dy)
        B, N, Fd = dy.shape
        call("tsg_nodebn_bwd", ptr(dy), ptr(y), ptr(rstd), ptr(dx), B, N, Fd, stream_ptr())
        return dx


def node_bn(x: torch.Tensor) -> torch.Tensor:
    """`apply_bn` (encoders.py:134-138) on the dense wire format [B,N,F] (any B)."""
    return _NodeBN.apply(x)


# ---------------------------------------------------------------------------------------------
# GraphConv on the packed layout
# ---------------------------------------------------------------------------------------------
class GraphConv(nn.Module):
    """Same parameters as the reference GraphConv (encoders.py:13-28): `weight [in,out]`, `bias [out]`."""

    def __init__(self, input_dim: int, output_dim: int, add_self: bool = False,
                 normalize_embedding: bool = False, dropout: float = 0.0, bias: bool = True):
        super().__init__()
        self.add_self, self.normalize_embedding, self.dropout = add_self, normalize_embedding, dropout
        self.input_dim, self.output_dim = input_dim, output_dim
        self.weight = nn.Parameter(torch.empty(input_dim, output_dim))
        self.bias = nn.Parameter(torch.empty(output_dim)) if bias else None
        nn.init.xavier_uniform_(self.weight, gain=nn.init.calculate_gain("relu"))   # encoders.py:91
        if self.bias is not None:
            nn.init.constant_(self.bias, 0.0)

    def forward(self, x: torch.Tensor, csr: CSR, act_bn: int = 0) -> torch.Tensor:
        """x [rows, F_in] packed; act_bn adds LIN_RELU / LIN_NODEBN to the fused epilogue (the
        reference applies them right after the conv, encoders.py:176-179)."""
        if self.dropout > 0.001 and self.training:
            x = F.dropout(x, self.dropout, True)
        y = ops.spmm(csr, x)                                   # adj @ x           (encoders.py:33)
        if self.add_self:
            y = y + x                                          #                   (:34-35)
        flags = (LIN_NORMALIZE if self.normalize_embedding else 0) | act_bn
        return ops.linear(y, self.weight, self.bias, flags)    # @W + b, normalise (:36-40)

    def virtual_row(self, act_bn: int) -> torch.Tensor:
        """Value of every zero-padded row after this layer: its adjacency row is zero, so u = b."""
        u = self.bias if self.bias is not None else self.weight.new_zeros(self.output_dim)
        if self.normalize_embedding:
            u = u / u.norm().clamp_min(1e-12)
        if act_bn & LIN_RELU:
            u = F.relu(u)
        if act_bn & LIN_NODEBN:
            u = (u - u.mean()) / torch.sqrt(u.var(unbiased=False) + 1e-5)
        return u


def _readout_max(x: torch.Tensor, graph_ptr: torch.Tensor, pad_value, has_pad: torch.Tensor):
    """max over a graph's real rows, then against the padded rows' value where the graph has any."""
    out = ops.readout(x, graph_ptr, READOUT_MAX)
    if pad_value is None:
        return out
    pv = pad_value.view(1, -1) if torch.is_tensor(pad_value) else out.new_full((1, out.size(1)), float(pad_value))
    return torch.where(has_pad.view(-1, 1), torch.maximum(out, pv.expand_as(out)), out)


class GcnStack(nn.Module):
    """conv_first / conv_block / conv_last with the reference's names (encoders.py:94-104)."""

    def __init__(self, input_dim, hidden_dim, embedding_dim, num_layers, add_self=False, normalize=True,
                 dropout=0.0, bias=True, names=("conv_first", "conv_block", "conv_last")):
        super().__init__()
        self.names = names
        setattr(self, names[0], GraphConv(input_dim, hidden_dim, add_self, normalize, bias=bias))
        setattr(self, names[1], nn.ModuleList([GraphConv(hidden_dim, hidden_dim, add_self, normalize, dropout, bias)
                                               for _ in range(num_layers - 2)]))
        setattr(self, names[2], GraphConv(hidden_dim, embedding_dim, add_self, normalize, bias=bias))

    def layers(self) -> List[GraphConv]:
        return [getattr(self, self.names[0])] + list(getattr(self, self.names[1])) + [getattr(self, self.names[2])]


def gcn_forward(x, csr: CSR, convs: List[GraphConv], bn: bool = True) -> torch.Tensor:
    """encoders.py:140-167 on packed rows (the mask only zeroes padded rows, which do not exist here)."""
    outs = []
    for i, c in enumerate(convs):
        last = i == len(convs) - 1
        x = c(x, csr, 0 if last else (LIN_RELU | (LIN_NODEBN if bn else 0)))
        outs.append(x)
    return torch.cat(outs, dim=1)


class PackedGcnEncoder(nn.Module):
    """GcnEncoderGraph (Code/sage+gat+diffpool/encoders.py:45-217; "GraphSAGE"/base) on packed graphs.
    State-dict keys match the reference (conv_first.weight, conv_block.0.bias, map_model.weight, ...)."""

    def __init__(self, input_dim, hidden_dim, embedding_dim, label_dim, num_layers, pred_hidden_dims=(),
                 concat=True, bn=True, dropout=0.0, bias=True, final_dim="output_dim"):
        super().__init__()
        self.concat, self.bn, self.num_layers, self.final_dim = concat, bn, num_layers, final_dim
        stack = GcnStack(input_dim, hidden_dim, embedding_dim, num_layers, not concat, True, dropout, bias)
        self.conv_first, self.conv_block, self.conv_last = stack.conv_first, stack.conv_block, stack.conv_last
        self.pred_input_dim = hidden_dim * (num_layers - 1) + embedding_dim if concat else embedding_dim
        self.pre_pred_model = _pred_layers(self.pred_input_dim, pred_hidden_dims, embedding_dim)
        self.pred_model = _pred_layers(embedding_dim, pred_hidden_dims, label_dim)
        self.map_model = _pred_layers(self.pred_input_dim, pred_hidden_dims, embedding_dim)
        self.map2_model = _pred_layers(embedding_dim, (), 2)

    def convs(self):
        return [self.conv_first] + list(self.conv_block) + [self.conv_last]

    def readout(self, x, csr: CSR, graph_ptr: torch.Tensor, has_pad: torch.Tensor) -> torch.Tensor:
        """encoders.py:175-203: per layer conv -> ReLU -> BN, max over all N rows (virtual padded row)."""
        outs = []
        convs = self.convs()
        for i, c in enumerate(convs):
            last = i == len(convs) - 1
            ab = 0 if last else (LIN_RELU | (LIN_NODEBN if self.bn else 0))
            x = c(x, csr, ab)
            outs.append(_readout_max(x, graph_ptr, c.virtual_row(ab), has_pad))
        return torch.cat(outs, dim=1) if self.concat else outs[-1]

    def forward(self, x, csr: CSR, graph_ptr: torch.Tensor, has_pad: torch.Tensor):
        output = self.readout(x, csr, graph_ptr, has_pad)
        if self.final_dim == "pretrain":                       # encoders.py:207-210
            out = self.map_model(output)
            return self.map2_model(out), out
        if self.final_dim != "output_dim":                     # :211-214
            ov = self.pre_pred_model(output)
            return ov, self.pred_model(ov)
        return output, self.map_model(output)                  # :215-217


def _pred_layers(inp, hidden, out):
    """build_pred_layers (encoders.py:105-119)."""
    if len(hidden) == 0:
        return nn.Linear(inp, out)
    layers = []
    for h in hidden:
        layers += [nn.Linear(inp, h), nn.ReLU()]
        inp = h
    layers.append(nn.Linear(inp, out))
    return nn.Sequential(*layers)


# ---------------------------------------------------------------------------------------------
# EigenPooling (Code/eigengcn/encoders.py:396-417) and the Wave encoder (:248-378)
# ---------------------------------------------------------------------------------------------
def eigen_pool(x: torch.Tensor, pool_csrs: List[CSR]) -> torch.Tensor:
    """K8: X_j = P_j^T X for every pooling operator, concatenated on the feature axis.  P_j^T is a
    CSR with one non-zero per node (its cluster's j-th Laplacian eigenvector entry), so forward is a
    segment-weighted sum and backward (dX = P_j dX_j) a pure gather -- both are K2 launches."""
    res = [ops.spmm(c, x) for c in pool_csrs]
    return torch.cat(res, dim=1) if len(res) > 1 else res[0]


class PackedWaveEncoder(nn.Module):
    """WavePoolingGcnEncoder (concat=True, mask=1, con_final=1) on packed graphs."""

    def __init__(self, input_dim, hidden_dim, embedding_dim, label_dim, num_layers, num_pool_matrix=2,
                 num_pool_final_matrix=0, pool_sizes=(4,), pred_hidden_dims=(50,), bn=True, dropout=0.0):
        super().__init__()
        self.bn, self.num_pool_matrix, self.num_pool_final_matrix = bn, num_pool_matrix, num_pool_final_matrix
        self.pool_sizes = list(pool_sizes)
        stack = GcnStack(input_dim, hidden_dim, embedding_dim, num_layers, False, True, dropout)
        self.conv_first, self.conv_block, self.conv_last = stack.conv_first, stack.conv_block, stack.conv_last
        D = hidden_dim * (num_layers - 1) + embedding_dim
        self.pred_input_dim = D
        self.conv_first_after_pool, self.conv_block_after_pool, self.conv_last_after_pool = (
            nn.ModuleList(), nn.ModuleList(), nn.ModuleList())
        for _ in self.pool_sizes:
            s = GcnStack(D * num_pool_matrix, hidden_dim, embedding_dim, num_layers, False, True, dropout)
            self.conv_first_after_pool.append(s.conv_first)
            self.conv_block_after_pool.append(s.conv_block)
            self.conv_last_after_pool.append(s.conv_last)
        width = D * (len(self.pool_sizes) + 1) + (D * num_pool_final_matrix if num_pool_final_matrix > 0 else 0)
        self.pred_model = _pred_layers(width, pred_hidden_dims, label_dim)      # eigengcn/encoders.py:294-296

    def readout(self, x, csr_adj: CSR, graph_ptr, pool_csrs: List[List[CSR]], csr_pooled: List[CSR],
                pooled_ptrs: List[torch.Tensor], final_ptr: Optional[torch.Tensor] = None,
                has_pad: Optional[Sequence[torch.Tensor]] = None) -> torch.Tensor:
        """The concatenated max-readouts (`output`, eigengcn/encoders.py:323-370): the input of pred_model.
        has_pad: per readout (level 0, every pooled level, then the final pooling if any) bool [graphs] -- whether the
        reference's max_nodes padding leaves a zero row there, so its max is taken against 0.  None: every graph is
        padded at every level (n < max_nodes, as bench config 5 assumes)."""
        outs = []
        ones = torch.ones(graph_ptr.numel() - 1, dtype=torch.bool, device=x.device) if has_pad is None else None
        pad = (lambda k: ones) if has_pad is None else (lambda k: has_pad[k])
        convs = [self.conv_first] + list(self.conv_block) + [self.conv_last]
        z = gcn_forward(x, csr_adj, convs, self.bn)
        outs.append(_readout_max(z, graph_ptr, 0.0, pad(0)))
        for i in range(len(self.pool_sizes)):
            z = eigen_pool(z, pool_csrs[i][:self.num_pool_matrix])
            convs = [self.conv_first_after_pool[i]] + list(self.conv_block_after_pool[i]) + [self.conv_last_after_pool[i]]
            z = gcn_forward(z, csr_pooled[i], convs, self.bn)
            outs.append(_readout_max(z, pooled_ptrs[i], 0.0, pad(i + 1)))
        if self.num_pool_final_matrix > 0:
            z = eigen_pool(z, pool_csrs[len(self.pool_sizes)][:self.num_pool_final_matrix])
            outs.append(_readout_max(z, final_ptr, 0.0, pad(len(self.pool_sizes) + 1)))
        return torch.cat(outs, dim=1)

    def forward(self, x, csr_adj: CSR, graph_ptr, pool_csrs: List[List[CSR]], csr_pooled: List[CSR],
                pooled_ptrs: List[torch.Tensor], final_ptr: Optional[torch.Tensor] = None,
                has_pad: Optional[Sequence[torch.Tensor]] = None):
        """x packed [sum n, F]; pool_csrs[i] = the P_j^T CSRs of level i (level len(pool_sizes) = final);
        csr_pooled[i] / pooled_ptrs[i] = coarsened adjacency / cluster offsets of level i; has_pad: see readout (None =
        every graph has n < N, padded rows exist, as in the reference's max_nodes padding)."""
        return self.pred_model(self.readout(x, csr_adj, graph_ptr, pool_csrs, csr_pooled, pooled_ptrs, final_ptr,
                                            has_pad))
