"""Synthetic EigenPooling operands for BASELINE config 5 (SURVEY 8d "Eigen-pool operands").

The reference builds them per graph on the CPU at load time (spectral clustering + per-cluster `eigh`,
Code/eigengcn/coarsen_pooling_with_last_eigen_padding.py:36-182, cached as a pickle): preprocessing,
outside the timed path.  For throughput runs the survey prescribes a cheap generator with the same
*format*: clusters = contiguous chunks of `pool_size` nodes in BFS order; P[:, c] = j-th eigenvector of
the cluster's unnormalised Laplacian (`--normalize 0`), sign-fixed so its first entry is >= 0
(coarsen...py:165-168), last eigenvector repeated when the cluster is smaller than j+1; coarsened
adjacency = Omega^T A_ext Omega (inter-cluster edge counts, :135,149); final pooling = the same
construction with ONE cluster holding every coarse node.  Pure numpy / scipy, seeded by the corpus.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List

import numpy as np

from .synth import Corpus


@dataclass
class EigenOperands:
    """Ragged per-corpus operands; ids local to each graph."""
    cluster_ptr: np.ndarray          # int64 [G+1] clusters per graph
    cluster_of: np.ndarray           # int64 [sum n] local cluster id of every node
    pool_w: List[np.ndarray]         # num_pool_matrix arrays f32 [sum n]: P_j[node, cluster_of[node]]
    coarse_ptr: np.ndarray           # int64 [G+1] non-zeros of every coarsened adjacency
    coarse_row: np.ndarray           # int64 local cluster ids (dst)
    coarse_col: np.ndarray           # int64 local cluster ids (src)
    coarse_w: np.ndarray             # f32
    final_w: List[np.ndarray]        # num_pool_final_matrix arrays f32 [sum n_c]


def _bfs_order(n: int, row: np.ndarray, col: np.ndarray) -> np.ndarray:
    import scipy.sparse as sp
    from scipy.sparse.csgraph import breadth_first_order
    if n == 1:
        return np.zeros(1, np.int64)
    a = sp.csr_matrix((np.ones(row.shape[0], np.int8), (row, col)), shape=(n, n))
    order = breadth_first_order(a, 0, directed=False, return_predecessors=False)
    if order.shape[0] < n:                      # disconnected (never for synth corpora): append the rest
        rest = np.setdiff1d(np.arange(n), order)
        order = np.concatenate([order, rest])
    return order.astype(np.int64)


def _eigvecs(adj: np.ndarray, num: int) -> np.ndarray:
    """first `num` eigenvectors (ascending eigenvalue) of D - A, sign-fixed, last one repeated."""
    lap = np.diag(adj.sum(1)) - adj
    _, v = np.linalg.eigh(lap.astype(np.float64))
    out = np.zeros((adj.shape[0], num), np.float64)
    for j in range(num):
        vec = v[:, min(j, v.shape[1] - 1)].copy()
        if vec[0] < 0:
            vec = -vec
        out[:, j] = vec
    return out


def bfs_clusters(c: Corpus, pool_size: int = 10):
    """The synthetic clustering: contiguous chunks of `pool_size` nodes in BFS order from node 0.  Returns
    (cluster_of int64 [sum n], order int64 [sum n]): graph-local cluster ids and every graph's BFS node order."""
    cluster_of = np.zeros(int(c.node_ptr[-1]), np.int64)
    order_all = np.zeros(int(c.node_ptr[-1]), np.int64)
    for g in range(c.num_graphs):
        n0, n1 = int(c.node_ptr[g]), int(c.node_ptr[g + 1])
        e0, e1 = int(c.edge_ptr[g]), int(c.edge_ptr[g + 1])
        n = n1 - n0
        order = _bfs_order(n, c.row[e0:e1], c.col[e0:e1])
        pos = np.empty(n, np.int64); pos[order] = np.arange(n)
        cluster_of[n0:n1] = pos // pool_size
        order_all[n0:n1] = order
    return cluster_of, order_all


def operands_from_clusters(c: Corpus, cluster_of, num_pool_matrix: int = 1, num_pool_final_matrix: int = 1,
                           member_order=None) -> EigenOperands:
    """EigenPooling operands of a corpus for a given clustering (e.g. the reference's SpectralClustering labels,
    coarsen_pooling_with_last_eigen_padding.py:36-60): `cluster_of` [sum n] graph-local cluster ids in [0, nc_g), every
    graph's clusters numbered from 0.  Per cluster, P_j[:, c] = the j-th eigenvector of its unnormalised Laplacian over
    its members listed in ascending node order, or in the order of `member_order` ([sum n], a per-graph permutation of
    the local node ids) when given; the coarsened adjacency and the final pooling follow (module docstring)."""
    cluster_of = np.asarray(cluster_of).reshape(-1)
    if cluster_of.shape[0] != int(c.node_ptr[-1]):
        raise ValueError(f"tsg: cluster_of has {cluster_of.shape[0]} entries, the corpus has {int(c.node_ptr[-1])} nodes")
    if cluster_of.size and not np.issubdtype(cluster_of.dtype, np.integer):
        raise ValueError("tsg: cluster_of must hold integer cluster ids")
    cluster_of = cluster_of.astype(np.int64)
    if cluster_of.size and int(cluster_of.min()) < 0:
        raise ValueError("tsg: cluster ids must be non-negative")
    G = c.num_graphs
    cluster_ptr = np.zeros(G + 1, np.int64)
    pool_w = [np.zeros(int(c.node_ptr[-1]), np.float32) for _ in range(num_pool_matrix)]
    c_rows, c_cols, c_ws, coarse_ptr = [], [], [], np.zeros(G + 1, np.int64)
    final_parts = [[] for _ in range(num_pool_final_matrix)]
    for g in range(G):
        n0, n1 = int(c.node_ptr[g]), int(c.node_ptr[g + 1])
        e0, e1 = int(c.edge_ptr[g]), int(c.edge_ptr[g + 1])
        n = n1 - n0
        row, col = c.row[e0:e1], c.col[e0:e1]
        cl = cluster_of[n0:n1]
        nc = int(cl.max()) + 1 if n else 0
        cluster_ptr[g + 1] = cluster_ptr[g] + nc
        order = np.arange(n, dtype=np.int64) if member_order is None else np.asarray(member_order[n0:n1], np.int64)
        members = order[np.argsort(cl[order], kind="stable")]           # by cluster, `order` within a cluster
        starts = np.searchsorted(cl[members], np.arange(nc + 1))
        adj = np.zeros((n, n), np.float32); adj[row, col] = 1.0
        for k in range(nc):
            nodes = members[starts[k]:starts[k + 1]]
            if nodes.size == 0:
                continue
            ev = _eigvecs(adj[np.ix_(nodes, nodes)], num_pool_matrix)
            for j in range(num_pool_matrix):
                pool_w[j][n0 + nodes] = ev[:, j].astype(np.float32)
        omega = np.zeros((n, nc), np.float32); omega[np.arange(n), cl] = 1.0
        ext = adj * (cl[:, None] != cl[None, :])
        coarse = omega.T @ ext @ omega
        rr, cc = np.nonzero(coarse)
        c_rows.append(rr.astype(np.int64)); c_cols.append(cc.astype(np.int64)); c_ws.append(coarse[rr, cc].astype(np.float32))
        coarse_ptr[g + 1] = coarse_ptr[g] + rr.shape[0]
        if num_pool_final_matrix > 0 and nc > 0:
            ev = _eigvecs((coarse > 0).astype(np.float32), num_pool_final_matrix)
            for j in range(num_pool_final_matrix):
                final_parts[j].append(ev[:, j].astype(np.float32))
    cat = lambda parts, dt: np.concatenate(parts).astype(dt) if parts else np.zeros(0, dt)
    return EigenOperands(cluster_ptr, cluster_of.copy(), pool_w, coarse_ptr, cat(c_rows, np.int64),
                         cat(c_cols, np.int64), cat(c_ws, np.float32), [cat(p, np.float32) for p in final_parts])


def make_operands(c: Corpus, pool_size: int = 10, num_pool_matrix: int = 1, num_pool_final_matrix: int = 1
                  ) -> EigenOperands:
    """Synthetic operands: bfs_clusters, members listed in BFS order (operands_from_clusters)."""
    cluster_of, order = bfs_clusters(c, pool_size)
    return operands_from_clusters(c, cluster_of, num_pool_matrix, num_pool_final_matrix, member_order=order)


def pack_operands(c: Corpus, op: EigenOperands, graph_ids) -> dict:
    """Operands of a packed batch (graphs `graph_ids` in order) as COO lists with batch-global ids:
    pool[j] = (src node, dst cluster, w); coarse = (src cluster, dst cluster, w); final[j] = (src cluster,
    dst graph, w); plus node_ptr / cluster_ptr of the batch."""
    ids = np.asarray(graph_ids, dtype=np.int64)
    n = c.node_ptr[ids + 1] - c.node_ptr[ids]
    nc = op.cluster_ptr[ids + 1] - op.cluster_ptr[ids]
    node_ptr = np.concatenate([[0], np.cumsum(n)]).astype(np.int64)
    cl_ptr = np.concatenate([[0], np.cumsum(nc)]).astype(np.int64)
    from .synth import _ragged_arange
    nidx = _ragged_arange(c.node_ptr[ids], n)
    cidx = _ragged_arange(op.cluster_ptr[ids], nc)
    node_src = np.arange(int(node_ptr[-1]), dtype=np.int64)
    node_dst = op.cluster_of[nidx] + np.repeat(cl_ptr[:-1], n)
    pool = [(node_src, node_dst, w[nidx]) for w in op.pool_w]
    ce = op.coarse_ptr[ids + 1] - op.coarse_ptr[ids]
    eidx = _ragged_arange(op.coarse_ptr[ids], ce)
    off = np.repeat(cl_ptr[:-1], ce)
    coarse = (op.coarse_col[eidx] + off, op.coarse_row[eidx] + off, op.coarse_w[eidx])
    cl_src = np.arange(int(cl_ptr[-1]), dtype=np.int64)
    cl_dst = np.repeat(np.arange(ids.shape[0], dtype=np.int64), nc)
    final = [(cl_src, cl_dst, w[cidx]) for w in op.final_w]
    return dict(node_ptr=node_ptr, cluster_ptr=cl_ptr, pool=pool, coarse=coarse, final=final)
