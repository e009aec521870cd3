"""Device-resident corpus + GPU batch assembly (SURVEY 8f n1).

The reference moves every graph of every triplet host->device each step (and, in the dense
directories, rebuilds 1000x1000 tensors from numpy: 115-125 ms per graph).  Here the corpus is uploaded
once (DD: 1,168 graphs = 14 MB) and a step ships only graph ids; `tsg_pack_batch` writes the packed
batch at HBM speed."""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch

from ._lib import call, ptr, stream_ptr
from .synth import Corpus


class _PinnedRing:
    """Four reusable page-locked int64 staging buffers: a per-step `.pin_memory()` on a fresh tensor is a host
    allocation + registration every call.  A slot is reused only after the upload issued from it has left it."""

    def __init__(self):
        self.slots, self.pos = [None] * 4, -1

    def stage(self, parts, device) -> torch.Tensor:
        need = sum(int(p.shape[0]) for p in parts)
        self.pos = (self.pos + 1) % 4
        slot = self.slots[self.pos]
        if slot is None or slot[0].numel() < need:
            slot = self.slots[self.pos] = [torch.empty(max(need, 1024), dtype=torch.int64, pin_memory=True), None]
        buf, busy = slot
        if busy is not None:
            busy.synchronize()
        host = buf[:need]
        np.concatenate(parts, out=host.numpy())
        dev = host.to(device, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        slot[1] = ev
        return dev


class DeviceCorpus:
    def __init__(self, corpus: Corpus, device, dense_x: np.ndarray | None = None):
        self.device = device
        self.n = np.diff(corpus.node_ptr).astype(np.int64)          # host copies: sizes drive the offsets
        self.e = np.diff(corpus.edge_ptr).astype(np.int64)
        self.num_graphs = corpus.num_graphs
        t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a.astype(dt))).to(device)
        self.node_ptr, self.edge_ptr = t(corpus.node_ptr, np.int64), t(corpus.edge_ptr, np.int64)
        self.row, self.col = t(corpus.row, np.int32), t(corpus.col, np.int32)
        from .synth import is_coalesced_symmetric
        self.coalesced = is_coalesced_symmetric(corpus)      # checked once, here; the kernels re-verify per graph
        if dense_x is None:
            self.label, self.x, self.feat = t(corpus.node_label, np.int32), None, corpus.num_node_labels
        else:
            self.label, self.x, self.feat = None, t(dense_x, np.float32), int(dense_x.shape[1])
        self.y_host = np.ascontiguousarray(corpus.y, dtype=np.int64)      # graph labels (the supervised setting)
        self.y = torch.from_numpy(self.y_host).to(device)
        self.labels_checked = None

    @classmethod
    def from_device(cls, label: torch.Tensor, row: torch.Tensor, col: torch.Tensor, node_ptr_host: np.ndarray,
                    edge_ptr_host: np.ndarray, num_labels: int, coalesced: bool,
                    y: torch.Tensor | None = None) -> "DeviceCorpus":
        """A corpus whose arrays already live in HBM (e.g. a shard assembled on the GPU from a smaller base corpus:
        bench.py's 1 M-graph config-5 corpus); only the two offset arrays come from the host.  `y`: optional int64
        [num_graphs] graph labels on the device."""
        self = cls.__new__(cls)
        self.device = label.device
        self.n = np.diff(node_ptr_host).astype(np.int64); self.e = np.diff(edge_ptr_host).astype(np.int64)
        self.num_graphs = int(self.n.shape[0])
        self.node_ptr = torch.from_numpy(np.ascontiguousarray(node_ptr_host, dtype=np.int64)).to(self.device)
        self.edge_ptr = torch.from_numpy(np.ascontiguousarray(edge_ptr_host, dtype=np.int64)).to(self.device)
        self.row, self.col, self.label, self.x, self.feat = row, col, label, None, int(num_labels)
        self.coalesced = bool(coalesced)
        if y is not None and tuple(y.shape) != (self.num_graphs,):
            raise ValueError(f"tsg: y has shape {tuple(y.shape)}, the corpus has {self.num_graphs} graphs")
        self.y = None if y is None else y.to(device=self.device, dtype=torch.int64).contiguous()
        self.y_host, self.labels_checked = None, None
        return self

    def check_labels(self, num_classes: int) -> None:
        """Raise ValueError unless every graph label lies in [0, num_classes): once per corpus and class count, on the
        host (a device-resident `y` is read back for it once).  An out-of-range label would otherwise reach ATen's
        nll_loss on the autograd path, which stops the process with a device assert."""
        if self.labels_checked == num_classes:
            return
        if self.y is None:
            raise ValueError("tsg: the corpus carries no graph labels (y)")
        y = self.y_host if self.y_host is not None else self.y.cpu().numpy()
        if y.size and (int(y.min()) < 0 or int(y.max()) >= num_classes):
            bad = int(np.flatnonzero((y < 0) | (y >= num_classes))[0])
            raise ValueError(f"tsg: graph {bad} has label {int(y[bad])}, outside [0, {num_classes})")
        self.labels_checked = num_classes

    def offsets(self, ids_host: np.ndarray):
        """Packed offsets for a list of graph ids (host numpy; int64 [B+1] each)."""
        ids = np.asarray(ids_host, dtype=np.int64)
        nptr = np.zeros(ids.shape[0] + 1, np.int64); np.cumsum(self.n[ids], out=nptr[1:])
        eptr = np.zeros(ids.shape[0] + 1, np.int64); np.cumsum(self.e[ids], out=eptr[1:])
        return ids, nptr, eptr

    def _upload(self, parts) -> torch.Tensor:
        """int64 host arrays -> their concatenation on the device, as ONE small upload through the pinned ring."""
        ring = self.__dict__.get("_ring")
        if ring is None:
            ring = self.__dict__["_ring"] = _PinnedRing()
        return ring.stage(parts, self.device)

    def _stage(self, ids_host: np.ndarray):
        """ids + packed offsets of the chosen graphs as ONE small pinned upload: (meta on the device, B, nptr, eptr)."""
        ids, nptr, eptr = self.offsets(ids_host)
        return self._upload([ids, nptr, eptr]), ids.shape[0], nptr, eptr

    def pack(self, ids_host: np.ndarray):
        """-> (x [sum n, F] f32, edge_index [2, sum E] i64, node_ptr_host).  One small H2D (ids + offsets)."""
        return self.pack_staged(*self._stage(ids_host))

    def pack_staged(self, meta: torch.Tensor, B: int, nptr: np.ndarray, eptr: np.ndarray):
        """`pack` when ids + offsets are already on the device (`meta` = [ids | nptr | eptr], int64)."""
        d_ids, d_nptr, d_eptr = meta[:B], meta[B:2 * B + 1], meta[2 * B + 1:]
        N, E = int(nptr[-1]), int(eptr[-1])
        x = torch.empty(N, self.feat, dtype=torch.float32, device=self.device)
        ei = torch.empty(2, E, dtype=torch.int64, device=self.device)
        call("tsg_pack_batch", ptr(d_ids), ptr(d_nptr), ptr(d_eptr), B, ptr(self.node_ptr), ptr(self.edge_ptr),
             ptr(self.row), ptr(self.col), ptr(self.label), ptr(self.x), self.feat, ptr(x), ptr(ei[0]), ptr(ei[1]),
             stream_ptr())
        return x, ei, nptr

    def pack_compact(self, ids_host: np.ndarray):
        """-> (ops.CompactBatch, node_ptr_host): labels + graph-local int32 endpoints of the chosen graphs, gathered
        on the GPU (4N + 8E bytes written; PackedSAGNet consumes the batch without expanding it)."""
        return self.pack_compact_staged(*self._stage(ids_host))

    def pack_compact_staged(self, meta: torch.Tensor, B: int, nptr: np.ndarray, eptr: np.ndarray):
        from .ops import CompactBatch
        if self.label is None:
            raise RuntimeError("tsg: the compact batch form needs categorical node labels (corpus holds dense features)")
        d_ids, d_nptr, d_eptr = meta[:B], meta[B:2 * B + 1], meta[2 * B + 1:]
        N, E = int(nptr[-1]), int(eptr[-1])
        label = torch.empty(N, dtype=torch.int32, device=self.device)
        rc = torch.empty(2, E, dtype=torch.int32, device=self.device)
        call("tsg_pack_batch_compact", ptr(d_ids), ptr(d_nptr), ptr(d_eptr), B, ptr(self.node_ptr), ptr(self.edge_ptr),
             ptr(self.row), ptr(self.col), ptr(self.label), ptr(label), ptr(rc[0]), ptr(rc[1]), stream_ptr())
        return CompactBatch(label, rc[0], rc[1], d_nptr, d_eptr, self.feat, int(np.diff(eptr).max()) if B else 0,
                            self.coalesced), nptr

    def check_dense(self, ids_host, table: torch.Tensor, max_nodes: int) -> np.ndarray:
        """The host-side checks of `pack_dense` (no device work): -> the ids as int64 numpy.  ValueError for a corpus with
        per-node feature rows, an empty id list, an id outside the corpus, a graph larger than `max_nodes` (named: the
        reference drops such graphs when it loads the dataset, load_data.py), a batch without any edge and a table that
        is not [>= max_nodes, F] fp32."""
        if self.x is not None:
            raise ValueError("tsg: pack_dense takes its features from the position-indexed table; this corpus carries "
                             "per-node feature rows (dense_x)")
        ids = np.asarray(ids_host, dtype=np.int64).reshape(-1)
        if ids.size == 0:
            raise ValueError("tsg: pack_dense needs at least one graph id")
        if int(ids.min()) < 0 or int(ids.max()) >= self.num_graphs:
            raise ValueError(f"tsg: graph ids must lie in [0, {self.num_graphs})")
        max_nodes = int(max_nodes)
        if max_nodes < 1:
            raise ValueError("tsg: max_nodes must be at least 1")
        n = self.n[ids]
        if int(n.max()) > max_nodes:
            at = int(np.argmax(n))
            raise ValueError(f"tsg: graph {int(ids[at])} has {int(n[at])} nodes, more than max_nodes = {max_nodes}")
        if int(self.e[ids].sum()) == 0:
            raise ValueError("tsg: the chosen graphs have no edges; the dense encoders' kernels need at least one edge "
                             "per batch (pack edge-free graphs together with others)")
        if table.dim() != 2 or table.size(0) < max_nodes:
            raise ValueError(f"tsg: the feature table must be [max_nodes = {max_nodes}, F], not {tuple(table.shape)}")
        if table.dtype != torch.float32:
            raise ValueError(f"tsg: the feature table must be float32, not {table.dtype}")
        return ids

    def pack_dense(self, ids_host, table: torch.Tensor, max_nodes: int, want_eid: bool = False) -> "DenseBatch":
        """-> DenseBatch: what the packed dense encoders (tsg.dense.PackedGcnEncoder, tsg.gat.PackedGatEncoder,
        tsg.diffpool.PackedSoftPoolEncoder) take for the graphs `ids_host` (duplicates allowed): x = rows of `table`
        ([>= max_nodes, F] fp32 on the device) by node position, the RAW 0/1 CSR of the packed adjacency in both
        orientations (eids with `want_eid`: GAT's backward needs them), graph offsets and has-padded-row flags.
        One small staged upload (ids + offsets), then one launch (K0d, tsg_pack_dense_batch), which verifies the
        coalesced promise per graph: a violation raises at the next tsg.nn.check_fused_status().  A corpus that is not
        coalesced takes the general path with the same result: K0 tsg_pack_batch + K1 build_csr(CSR_RAW)."""
        ids = self.check_dense(ids_host, table, max_nodes)
        return self.pack_dense_staged(*self._stage(ids), table, max_nodes, want_eid)

    def pack_dense_staged(self, meta: torch.Tensor, B: int, nptr: np.ndarray, eptr: np.ndarray, table: torch.Tensor,
                          max_nodes: int, want_eid: bool = False) -> "DenseBatch":
        """`pack_dense` when ids + offsets are already on the device (`meta` = [ids | nptr | eptr], int64) and the ids
        passed `check_dense`."""
        from . import nn as tnn, ops
        d_ids, d_nptr, d_eptr = meta[:B], meta[B:2 * B + 1], meta[2 * B + 1:]
        N, E, F = int(nptr[-1]), int(eptr[-1]), int(table.size(1))
        dev = self.device
        table = table.contiguous()
        x = torch.empty(N, F, dtype=torch.float32, device=dev)
        has_pad = torch.empty(B, dtype=torch.bool, device=dev)
        i32 = dict(dtype=torch.int32, device=dev)
        if self.coalesced:
            rowptr, colidx = torch.empty(N + 1, **i32), torch.empty(E, **i32)
            val = torch.empty(E, dtype=torch.float32, device=dev)
            eid, t_eid = (torch.empty(E, **i32), torch.empty(E, **i32)) if want_eid else (None, None)
            status = tnn._status_word(dev)
            call("tsg_pack_dense_batch", ptr(d_ids), ptr(d_nptr), ptr(d_eptr), B, N, E, ptr(self.node_ptr),
                 ptr(self.edge_ptr), ptr(self.row), ptr(self.col), ptr(table), int(max_nodes), F, ptr(x), ptr(has_pad),
                 ptr(rowptr), ptr(colidx), ptr(val), ptr(eid), ptr(t_eid), ptr(status), stream_ptr())
            # symmetric lists: the src-major orientation is the same arrays; only the eids differ
            csr = ops.CSR(rowptr, colidx, val, eid, rowptr, colidx, val, t_eid, N)
        else:
            _, ei, _ = self.pack_staged(meta, B, nptr, eptr)
            csr = ops.build_csr(ops.EdgeList.from_edge_index(ei), N, mode=ops.CSR_RAW, want_eid=want_eid)
            call("tsg_pack_dense_batch", ptr(d_ids), ptr(d_nptr), ptr(d_eptr), B, N, E, ptr(self.node_ptr),
                 ptr(self.edge_ptr), None, None, ptr(table), int(max_nodes), F, ptr(x), ptr(has_pad),
                 None, None, None, None, None, None, stream_ptr())
        return DenseBatch(x, csr, d_nptr, has_pad, nptr, int(max_nodes))

    def attach_eigen(self, operands) -> None:
        """Make the EigenPooling operands of this corpus (tsg.eigen_synth.EigenOperands: make_operands, or
        operands_from_clusters for a clustering of your own) resident in HBM for `pack_eigen`.  Checked on the host
        against the corpus: array lengths, the cluster and coarse-entry offsets (1 <= clusters <= nodes for every graph
        with nodes, none for an empty one) and J >= 1.  What the kernel relies on per graph -- cluster ids in range, the
        coarse list sorted, loop free and symmetric -- is verified on the device at every pack (status bit 16).
        Uploaded once; the per-graph cluster and coarse-entry counts stay on the host for the packed offsets."""
        G, Nt = self.num_graphs, int(self.n.sum())
        i64 = lambda a: np.ascontiguousarray(np.asarray(a), dtype=np.int64).reshape(-1)
        cptr, qptr = i64(operands.cluster_ptr), i64(operands.coarse_ptr)
        for name, p in (("cluster_ptr", cptr), ("coarse_ptr", qptr)):
            if p.shape[0] != G + 1 or int(p[0]) != 0 or (np.diff(p) < 0).any():
                raise ValueError(f"tsg: {name} must be non-decreasing offsets [num_graphs + 1 = {G + 1}] from 0")
        nc = np.diff(cptr)
        bad = np.flatnonzero(((self.n > 0) & ((nc < 1) | (nc > self.n))) | ((self.n == 0) & (nc != 0)))
        if bad.size:
            g = int(bad[0])
            raise ValueError(f"tsg: graph {g} has {int(self.n[g])} nodes and {int(nc[g])} clusters; every graph with "
                             "nodes needs between 1 and that many clusters")
        NCt, ECt = int(cptr[-1]), int(qptr[-1])
        pool_w, final_w = list(operands.pool_w), list(operands.final_w)
        if len(pool_w) < 1:
            raise ValueError("tsg: the operands carry no pooling matrix (J = 0)")
        lens = [("cluster_of", operands.cluster_of, Nt), ("coarse_row", operands.coarse_row, ECt),
                ("coarse_col", operands.coarse_col, ECt), ("coarse_w", operands.coarse_w, ECt)]
        lens += [(f"pool_w[{j}]", w, Nt) for j, w in enumerate(pool_w)]
        lens += [(f"final_w[{j}]", w, NCt) for j, w in enumerate(final_w)]
        for name, a, want in lens:
            if np.asarray(a).reshape(-1).shape[0] != want:
                raise ValueError(f"tsg: {name} has {np.asarray(a).size} entries, the corpus needs {want}")
        if max(NCt, ECt, Nt) >= 2 ** 31:
            raise ValueError("tsg: the operands exceed 32-bit indexing")
        t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(np.asarray(a), dtype=dt).reshape(-1)).to(self.device)
        stack = lambda ws, m: (torch.from_numpy(np.ascontiguousarray(np.stack([np.asarray(w, np.float32).reshape(-1)
                               for w in ws]))).to(self.device) if ws else torch.zeros(1, m, dtype=torch.float32,
                               device=self.device))
        self.eigen = dict(cluster_ptr=t(cptr, np.int64), coarse_ptr=t(qptr, np.int64),
                          cluster_of=t(operands.cluster_of, np.int32), coarse_row=t(operands.coarse_row, np.int32),
                          coarse_col=t(operands.coarse_col, np.int32), coarse_w=t(operands.coarse_w, np.float32),
                          pool_w=stack(pool_w, Nt), final_w=stack(final_w, NCt), J=len(pool_w), Jf=len(final_w),
                          nc=nc, ncoarse=np.diff(qptr))

    def build_eigen(self, pool_size: int = 10, num_pool_matrix: int = 1, num_pool_final_matrix: int = 1,
                    cluster_of=None, chunk_size: int = 1 << 24) -> int:
        """Build this corpus's EigenPooling operands on the GPU (K17 + K11's per-cluster eigensolver) and leave them as
        `attach_eigen` does.  Without `cluster_of`: the device form of eigen_synth.make_operands(corpus, pool_size,
        num_pool_matrix, num_pool_final_matrix) -- BFS chunks of `pool_size` nodes, members in BFS order.  With
        `cluster_of` (integer [sum n] graph-local ids, numpy or a tensor): the device form of operands_from_clusters,
        members in ascending node order; clusters may have at most TSG_EIG_MAX = 32 members, ids lie in [0, n).
        Works on `from_device` corpora (no host copy of the corpus); graphs are processed in chunks of about
        `chunk_size` nodes + edges, so scratch memory does not grow with the corpus.  One device-to-host read of the
        per-graph cluster and coarse-entry counts; the final pooling of graphs with more than TSG_EIGEN_FINAL_MAX = 112
        clusters is computed on the host from their coarse lists (eigen_synth._eigvecs) and uploaded.  Returns the
        number of such graphs.  Nothing collective: each rank builds its own shard.
        Integer arrays equal the host operands exactly.  Eigenvectors of simple eigenvalues match the host's; where an
        eigenvalue is repeated, the vector is another unit vector of the same eigenspace (sign and repeat rules kept),
        so training from a device build follows a different trajectory than from host operands.
        ValueError, before any device work, for a corpus that is not coalesced and symmetric (attach_eigen takes host
        operands for those), a dense_x corpus, pool_size outside [1, 32], J < 1 or Jf < 0, a cluster_of of the wrong
        length or with a negative id, and a graph of more than TSG_EIGEN_BUILD_MAX_NODES = 19,370 nodes; after the
        device work (nothing attached) for a label >= its graph's node count, a cluster of more than 32 members and an
        edge list that breaks the coalesced promise."""
        from . import eigen_synth
        max_nodes_cap, final_cap, i32_max = 19370, 112, 2 ** 31 - 1
        G, Nt, Et = self.num_graphs, int(self.n.sum()), int(self.e.sum())
        ps, J, Jf = int(pool_size), int(num_pool_matrix), int(num_pool_final_matrix)
        if not self.coalesced:
            raise ValueError("tsg: build_eigen needs a coalesced, symmetric corpus; build the operands on the host "
                             "(eigen_synth) and attach_eigen them")
        if self.x is not None:
            raise ValueError("tsg: build_eigen is for one-hot node label corpora; this one carries per-node feature rows "
                             "(dense_x)")
        if not 1 <= ps <= 32:
            raise ValueError(f"tsg: pool_size = {ps}, outside [1, 32]")
        if J < 1 or Jf < 0:
            raise ValueError(f"tsg: num_pool_matrix = {J} (>= 1) and num_pool_final_matrix = {Jf} (>= 0)")
        if G and int(self.n.max()) > max_nodes_cap:
            g = int(np.argmax(self.n))
            raise ValueError(f"tsg: graph {g} has {int(self.n[g])} nodes, more than build_eigen's {max_nodes_cap}")
        if Nt + Et > i32_max:
            raise ValueError("tsg: the corpus exceeds 32-bit indexing")
        dev = self.device
        i32 = dict(dtype=torch.int32, device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        labels = None
        if cluster_of is not None:
            if isinstance(cluster_of, torch.Tensor):
                if cluster_of.numel() != Nt:
                    raise ValueError(f"tsg: cluster_of has {cluster_of.numel()} entries, the corpus has {Nt} nodes")
                if cluster_of.is_floating_point() or cluster_of.is_complex() or cluster_of.dtype == torch.bool:
                    raise ValueError("tsg: cluster_of must hold integer cluster ids")
                if Nt and int(cluster_of.min()) < 0:
                    raise ValueError("tsg: cluster ids must be non-negative")
                labels = cluster_of.reshape(-1).clamp(max=i32_max).to(**i32, copy=True)
            else:
                host = np.asarray(cluster_of).reshape(-1)
                if host.shape[0] != Nt:
                    raise ValueError(f"tsg: cluster_of has {host.shape[0]} entries, the corpus has {Nt} nodes")
                if host.size and not np.issubdtype(host.dtype, np.integer):
                    raise ValueError("tsg: cluster_of must hold integer cluster ids")
                if host.size and int(host.min()) < 0:
                    raise ValueError("tsg: cluster ids must be non-negative")
                labels = torch.from_numpy(np.clip(host, 0, i32_max).astype(np.int32)).to(dev)

        nptr = np.zeros(G + 1, np.int64); np.cumsum(self.n, out=nptr[1:])
        eptr = np.zeros(G + 1, np.int64); np.cumsum(self.e, out=eptr[1:])
        w = self.n + self.e
        cid = (np.cumsum(w) - w) // max(int(chunk_size), 1)
        starts = np.concatenate([[0], np.flatnonzero(np.diff(cid)) + 1]) if G else np.zeros(0, np.int64)
        chunks = [(int(a), int(b)) for a, b in zip(starts, np.append(starts[1:], G))]
        cap_n = max([int(nptr[b] - nptr[a]) for a, b in chunks], default=0)
        cap_e = max([int(eptr[b] - eptr[a]) for a, b in chunks], default=0)
        rowptr, colidx = torch.empty(cap_n + 1, **i32), torch.empty(max(cap_e, 1), **i32)
        cluster_g, member_ptr, member = torch.empty(max(cap_n, 1), **i32), torch.empty(cap_n + 1, **i32), \
            torch.empty(max(cap_n, 1), **i32)
        pool_val, pool_nodes = torch.empty(max(J * cap_n, 1), **f32), torch.empty(max(J * cap_n, 1), **f32)
        row_off = torch.empty(max(cap_n, 1), **i32)
        counts = torch.empty(2 * G + 4, **i32)          # clusters [G] | coarse entries [G] | status [4]
        nc_d, nq_d, status = counts[:G], counts[G:2 * G], counts[2 * G:]
        status.fill_(i32_max)
        cl = labels if labels is not None else torch.empty(max(Nt, 1), **i32)
        pool_w = torch.empty(J, Nt, **f32)
        st = stream_ptr()
        corpus = (ptr(self.node_ptr), ptr(self.edge_ptr), ptr(self.row), ptr(self.col))
        chunk_bufs = (ptr(rowptr), ptr(colidx), ptr(cluster_g), ptr(member_ptr), ptr(member), ptr(status))

        def group(g0, g1, nc_out):
            Nc, Ec = int(nptr[g1] - nptr[g0]), int(eptr[g1] - eptr[g0])
            call("tsg_eigen_group_clusters", *corpus, g0, g1 - g0, Nc, Ec, int(self.n[g0:g1].max()), ptr(cl), nc_out,
                 *chunk_bufs, st)

        def coarse(g0, g1, write):
            out = (ptr(row_off), None, ptr(d_qptr), ptr(coarse_row), ptr(coarse_col), ptr(coarse_w)) if write else \
                (None, ptr(nq_d), None, None, None, None)
            call("tsg_eigen_coarse", ptr(self.node_ptr), g0, g1 - g0, ptr(nc_d), ptr(rowptr), ptr(colidx),
                 ptr(cluster_g), ptr(member_ptr), ptr(member), *out, st)

        # pass 1: clusters, per-cluster eigenvectors (K11), coarse-entry counts
        for g0, g1 in chunks:
            n0, n1 = int(nptr[g0]), int(nptr[g1])
            Nc, Ec = n1 - n0, int(eptr[g1] - eptr[g0])
            if labels is None:
                call("tsg_eigen_bfs_clusters", *corpus, g0, g1 - g0, Nc, Ec, int(self.n[g0:g1].max()), ps, ptr(cl),
                     ptr(nc_d), *chunk_bufs, st)
            else:
                group(g0, g1, ptr(nc_d))
            if Nc:
                call("tsg_eigpool_build", ptr(rowptr), ptr(colidx), None, ptr(cluster_g), ptr(member_ptr), ptr(member),
                     Nc, Nc, J, ptr(pool_val), ptr(pool_nodes), None, ptr(status[3:]), st)
                pool_w[:, n0:n1].copy_(pool_nodes[:J * Nc].view(J, Nc))
            coarse(g0, g1, False)
        host = counts.cpu().numpy()
        bad = host[2 * G:2 * G + 3]
        if bad[0] != i32_max:
            raise ValueError(f"tsg: graph {int(bad[0])}'s edge list is not coalesced and symmetric")
        if bad[2] != i32_max:
            g = int(bad[2])
            raise ValueError(f"tsg: graph {g} has a cluster id outside [0, {int(self.n[g])}) (at most one cluster per "
                             "node)")
        if bad[1] != i32_max:
            raise ValueError(f"tsg: graph {int(bad[1])} has a cluster of more than 32 members")
        nc, ncoarse = host[:G].astype(np.int64), host[G:2 * G].astype(np.int64)
        cptr = np.zeros(G + 1, np.int64); np.cumsum(nc, out=cptr[1:])
        qptr = np.zeros(G + 1, np.int64); np.cumsum(ncoarse, out=qptr[1:])
        NCt, ECt = int(cptr[-1]), int(qptr[-1])
        if NCt + ECt > i32_max:
            raise ValueError("tsg: the operands exceed 32-bit indexing")
        t64 = lambda a: torch.from_numpy(a).to(dev)
        d_cptr, d_qptr = t64(cptr), t64(qptr)
        coarse_row, coarse_col, coarse_w = torch.empty(ECt, **i32), torch.empty(ECt, **i32), torch.empty(ECt, **f32)
        final_w = torch.empty(Jf, NCt, **f32) if Jf else torch.zeros(1, NCt, **f32)

        # pass 2: the coarse lists at their corpus offsets, then the final pooling
        for g0, g1 in chunks:
            if ECt:
                group(g0, g1, None)
                coarse(g0, g1, True)
            for lo, hi in ((0, 32), (32, 64), (64, final_cap)) if Jf else ():     # shared memory per size class
                sel = nc[g0:g1][(nc[g0:g1] > lo) & (nc[g0:g1] <= hi)]
                if sel.size:
                    call("tsg_eigen_final", ptr(d_cptr), ptr(d_qptr), ptr(coarse_row), ptr(coarse_col), g0, g1 - g0,
                         lo, int(sel.max()), Jf, ptr(final_w), NCt, st)
        fallback = np.flatnonzero(nc > final_cap) if Jf else np.zeros(0, np.int64)
        if fallback.size:
            from .synth import _ragged_arange
            idx = torch.from_numpy(_ragged_arange(qptr[fallback], ncoarse[fallback])).to(dev)
            rows, cols = coarse_row[idx].cpu().numpy(), coarse_col[idx].cpu().numpy()
            o = 0
            for g in fallback.tolist():
                k, m = int(nc[g]), int(ncoarse[g])
                adj = np.zeros((k, k), np.float32)
                adj[rows[o:o + m], cols[o:o + m]] = 1.0
                o += m
                ev = eigen_synth._eigvecs(adj, Jf)
                final_w[:, int(cptr[g]):int(cptr[g + 1])] = torch.from_numpy(np.ascontiguousarray(ev.T, np.float32)).to(dev)
        self.eigen = dict(cluster_ptr=d_cptr, coarse_ptr=d_qptr, cluster_of=cl[:Nt], coarse_row=coarse_row,
                          coarse_col=coarse_col, coarse_w=coarse_w, pool_w=pool_w, final_w=final_w, J=J, Jf=Jf, nc=nc,
                          ncoarse=ncoarse)
        return int(fallback.size)

    def check_eigen(self, ids_host, max_nodes: int, num_pool_matrix=None, num_pool_final_matrix=None):
        """The host-side checks of `pack_eigen` (no device work): -> (ids int64 numpy, J, Jf).  ValueError when no
        operands are attached, for a corpus with per-node feature rows, an empty id list, an id outside the corpus, a
        graph larger than `max_nodes` (named), J / Jf beyond what the operands carry and a batch without any edge."""
        op = self.__dict__.get("eigen")
        if op is None:
            raise ValueError("tsg: no EigenPooling operands attached to this corpus (DeviceCorpus.attach_eigen)")
        if self.x is not None:
            raise ValueError("tsg: pack_eigen takes one-hot node labels; this corpus carries per-node feature rows "
                             "(dense_x)")
        ids = np.asarray(ids_host, dtype=np.int64).reshape(-1)
        if ids.size == 0:
            raise ValueError("tsg: pack_eigen needs at least one graph id")
        if int(ids.min()) < 0 or int(ids.max()) >= self.num_graphs:
            raise ValueError(f"tsg: graph ids must lie in [0, {self.num_graphs})")
        max_nodes = int(max_nodes)
        if max_nodes < 1:
            raise ValueError("tsg: max_nodes must be at least 1")
        n = self.n[ids]
        if int(n.max()) > max_nodes:
            at = int(np.argmax(n))
            raise ValueError(f"tsg: graph {int(ids[at])} has {int(n[at])} nodes, more than max_nodes = {max_nodes}")
        J = op["J"] if num_pool_matrix is None else int(num_pool_matrix)
        Jf = op["Jf"] if num_pool_final_matrix is None else int(num_pool_final_matrix)
        if not 1 <= J <= op["J"]:
            raise ValueError(f"tsg: num_pool_matrix = {J}; the attached operands carry 1 .. {op['J']}")
        if not 0 <= Jf <= op["Jf"]:
            raise ValueError(f"tsg: num_pool_final_matrix = {Jf}; the attached operands carry 0 .. {op['Jf']}")
        if int(self.e[ids].sum()) == 0:
            raise ValueError("tsg: the chosen graphs have no edges; the encoder's kernels need at least one adjacency "
                             "edge per batch (pack edge-free graphs together with others)")
        return ids, J, Jf

    def pack_eigen(self, ids_host, max_nodes: int, num_pool_matrix=None, num_pool_final_matrix=None) -> "EigenBatch":
        """-> EigenBatch: everything tsg.dense.PackedWaveEncoder takes for the graphs `ids_host` (duplicates allowed),
        from the operands attached with `attach_eigen`: one-hot x, the RAW adjacency CSR, P_j^T for j < J, the
        coarsened adjacency, the final pooling for j < Jf (defaults: all the operands carry), the offsets and the
        per-level padded-row flags for `max_nodes`.  One small staged upload (ids + node / edge / cluster / coarse-entry
        offsets), then one launch (K0e, tsg_pack_eigen_batch), which verifies the adjacency and operand promises per
        graph: a violation raises at the next tsg.nn.check_fused_status().  A corpus that is not coalesced gets its
        adjacency from K0 tsg_pack_batch + K1 build_csr(CSR_RAW) instead, with the same result.
        A batch whose graphs are single clusters has an empty coarsened adjacency (rowptr all zero; its colidx / val
        hold one zero slot that no row reaches, because K2 takes no NULL array): the pooled tower then sees no edges,
        each cluster row being its bias-derived epilogue, as with the reference's zero coarse matrix."""
        ids, J, Jf = self.check_eigen(ids_host, max_nodes, num_pool_matrix, num_pool_final_matrix)
        return self.pack_eigen_checked(ids, max_nodes, J, Jf)

    def pack_eigen_checked(self, ids: np.ndarray, max_nodes: int, J: int, Jf: int) -> "EigenBatch":
        """`pack_eigen` for ids, J and Jf that passed `check_eigen`."""
        from . import nn as tnn, ops
        op = self.eigen
        ids, nptr, eptr = self.offsets(ids)
        B = ids.shape[0]
        cptr = np.zeros(B + 1, np.int64); np.cumsum(op["nc"][ids], out=cptr[1:])
        qptr = np.zeros(B + 1, np.int64); np.cumsum(op["ncoarse"][ids], out=qptr[1:])
        meta = self._upload([ids, nptr, eptr, cptr, qptr])
        d_ids, d_nptr, d_eptr = meta[:B], meta[B:2 * B + 1], meta[2 * B + 1:3 * B + 2]
        d_cptr, d_qptr = meta[3 * B + 2:4 * B + 3], meta[4 * B + 3:]
        N, E, NC, EC = int(nptr[-1]), int(eptr[-1]), int(cptr[-1]), int(qptr[-1])
        dev = self.device
        i32 = dict(dtype=torch.int32, device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        x = torch.empty(N, self.feat, **f32)
        has_pad = torch.empty(3, B, dtype=torch.bool, device=dev)
        member_ptr, member, node_iota, node_cluster = (torch.empty(NC + 1, **i32), torch.empty(N, **i32),
                                                       torch.empty(N + 1, **i32), torch.empty(N, **i32))
        pool_val, pool_val_nodes = torch.empty(J, N, **f32), torch.empty(J, N, **f32)
        coarse_rowptr = torch.empty(NC + 1, **i32)
        if EC:
            coarse_colidx, coarse_val = torch.empty(EC, **i32), torch.empty(EC, **f32)
        else:   # single-cluster graphs only: one zero slot that rowptr never reaches (K2 takes no NULL colidx)
            coarse_colidx, coarse_val = torch.zeros(1, **i32), torch.zeros(1, **f32)
        if Jf > 0:
            final_rowptr, cluster_iota = torch.empty(B + 1, **i32), torch.empty(NC + 1, **i32)
            cluster_graph, final_val = torch.empty(NC, **i32), torch.empty(Jf, NC, **f32)
        else:
            final_rowptr = cluster_iota = cluster_graph = final_val = None
        graph_iota = torch.empty(B + 1, dtype=torch.int64, device=dev)
        status = tnn._status_word(dev)
        if self.coalesced:
            rowptr, colidx, val = torch.empty(N + 1, **i32), torch.empty(E, **i32), torch.empty(E, **f32)
            adj = (ptr(rowptr), ptr(colidx), ptr(val))
        else:
            _, ei, _ = self.pack_staged(meta[:3 * B + 2], B, nptr, eptr)
            csr = ops.build_csr(ops.EdgeList.from_edge_index(ei), N, mode=ops.CSR_RAW)
            adj = (None, None, None)
        call("tsg_pack_eigen_batch", ptr(d_ids), ptr(d_nptr), ptr(d_eptr), ptr(d_cptr), ptr(d_qptr), B, N, E, NC, EC,
             ptr(self.node_ptr), ptr(self.edge_ptr), ptr(self.label), ptr(self.row), ptr(self.col), self.feat,
             ptr(op["cluster_ptr"]), ptr(op["coarse_ptr"]), ptr(op["cluster_of"]), ptr(op["pool_w"]),
             int(op["pool_w"].size(1)), J, ptr(op["coarse_row"]), ptr(op["coarse_col"]), ptr(op["coarse_w"]),
             ptr(op["final_w"]), int(op["final_w"].size(1)), Jf, int(max_nodes), ptr(x), ptr(has_pad), *adj,
             ptr(member_ptr), ptr(member), ptr(pool_val), ptr(node_iota), ptr(node_cluster), ptr(pool_val_nodes),
             ptr(coarse_rowptr), ptr(coarse_colidx), ptr(coarse_val), ptr(final_rowptr), ptr(cluster_iota),
             ptr(cluster_graph), ptr(final_val), ptr(graph_iota), ptr(status), stream_ptr())
        if self.coalesced:       # symmetric lists: the transposed orientation is the same arrays
            csr = ops.CSR(rowptr, colidx, val, None, rowptr, colidx, val, None, N)
        pool = [ops.CSR(member_ptr, member, pool_val[j], None, node_iota, node_cluster, pool_val_nodes[j], None, NC)
                for j in range(J)]
        coarse = ops.CSR(coarse_rowptr, coarse_colidx, coarse_val, None, coarse_rowptr, coarse_colidx, coarse_val,
                         None, NC)
        final = [ops.CSR(final_rowptr, cluster_iota[:NC], final_val[j], None, cluster_iota, cluster_graph, final_val[j],
                         None, B) for j in range(Jf)]
        return EigenBatch(x, csr, d_nptr, pool, coarse, d_cptr, final, graph_iota, has_pad, nptr, cptr, int(max_nodes))


@dataclass
class EigenBatch:
    """A packed batch in the form tsg.dense.PackedWaveEncoder takes (DeviceCorpus.pack_eigen).  Each CSR equals what the
    host path builds (tile_ptr / tma_ok unset): `csr` the RAW adjacency (ops.build_csr(CSR_RAW)), `pool[j]` P_j^T and
    `final[j]` the final pooling (dense.build_rect_csr), `coarse` the coarsened adjacency (build_csr(CSR_RAW,
    edge_weight)).  `graph_ptr` / `cluster_ptr` / `final_ptr` are the int64 row offsets of level 0, the pooled level and
    the final level, and `has_pad` bool [3, B] the padded-row flags of the three readouts, all on the device;
    `node_ptr_host` / `cluster_ptr_host` are the first two offsets in host memory."""
    x: torch.Tensor
    csr: "ops.CSR"
    graph_ptr: torch.Tensor
    pool: list
    coarse: "ops.CSR"
    cluster_ptr: torch.Tensor
    final: list
    final_ptr: torch.Tensor
    has_pad: torch.Tensor
    node_ptr_host: np.ndarray
    cluster_ptr_host: np.ndarray
    max_nodes: int

    def readout_args(self):
        """The positional arguments of PackedWaveEncoder.forward / readout (one pooling level), and its has_pad."""
        return ((self.x, self.csr, self.graph_ptr, [self.pool, self.final], [self.coarse], [self.cluster_ptr],
                 self.final_ptr), dict(has_pad=[self.has_pad[0], self.has_pad[1], self.has_pad[2]]))


@dataclass
class DenseBatch:
    """A packed batch in the form the dense encoders take (DeviceCorpus.pack_dense).  `csr` is what
    ops.build_csr(CSR_RAW) returns for the expanded edge list (tile_ptr / tma_ok unset); `graph_ptr` int64 [B+1] and
    `has_pad` bool [B] (n_b < max_nodes) live on the device, `node_ptr_host` is the same offsets in host memory."""
    x: torch.Tensor
    csr: "ops.CSR"
    graph_ptr: torch.Tensor
    has_pad: torch.Tensor
    node_ptr_host: np.ndarray
    max_nodes: int


class DeviceRagged:
    """Per-graph variable-length rows of 32-bit values resident in HBM (cluster labels per node, pooling weights per
    cluster, ...), gathered by graph id with the same kernel as the corpus itself (K0 compact with no edges)."""

    def __init__(self, ptr_host: np.ndarray, values: torch.Tensor):
        assert values.dtype in (torch.int32, torch.float32)
        self.device = values.device
        self.len = np.diff(ptr_host).astype(np.int64)
        self.ptr = torch.from_numpy(np.ascontiguousarray(ptr_host, dtype=np.int64)).to(self.device)
        self.values = values.contiguous()
        self._zero_ptr = torch.zeros(self.len.shape[0] + 1, dtype=torch.int64, device=self.device)
        self._dummy = torch.zeros(4, dtype=torch.int32, device=self.device)
        self._ring = _PinnedRing()

    def gather(self, ids_host: np.ndarray):
        """-> (values of the chosen graphs, concatenated; their offsets on the host [B+1])."""
        ids = np.asarray(ids_host, dtype=np.int64)
        B = ids.shape[0]
        optr = np.zeros(B + 1, np.int64); np.cumsum(self.len[ids], out=optr[1:])
        meta = self._ring.stage([ids, optr, np.zeros(B + 1, np.int64)], self.device)
        out = torch.empty(int(optr[-1]), dtype=torch.int32, device=self.device)
        call("tsg_pack_batch_compact", ptr(meta[:B]), ptr(meta[B:2 * B + 1]), ptr(meta[2 * B + 1:]), B, ptr(self.ptr),
             ptr(self._zero_ptr), ptr(self._dummy), ptr(self._dummy), ptr(self.values.view(torch.int32)), ptr(out),
             ptr(self._dummy), ptr(self._dummy), stream_ptr())
        return (out.view(self.values.dtype), optr)


def compact_host_batch(corpus: Corpus, graph_ids, triplets: np.ndarray, pin: bool | None = None,
                       coalesced: bool | None = None) -> dict:
    """One step's HOST batch in the compact form `TripletTrainer.run_from_host_compact` consumes: the chosen graphs'
    node labels (int32), graph-local edge endpoints (int32), node / edge offsets (int64 numpy) and the triplet index
    rows [T, 3] into `graph_ids` (int64).  What a TU file stores, nothing expanded: 4 n + 8 E bytes per graph.
    `pin` (default: when CUDA is available) page-locks the tensors so the feeder's H2D copies are asynchronous."""
    from .synth import select
    sel = select(corpus, np.asarray(graph_ids, dtype=np.int64))
    n_max = int(np.diff(sel.node_ptr).max()) if sel.num_graphs else 0
    if n_max >= 2 ** 31:
        raise ValueError("tsg: graph too large for int32 local node ids")
    trip = np.ascontiguousarray(np.asarray(triplets, dtype=np.int64).reshape(-1, 3))
    if trip.size and (trip.min() < 0 or trip.max() >= sel.num_graphs):
        raise ValueError("tsg: triplet index outside the batch")
    pin = torch.cuda.is_available() if pin is None else pin
    t = lambda a: (torch.from_numpy(np.ascontiguousarray(a)).pin_memory() if pin else torch.from_numpy(np.ascontiguousarray(a)))
    if coalesced is None:
        from .synth import is_coalesced_symmetric
        coalesced = is_coalesced_symmetric(sel)
    return dict(label=t(sel.node_label.astype(np.int32)), row=t(sel.row.astype(np.int32)), col=t(sel.col.astype(np.int32)),
                node_ptr=sel.node_ptr.astype(np.int64).copy(), edge_ptr=sel.edge_ptr.astype(np.int64).copy(),
                triplets=t(trip), coalesced=bool(coalesced))
