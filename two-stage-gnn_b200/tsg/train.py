"""2stg training step over packed batches: the public call a user of this framework makes (ClassifierTrainer, at the
end, is the supervised "original" setting of Code/sag/train.py).

Mirrors the loop of Code/sag/train_triplet.py:198-214 (TNet forward -> MarginRankingLoss ->
backward -> Adam step) with two differences that are the point of this framework: the step runs
ONE packed forward over all 3T graphs of T triplets instead of 3 single-graph forwards per
triplet, and it is data-parallel: every rank embeds its own graphs and evaluates its own triplets; ONE
all-reduce (NCCL) per step of the flat bucket [T_r * gradients, T_r * loss, T_r] yields the global-batch mean
loss and its gradient on every rank.  Graphs are independent, so there is no other exchange step
(`all_gather_rows` stays for triplets that reference graphs of other ranks).
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch
import torch.distributed as dist
import torch.nn.functional as F

from . import ops


class _AllGatherRows(torch.autograd.Function):
    """emb_local [M, D] -> emb_global [world*M, D].  Every rank evaluates the SAME global loss on
    the gathered matrix, so d(loss)/d(emb_global) is complete on every rank and the backward is a
    slice (no reduce-scatter needed)."""

    @staticmethod
    def forward(ctx, emb, group):
        world = dist.get_world_size(group)
        ctx.rank, ctx.m = dist.get_rank(group), emb.size(0)
        out = torch.empty(world * emb.size(0), emb.size(1), dtype=emb.dtype, device=emb.device)
        dist.all_gather_into_tensor(out, emb.contiguous(), group=group)
        return out

    @staticmethod
    def backward(ctx, g):
        return g[ctx.rank * ctx.m:(ctx.rank + 1) * ctx.m].contiguous(), None


def all_gather_rows(emb: torch.Tensor, group=None) -> torch.Tensor:
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return emb
    return _AllGatherRows.apply(emb, group)


def all_reduce_grads(params, group=None) -> None:
    """One flat-bucket all-reduce(SUM) of every parameter gradient (33-361 KB: latency bound)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return
    grads = [p.grad for p in params if p.grad is not None]
    if not grads:
        return
    flat = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    views, off = [], 0
    for g in grads:
        n = g.numel()
        views.append(flat[off:off + n].view_as(g)); off += n
    torch._foreach_copy_(grads, views)          # one multi-tensor kernel instead of one copy per parameter


def all_reduce_grads_and_loss(params, loss_local: torch.Tensor, num_local: int, group=None) -> torch.Tensor:
    """The step's ONE collective when every rank's triplets index its own graphs.  `loss_local` is the MEAN hinge over
    this rank's `num_local` triplets and the parameters hold its gradient; the global batch's mean loss is
    sum_r(T_r * loss_r) / sum_r(T_r) and its gradient the same combination of the per-rank gradients, so one
    all-reduce(SUM) of [T_r * grads..., T_r * loss_r, T_r] carries everything -- no embedding all-gather, no triplet
    all-gather, nothing to wait for before the backward pass.  Returns the global mean loss (on the device)."""
    grads = [p.grad for p in params if p.grad is not None]
    tail = torch.stack([loss_local.detach().reshape(()), torch.ones((), dtype=loss_local.dtype, device=loss_local.device)])
    flat = torch.cat([g.reshape(-1) for g in grads] + [tail])
    flat.mul_(float(num_local))
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    flat.div_(flat[-1].clone())
    views, off = [], 0
    for g in grads:
        n = g.numel()
        views.append(flat[off:off + n].view_as(g)); off += n
    if grads:
        torch._foreach_copy_(grads, views)
    return flat[-2]


class CapturedStep:
    """A whole training step (forward through the tsg operators, loss, backward, clipping, optimiser) captured ONCE into a
    CUDA graph and replayed -- for steps whose shapes do not change between iterations (the reference's "original"
    setting trains on the same packed corpus every epoch, Code/sage+gat+diffpool/train.py:85-152): ~200 launches of a few
    microseconds each become one graph launch.  This is what the C ABI's contract buys (include/tsg.h: every compute
    entry point only enqueues on the caller's stream, never allocates, never synchronises; tsg_init_device() runs
    before the capture): the library's kernels, memsets and last-CTA reduction tickets are all capturable.

    `body()` must read its inputs from tensors that stay alive and in place (update them with copy_()), use an optimiser
    built with `capturable=True`, and return a tensor (the loss); its value after each replay() is in `.out`."""

    def __init__(self, body, warmup: int = 3):
        from . import _lib
        _lib.init_device()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):                    # warm-up on a side stream (allocator, lazy inits, autotuned paths)
            for _ in range(warmup):
                body()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out = body()

    def replay(self) -> torch.Tensor:
        self.graph.replay()
        return self.out


def _check_status():
    from . import nn as _nn
    _nn.check_fused_status()


def _all_reduce_native_flat(model, num_local: int, group) -> None:
    """The native step's ONE collective: the model's flat buffer [grads | loss | weight] becomes
    [n_r * grads, n_r * loss, n_r], is summed over the ranks and divided by sum_r n_r -- the global batch's mean loss and
    its gradient, in place (n_r = this rank's triplets or graphs)."""
    flat, _ = model._flat_grads()
    flat[-1:].fill_(1.0)           # (NOT flat[-1] = 1.0: a Python scalar store is a blocking H2D copy -- measured
                                   # 1.2 ms of host stall per step, 1.43 -> 1.87 ms at any N > 1: profiles/tools/scale_probe2.py)
    flat.mul_(float(num_local))
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    flat.div_(flat[-1].clone())


def _native_ok(model, x, edge_index, node_ptr_host) -> bool:
    """The batch runs on the model's native (K14) entries: compact input the model's shape checks accept."""
    return (edge_index is None and getattr(model, "native_step_supported", None) is not None
            and model.native_step_supported(x, node_ptr_host))


def gather_score_reduce(train_emb: torch.Tensor, train_y: torch.Tensor, query_emb: torch.Tensor, query_y: torch.Tensor,
                        score, group=None) -> torch.Tensor:
    """Stage-2 scoring of a sharded evaluation: every rank holds its own train rows (embeddings [M_r, D], labels [M_r])
    and its own queries.  The train rows of all ranks are all-gathered in rank order (the shard sizes first: they may
    differ, so each shard travels padded to the largest), `score(train_emb, train_y, query_emb, query_y)` -> int64 [1]
    correct count runs against the gathered set on every rank, and [correct, count] is all-reduced.  Returns int64 [2]
    = [correct, count] over all ranks.  Without a process group (or at world size 1) nothing is exchanged."""
    world = dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1
    if world > 1:
        dev = train_emb.device
        n = torch.full((1,), train_emb.size(0), dtype=torch.int64, device=dev)
        sizes = [torch.empty_like(n) for _ in range(world)]
        dist.all_gather(sizes, n, group=group)
        sizes = torch.cat(sizes).tolist()
        m = max(sizes)

        def gather(t):
            padded = torch.cat([t, t.new_zeros((m - t.size(0),) + tuple(t.shape[1:]))]) if t.size(0) < m else t.contiguous()
            parts = [torch.empty_like(padded) for _ in range(world)]
            dist.all_gather(parts, padded, group=group)
            return torch.cat([p[:s] for p, s in zip(parts, sizes)])
        train_emb, train_y = gather(train_emb), gather(train_y)
    correct = score(train_emb, train_y, query_emb, query_y).reshape(1).to(torch.int64)
    tot = torch.cat([correct, torch.full((1,), query_emb.size(0), dtype=torch.int64, device=correct.device)])
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.SUM, group=group)
    return tot


def _stage2_args(corpus, train_ids, eval_ids, head, k, mlp_epochs, num_classes, batch_graphs):
    """The host-side validation of a 2stg evaluation (before any device work): -> (train ids, eval ids, class count)."""
    if head not in ("knn", "mlp"):
        raise ValueError(f"tsg: head must be 'knn' or 'mlp', not {head!r}")
    train_ids = np.asarray(train_ids, dtype=np.int64).reshape(-1)
    eval_ids = np.asarray(eval_ids, dtype=np.int64).reshape(-1)
    if train_ids.size == 0 or eval_ids.size == 0:
        raise ValueError("tsg: evaluate needs at least one train id and one eval id")
    if not 1 <= int(k) <= 32:
        raise ValueError(f"tsg: k must be in [1, 32], not {k}")
    if head == "mlp" and int(mlp_epochs) < 1:
        raise ValueError("tsg: mlp_epochs must be at least 1")
    if batch_graphs < 1:
        raise ValueError("tsg: batch_graphs must be at least 1")
    if corpus.y is None:
        raise ValueError("tsg: the corpus carries no graph labels (y)")
    if num_classes is None:
        y_all = corpus.y_host if corpus.y_host is not None else corpus.y.cpu().numpy()
        num_classes = int(y_all.max()) + 1 if y_all.size else 1
    C = int(num_classes)
    corpus.check_labels(C)
    return train_ids, eval_ids, C


def _stage2_accuracy(corpus, status, train_emb, eval_emb, train_ids, eval_ids, head, k, mlp_epochs, seed, C, group):
    """The scoring half of a 2stg evaluation on embeddings already computed: labels gathered from `corpus.y`, the kNN or
    MLP head (K12), gather_score_reduce under a process group, and ONE device-to-host read of the totals together with
    the status word (`status`, which the embedding passes may also have written)."""
    from . import heads, nn as tnn
    dev = corpus.device
    take = lambda ids: corpus.y.index_select(0, torch.from_numpy(ids).to(dev))
    train_y, eval_y = take(train_ids), take(eval_ids)
    if head == "knn":
        def score(a, ya, q, yq):
            return heads.knn_classify(a, ya, q, yq, k=int(k), num_classes=C, status=status)[1]
    else:
        def score(a, ya, q, yq):
            with torch.random.fork_rng(devices=[]):
                torch.manual_seed(int(seed))
                clf = heads.Mlp1Classifier(a.size(1), dev, num_classes=C)
            for _ in range(int(mlp_epochs)):
                clf.fit(a, ya)
            return clf.score(q, yq, status=status)
    tot = gather_score_reduce(train_emb, train_y, eval_emb, eval_y, score, group)
    host = torch.cat([tot, status.to(torch.int64)]).cpu()            # the one read: totals and the status word
    tnn.check_fused_status({status.device.index: int(host[2])})
    return float(host[0]) / max(float(host[1]), 1.0)


class TripletTrainer:
    """model: tsg.nn.PackedSAGNet (or any module with the same forward signature)."""

    def __init__(self, model: torch.nn.Module, lr: float = 5e-4, weight_decay: float = 1e-4,
                 margin: float = 1.5, group=None):
        self.model, self.margin, self.group = model, margin, group
        # Code/sag/train_triplet.py:191
        params = list(model.parameters())
        # one fused multi-tensor kernel per step when the parameters live on the GPU (same update rule as the
        # reference's torch.optim.Adam; the foreach path costs ~8 launches and 0.15 ms of host time per step)
        fused = bool(params) and all(p.is_cuda for p in params)
        self.opt = torch.optim.Adam(params, lr=lr, weight_decay=weight_decay, fused=fused)

    def step(self, x: torch.Tensor, edge_index: torch.Tensor, node_ptr_host: np.ndarray,
             triplets: torch.Tensor) -> torch.Tensor:
        """x/edge_index/triplets on the device.  `triplets` [T,3] index rows of THIS rank's embedding matrix; with
        world > 1 the returned loss is the mean over the GLOBAL batch and the parameters receive its gradient."""
        self.model.train()
        world = dist.get_world_size(self.group) if dist.is_initialized() else 1
        if (edge_index is None and getattr(self.model, "native_step_supported", None)
                and self.model.native_step_supported(x, node_ptr_host)):
            # K14: forward, loss and backward are ONE C-ABI call; gradients land in views of one flat buffer
            loss = self.model.native_step(x, node_ptr_host, triplets, self.margin)
            if world > 1:
                _all_reduce_native_flat(self.model, int(triplets.size(0)), self.group)     # [T_r * grads, T_r * loss, T_r]
            loss = loss.clone()                                           # the buffer is rewritten by the next step
            self.opt.step()
            return loss
        emb = self.model(x, edge_index, node_ptr_host)
        loss, _, _ = ops.triplet_loss(emb, triplets, self.margin)         # mean over THIS rank's triplets
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        if world > 1:
            # triplets are rank-local by contract, so the global-batch loss and gradient are the T_r-weighted means of
            # the per-rank ones: one all-reduce per step (the all-gather formulation, kept as all_gather_rows for
            # triplets that cross ranks, cost two more collectives and a synchronisation before the backward pass)
            loss = all_reduce_grads_and_loss(list(self.model.parameters()), loss, int(triplets.size(0)), self.group)
        self.opt.step()
        return loss.detach()

    def step_allgather(self, x, edge_index, node_ptr_host: np.ndarray, triplets_global: torch.Tensor) -> torch.Tensor:
        """The north-star's formulation for triplets that CROSS ranks (the reference sampler draws positives and negatives
        from the whole training set, Code/sag/triplet_sampler.py:36-56): every rank embeds its own M graphs, the
        embeddings are all-gathered into [world * M, D] (row r * M + i = graph i of rank r), every rank evaluates the SAME
        global loss over `triplets_global` [T_g, 3] (indices into the gathered matrix, identical on all ranks), backward
        takes this rank's slice of d(loss)/d(embeddings), and one all-reduce(SUM) completes the parameter gradient."""
        self.model.train()
        if (edge_index is None and getattr(self.model, "native_step_supported", None)
                and self.model.native_step_supported(x, node_ptr_host)):
            # native halves (K14): forward to the embeddings, gather, loss + its gradient on the gathered matrix (K9),
            # this rank's slice back into the native backward
            emb, ctx = self.model.native_forward(x, node_ptr_host)
            world = dist.get_world_size(self.group) if dist.is_initialized() else 1
            if world > 1:
                emb_g = torch.empty(world * emb.size(0), emb.size(1), dtype=emb.dtype, device=emb.device)
                dist.all_gather_into_tensor(emb_g, emb, group=self.group)
            else:
                emb_g = emb.clone()
            emb_g.requires_grad_(True)
            loss, _, _ = ops.triplet_loss(emb_g, triplets_global, self.margin)
            loss.backward()
            r = dist.get_rank(self.group) if world > 1 else 0
            self.model.native_backward(ctx, emb_g.grad[r * emb.size(0):(r + 1) * emb.size(0)])
            if world > 1:
                flat, _ = self.model._flat_grads()
                dist.all_reduce(flat[:-2], op=dist.ReduceOp.SUM, group=self.group)
            self.opt.step()
            return loss.detach()
        emb = self.model(x, edge_index, node_ptr_host)
        emb_g = all_gather_rows(emb, self.group)
        loss, _, _ = ops.triplet_loss(emb_g, triplets_global, self.margin)
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        all_reduce_grads(list(self.model.parameters()), self.group)
        self.opt.step()
        return loss.detach()

    def step_from_host(self, x_host: torch.Tensor, edge_index_host: torch.Tensor,
                       node_ptr_host: np.ndarray, triplets_host: torch.Tensor, device) -> float:
        """End-to-end call with (pinned) HOST buffers: H2D copies, the step, and the loss read back."""
        x = x_host.to(device, non_blocking=True)
        ei = edge_index_host.to(device, non_blocking=True)
        tr = triplets_host.to(device, non_blocking=True)
        return float(self.step(x, ei, node_ptr_host, tr).item())

    def run_from_host(self, host_batches, device) -> list:
        """Pipelined end-to-end loop over an iterable of HOST batches (dicts with pinned `x`, `edge_index`,
        `triplets` and numpy `node_ptr`): the H2D copies of batch i+1 run on a copy stream while the step
        on batch i computes, and every step's loss is read back into pinned host memory without stalling
        the enqueue thread.  Same arithmetic as step_from_host; returns the per-step losses."""
        cur = torch.cuda.current_stream(device)
        copy = getattr(self, "_copy_stream", None)
        if copy is None:
            copy = self._copy_stream = torch.cuda.Stream(device)

        def upload(b):
            copy.wait_stream(cur)      # staging memory freed by earlier steps must be done being read
            with torch.cuda.stream(copy):
                x = b["x"].to(device, non_blocking=True)
                ei = b["edge_index"].to(device, non_blocking=True)
                tr = b["triplets"].to(device, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy)
            return x, ei, b["node_ptr"], tr, ev

        it = iter(host_batches)
        try:
            nxt = upload(next(it))
        except StopIteration:
            return []
        host_losses = []
        while nxt is not None:
            x, ei, nptr, tr, ev = nxt
            try:
                nxt = upload(next(it))
            except StopIteration:
                nxt = None
            cur.wait_event(ev)
            for t in (x, ei, tr):
                t.record_stream(cur)
            loss = self.step(x, ei, nptr, tr)
            h = torch.empty((), dtype=torch.float32, pin_memory=True)
            h.copy_(loss, non_blocking=True)
            host_losses.append(h)
        cur.synchronize()
        _check_status()
        return [float(h) for h in host_losses]

    def run_from_host_compact(self, host_batches, device, num_node_labels: int, expand: bool = False) -> list:
        """Pipelined end-to-end loop over COMPACT host batches: what a TU dataset actually stores for a graph --
        node labels and the edge list -- instead of the fp32 one-hot matrix and int64 edge_index the PyG surface
        materialises.  Each batch: dict(label int32 [N], row / col int32 [E] LOCAL node ids, node_ptr / edge_ptr
        int64 numpy [G+1], triplets int64 [T,3]), tensors pinned.  Per step the H2D is 4N + 8E + 16G bytes
        (43 MB instead of 423 MB for the bench batch).  The batch goes to the model as an `ops.CompactBatch`:
        PackedSAGNet's executor consumes labels and local endpoints directly (K3c gather / segment sum for conv1,
        K1b on int32 local ids), so neither the fp32 one-hot x nor the int64 edge_index is ever written.
        `expand=True` restores the earlier behaviour: `tsg_pack_batch` (K0) materialises both on the GPU first
        (models without a compact path do that themselves through `CompactBatch.expand`)."""
        from ._lib import call, ptr, stream_ptr
        cur = torch.cuda.current_stream(device)
        copy = getattr(self, "_copy_stream", None)
        if copy is None:
            copy = self._copy_stream = torch.cuda.Stream(device)

        def upload(b):
            copy.wait_stream(cur)
            G = b["node_ptr"].shape[0] - 1
            meta = b.get("_meta")
            if meta is None:          # pinned once per host batch, reused when the batch comes round again
                meta = b["_meta"] = torch.from_numpy(np.concatenate([b["node_ptr"], b["edge_ptr"]])).pin_memory()
            with torch.cuda.stream(copy):
                t = {k: b[k].to(device, non_blocking=True) for k in ("label", "row", "col", "triplets")}
                t["meta"] = meta.to(device, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy)
            return t, b["node_ptr"], b["edge_ptr"], ev, b.get("coalesced", False)

        it = iter(host_batches)
        try:
            nxt = upload(next(it))
        except StopIteration:
            return []
        host_losses = []
        while nxt is not None:
            t, nptr, eptr, ev, b_coalesced = nxt
            try:
                nxt = upload(next(it))
            except StopIteration:
                nxt = None
            cur.wait_event(ev)
            for v in t.values():
                v.record_stream(cur)
            G, N, E = nptr.shape[0] - 1, int(nptr[-1]), int(eptr[-1])
            d_nptr, d_eptr = t["meta"][:G + 1], t["meta"][G + 1:]
            cb = ops.CompactBatch(t["label"], t["row"], t["col"], d_nptr, d_eptr, num_node_labels,
                                  int(np.diff(eptr).max()) if G else 0, bool(b_coalesced))
            if expand or not getattr(self.model, "accepts_compact", False):
                x, ei = cb.expand()
            else:
                x, ei = cb, None
            loss = self.step(x, ei, nptr, t["triplets"])
            h = torch.empty((), dtype=torch.float32, pin_memory=True)
            h.copy_(loss, non_blocking=True)
            host_losses.append(h)
        cur.synchronize()
        _check_status()
        return [float(h) for h in host_losses]

    def run_from_ids(self, corpus, id_batches) -> list:
        """Pipelined end-to-end loop against an HBM-resident corpus (tsg.feeder.DeviceCorpus): every step the host
        provides only what a sampler produces -- the step's graph ids and its triplet index rows -- as
        (graph_ids int64 numpy [B], triplets int64 pinned tensor [T, 3]).  Per step, INSIDE the loop: the packed
        offsets of the chosen graphs are computed on the host (two cumsums over B sizes), ids + offsets + triplets go
        up on the copy stream, the batch is assembled on the GPU from the resident corpus (K0 compact gather), the
        training step runs, and the loss is read back into pinned memory without stalling the enqueue thread.
        Nothing is pre-packed or cached across steps.  Returns the per-step losses."""
        dev = corpus.device
        cur = torch.cuda.current_stream(dev)
        copy = getattr(self, "_copy_stream", None)
        if copy is None:
            copy = self._copy_stream = torch.cuda.Stream(dev)
        compact = corpus.label is not None and getattr(self.model, "accepts_compact", False)

        def stage(item):
            ids_host, trip_host = item
            ids, nptr, eptr = corpus.offsets(ids_host)
            need = ids.shape[0] + nptr.shape[0] + eptr.shape[0]
            slot = self._ring_pos = (getattr(self, "_ring_pos", -1) + 1) % 4
            ring = self.__dict__.setdefault("_meta_ring", [None] * 4)
            if ring[slot] is None or ring[slot][0].numel() < need:       # pinned staging ring: allocated once, reused
                ring[slot] = [torch.empty(max(need, 1024), dtype=torch.int64, pin_memory=True), None]
            buf, busy = ring[slot]
            if busy is not None:
                busy.synchronize()             # the upload issued from this slot four stages ago has left it
            meta_h = buf[:need]
            np.concatenate([ids, nptr, eptr], out=meta_h.numpy())
            copy.wait_stream(cur)
            with torch.cuda.stream(copy):
                meta = meta_h.to(dev, non_blocking=True)
                tr = trip_host.to(dev, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy)
            ring[slot][1] = ev
            return meta, tr, ids.shape[0], nptr, eptr, ev, meta_h

        it = iter(id_batches)
        try:
            nxt = stage(next(it))
        except StopIteration:
            return []
        host_losses = []
        while nxt is not None:
            meta, tr, B, nptr, eptr, ev, keep = nxt
            try:
                nxt = stage(next(it))
            except StopIteration:
                nxt = None
            cur.wait_event(ev)
            meta.record_stream(cur); tr.record_stream(cur)
            if compact:
                (x, _), ei = corpus.pack_compact_staged(meta, B, nptr, eptr), None
            else:
                x, ei, _ = corpus.pack_staged(meta, B, nptr, eptr)
            loss = self.step(x, ei, nptr, tr)
            h = torch.empty((), dtype=torch.float32, pin_memory=True)
            h.copy_(loss, non_blocking=True)
            host_losses.append(h)
        cur.synchronize()
        _check_status()
        return [float(h) for h in host_losses]

    def step_from_ids(self, corpus, graph_ids_host: np.ndarray, triplets_host: torch.Tensor) -> float:
        """End-to-end call against an HBM-resident corpus (tsg.feeder.DeviceCorpus): the host sends the
        step's graph ids + triplet index list, the batch is assembled on the GPU, the loss is read back."""
        if corpus.label is not None and getattr(self.model, "accepts_compact", False):
            (x, nptr), ei = corpus.pack_compact(graph_ids_host), None
        else:
            x, ei, nptr = corpus.pack(graph_ids_host)
        tr = triplets_host.to(corpus.device, non_blocking=True)
        loss = float(self.step(x, ei, nptr, tr).item())
        _check_status()
        return loss

    def _pack(self, corpus, ids_host):
        """ids -> (x or an ops.CompactBatch, edge_index or None, node_ptr_host), assembled on the GPU from the corpus."""
        if corpus.label is not None and getattr(self.model, "accepts_compact", False):
            (x, nptr), ei = corpus.pack_compact(ids_host), None
        else:
            x, ei, nptr = corpus.pack(ids_host)
        return x, ei, nptr

    def _embed(self, corpus, ids: np.ndarray, batch_graphs: int) -> torch.Tensor:
        model = self.model
        was_training = model.training
        model.eval()
        parts = []
        try:
            with torch.no_grad():
                for s in range(0, ids.shape[0], batch_graphs):
                    x, ei, nptr = self._pack(corpus, ids[s:s + batch_graphs])
                    if _native_ok(model, x, ei, nptr):
                        parts.append(model.native_classify(x, nptr)[1])      # the head's log-softmax output = embedding
                    else:
                        if ei is None and not getattr(model, "accepts_compact", False):
                            x, ei = x.expand()
                        parts.append(model(x, ei, nptr))
        finally:
            model.train(was_training)
        if not parts:
            return torch.empty(0, model.num_classes, dtype=torch.float32, device=corpus.device)
        return parts[0] if len(parts) == 1 else torch.cat(parts)

    def embed(self, corpus, ids, batch_graphs: int = 4096) -> torch.Tensor:
        """Embeddings [len(ids), D] on the device of the graphs `ids` of an HBM-resident corpus (tsg.feeder.DeviceCorpus),
        row i = graph ids[i] (duplicates allowed): what the stage-2 loops of Code/sag/train_triplet.py:36-58,86-99 feed
        their classifiers.  The model runs in eval mode (dropout off, as in ClassifierTrainer.evaluate) in packed batches
        of `batch_graphs`, natively (tsg_sag_classify_compact: K13 where the shape allows, then the head) where
        native_step_supported holds, else through a torch.no_grad() forward; the caller's training flag is restored.
        The status word is checked once, at the end."""
        if batch_graphs < 1:
            raise ValueError("tsg: batch_graphs must be at least 1")
        out = self._embed(corpus, np.asarray(ids, dtype=np.int64).reshape(-1), int(batch_graphs))
        _check_status()
        return out

    def evaluate(self, corpus, train_ids, eval_ids, head: str = "knn", k: int = 3, mlp_epochs: int = 1, seed: int = 0,
                 num_classes: Optional[int] = None, batch_graphs: int = 4096) -> float:
        """The 2stg accuracy: the encoder's embeddings (`embed`) of `train_ids` fit a stage-2 classifier that labels
        `eval_ids`; labels come from `corpus.y`.
          head="knn": KNeighborsClassifier(n_neighbors=k) on the train embeddings (Code/sage+gat+diffpool/
            train_triplet.py:80-85) -- tsg_knn_classify, k <= 32, up to 1,024 classes.
          head="mlp": evaluate_mlp's classifier (tsg.heads.Mlp1Classifier) trained one sample per step in the order of
            `train_ids` for `mlp_epochs` passes, then scored with tsg_mlp1_predict.  Its initial weights are drawn from
            `seed` under torch.random.fork_rng, so evaluating does not move the caller's RNG stream.
        `num_classes` = the graph-class count (default: 1 + the corpus's largest label; NOT model.num_classes, which for
        a triplet model is the embedding width); every label is checked against it on the host, once per corpus.
        Under a process group each rank passes its own ids: train rows are all-gathered in rank order, every rank fits
        the same classifier on them and scores its own queries, and [correct, count] is all-reduced
        (gather_score_reduce).  One device-to-host read, at the end (plus the shard sizes under a process group)."""
        from . import nn as tnn
        train_ids, eval_ids, C = _stage2_args(corpus, train_ids, eval_ids, head, k, mlp_epochs, num_classes, batch_graphs)
        status = tnn._status_word(corpus.device)
        train_emb = self._embed(corpus, train_ids, int(batch_graphs))
        eval_emb = self._embed(corpus, eval_ids, int(batch_graphs))
        return _stage2_accuracy(corpus, status, train_emb, eval_emb, train_ids, eval_ids, head, k, mlp_epochs, seed, C,
                                self.group)


class ClassifierTrainer:
    """The "original" setting of Code/sag/train.py: the classifier trained end to end with F.nll_loss on its own
    log-softmax output (the baseline 2stg is compared with).  model: tsg.nn.PackedSAGNet, or any module with the same
    forward signature that returns log-probabilities [G, C] and has `num_classes`."""

    def __init__(self, model: torch.nn.Module, lr: float = 5e-4, weight_decay: float = 1e-4, group=None):
        self.model, self.group = model, group
        # Code/sag/train.py's torch.optim.Adam(lr, weight_decay); fused on the GPU as in TripletTrainer
        params = list(model.parameters())
        fused = bool(params) and all(p.is_cuda for p in params)
        self.opt = torch.optim.Adam(params, lr=lr, weight_decay=weight_decay, fused=fused)

    def _world(self) -> int:
        return dist.get_world_size(self.group) if dist.is_initialized() else 1

    def _native(self, x, edge_index, node_ptr_host) -> bool:
        return _native_ok(self.model, x, edge_index, node_ptr_host)

    def step(self, x, edge_index, node_ptr_host: np.ndarray, y: torch.Tensor) -> torch.Tensor:
        """One step of Code/sag/train.py:190-197 on a packed batch: F.nll_loss(model(data), data.y), backward, Adam.
        x / edge_index (or an ops.CompactBatch and None) and y (int64 [G]) on the device.  Native (one C-ABI call for
        forward, loss and backward) when the model supports the batch, else through autograd; TSG_NATIVE_STEP=0 forces
        the latter.  With world > 1 the returned loss is the mean over the GLOBAL batch and the parameters receive its
        gradient: one all-reduce of [G_r * grads, G_r * loss, G_r]."""
        self.model.train()
        world = self._world()
        G = int(y.shape[0])
        if self._native(x, edge_index, node_ptr_host):
            loss = self.model.native_nll_step(x, node_ptr_host, y)
            if world > 1:
                _all_reduce_native_flat(self.model, G, self.group)
            loss = loss.clone()                                           # the buffer is rewritten by the next step
            self.opt.step()
            return loss
        out = self.model(x, edge_index, node_ptr_host)
        loss = F.nll_loss(out, y)                                         # mean over THIS rank's graphs
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        if world > 1:
            loss = all_reduce_grads_and_loss(list(self.model.parameters()), loss, G, self.group)
        self.opt.step()
        return loss.detach()

    def _batch(self, corpus, ids_host):
        """ids -> (x, edge_index, node_ptr_host, y): the batch assembled on the GPU from the resident corpus (one small
        upload of ids + offsets), its labels gathered on the device from the same staged ids."""
        meta, B, nptr, eptr = corpus._stage(ids_host)
        y = corpus.y.index_select(0, meta[:B])
        if corpus.label is not None and getattr(self.model, "accepts_compact", False):
            (x, _), ei = corpus.pack_compact_staged(meta, B, nptr, eptr), None
        else:
            x, ei, _ = corpus.pack_staged(meta, B, nptr, eptr)
        return x, ei, nptr, y

    def run_from_ids(self, corpus, id_batches) -> list:
        """Training loop against an HBM-resident corpus (tsg.feeder.DeviceCorpus with labels): the host provides only
        each step's graph ids (int64 numpy [B]); batch and labels are assembled on the GPU, and every step's loss is read
        back into pinned memory without stalling the enqueue thread.  Returns the per-step losses."""
        corpus.check_labels(self.model.num_classes)
        host_losses = []
        for ids in id_batches:
            loss = self.step(*self._batch(corpus, ids))
            h = torch.empty((), dtype=torch.float32, pin_memory=True)
            h.copy_(loss, non_blocking=True)
            host_losses.append(h)
        torch.cuda.current_stream(corpus.device).synchronize()
        _check_status()
        return [float(h) for h in host_losses]

    def evaluate(self, corpus, ids, batch_graphs: int = 4096):
        """`test()` of Code/sag/train.py:19-29 over the graphs `ids` of the corpus in packed batches of `batch_graphs`:
        (accuracy, mean NLL) of the model in eval mode, pred = out.max(dim=1)[1].  Per-batch totals stay on the device
        and are read back once at the end, then summed in float64; under a process group every rank passes its own ids
        and [correct, loss_sum, count] is all-reduced."""
        corpus.check_labels(self.model.num_classes)
        ids = np.asarray(ids, dtype=np.int64)
        was_training = self.model.training
        self.model.eval()
        totals = []
        try:
            with torch.no_grad():
                for s in range(0, ids.shape[0], batch_graphs):
                    x, ei, nptr, y = self._batch(corpus, ids[s:s + batch_graphs])
                    if self._native(x, ei, nptr):
                        _, _, correct, nll_sum = self.model.native_classify(x, nptr, y)
                    else:
                        if ei is None and not getattr(self.model, "accepts_compact", False):
                            x, ei = x.expand()
                        out = self.model(x, ei, nptr)
                        correct = (out.max(dim=1)[1] == y).sum().view(1)
                        nll_sum = F.nll_loss(out, y, reduction="sum").view(1)
                    totals.append(torch.cat([correct.double(), nll_sum.double()]))
        finally:
            self.model.train(was_training)
        t = torch.stack(totals).cpu().numpy() if totals else np.zeros((0, 2))
        _check_status()
        acc = np.array([t[:, 0].sum(), t[:, 1].sum(), float(ids.shape[0])], dtype=np.float64)
        if self._world() > 1:
            red = torch.from_numpy(acc).to(corpus.device)
            dist.all_reduce(red, op=dist.ReduceOp.SUM, group=self.group)
            acc = red.cpu().numpy()
        n = max(acc[2], 1.0)
        return float(acc[0] / n), float(acc[1] / n)


class _DenseEncoderTrainer:
    """What the trainers of the dense encoders share: the model / feature-table checks, the batch assembled on the GPU
    from an HBM-resident corpus (DeviceCorpus.pack_dense, after the host-side `_check`) and the forward up to the graph
    readout.  Subclasses call `_bind` first."""

    def _bind(self, model: torch.nn.Module, table: torch.Tensor, max_nodes: int) -> list:
        """Check the model and the table and keep them: -> the model's parameters."""
        from . import dense, diffpool, gat
        if isinstance(model, gat.PackedGatEncoder):
            self.kind, in_dim = "gat", model.conv_first.heads()[0].input_dim
        elif isinstance(model, diffpool.PackedSoftPoolEncoder):
            self.kind, in_dim = "diffpool", model.conv_first.input_dim
            if int(model.max_num_nodes) != int(max_nodes):
                raise ValueError(f"tsg: the DiffPool model was built for max_num_nodes = {model.max_num_nodes}, the trainer "
                                 f"pads to max_nodes = {max_nodes}")
        elif isinstance(model, dense.PackedGcnEncoder):
            self.kind, in_dim = "base", model.conv_first.input_dim
        else:
            raise TypeError(f"tsg: {type(self).__name__} takes a PackedGcnEncoder, PackedGatEncoder or PackedSoftPoolEncoder")
        if int(max_nodes) < 1:
            raise ValueError("tsg: max_nodes must be at least 1")
        if table.dim() != 2 or table.size(0) < int(max_nodes):
            raise ValueError(f"tsg: the feature table must be [max_nodes = {max_nodes}, F], not {tuple(table.shape)}")
        if table.size(1) != in_dim:
            raise ValueError(f"tsg: the feature table has {table.size(1)} columns, the model takes {in_dim}")
        params = list(model.parameters())
        dev = params[0].device if params else table.device
        self.model, self.max_nodes = model, int(max_nodes)
        self.table = table.to(device=dev, dtype=torch.float32).contiguous()
        self.want_eid = self.kind == "gat"                 # GAT's backward walks both orientations by edge id
        return params

    def _forward(self, batch):
        if self.kind == "gat":
            return self.model(batch.x, batch.csr, batch.graph_ptr, batch.max_nodes)
        return self.model(batch.x, batch.csr, batch.graph_ptr, batch.has_pad)

    def _readout(self, batch):
        """The model's forward up to its graph readout (the input of its heads)."""
        if self.kind == "gat":
            return self.model.readout(batch.x, batch.csr, batch.graph_ptr, batch.max_nodes)
        return self.model.readout(batch.x, batch.csr, batch.graph_ptr, batch.has_pad)

    def pack(self, corpus, ids_host):
        """ids -> tsg.feeder.DenseBatch for this trainer's model (eids for GAT), assembled on the GPU."""
        return corpus.pack_dense(ids_host, self.table, self.max_nodes, want_eid=self.want_eid)

    def _check(self, corpus, ids_host) -> np.ndarray:
        """The host-side checks of a pack (no device work): -> the ids as int64 numpy."""
        return corpus.check_dense(ids_host, self.table, self.max_nodes)

    def _pack_checked(self, corpus, ids: np.ndarray):
        """`pack` for ids that passed `_check`: one staged upload, one launch."""
        return corpus.pack_dense_staged(*corpus._stage(ids), self.table, self.max_nodes, self.want_eid)

    def _batch(self, corpus, ids: np.ndarray):
        """`_pack_checked` and the graphs' labels (int64 [B], gathered on the device from corpus.y by the staged ids)."""
        meta, B, nptr, eptr = corpus._stage(ids)
        batch = corpus.pack_dense_staged(meta, B, nptr, eptr, self.table, self.max_nodes, self.want_eid)
        return batch, corpus.y.index_select(0, meta[:B])


class _WaveEncoderTrainer(_DenseEncoderTrainer):
    """`_DenseEncoderTrainer` for the EigenGCN encoder (tsg.dense.PackedWaveEncoder = Code/eigengcn's
    WavePoolingGcnEncoder with one pooling level) against a corpus whose EigenPooling operands are attached
    (DeviceCorpus.attach_eigen): every batch is assembled on the GPU by DeviceCorpus.pack_eigen in one launch.
    Refused on the host: a model with more than one pooling level (the operands describe one), operands with fewer
    pooling matrices than the model uses, and a corpus whose node-label count differs from the model's input_dim."""

    def _bind(self, model: torch.nn.Module, table, max_nodes: int) -> list:
        from . import dense
        if not isinstance(model, dense.PackedWaveEncoder):
            raise TypeError(f"tsg: {type(self).__name__} takes a PackedWaveEncoder")
        if len(model.pool_sizes) != 1:
            raise ValueError(f"tsg: the model has {len(model.pool_sizes)} pooling levels; the EigenPooling operands "
                             "describe one")
        if int(max_nodes) < 1:
            raise ValueError("tsg: max_nodes must be at least 1")
        self.kind, self.table, self.want_eid = "wave", None, False
        self.model, self.max_nodes = model, int(max_nodes)
        return list(model.parameters())

    def _check(self, corpus, ids_host) -> np.ndarray:
        m = self.model
        if corpus.feat != m.conv_first.input_dim:
            raise ValueError(f"tsg: the corpus has {corpus.feat} node labels, the model takes input_dim = "
                             f"{m.conv_first.input_dim}")
        ids, _, _ = corpus.check_eigen(ids_host, self.max_nodes, m.num_pool_matrix, m.num_pool_final_matrix)
        return ids

    def _pack_checked(self, corpus, ids: np.ndarray):
        return corpus.pack_eigen_checked(ids, self.max_nodes, self.model.num_pool_matrix,
                                         self.model.num_pool_final_matrix)

    def _batch(self, corpus, ids: np.ndarray):
        return self._pack_checked(corpus, ids), corpus.y.index_select(0, corpus._upload([ids]))

    def pack(self, corpus, ids_host):
        """ids -> tsg.feeder.EigenBatch for this trainer's model, assembled on the GPU."""
        return self._pack_checked(corpus, self._check(corpus, ids_host))

    def _forward(self, batch):
        args, kw = batch.readout_args()
        return self.model(*args, **kw)

    def _readout(self, batch):
        args, kw = batch.readout_args()
        return self.model.readout(*args, **kw)


class DenseTripletTrainer(_DenseEncoderTrainer):
    """2stg stage-1 training and scoring of the dense encoders of Code/sage+gat+diffpool against an HBM-resident corpus
    (tsg.feeder.DeviceCorpus): tsg.dense.PackedGcnEncoder ("base" / GraphSAGE), tsg.gat.PackedGatEncoder and
    tsg.diffpool.PackedSoftPoolEncoder.  Every batch is assembled on the GPU by DeviceCorpus.pack_dense: node features are
    the rows of `table` ([>= max_nodes, F], the shared N(0, 2^2) table indexed by node position,
    train_triplet.py:379-385), the adjacency is the RAW 0/1 CSR.  The embedding is element [1] of the model's output, the
    one the triplet loss sees (tripletnet.py:36-38).

    The step is the reference's dense stage-1 setting: MarginRankingLoss(margin) on the embedding distances, Adam(lr)
    (train_triplet.py:216) and clip_grad_norm(clip_norm) (:286); clip_norm=None skips the clip.  Documented deviation:
    the reference's dense triplet loss also adds L1 / L2 norms of the embeddings (SURVEY section 3b); their coefficients
    are not recorded, so this trainer leaves those terms out rather than guess them.

    `max_nodes` is the reference's padding size: a graph with fewer nodes has zero-padded rows (has_pad, or GAT's
    max_nodes argument), one with more is refused.  A DiffPool model's `max_num_nodes` must equal it."""

    def __init__(self, model: torch.nn.Module, table: torch.Tensor, max_nodes: int = 1000, lr: float = 1e-3,
                 margin: float = 1.5, clip_norm: Optional[float] = 2.0, group=None):
        params = self._bind(model, table, max_nodes)
        self.margin, self.group, self.clip_norm = margin, group, clip_norm
        self.opt = torch.optim.Adam(params, lr=lr)          # train_triplet.py:216

    def _head(self, r):
        """Element [1] of the model's forward from its readout `r` (encoders.py:207-217, encoders_GAT.py:191-198)."""
        m = self.model
        if self.kind == "gat":
            return (m.pred_model if m.final_dim != "output_dim" else m.map_model)(r)
        if m.final_dim not in ("pretrain", "output_dim"):
            return m.pred_model(m.pre_pred_model(r))
        return m.map_model(r)

    def _embedding(self, batch) -> torch.Tensor:
        """The embedding the triplet loss sees (element [1] of the model's output)."""
        return self._forward(batch)[1]

    def step(self, batch, triplets: torch.Tensor) -> torch.Tensor:
        """One stage-1 step on a DenseBatch: embeddings, the triplet loss over `triplets` [T, 3] (rows of this batch),
        backward, the optional clip, Adam.  With world > 1 one all-reduce of [T_r * grads, T_r * loss, T_r] makes the loss
        and gradient those of the global batch (triplets are rank-local); the clip then applies to that gradient."""
        self.model.train()
        emb = self._embedding(batch)
        loss, _, _ = ops.triplet_loss(emb, triplets, self.margin)
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        params = list(self.model.parameters())
        world = dist.get_world_size(self.group) if dist.is_initialized() else 1
        if world > 1:
            loss = all_reduce_grads_and_loss(params, loss, int(triplets.size(0)), self.group)
        if self.clip_norm is not None:
            torch.nn.utils.clip_grad_norm_(params, self.clip_norm)
        self.opt.step()
        return loss.detach()

    def run_from_ids(self, corpus, id_batches) -> list:
        """Training loop against an HBM-resident corpus, with TripletTrainer.run_from_ids's contract: per step the host
        provides (graph_ids int64 numpy [B], triplets int64 pinned tensor [T, 3] into graph_ids).  Inside the loop the ids
        and offsets go up in one small staged upload, pack_dense assembles the batch in one launch, the step runs and its
        loss is read back into pinned memory without stalling the enqueue thread.  The status word is checked once, at
        the end.  Returns the per-step losses."""
        dev = corpus.device
        host_losses = []
        for ids_host, trip_host in id_batches:
            batch = self._pack_checked(corpus, self._check(corpus, ids_host))
            loss = self.step(batch, trip_host.to(dev, non_blocking=True))
            h = torch.empty((), dtype=torch.float32, pin_memory=True)
            h.copy_(loss, non_blocking=True)
            host_losses.append(h)
        torch.cuda.current_stream(dev).synchronize()
        _check_status()
        return [float(h) for h in host_losses]

    def _embed(self, corpus, ids: np.ndarray, batch_graphs: int) -> torch.Tensor:
        model = self.model
        was_training = model.training
        model.eval()
        parts = []
        try:
            with torch.no_grad():
                for s in range(0, ids.shape[0], batch_graphs):
                    parts.append(self._readout(self.pack(corpus, ids[s:s + batch_graphs])))
                # the head runs ONCE over all rows: the ATen GEMM picks its algorithm by row count, so one call per
                # packed batch would make a row's last bits depend on batch_graphs
                return self._head(parts[0] if len(parts) == 1 else torch.cat(parts))
        finally:
            model.train(was_training)

    def embed(self, corpus, ids, batch_graphs: int = 4096) -> torch.Tensor:
        """Embeddings [len(ids), D] on the device, row i = graph ids[i] (duplicates allowed): the model in eval mode under
        torch.no_grad(): readouts in packed batches of `batch_graphs`, then the model's head over all of them in one call, so
        the result does not depend on `batch_graphs`; the caller's training flag is restored.  The status word is checked
        once, at the end."""
        if batch_graphs < 1:
            raise ValueError("tsg: batch_graphs must be at least 1")
        ids = self._check(corpus, ids)
        out = self._embed(corpus, ids, int(batch_graphs))
        _check_status()
        return out

    def evaluate(self, corpus, train_ids, eval_ids, head: str = "knn", k: int = 3, mlp_epochs: int = 1, seed: int = 0,
                 num_classes: Optional[int] = None, batch_graphs: int = 4096) -> float:
        """The 2stg accuracy of the encoder (Code/sage+gat+diffpool/train_triplet.py:80-85 kNN, evaluate_mlp's MLP):
        TripletTrainer.evaluate's contract, validation and scoring (K12 heads, the MLP's initial weights drawn from `seed`
        under fork_rng, gather_score_reduce under a process group, one device-to-host read) on this trainer's
        embeddings."""
        from . import nn as tnn
        train_ids, eval_ids, C = _stage2_args(corpus, train_ids, eval_ids, head, k, mlp_epochs, num_classes, batch_graphs)
        self._check(corpus, train_ids)
        self._check(corpus, eval_ids)
        status = tnn._status_word(corpus.device)
        train_emb = self._embed(corpus, train_ids, int(batch_graphs))
        eval_emb = self._embed(corpus, eval_ids, int(batch_graphs))
        return _stage2_accuracy(corpus, status, train_emb, eval_emb, train_ids, eval_ids, head, k, mlp_epochs, seed, C,
                                self.group)


class WaveTripletTrainer(_WaveEncoderTrainer, DenseTripletTrainer):
    """2stg stage-1 training and scoring of the EigenGCN encoder (see _WaveEncoderTrainer for the batches and what is
    refused on the host).  The embedding is the model's output, the one bench config 5 feeds the triplet loss;
    DenseTripletTrainer's step / run_from_ids / embed / evaluate contract applies (embed: readouts in packed batches,
    pred_model once over all rows).  Defaults: Adam 1e-3, margin 1.5, no clip (bench config 5's step)."""

    def __init__(self, model: torch.nn.Module, max_nodes: int = 1000, lr: float = 1e-3, margin: float = 1.5,
                 clip_norm: Optional[float] = None, group=None):
        params = self._bind(model, None, max_nodes)
        self.margin, self.group, self.clip_norm = margin, group, clip_norm
        self.opt = torch.optim.Adam(params, lr=lr)

    def _embedding(self, batch) -> torch.Tensor:
        return self._forward(batch)

    def _head(self, r):
        return self.model.pred_model(r)


def _linear_chain(*mods) -> list:
    """nn.Linear / nn.ReLU / nn.Sequential modules in call order -> K16's layers [(weight, bias, relu_after), ...]."""
    out = []
    for m in mods:
        for c in (m if isinstance(m, torch.nn.Sequential) else [m]):
            if isinstance(c, torch.nn.Linear):
                out.append([c.weight, c.bias, False])
            elif isinstance(c, torch.nn.ReLU) and out:
                out[-1][2] = True
            else:
                raise ValueError(f"tsg: the prediction head holds a {type(c).__name__}; K16 runs Linear and ReLU layers")
    return [tuple(x) for x in out]


class DenseClassifierTrainer(_DenseEncoderTrainer):
    """Supervised training and evaluation of the dense encoders (tsg.dense.PackedGcnEncoder "base", tsg.gat.PackedGatEncoder,
    tsg.diffpool.PackedSoftPoolEncoder) against an HBM-resident corpus with graph labels, batches assembled as for
    DenseTripletTrainer.  The head over the readout and the cross-entropy are K16 (tsg.ops.pred_ce); the encoder's
    backward continues from the readout gradient.  The logits per setting (Code/sage+gat+diffpool, SURVEY A.2):

      setting="original" (train.py:85-152; the model's final_dim must not be "output_dim" or "pretrain"):
        base / DiffPool: pred_model(pre_pred_model(readout)); GAT: pred_model(readout); plain cross-entropy.
      setting="2stg+" (stage 2 of train_triplet_pre_train.py:249-256, after stage 1 with DenseTripletTrainer):
        base / DiffPool (final_dim="pretrain"): map2_model(map_model(readout)), 2 classes; GAT (any final_dim): the raw
        readout, embedding_dim classes, no head parameters.  The reference applies softmax to these logits before
        F.cross_entropy; so does this trainer.

    The step is the reference's: the loss (plus the DiffPool link-prediction term with linkpred=True, original only),
    backward, clip_grad_norm(clip_norm) (None: no clip), Adam(lr) -- or `optimizer`, e.g. the stage-1 trainer's `opt`,
    whose state then carries on.  Under a process group one all-reduce of [G_r * grads, G_r * loss, G_r] per step makes
    the loss and gradient those of the global batch, before the clip.

    Refused on the host (ValueError): a final_dim that does not fit the setting, linkpred on anything but DiffPool
    original, a head beyond K16's limits (at most 8 layers, widths <= 256), and a corpus label outside the class count."""

    def __init__(self, model: torch.nn.Module, table: torch.Tensor, max_nodes: int = 1000, setting: str = "original",
                 lr: float = 1e-3, clip_norm: Optional[float] = 2.0, linkpred: bool = False, optimizer=None, group=None):
        params = self._bind(model, table, max_nodes)
        self._setup(setting, linkpred)
        self.clip_norm, self.group = clip_norm, group
        self.opt = optimizer if optimizer is not None else torch.optim.Adam(params, lr=lr)     # train.py: Adam 1e-3

    def _setup(self, setting: str, linkpred: bool) -> None:
        """The head modules, softmax_first and the class count of (model, setting), checked against K16's limits."""
        if setting not in ("original", "2stg+"):
            raise ValueError(f"tsg: setting must be 'original' or '2stg+', not {setting!r}")
        m, kind = self.model, self.kind
        fd = getattr(m, "final_dim", None)
        note = ""
        if kind == "wave":                          # EigenGCN: pred_model in both settings, no softmax (SURVEY 3c, a13)
            mods, softmax_first = (m.pred_model,), False
        elif setting == "original":
            if fd in ("output_dim", "pretrain"):
                raise ValueError(f"tsg: the original setting classifies with pred_model: the model's final_dim must not be "
                                 f"'output_dim' or 'pretrain' (it is {fd!r})")
            mods = (m.pred_model,) if kind == "gat" else (m.pre_pred_model, m.pred_model)
            softmax_first = False
        elif kind == "gat":
            mods, softmax_first = (), True
            note = f"2stg+ takes the GAT readout's embedding_dim = {m.map_model.in_features} columns as the logits"
        else:
            if fd != "pretrain":
                raise ValueError(f"tsg: 2stg+ classifies with map2_model(map_model(readout)): the model's final_dim must be "
                                 f"'pretrain' (it is {fd!r})")
            mods, softmax_first = (m.map_model, m.map2_model), True
            note = "2stg+ takes map2_model's 2 outputs as the logits"
        if linkpred and not (kind == "diffpool" and setting == "original"):
            raise ValueError("tsg: linkpred adds DiffPool's link-prediction loss: it needs a PackedSoftPoolEncoder in the "
                             "original setting")
        self.setting, self.linkpred, self.softmax_first = setting, bool(linkpred), softmax_first
        self._head_mods, self._label_note = mods, note
        layers = self._layers()
        in_dim = layers[0][0].size(1) if layers else m.map_model.in_features
        ops.check_pred_head(in_dim, [w.size(0) for w, _, _ in layers])
        self.num_classes = int(layers[-1][0].size(0)) if layers else int(in_dim)

    def _layers(self) -> list:
        return _linear_chain(*self._head_mods)

    def _check_labels(self, corpus) -> None:
        try:
            corpus.check_labels(self.num_classes)
        except ValueError as e:
            if not self._label_note or corpus.y is None:
                raise
            raise ValueError(f"{e}: {self._label_note}") from None

    def step(self, batch, y: torch.Tensor) -> torch.Tensor:
        """One training step on a packed batch (DenseBatch, or EigenBatch for WaveClassifierTrainer) with its labels y
        (int64 [G], on the device).  Returns the loss (the global batch's mean under a process group)."""
        self.model.train()
        if self.linkpred:
            b = batch
            r, aux = self.model.readout(b.x, b.csr, b.graph_ptr, b.has_pad, return_aux=True)
        else:
            r = self._readout(batch)
        loss = ops.pred_ce(r, self._layers(), y, self.softmax_first)
        if self.linkpred:                                                  # encoders.py:409-441
            loss = loss + self.model.link_loss(aux["s"], batch.csr, batch.graph_ptr, np.diff(batch.node_ptr_host))
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        params = list(self.model.parameters())
        world = dist.get_world_size(self.group) if dist.is_initialized() else 1
        if world > 1:
            loss = all_reduce_grads_and_loss(params, loss, int(y.shape[0]), self.group)
        if self.clip_norm is not None:
            torch.nn.utils.clip_grad_norm_(params, self.clip_norm)
        self.opt.step()
        return loss.detach()

    def run_from_ids(self, corpus, id_batches) -> list:
        """Training loop against an HBM-resident corpus with labels: per step the host provides only the graph ids (int64
        numpy [B]); the batch is assembled on the GPU, its labels gathered there from corpus.y, and the loss is read
        back into pinned memory without stalling the enqueue thread.  Labels are checked against the class count on
        the host once; the status word once, at the end.  Returns the per-step losses."""
        self._check_labels(corpus)
        host_losses = []
        for ids_host in id_batches:
            loss = self.step(*self._batch(corpus, self._check(corpus, ids_host)))
            h = torch.empty((), dtype=torch.float32, pin_memory=True)
            h.copy_(loss, non_blocking=True)
            host_losses.append(h)
        torch.cuda.current_stream(corpus.device).synchronize()
        _check_status()
        return [float(h) for h in host_losses]

    def evaluate(self, corpus, ids, batch_graphs: int = 4096):
        """(accuracy, mean cross-entropy) over the graphs `ids` in eval mode, the caller's mode restored: readouts in
        packed batches of `batch_graphs`, then K16's classify over all rows at once (tsg_pred_classify: pred = the
        first-index argmax of the logits, the loss as in training, softmax_first included), so the totals do not depend
        on `batch_graphs`.  One device-to-host read of [correct, loss sum, status]; under a process group every rank
        passes its own ids and [correct, loss sum, count] is all-reduced."""
        from . import nn as tnn
        if batch_graphs < 1:
            raise ValueError("tsg: batch_graphs must be at least 1")
        ids = self._check(corpus, ids)
        self._check_labels(corpus)
        dev = corpus.device
        status = tnn._status_word(dev)
        was_training = self.model.training
        self.model.eval()
        try:
            with torch.no_grad():
                parts = [self._readout(self._pack_checked(corpus, ids[s:s + batch_graphs]))
                         for s in range(0, ids.shape[0], batch_graphs)]
                r = parts[0] if len(parts) == 1 else torch.cat(parts)
                y = corpus.y.index_select(0, corpus._upload([ids]))
                _, _, correct, ce_sum = ops.pred_classify(r, self._layers(), y, self.softmax_first)
        finally:
            self.model.train(was_training)
        host = torch.cat([correct.double(), ce_sum.double(), status.double()]).cpu().numpy()
        tnn.check_fused_status({status.device.index: int(host[2])})
        acc = np.array([host[0], host[1], float(ids.shape[0])], dtype=np.float64)
        if dist.is_initialized() and dist.get_world_size(self.group) > 1:
            red = torch.from_numpy(acc).to(dev)
            dist.all_reduce(red, op=dist.ReduceOp.SUM, group=self.group)
            acc = red.cpu().numpy()
        n = max(acc[2], 1.0)
        return float(acc[0] / n), float(acc[1] / n)


class WaveClassifierTrainer(_WaveEncoderTrainer, DenseClassifierTrainer):
    """DenseClassifierTrainer for the EigenGCN encoder (tsg.dense.PackedWaveEncoder, batches as for WaveTripletTrainer).
    The logits are pred_model(readout) in both settings, with plain cross-entropy: in 2stg+ the reference swaps in a
    map_model that the forward never reaches (SURVEY 3c, row a13), and SURVEY records no softmax before its loss.  The
    reference's stage 2 steps the stage-1 optimiser: pass WaveTripletTrainer's `opt` as `optimizer` for that.  Defaults
    as WaveTripletTrainer: Adam 1e-3, no clip."""

    def __init__(self, model: torch.nn.Module, max_nodes: int = 1000, setting: str = "original", lr: float = 1e-3,
                 clip_norm: Optional[float] = None, optimizer=None, group=None):
        params = self._bind(model, None, max_nodes)
        self._setup(setting, False)
        self.clip_norm, self.group = clip_norm, group
        self.opt = optimizer if optimizer is not None else torch.optim.Adam(params, lr=lr)
