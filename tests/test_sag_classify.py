"""Host-side checks of the supervised ("original") setting: the head workspace queries of the native NLL step and the
classification forward (pure host functions of the shape), the host label check, and ClassifierTrainer's data-parallel
reduction on its autograd branch (gloo, world size 2, CPU stand-in model) against the single-process union batch."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _queries(H, C):
    from tsg import _lib
    shape = _lib.SagShape(3504, 89, H, 0)
    head = _lib.SagHead(C, 1, 1.5, 1e-6, 0.5, 0)
    return [getattr(_lib.lib, q)(ctypes.byref(shape), ctypes.byref(head)) for q in
            ("tsg_sag_nll_step_workspace_bytes", "tsg_sag_classify_workspace_bytes", "tsg_sag_triplet_step_workspace_bytes")]


@pytest.mark.parametrize("H,C", [(32, 2), (64, 8), (128, 2), (128, 64)])
def test_workspace_queries_cover_the_reference_widths(H, C):
    # nhid 128 is Code/sag/train.py's default; the triplet step at that width runs the same wide head backward
    assert all(q > 0 for q in _queries(H, C))


@pytest.mark.parametrize("H,C", [(33, 2), (127, 64), (128, 0)])
def test_workspace_queries_refuse_shapes_the_head_cannot_run(H, C):
    assert _queries(H, C) == [0, 0, 0]


class _StandIn(torch.nn.Module):
    """CPU stand-in for PackedSAGNet: log-probabilities of one linear layer over per-graph mean features."""

    def __init__(self, fin=5, num_classes=3):
        super().__init__()
        g = torch.Generator().manual_seed(0)
        self.num_classes = num_classes
        self.w = torch.nn.Parameter(torch.randn(fin, num_classes, generator=g))
        self.b = torch.nn.Parameter(torch.randn(num_classes, generator=g))

    def forward(self, x, edge_index, node_ptr_host):
        ptr = torch.from_numpy(np.asarray(node_ptr_host, dtype=np.int64))
        seg = torch.repeat_interleave(torch.arange(ptr.numel() - 1), ptr.diff())
        pooled = torch.zeros(ptr.numel() - 1, x.size(1)).index_add_(0, seg, x) / ptr.diff().unsqueeze(1)
        return torch.log_softmax(pooled @ self.w + self.b, dim=-1)


def test_invalid_label_raises_on_the_host():
    from tsg import synth
    from tsg.feeder import DeviceCorpus
    from tsg.train import ClassifierTrainer
    corpus = synth.make_corpus("PROTEINS", 6, seed=3)
    corpus.y = np.array([0, 1, 2, 1, 3, 0], np.int64)              # 3 is outside [0, 3)
    dc = DeviceCorpus(corpus, torch.device("cpu"))
    trainer = ClassifierTrainer(_StandIn(num_classes=3))
    with pytest.raises(ValueError, match="graph 4 has label 3"):
        trainer.evaluate(dc, np.arange(6))
    with pytest.raises(ValueError, match="outside"):
        trainer.run_from_ids(dc, [np.arange(6)])
    corpus.y[4] = 2
    DeviceCorpus(corpus, torch.device("cpu")).check_labels(3)
    # a corpus assembled on the device carries its labels as a tensor: the same check reads them back once
    shard = DeviceCorpus.from_device(dc.label, dc.row, dc.col, corpus.node_ptr, corpus.edge_ptr, corpus.num_node_labels,
                                     True, y=torch.tensor([0, 1, -1, 0, 0, 2]))
    with pytest.raises(ValueError, match="graph 2 has label -1"):
        shard.check_labels(3)
    with pytest.raises(ValueError, match="shape"):
        DeviceCorpus.from_device(dc.label, dc.row, dc.col, corpus.node_ptr, corpus.edge_ptr, corpus.num_node_labels,
                                 True, y=torch.zeros(5, dtype=torch.int64))


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


SIZES = [[3, 5, 2, 4], [6, 1, 2]]           # nodes per graph on each rank: different graph counts per rank


def _rank_batch(rank):
    g = torch.Generator().manual_seed(10 + rank)
    n = SIZES[rank]
    x = torch.randn(sum(n), 5, generator=g)
    y = torch.randint(0, 3, (len(n),), generator=g)
    return x, np.concatenate([[0], np.cumsum(n)]).astype(np.int64), y


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, os.path.join(root, "two-stage-gnn_b200"))
    from tsg.train import ClassifierTrainer
    model = _StandIn()
    trainer = ClassifierTrainer(model, lr=1e-2, weight_decay=1e-4)
    x, ptr, y = _rank_batch(rank)
    loss = trainer.step(x, None, ptr, y)
    if rank == 1:
        torch.save(dict(loss=loss.clone(), w=model.w.detach().clone(), b=model.b.detach().clone(),
                        gw=model.w.grad.clone(), gb=model.b.grad.clone()), out)
    dist.barrier()
    dist.destroy_process_group()


def test_data_parallel_step_equals_the_union_batch(tmp_path):
    """graph-weighted all-reduce of [G_r * grads, G_r * loss, G_r] == loss, gradient and Adam step of the union batch"""
    from tsg.train import ClassifierTrainer
    world, port, out = 2, _free_port(), str(tmp_path / "r1.pt")
    mp.spawn(_worker, args=(world, port, out), nprocs=world, join=True)
    got = torch.load(out)
    parts = [_rank_batch(r) for r in range(world)]
    x = torch.cat([p[0] for p in parts])
    ptr = np.concatenate([[0], np.cumsum(SIZES[0] + SIZES[1])]).astype(np.int64)
    y = torch.cat([p[2] for p in parts])
    model = _StandIn()
    loss = ClassifierTrainer(model, lr=1e-2, weight_decay=1e-4).step(x, None, ptr, y)
    assert torch.allclose(got["loss"], loss, atol=1e-6)
    for k in ("w", "b"):
        assert torch.allclose(got["g" + k], getattr(model, k).grad, atol=1e-6, rtol=1e-5), k
        assert torch.allclose(got[k], getattr(model, k).detach(), atol=1e-6, rtol=1e-5), k
