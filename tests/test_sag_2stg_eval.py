"""Host-side checks of the 2stg evaluation (TripletTrainer.embed / evaluate): the C ABI of the stage-2 entries as the
ctypes layer declares it, evaluate's argument validation (which runs before any device work), and the data-parallel
gather-and-reduce helper under gloo at world size 2 with shards of different sizes, against one process holding the
union."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import heads_ref as H


def test_stage2_abi_signatures():
    from tsg import _lib
    P, I64, I, F32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_float
    # tsg_knn_classify(train, train_labels, query, query_labels, M, Q, D, k, C, pred, correct, status, stream)
    assert _lib.lib.tsg_knn_classify.argtypes == [P, P, P, P, I64, I64, I64, I, I, P, P, P, P]
    # tsg_mlp1_predict(emb, labels, Q, D, H1, H2, C, params, slope, pred, logits, correct, status, stream)
    assert _lib.lib.tsg_mlp1_predict.argtypes == [P, P, I64, I64, I64, I64, I64, P, F32, P, P, P, P, P]
    # the old entry keeps its signature
    assert _lib.lib.tsg_knn_predict.argtypes == [P, P, P, I64, I64, I64, I, I, P, P]
    for name in ("tsg_knn_classify", "tsg_mlp1_predict"):
        assert _lib.lib[name].restype is ctypes.c_int


def _trainer_and_corpus(y):
    from tsg import nn as tnn, synth
    from tsg.feeder import DeviceCorpus
    from tsg.train import TripletTrainer
    corpus = synth.make_corpus("PROTEINS", len(y), seed=3)
    corpus.y = np.asarray(y, np.int64)
    model = tnn.PackedSAGNet(corpus.num_node_labels, 8, 4, 0.5, 0.0)
    return TripletTrainer(model), DeviceCorpus(corpus, torch.device("cpu"))


def test_evaluate_validates_its_arguments():
    tt, dc = _trainer_and_corpus([0, 1, 2, 1, 0, 1])
    with pytest.raises(ValueError, match="head"):
        tt.evaluate(dc, [0, 1, 2], [3, 4], head="svm")
    with pytest.raises(ValueError, match="at least one"):
        tt.evaluate(dc, [], [3, 4])
    with pytest.raises(ValueError, match="at least one"):
        tt.evaluate(dc, [0, 1], np.zeros(0, np.int64), head="mlp")
    with pytest.raises(ValueError, match="k must"):
        tt.evaluate(dc, [0, 1], [3], k=33)
    with pytest.raises(ValueError, match="k must"):
        tt.evaluate(dc, [0, 1], [3], k=0)
    with pytest.raises(ValueError, match="mlp_epochs"):
        tt.evaluate(dc, [0, 1], [3], head="mlp", mlp_epochs=0)
    # the graph-class count, not the embedding width (4 here), bounds the labels
    with pytest.raises(ValueError, match="graph 2 has label 2"):
        tt.evaluate(dc, [0, 1], [3], num_classes=2)
    with pytest.raises(ValueError, match="batch_graphs"):
        tt.embed(dc, [0, 1], batch_graphs=0)


def test_evaluate_rejects_negative_labels():
    tt, dc = _trainer_and_corpus([0, 1, -1, 1])
    with pytest.raises(ValueError, match="graph 2 has label -1"):
        tt.evaluate(dc, [0, 1], [3])


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


# (train rows, queries) per rank: unequal shards, and one rank without queries
SHARDS = [(7, 5), (3, 0)]
D, C, K = 6, 5, 3


def _shard(rank):
    g = np.random.default_rng(100 + rank)
    m, q = SHARDS[rank]
    # small integer coordinates: exact distances, so ties are decided by the train index alone
    return (torch.from_numpy(g.integers(-2, 3, (m, D)).astype(np.float32)), torch.from_numpy(g.integers(0, C, m)),
            torch.from_numpy(g.integers(-2, 3, (q, D)).astype(np.float32)), torch.from_numpy(g.integers(0, C, q)))


def _knn_score(a, ya, q, yq):
    if q.size(0) == 0:
        return torch.zeros(1, dtype=torch.int64)
    pred = H.knn_predict(a.numpy(), ya.numpy(), q.numpy(), K)
    return torch.tensor([int((torch.from_numpy(pred) == yq).sum())])


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path[:0] = [os.path.join(root, "two-stage-gnn_b200"), root]
    from tsg.train import gather_score_reduce
    seen = {}

    def score(a, ya, q, yq):
        seen["train"], seen["train_y"] = a.clone(), ya.clone()
        return _knn_score(a, ya, q, yq)
    tot = gather_score_reduce(*_shard(rank), score)
    torch.save(dict(tot=tot, **seen), out + f".{rank}")
    dist.barrier()
    dist.destroy_process_group()


def test_gather_score_reduce_equals_one_process(tmp_path):
    """Train rows gathered in rank order with unequal shard sizes; [correct, count] summed over ranks == the union's"""
    from tsg.train import gather_score_reduce
    world, port, out = 2, _free_port(), str(tmp_path / "r")
    mp.spawn(_worker, args=(world, port, out), nprocs=world, join=True)
    got = [torch.load(out + f".{r}") for r in range(world)]
    parts = [_shard(r) for r in range(world)]
    train = torch.cat([p[0] for p in parts]); train_y = torch.cat([p[1] for p in parts])
    query = torch.cat([p[2] for p in parts]); query_y = torch.cat([p[3] for p in parts])
    for g in got:
        assert torch.equal(g["train"], train) and torch.equal(g["train_y"], train_y), "gathered in rank order"
        assert g["tot"].tolist() == got[0]["tot"].tolist()
    single = gather_score_reduce(train, train_y, query, query_y, _knn_score)          # no process group: no exchange
    assert single.tolist() == got[0]["tot"].tolist()
    assert single[1] == sum(q for _, q in SHARDS)
