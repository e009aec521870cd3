"""Host-side checks of the dense-encoder 2stg path (DeviceCorpus.pack_dense, DenseTripletTrainer): the C ABI of
tsg_pack_dense_batch as the ctypes layer declares it, and the argument validation, which raises ValueError before any
device work (the corpus here lives in host memory, so any device call would fail differently)."""
import ctypes

import numpy as np
import pytest
import torch

from tsg import synth


def test_pack_dense_abi_signature():
    from tsg import _lib
    P, I64 = ctypes.c_void_p, ctypes.c_int64
    # (ids, out_node_ptr, out_edge_ptr, B, N, E, corpus_node_ptr, corpus_edge_ptr, corpus_row, corpus_col, table,
    #  max_nodes, feat, x_out, has_pad, rowptr, colidx, val, eid, t_eid, status, stream)
    assert _lib.lib.tsg_pack_dense_batch.argtypes == [P, P, P, I64, I64, I64, P, P, P, P, P, I64, I64,
                                                      P, P, P, P, P, P, P, P, P]
    assert _lib.lib.tsg_pack_dense_batch.restype is ctypes.c_int
    assert _lib.KERNELS_PER_CALL["tsg_pack_dense_batch"] == 1


def _setup(kind="gat", max_nodes=1000, model_max_nodes=None, F=32):
    from tsg import dense, diffpool, gat
    from tsg.feeder import DeviceCorpus
    from tsg.train import DenseTripletTrainer
    corpus = synth.make_corpus("DD", 8, seed=4)
    corpus.y = np.array([0, 1, 2, 1, 0, 1, 2, 0], np.int64)
    if kind == "gat":
        model = gat.PackedGatEncoder(32, 8, 8, 2, num_layers=2, num_heads=[2, 2])
    elif kind == "base":
        model = dense.PackedGcnEncoder(32, 8, 8, 2, 2)
    else:
        model = diffpool.PackedSoftPoolEncoder(model_max_nodes or max_nodes, 32, 8, 8, 2, 2, 8, assign_ratio=0.1)
    table = torch.zeros(max_nodes, F)
    return corpus, DeviceCorpus(corpus, torch.device("cpu")), model, table, DenseTripletTrainer


def test_pack_dense_validates_on_the_host():
    from tsg.feeder import DeviceCorpus
    corpus, dc, _, table, _ = _setup()
    with pytest.raises(ValueError, match="at least one graph id"):
        dc.pack_dense([], table, 1000)
    with pytest.raises(ValueError, match="ids must lie"):
        dc.pack_dense([0, 8], table, 1000)
    big = int(np.argmax(np.diff(corpus.node_ptr)))
    nb = corpus.num_nodes(big)
    with pytest.raises(ValueError, match=f"graph {big} has {nb} nodes, more than max_nodes = {nb - 1}"):
        dc.pack_dense([0, big, 1], table[: nb - 1], nb - 1)
    with pytest.raises(ValueError, match="feature table must be"):
        dc.pack_dense([0, 1], table[:999], 1000)
    edge_free = synth.Corpus("one-node", np.array([0, 1, 3]), np.array([0, 0, 2]), np.array([0, 1]), np.array([1, 0]),
                             np.zeros(3, np.int32), np.array([0, 1]), 3)
    ef = DeviceCorpus(edge_free, torch.device("cpu"))
    with pytest.raises(ValueError, match="no edges"):
        ef.pack_dense([0, 0], table, 1000)
    with pytest.raises(ValueError, match="float32"):
        dc.pack_dense([0, 1], table.double(), 1000)
    dense_x = DeviceCorpus(corpus, torch.device("cpu"), dense_x=np.zeros((int(corpus.node_ptr[-1]), 4), np.float32))
    with pytest.raises(ValueError, match="dense_x"):
        dense_x.pack_dense([0], table, 1000)


def test_trainer_validates_its_model_and_table():
    _, _, model, table, T = _setup("diffpool", max_nodes=1000, model_max_nodes=500)
    with pytest.raises(ValueError, match="max_num_nodes = 500"):
        T(model, table, 1000)
    T(model, table[:500], 500)
    _, _, model, table, T = _setup("base", F=16)
    with pytest.raises(ValueError, match="16 columns, the model takes 32"):
        T(model, table, 1000)
    _, _, model, table, T = _setup("gat")
    with pytest.raises(ValueError, match="feature table must be"):
        T(model, table[:100], 1000)
    with pytest.raises(TypeError):
        T(torch.nn.Linear(32, 4), table, 1000)


def test_evaluate_and_embed_validate_their_arguments():
    corpus, dc, model, table, T = _setup("gat")
    tt = T(model, table, 1000)
    with pytest.raises(ValueError, match="head"):
        tt.evaluate(dc, [0, 1, 2], [3, 4], head="svm")
    with pytest.raises(ValueError, match="at least one"):
        tt.evaluate(dc, [], [3, 4])
    with pytest.raises(ValueError, match="k must"):
        tt.evaluate(dc, [0, 1], [3], k=33)
    with pytest.raises(ValueError, match="k must"):
        tt.evaluate(dc, [0, 1], [3], k=0)
    with pytest.raises(ValueError, match="mlp_epochs"):
        tt.evaluate(dc, [0, 1], [3], head="mlp", mlp_epochs=0)
    with pytest.raises(ValueError, match="graph 2 has label 2"):
        tt.evaluate(dc, [0, 1], [3], num_classes=2)
    with pytest.raises(ValueError, match="batch_graphs"):
        tt.embed(dc, [0, 1], batch_graphs=0)
    with pytest.raises(ValueError, match="at least one graph id"):
        tt.embed(dc, [])
    small = T(model, table[:30], 30)
    with pytest.raises(ValueError, match="more than max_nodes = 30"):
        small.evaluate(dc, [0, 1], [3])
    with pytest.raises(ValueError, match="more than max_nodes = 30"):
        small.run_from_ids(dc, [(np.array([0, 1, 2]), torch.zeros(1, 3, dtype=torch.int64))])
