"""Host-side checks of the EigenGCN 2stg path (DeviceCorpus.attach_eigen / pack_eigen, WaveTripletTrainer): the C ABI
of tsg_pack_eigen_batch as the ctypes layer declares it, the argument validation, which raises ValueError before any
device work (the corpus here lives in host memory, so any device call would fail differently), and the split of
eigen_synth.make_operands into its clustering and operands_from_clusters."""
import ctypes

import numpy as np
import pytest
import torch

from tsg import eigen_synth, synth


def test_pack_eigen_abi_signature():
    from tsg import _lib
    P, I64 = ctypes.c_void_p, ctypes.c_int64
    # (ids, out node / edge / cluster / coarse ptrs, B, N, E, NC, EC, corpus node_ptr, edge_ptr, label, row, col, F,
    #  corpus cluster_ptr, coarse_ptr, cluster_of, pool_w, pool_stride, J, coarse_row, coarse_col, coarse_w, final_w,
    #  final_stride, Jf, max_nodes, then 20 output pointers and the stream)
    want = [P] * 5 + [I64] * 5 + [P] * 5 + [I64] + [P] * 4 + [I64] * 2 + [P] * 4 + [I64] * 3 + [P] * 21
    assert _lib.lib.tsg_pack_eigen_batch.argtypes == want
    assert _lib.lib.tsg_pack_eigen_batch.restype is ctypes.c_int
    assert _lib.KERNELS_PER_CALL["tsg_pack_eigen_batch"] == 1


@pytest.mark.parametrize("shape,G,pool_size,J,Jf", [("DD", 12, 10, 1, 1), ("PROTEINS", 40, 4, 2, 2),
                                                    ("PROTEINS", 15, 3, 2, 0)])
def test_make_operands_is_bfs_clusters_through_operands_from_clusters(shape, G, pool_size, J, Jf):
    c = synth.make_corpus(shape, G, seed=11)
    ref = eigen_synth.make_operands(c, pool_size, J, Jf)
    cl, order = eigen_synth.bfs_clusters(c, pool_size)
    got = eigen_synth.operands_from_clusters(c, cl, J, Jf, member_order=order)
    for f in ("cluster_ptr", "cluster_of", "coarse_ptr", "coarse_row", "coarse_col", "coarse_w"):
        a, b = getattr(ref, f), getattr(got, f)
        assert a.dtype == b.dtype and np.array_equal(a, b), f
    for f in ("pool_w", "final_w"):
        a, b = getattr(ref, f), getattr(got, f)
        assert len(a) == len(b) and all(x.dtype == y.dtype and np.array_equal(x, y) for x, y in zip(a, b)), f
    # the BFS chunks: cluster k of a graph holds positions k * pool_size .. of its BFS order
    for g in range(G):
        n0, n1 = int(c.node_ptr[g]), int(c.node_ptr[g + 1])
        pos = np.empty(n1 - n0, np.int64); pos[order[n0:n1]] = np.arange(n1 - n0)
        assert np.array_equal(cl[n0:n1], pos // pool_size)


def test_operands_from_clusters_takes_any_clustering():
    c = synth.make_corpus("PROTEINS", 6, seed=2)
    cl = np.concatenate([np.arange(c.num_nodes(g)) % 3 for g in range(6)])     # not contiguous in any order
    op = eigen_synth.operands_from_clusters(c, cl, 2, 1)
    assert np.array_equal(np.diff(op.cluster_ptr), [3] * 6)
    for g in range(6):
        q0, q1 = int(op.coarse_ptr[g]), int(op.coarse_ptr[g + 1])
        r, s, w = op.coarse_row[q0:q1], op.coarse_col[q0:q1], op.coarse_w[q0:q1]
        assert (r != s).all() and (np.diff(r * 3 + s) > 0).all()
        dense = np.zeros((3, 3), np.float32); dense[r, s] = w
        assert np.array_equal(dense, dense.T)
    with pytest.raises(ValueError, match="entries"):
        eigen_synth.operands_from_clusters(c, cl[:-1])
    with pytest.raises(ValueError, match="non-negative"):
        eigen_synth.operands_from_clusters(c, cl - 1)


def _setup(G=8):
    from tsg.feeder import DeviceCorpus
    corpus = synth.make_corpus("PROTEINS", G, seed=4)
    op = eigen_synth.make_operands(corpus, 4, 2, 1)
    dc = DeviceCorpus(corpus, torch.device("cpu"))
    return corpus, op, dc


def test_attach_eigen_checks_the_operands_against_the_corpus():
    import dataclasses
    corpus, op, dc = _setup()
    dc.attach_eigen(op)
    assert dc.eigen["J"] == 2 and dc.eigen["Jf"] == 1
    assert np.array_equal(dc.eigen["nc"], np.diff(op.cluster_ptr))
    assert np.array_equal(dc.eigen["ncoarse"], np.diff(op.coarse_ptr))
    bad = lambda **kw: dataclasses.replace(op, **kw)
    with pytest.raises(ValueError, match="J = 0"):
        dc.attach_eigen(bad(pool_w=[]))
    with pytest.raises(ValueError, match="cluster_of has"):
        dc.attach_eigen(bad(cluster_of=op.cluster_of[:-1]))
    with pytest.raises(ValueError, match=r"pool_w\[1\] has"):
        dc.attach_eigen(bad(pool_w=[op.pool_w[0], op.pool_w[1][:-1]]))
    with pytest.raises(ValueError, match="coarse_w has"):
        dc.attach_eigen(bad(coarse_w=op.coarse_w[:-1]))
    with pytest.raises(ValueError, match=r"final_w\[0\] has"):
        dc.attach_eigen(bad(final_w=[op.final_w[0][1:]]))
    with pytest.raises(ValueError, match="cluster_ptr must be"):
        dc.attach_eigen(bad(cluster_ptr=op.cluster_ptr[:-1]))
    with pytest.raises(ValueError, match="coarse_ptr must be"):
        dc.attach_eigen(bad(coarse_ptr=op.coarse_ptr[::-1].copy()))
    cp = op.cluster_ptr.copy(); cp[1:] += corpus.num_nodes(0)                  # graph 0: more clusters than nodes
    with pytest.raises(ValueError, match="graph 0 has"):
        dc.attach_eigen(bad(cluster_ptr=cp))


def test_pack_eigen_validates_on_the_host():
    from tsg.feeder import DeviceCorpus
    corpus, op, dc = _setup()
    with pytest.raises(ValueError, match="no EigenPooling operands"):
        dc.pack_eigen([0], 1000)
    dc.attach_eigen(op)
    with pytest.raises(ValueError, match="at least one graph id"):
        dc.pack_eigen([], 1000)
    with pytest.raises(ValueError, match="ids must lie"):
        dc.pack_eigen([0, 8], 1000)
    big = int(np.argmax(np.diff(corpus.node_ptr)))
    nb = corpus.num_nodes(big)
    with pytest.raises(ValueError, match=f"graph {big} has {nb} nodes, more than max_nodes = {nb - 1}"):
        dc.pack_eigen([0, big, 1], nb - 1)
    with pytest.raises(ValueError, match="num_pool_matrix = 3"):
        dc.pack_eigen([0], 1000, num_pool_matrix=3)
    with pytest.raises(ValueError, match="num_pool_matrix = 0"):
        dc.pack_eigen([0], 1000, num_pool_matrix=0)
    with pytest.raises(ValueError, match="num_pool_final_matrix = 2"):
        dc.pack_eigen([0], 1000, num_pool_final_matrix=2)
    edge_free = synth.Corpus("one-node", np.array([0, 1, 3]), np.array([0, 0, 2]), np.array([0, 1]), np.array([1, 0]),
                             np.zeros(3, np.int32), np.array([0, 1]), 3)
    ef = DeviceCorpus(edge_free, torch.device("cpu"))
    ef.attach_eigen(eigen_synth.make_operands(edge_free, 4, 1, 1))
    with pytest.raises(ValueError, match="no edges"):
        ef.pack_eigen([0, 0], 1000)
    dense_x = DeviceCorpus(corpus, torch.device("cpu"), dense_x=np.zeros((int(corpus.node_ptr[-1]), 4), np.float32))
    dense_x.attach_eigen(op)
    with pytest.raises(ValueError, match="dense_x"):
        dense_x.pack_eigen([0], 1000)


def test_wave_trainer_refuses_what_the_operands_cannot_feed():
    from tsg import dense
    from tsg.train import WaveTripletTrainer
    corpus, op, dc = _setup()
    two_levels = dense.PackedWaveEncoder(3, 8, 8, 2, 2, num_pool_matrix=1, num_pool_final_matrix=1, pool_sizes=[4, 4])
    with pytest.raises(ValueError, match="2 pooling levels"):
        WaveTripletTrainer(two_levels)
    with pytest.raises(TypeError):
        WaveTripletTrainer(torch.nn.Linear(3, 2))
    dc.attach_eigen(op)
    for J, Jf, what in ((3, 1, "num_pool_matrix = 3"), (1, 2, "num_pool_final_matrix = 2")):
        tt = WaveTripletTrainer(dense.PackedWaveEncoder(3, 8, 8, 2, 2, num_pool_matrix=J, num_pool_final_matrix=Jf,
                                                        pool_sizes=[4]))
        with pytest.raises(ValueError, match=what):
            tt.embed(dc, [0, 1])
        with pytest.raises(ValueError, match=what):
            tt.run_from_ids(dc, [(np.array([0, 1, 2]), torch.zeros(1, 3, dtype=torch.int64))])
    tt = WaveTripletTrainer(dense.PackedWaveEncoder(5, 8, 8, 2, 2, num_pool_matrix=1, num_pool_final_matrix=1,
                                                    pool_sizes=[4]))
    with pytest.raises(ValueError, match="3 node labels, the model takes input_dim = 5"):
        tt.evaluate(dc, [0, 1], [2])
    tt = WaveTripletTrainer(dense.PackedWaveEncoder(3, 8, 8, 2, 2, num_pool_matrix=2, num_pool_final_matrix=1,
                                                    pool_sizes=[4]), max_nodes=10)
    with pytest.raises(ValueError, match="more than max_nodes = 10"):
        tt.embed(dc, np.arange(8))
    with pytest.raises(ValueError, match="batch_graphs"):
        tt.embed(dc, [0], batch_graphs=0)
    with pytest.raises(ValueError, match="head"):
        tt.evaluate(dc, [0, 1], [2], head="svm")
