"""Host-side refusals of DeviceCorpus.build_eigen: every one raises ValueError before any device work, so they run on
a CPU-resident DeviceCorpus; and the C ABI of the K17 entries."""
import ctypes

import numpy as np
import pytest
import torch

from tsg import synth
from test_eigen_2stg_gpu import _corpus_of, _sym


def _dc(corpus, **kw):
    from tsg.feeder import DeviceCorpus
    return DeviceCorpus(corpus, torch.device("cpu"), **kw)


def test_k17_abi_signatures():
    from tsg import _lib
    P, I64 = ctypes.c_void_p, ctypes.c_int64
    assert _lib.lib.tsg_eigen_bfs_clusters.argtypes == [P] * 4 + [I64] * 6 + [P] * 9
    assert _lib.lib.tsg_eigen_group_clusters.argtypes == [P] * 4 + [I64] * 5 + [P] * 9
    assert _lib.lib.tsg_eigen_coarse.argtypes == [P, I64, I64] + [P] * 13
    assert _lib.lib.tsg_eigen_final.argtypes == [P] * 4 + [I64] * 5 + [P, I64, P]


def test_build_eigen_refuses_on_the_host():
    corpus = synth.make_corpus("PROTEINS", 6, seed=4)
    Nt = int(corpus.node_ptr[-1])
    dc = _dc(corpus)
    for kw, msg in [(dict(pool_size=0), "pool_size = 0"), (dict(pool_size=33), "pool_size = 33"),
                    (dict(num_pool_matrix=0), "num_pool_matrix = 0"), (dict(num_pool_final_matrix=-1), "= -1"),
                    (dict(cluster_of=np.zeros(Nt - 1, np.int64)), f"has {Nt - 1} entries"),
                    (dict(cluster_of=torch.zeros(Nt + 1, dtype=torch.int64)), f"has {Nt + 1} entries"),
                    (dict(cluster_of=-np.ones(Nt, np.int64)), "non-negative"),
                    (dict(cluster_of=-torch.ones(Nt, dtype=torch.int32)), "non-negative"),
                    (dict(cluster_of=np.zeros(Nt, np.float32)), "integer"),
                    (dict(cluster_of=torch.zeros(Nt)), "integer")]:
        with pytest.raises(ValueError, match=msg):
            dc.build_eigen(**kw)
    with pytest.raises(ValueError, match="dense_x"):
        _dc(corpus, dense_x=np.zeros((Nt, 4), np.float32)).build_eigen()
    unsorted = synth.Corpus("x", corpus.node_ptr, corpus.edge_ptr, corpus.row[::-1].copy(), corpus.col[::-1].copy(),
                            corpus.node_label, corpus.y, corpus.num_node_labels)
    with pytest.raises(ValueError, match="coalesced"):
        _dc(unsorted).build_eigen()
    big = _corpus_of([(3,) + _sym([(0, 1), (1, 2)]), (19371, [], [])])
    with pytest.raises(ValueError, match="graph 1 has 19371 nodes"):
        _dc(big).build_eigen()
    assert "eigen" not in dc.__dict__
