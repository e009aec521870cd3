"""Host-side checks of the dense encoders' supervised settings (K16, DenseClassifierTrainer, WaveClassifierTrainer): the
C ABI of the K16 entries as the ctypes layer declares it, their refusal of bad descriptors before any device work (the
workspace queries are pure host code), and the trainers' argument validation, which raises ValueError / TypeError on the
host (the corpus here lives in host memory, so any device call would fail differently)."""
import ctypes

import numpy as np
import pytest
import torch

from tsg import synth

EINVAL = -1


def test_pred_ce_abi_signatures():
    from tsg import _lib
    P, I64, SZ = ctypes.c_void_p, ctypes.c_int64, ctypes.c_size_t
    L = _lib.lib
    assert L.tsg_pred_ce_workspace_bytes.argtypes == [P, I64] and L.tsg_pred_ce_workspace_bytes.restype is SZ
    assert L.tsg_pred_classify_workspace_bytes.argtypes == [P, I64]
    # (head, r, y, G, loss, logits_out, status, workspace, workspace_bytes, stream)
    assert L.tsg_pred_ce_fwd.argtypes == [P, P, P, I64, P, P, P, P, SZ, P]
    # (head, r, y, G, dloss, dr, dweight[], dbias[], workspace, workspace_bytes, stream)
    assert L.tsg_pred_ce_bwd.argtypes == [P, P, P, I64, P, P, P, P, P, SZ, P]
    # (head, r, y, G, pred, logits_out, correct, ce_sum, status, workspace, workspace_bytes, stream)
    assert L.tsg_pred_classify.argtypes == [P, P, P, I64, P, P, P, P, P, P, SZ, P]
    for n in ("tsg_pred_ce_fwd", "tsg_pred_ce_bwd", "tsg_pred_classify"):
        assert getattr(L, n).restype is ctypes.c_int
    assert ctypes.sizeof(_lib.PredHead) == 8 * (2 + 8 + 2 + 8 + 8)


def _head(in_dim, outs, relu_mask=0, softmax_first=0):
    """a descriptor with fake (never dereferenced) weight pointers; num_layers = len(outs), the struct holds 8"""
    from tsg import _lib
    h = _lib.PredHead()
    h.num_layers, h.in_dim, h.relu_mask, h.softmax_first = len(outs), in_dim, relu_mask, softmax_first
    for l, o in enumerate(outs[:8]):
        h.out_dim[l], h.weight[l], h.bias[l] = o, 4096 * (l + 1), None
    return h


GOOD = [(64, [32, 2]), (192, [50, 2]), (32, []), (256, [256] * 8), (1, [1])]
BAD = [(64, [32] * 8 + [2], "9 layers"), (64, [257, 2], "width 257"), (257, [2], "input width 257"),
       (64, [32, 0], "C 0"), (0, [], "C 0 without layers"), (64, [-1, 2], "negative width")]


def test_pred_ce_workspace_queries_are_pure_host():
    from tsg import _lib
    for in_dim, outs in GOOD:
        h = _head(in_dim, outs)
        for G in (1, 7, 3504):
            assert _lib.lib.tsg_pred_ce_workspace_bytes(ctypes.byref(h), G) > 0
            assert _lib.lib.tsg_pred_classify_workspace_bytes(ctypes.byref(h), G) > 0
        # activations and deltas: G rows of every layer's width
        small, big = (_lib.lib.tsg_pred_ce_workspace_bytes(ctypes.byref(h), G) for G in (1, 100000))
        assert big - small >= 2 * 4 * 99999 * sum(outs)
    for in_dim, outs, what in BAD:
        h = _head(in_dim, outs)
        assert _lib.lib.tsg_pred_ce_workspace_bytes(ctypes.byref(h), 7) == 0, what
        assert _lib.lib.tsg_pred_classify_workspace_bytes(ctypes.byref(h), 7) == 0, what
    assert _lib.lib.tsg_pred_ce_workspace_bytes(None, 7) == 0
    assert _lib.lib.tsg_pred_ce_workspace_bytes(ctypes.byref(_head(64, [2])), 0) == 0


def test_pred_ce_entries_refuse_bad_arguments_before_any_device_work():
    from tsg import _lib
    L = _lib.lib
    fake = 1 << 20
    arr = (ctypes.c_void_p * 8)(*([fake] * 8))

    def calls(h, G, r=fake, y=fake, out=fake, ws=fake):
        yield L.tsg_pred_ce_fwd(ctypes.byref(h), r, y, G, out, None, None, ws, 1 << 30, None)
        yield L.tsg_pred_ce_bwd(ctypes.byref(h), r, y, G, None, None, arr, arr, ws, 1 << 30, None)
        yield L.tsg_pred_classify(ctypes.byref(h), r, None, G, out, None, None, None, None, ws, 1 << 30, None)

    for in_dim, outs, what in BAD:
        assert all(rc == EINVAL for rc in calls(_head(in_dim, outs), 7)), what
        assert "bad head" in _lib.last_error()
    for G in (0, -3):
        assert all(rc == EINVAL for rc in calls(_head(64, [32, 2]), G)), G
    assert all(rc == EINVAL for rc in calls(_head(64, [32, 2]), 7, r=None))
    assert all(rc == EINVAL for rc in calls(_head(64, [32, 2]), 7, out=None))
    assert all(rc == EINVAL for rc in calls(_head(64, [32, 2]), 7, ws=None))
    missing_weight = _head(64, [32, 2]); missing_weight.weight[1] = None
    assert all(rc == EINVAL for rc in calls(missing_weight, 7))
    h = _head(64, [32, 2])
    assert L.tsg_pred_ce_bwd(ctypes.byref(h), fake, fake, 7, None, None, None, None, fake, 1 << 30, None) == EINVAL
    # correct / ce_sum without labels
    assert L.tsg_pred_classify(ctypes.byref(h), fake, None, 7, fake, None, fake, None, None, fake, 1 << 30, None) == EINVAL
    assert "labels" in _lib.last_error()


def test_check_pred_head_limits():
    from tsg import ops
    ops.check_pred_head(256, [256] * 8)
    ops.check_pred_head(32, [])
    for in_dim, outs, what in BAD:
        with pytest.raises(ValueError, match="beyond K16's limits"):
            ops.check_pred_head(in_dim, outs)


# ------------------------------------------------------------------------------------------ trainers
def _corpus(y, shape="DD"):
    from tsg.feeder import DeviceCorpus
    corpus = synth.make_corpus(shape, len(y), seed=4)
    corpus.y = np.asarray(y, np.int64)
    return corpus, DeviceCorpus(corpus, torch.device("cpu"))


def _model(kind, final_dim, pred_hidden_dims=(), embedding_dim=8, label_dim=2):
    from tsg import dense, diffpool, gat
    if kind == "gat":
        return gat.PackedGatEncoder(32, 8, embedding_dim, label_dim, num_layers=2, num_heads=[2, 2], final_dim=final_dim)
    if kind == "base":
        return dense.PackedGcnEncoder(32, 8, embedding_dim, label_dim, 2, pred_hidden_dims=pred_hidden_dims,
                                      final_dim=final_dim)
    return diffpool.PackedSoftPoolEncoder(1000, 32, 8, embedding_dim, label_dim, 2, 8, assign_ratio=0.1,
                                          pred_hidden_dims=pred_hidden_dims, final_dim=final_dim)


TABLE = torch.zeros(1000, 32)


@pytest.mark.parametrize("kind", ["base", "diffpool", "gat"])
def test_classifier_setups(kind):
    from tsg.train import DenseClassifierTrainer as T
    t = T(_model(kind, "number_classes", label_dim=3), TABLE, setting="original")
    assert (t.num_classes, t.softmax_first) == (3, False)
    assert [w.shape[0] for w, _, _ in t._layers()] == ([3] if kind == "gat" else [8, 3])
    t = T(_model(kind, "pretrain" if kind != "gat" else "output_dim"), TABLE, setting="2stg+")
    assert t.softmax_first
    assert t.num_classes == (8 if kind == "gat" else 2)
    assert [tuple(w.shape) for w, _, _ in t._layers()] == ([] if kind == "gat" else [(8, t.model.map_model.in_features), (2, 8)])
    if kind != "gat":
        relus = [r for _, _, r in T(_model(kind, "number_classes", pred_hidden_dims=(50,)), TABLE)._layers()]
        assert relus == [True, False, True, False]          # pre_pred_model: Linear ReLU Linear, pred_model: the same


@pytest.mark.parametrize("kind", ["base", "diffpool", "gat"])
def test_classifier_refuses_a_final_dim_that_does_not_fit_the_setting(kind):
    from tsg.train import DenseClassifierTrainer as T
    for fd in ("output_dim", "pretrain"):
        with pytest.raises(ValueError, match="must not be 'output_dim' or 'pretrain'"):
            T(_model(kind, fd), TABLE, setting="original")
    if kind != "gat":
        for fd in ("output_dim", "number_classes"):
            with pytest.raises(ValueError, match="final_dim must be 'pretrain'"):
                T(_model(kind, fd), TABLE, setting="2stg+")
    else:                                                   # GAT's 2stg+ logits are the readout, whatever final_dim
        for fd in ("output_dim", "pretrain", "number_classes"):
            T(_model(kind, fd), TABLE, setting="2stg+")
    with pytest.raises(ValueError, match="setting must be"):
        T(_model(kind, "number_classes"), TABLE, setting="2stg")
    with pytest.raises(TypeError):
        T(torch.nn.Linear(32, 2), TABLE)


def test_classifier_refuses_linkpred_outside_diffpool_original():
    from tsg.train import DenseClassifierTrainer as T
    T(_model("diffpool", "number_classes"), TABLE, linkpred=True)
    for kind, fd, setting in (("base", "number_classes", "original"), ("gat", "number_classes", "original"),
                              ("diffpool", "pretrain", "2stg+"), ("base", "pretrain", "2stg+")):
        with pytest.raises(ValueError, match="linkpred"):
            T(_model(kind, fd), TABLE, setting=setting, linkpred=True)


def test_classifier_refuses_a_head_beyond_k16():
    from tsg import dense
    from tsg.train import DenseClassifierTrainer as T, WaveClassifierTrainer as W
    with pytest.raises(ValueError, match="beyond K16's limits"):
        T(_model("base", "number_classes", pred_hidden_dims=(300,)), TABLE)
    with pytest.raises(ValueError, match="beyond K16's limits"):
        T(_model("base", "number_classes", pred_hidden_dims=(8,) * 4), TABLE)         # 10 layers
    with pytest.raises(ValueError, match="beyond K16's limits"):
        T(_model("gat", "output_dim", embedding_dim=300), TABLE, setting="2stg+")      # 300 classes
    with pytest.raises(ValueError, match="beyond K16's limits"):
        T(_model("base", "number_classes", label_dim=257), TABLE)
    T(_model("base", "number_classes", label_dim=256), TABLE)
    with pytest.raises(ValueError, match="beyond K16's limits"):                     # readout width 3 * (50 + 50) = 300
        W(dense.PackedWaveEncoder(3, 50, 50, 2, 2, num_pool_matrix=2, num_pool_final_matrix=1, pool_sizes=[4]))


def test_classifier_refuses_labels_outside_the_class_count():
    from tsg.train import DenseClassifierTrainer as T
    corpus, dc = _corpus([0, 1, 2, 1, 0, 1, 2, 0])
    t = T(_model("base", "pretrain"), TABLE, setting="2stg+")
    with pytest.raises(ValueError, match="graph 2 has label 2, outside \\[0, 2\\): 2stg\\+ takes map2_model's 2 outputs"):
        t.evaluate(dc, [0, 1])
    with pytest.raises(ValueError, match="map2_model's 2 outputs"):
        t.run_from_ids(dc, [np.array([0, 1])])
    with pytest.raises(ValueError, match="map2_model's 2 outputs"):
        T(_model("diffpool", "pretrain"), TABLE, setting="2stg+").evaluate(dc, [0])
    with pytest.raises(ValueError, match="graph 2 has label 2, outside \\[0, 2\\)$"):
        T(_model("base", "number_classes"), TABLE).run_from_ids(dc, [np.array([0, 1])])
    T(_model("base", "number_classes", label_dim=3), TABLE)._check_labels(dc)
    corpus, dc = _corpus([0, 1, 8, 1])
    g = T(_model("gat", "output_dim"), TABLE, setting="2stg+")
    with pytest.raises(ValueError, match="graph 2 has label 8, outside \\[0, 8\\): 2stg\\+ takes the GAT readout's "
                                         "embedding_dim = 8 columns"):
        g.evaluate(dc, [0, 1])
    T(_model("gat", "output_dim", embedding_dim=9), TABLE, setting="2stg+")._check_labels(dc)
    dc.y, dc.y_host, dc.labels_checked = None, None, None
    with pytest.raises(ValueError, match="no graph labels"):
        g.run_from_ids(dc, [np.array([0])])


def test_classifier_validates_batches_and_tables():
    from tsg.train import DenseClassifierTrainer as T
    corpus, dc = _corpus([0, 1, 1, 0])
    t = T(_model("base", "number_classes"), TABLE)
    with pytest.raises(ValueError, match="batch_graphs"):
        t.evaluate(dc, [0, 1], batch_graphs=0)
    with pytest.raises(ValueError, match="at least one graph id"):
        t.evaluate(dc, [])
    with pytest.raises(ValueError, match="ids must lie"):
        t.run_from_ids(dc, [np.array([0, 4])])
    small = T(_model("base", "number_classes"), TABLE[:30], 30)
    with pytest.raises(ValueError, match="more than max_nodes = 30"):
        small.evaluate(dc, [0, 1])
    with pytest.raises(ValueError, match="16 columns, the model takes 32"):
        T(_model("base", "number_classes"), torch.zeros(1000, 16))
    with pytest.raises(ValueError, match="max_num_nodes = 1000"):
        T(_model("diffpool", "number_classes"), TABLE[:500], 500)


def test_wave_classifier_refusals():
    from tsg import dense, eigen_synth
    from tsg.train import WaveClassifierTrainer as W
    corpus, dc = _corpus([0, 1, 2, 1, 0, 1, 2, 0], "PROTEINS")
    dc.attach_eigen(eigen_synth.make_operands(corpus, 4, 2, 1))
    with pytest.raises(TypeError):
        W(_model("base", "number_classes"))
    with pytest.raises(ValueError, match="2 pooling levels"):
        W(dense.PackedWaveEncoder(3, 8, 8, 2, 2, num_pool_matrix=1, num_pool_final_matrix=1, pool_sizes=[4, 4]))
    with pytest.raises(TypeError):                          # no link-prediction term for EigenGCN
        W(dense.PackedWaveEncoder(3, 8, 8, 2, 2, pool_sizes=[4]), linkpred=True)
    for setting in ("original", "2stg+"):
        w = W(dense.PackedWaveEncoder(3, 8, 8, 2, 2, num_pool_matrix=2, num_pool_final_matrix=1, pool_sizes=[4]),
              setting=setting)
        assert (w.num_classes, w.softmax_first) == (2, False)
        with pytest.raises(ValueError, match="graph 2 has label 2, outside \\[0, 2\\)"):
            w.evaluate(dc, [0, 1])
        with pytest.raises(ValueError, match="graph 2 has label 2"):
            w.run_from_ids(dc, [np.array([0, 1])])
    w = W(dense.PackedWaveEncoder(5, 8, 8, 3, 2, num_pool_matrix=1, num_pool_final_matrix=1, pool_sizes=[4]))
    with pytest.raises(ValueError, match="3 node labels, the model takes input_dim = 5"):
        w.evaluate(dc, [0, 1])
    w = W(dense.PackedWaveEncoder(3, 8, 8, 3, 2, num_pool_matrix=3, num_pool_final_matrix=1, pool_sizes=[4]))
    with pytest.raises(ValueError, match="num_pool_matrix = 3"):
        w.run_from_ids(dc, [np.array([0, 1])])
