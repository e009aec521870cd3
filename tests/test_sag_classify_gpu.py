"""The supervised ("original") setting of Code/sag/train.py on the GPU: the native NLL step (tsg_sag_nll_step_compact)
against the oracle, against its own halves and against the autograd path; the classification forward
(tsg_sag_classify_compact) against the unmodified reference glue's output and a graph-by-graph oracle `test()` loop;
ClassifierTrainer; the wide head backward (nhid 128) in both the NLL and the triplet step; the label range check."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import grad_check, rel_err
from golden_util import load_sag_glue
from oracle import pyg_ref as R
from tsg import synth

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _compact(corpus, dev):
    from tsg import ops
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a).astype(dt)).to(dev)
    return ops.CompactBatch(t(corpus.node_label, np.int32), t(corpus.row, np.int32), t(corpus.col, np.int32),
                            t(corpus.node_ptr, np.int64), t(corpus.edge_ptr, np.int64), corpus.num_node_labels,
                            int(np.diff(corpus.edge_ptr).max()), True)


def _corpus(shape, G, C, seed):
    corpus = synth.make_corpus(shape, G, seed=seed)
    if shape == "PROTEINS":          # 3 node labels make exact score ties (DESIGN 2): widen the alphabet
        corpus.node_label[:] = np.random.default_rng(1).integers(0, 89, corpus.node_label.shape[0]); corpus.num_node_labels = 89
    corpus.y = np.random.default_rng(seed).integers(0, C, G).astype(np.int64)
    return corpus


def _model(corpus, nhid, C, dev, dropout=0.5, seed=9):
    from tsg import nn as tnn
    params = R.init_sag_params(corpus.num_node_labels, nhid, C, seed=seed)
    model = tnn.PackedSAGNet(corpus.num_node_labels, nhid, C, 0.5, dropout).to(dev)
    model.load_state_dict(params)
    return model, params


def _mask(G, nhid, seed=3):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(G, nhid, generator=g) >= 0.5).float() * 2.0


@pytest.mark.parametrize("shape,G,nhid,C", [("DD", 24, 32, 2), ("PROTEINS", 120, 32, 6), ("DD", 6, 128, 2)])
def test_nll_step_matches_oracle_and_autograd(cuda, shape, G, nhid, C):
    from tsg import nn as tnn, ops
    corpus = _corpus(shape, G, C, 41)
    b = synth.pack(corpus)
    cb = _compact(corpus, cuda)
    model, params = _model(corpus, nhid, C, cuda)
    model.train()
    y = torch.from_numpy(corpus.y)
    mask = _mask(G, nhid)
    assert model.native_step_supported(cb, corpus.node_ptr)
    loss, emb = model.native_nll_step(cb, corpus.node_ptr, y.to(cuda), dropout_mask=mask.to(cuda), return_emb=True)
    grads = {k: p.grad.clone() for k, p in model.named_parameters()}
    tnn.check_fused_status()
    res = {}
    for dt in (torch.float32, torch.float64):
        po = {k: v.clone().to(dt).requires_grad_(True) for k, v in params.items()}
        emb_o = R.sag_net_forward(po, torch.from_numpy(b["x"]).to(dt), torch.from_numpy(b["edge_index"]),
                                  torch.from_numpy(b["batch"]), 0.5, dropout_mask=mask.to(dt))
        loss_o = F.nll_loss(emb_o, y)
        loss_o.backward()
        res[dt] = (emb_o.detach(), loss_o.detach(), {k: v.grad for k, v in po.items()})
    assert rel_err(emb, res[torch.float32][0]) <= TOL
    assert rel_err(loss, res[torch.float32][1]) <= TOL
    fwd_noise = max(rel_err(res[torch.float32][0], res[torch.float64][0]), 1e-7)
    for k in grads:
        grad_check(grads[k], res[torch.float32][2][k], res[torch.float64][2][k], TOL, k, fwd_noise)
    # the autograd path: K10 through autograd + the ops.linear head + ATen nll_loss
    model.zero_grad(set_to_none=True)
    plan, ptrs = model._level_plan(corpus.node_ptr, cuda)
    zenc = model._encode_compact(cb, plan, ptrs)
    lin = lambda layer, t: ops.linear(t, layer.weight.t().contiguous(), layer.bias)
    h1 = torch.relu(lin(model.lin1, zenc)) * mask.to(cuda)
    emb_a = torch.log_softmax(lin(model.lin3, torch.relu(lin(model.lin2, h1))), dim=-1)
    loss_a = F.nll_loss(emb_a, y.to(cuda))
    loss_a.backward()
    assert rel_err(emb, emb_a) <= 2e-6 and rel_err(loss, loss_a) <= 2e-6
    for k, p in model.named_parameters():
        grad_check(grads[k], p.grad, res[torch.float64][2][k], 5e-5, "vs autograd " + k, fwd_noise)


@pytest.mark.parametrize("nhid,C", [(32, 2), (128, 64)])
def test_nll_step_equals_its_halves_bitwise(cuda, nhid, C):
    """tsg_sag_nll_step_compact == tsg_sag_step_fwd_compact + F.nll_loss through autograd + tsg_sag_step_bwd_compact:
    identical embeddings and gradients (the same demb enters the same backward), and run to run reproducible."""
    from tsg import nn as tnn
    corpus = _corpus("DD", 18, C, 77)
    cb = _compact(corpus, cuda)
    model, _ = _model(corpus, nhid, C, cuda)
    model.train()
    y = torch.from_numpy(corpus.y).to(cuda)
    mask = _mask(18, nhid).to(cuda)
    loss1, emb1 = model.native_nll_step(cb, corpus.node_ptr, y, dropout_mask=mask, return_emb=True)
    loss1 = loss1.clone()
    g1 = {k: p.grad.clone() for k, p in model.named_parameters()}
    emb2, ctx = model.native_forward(cb, corpus.node_ptr, dropout_mask=mask)
    e = emb2.clone().requires_grad_(True)
    loss2 = F.nll_loss(e, y)
    loss2.backward()
    model.native_backward(ctx, e.grad)
    assert torch.equal(emb1, emb2)
    assert abs(float(loss1) - float(loss2)) <= 1e-6 * abs(float(loss2))          # two summation orders of the same mean
    for k, p in model.named_parameters():
        assert torch.equal(g1[k], p.grad), k
    loss3 = model.native_nll_step(cb, corpus.node_ptr, y, dropout_mask=mask).clone()
    assert torch.equal(loss1, loss3)
    for k, p in model.named_parameters():
        assert torch.equal(g1[k], p.grad), "rerun " + k
    tnn.check_fused_status()


def test_classify_matches_the_reference_glue_fixture(cuda):
    """log-probabilities vs the unmodified network.py's output (tests/golden/sag_glue.npz), argmax equal; pred / logp
    bitwise equal with the graph-resident kernels (K13) on and off; totals == the reference's test() loop over it."""
    from tsg import _lib, nn as tnn, ops
    d = load_sag_glue()
    model = tnn.PackedSAGNet(d["F"], d["nhid"], d["C"], 0.5, 0.5).to(cuda)
    model.load_state_dict(d["params"])
    model.train()                                   # native_classify is the eval-mode forward whatever the flag says
    t = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a)).to(dt).to(cuda)
    cb = ops.CompactBatch(t(d["label"], torch.int32), t(d["local_row"], torch.int32), t(d["local_col"], torch.int32),
                          t(d["node_ptr"], torch.int64), t(d["edge_ptr"], torch.int64), d["F"],
                          int(np.diff(d["edge_ptr"]).max()), True)
    y = torch.from_numpy(np.random.default_rng(5).integers(0, d["C"], d["G"]).astype(np.int64))
    pred, logp, correct, nll_sum = model.native_classify(cb, d["node_ptr"], y.to(cuda))
    tnn.check_fused_status()
    assert rel_err(logp, d["emb"]) <= TOL
    pred_ref = d["emb"].max(dim=1)[1]
    assert torch.equal(pred.cpu(), pred_ref)
    correct_ref, loss_ref = 0, 0.0
    for g in range(d["G"]):                         # Code/sag/train.py:19-29, one graph per batch
        out = d["emb"][g:g + 1]
        correct_ref += int(out.max(dim=1)[1].eq(y[g:g + 1]).sum().item())
        loss_ref += F.nll_loss(out, y[g:g + 1], reduction="sum").item()
    assert int(correct.item()) == correct_ref
    assert abs(float(nll_sum.item()) - loss_ref) <= TOL * abs(loss_ref)
    prev = _lib.lib.tsg_sag_set_fused(0)
    try:
        pred0, logp0, correct0, nll0 = model.native_classify(cb, d["node_ptr"], y.to(cuda))
    finally:
        _lib.lib.tsg_sag_set_fused(prev)
    assert torch.equal(pred0, pred) and torch.equal(logp0, logp)
    assert torch.equal(correct0, correct) and torch.equal(nll0, nll_sum)


@pytest.mark.parametrize("nhid,C", [(32, 2), (128, 6)])
def test_evaluate_matches_the_oracle_test_loop(cuda, nhid, C, monkeypatch):
    """ClassifierTrainer.evaluate over several packed batches == test() of Code/sag/train.py:19-29 run graph by graph on
    the oracle: correct count exactly, mean NLL to 1e-5; the autograd evaluation agrees."""
    from tsg import nn as tnn
    from tsg.feeder import DeviceCorpus
    from tsg.train import ClassifierTrainer
    G = 40
    corpus = _corpus("DD", G, C, 12)
    model, params = _model(corpus, nhid, C, cuda)
    trainer = ClassifierTrainer(model)
    dc = DeviceCorpus(corpus, cuda)
    ids = np.random.default_rng(2).permutation(G)[:33]
    acc, nll = trainer.evaluate(dc, ids, batch_graphs=8)
    assert model.training, "evaluate restores the training flag"
    correct_ref, loss_ref = 0, 0.0
    for g in ids.tolist():
        one = synth.pack(corpus, [g])
        out = R.sag_net_forward(params, torch.from_numpy(one["x"]), torch.from_numpy(one["edge_index"]),
                                torch.from_numpy(one["batch"]), 0.5)
        yg = torch.from_numpy(corpus.y[g:g + 1])
        correct_ref += int(out.max(dim=1)[1].eq(yg).sum().item())
        loss_ref += F.nll_loss(out, yg, reduction="sum").item()
    assert round(acc * len(ids)) == correct_ref
    assert abs(nll - loss_ref / len(ids)) <= TOL * abs(loss_ref / len(ids))
    monkeypatch.setattr(tnn, "USE_NATIVE_STEP", False)
    acc_a, nll_a = trainer.evaluate(dc, ids, batch_graphs=8)
    assert acc_a == acc and abs(nll_a - nll) <= TOL * abs(nll)


def test_trainer_takes_the_native_path_and_learns(cuda):
    from tsg import _lib
    from tsg.feeder import DeviceCorpus
    from tsg.train import ClassifierTrainer
    corpus = _corpus("DD", 30, 2, 5)
    cb = _compact(corpus, cuda)
    torch.manual_seed(0)
    from tsg import nn as tnn
    model = tnn.PackedSAGNet(corpus.num_node_labels, 32, 2, 0.5, 0.0).to(cuda)
    trainer = ClassifierTrainer(model, lr=5e-3, weight_decay=0.0)
    y = torch.from_numpy(corpus.y).to(cuda)
    calls = _lib.launch_calls
    losses = [float(trainer.step(cb, None, corpus.node_ptr, y)) for _ in range(25)]
    assert _lib.launch_calls - calls == 25, "one C-ABI call per step"
    assert all(np.isfinite(losses)) and losses[-1] < losses[0]
    # the id-driven loop: batches and labels assembled on the device
    dc = DeviceCorpus(corpus, cuda)
    out = trainer.run_from_ids(dc, [np.arange(30), np.arange(30)[::-1].copy(), np.arange(0, 30, 2)])
    assert len(out) == 3 and all(np.isfinite(out))


def test_trainer_falls_back_when_a_graph_exceeds_the_executor_limits(cuda, monkeypatch):
    from tsg import nn as tnn, ops
    from tsg.train import ClassifierTrainer
    corpus = _corpus("DD", 12, 2, 6)
    cb = _compact(corpus, cuda)
    y = torch.from_numpy(corpus.y).to(cuda)
    torch.manual_seed(0)
    model = tnn.PackedSAGNet(corpus.num_node_labels, 32, 2, 0.5, 0.0).to(cuda)
    assert model.native_step_supported(cb, corpus.node_ptr)
    ref = float(ClassifierTrainer(model, lr=1e-3).step(cb, None, corpus.node_ptr, y))
    monkeypatch.setattr(ops, "GRAPH_CSR_MAX_NODES", int(np.diff(corpus.node_ptr).max()) - 1)
    torch.manual_seed(0)
    model2 = tnn.PackedSAGNet(corpus.num_node_labels, 32, 2, 0.5, 0.0).to(cuda)
    assert not model2.native_step_supported(cb, corpus.node_ptr)
    got = float(ClassifierTrainer(model2, lr=1e-3).step(cb, None, corpus.node_ptr, y))
    assert abs(got - ref) <= 1e-5 * max(abs(ref), 1.0)


def test_two_shards_combined_equal_the_union_batch(cuda):
    """what the data-parallel step all-reduces: G_r-weighted shard losses and gradients == the union batch's"""
    from tsg import synth as S
    corpus = _corpus("DD", 20, 3, 31)
    model, _ = _model(corpus, 32, 3, cuda, dropout=0.0)
    model.train()
    y = torch.from_numpy(corpus.y).to(cuda)
    loss_u = model.native_nll_step(_compact(corpus, cuda), corpus.node_ptr, y).clone()
    g_u = {k: p.grad.clone() for k, p in model.named_parameters()}
    parts = []
    for ids in (np.arange(0, 7), np.arange(7, 20)):
        sub = S.select(corpus, ids)
        loss = model.native_nll_step(_compact(sub, cuda), sub.node_ptr, y[torch.from_numpy(ids).to(cuda)]).clone()
        parts.append((len(ids), loss, {k: p.grad.clone() for k, p in model.named_parameters()}))
    n = sum(p[0] for p in parts)
    assert rel_err(sum(p[0] * p[1] for p in parts) / n, loss_u) <= TOL
    for k in g_u:
        assert rel_err(sum(p[0] * p[2][k] for p in parts) / n, g_u[k]) <= TOL, k


def test_triplet_step_at_the_reference_default_widths(cuda):
    """nhid 128, final_dim 64 (Code/sag/train_triplet.py's defaults): the triplet step runs natively through the wide
    head backward and matches the oracle; before it, the step raised at this width."""
    from tsg import _lib
    from tsg.train import TripletTrainer
    G, nhid, C, margin = 6, 128, 64, 50.0
    corpus = _corpus("DD", G, 2, 41)
    b = synth.pack(corpus)
    cb = _compact(corpus, cuda)
    model, params = _model(corpus, nhid, C, cuda)
    model.train()
    assert model.native_step_supported(cb, corpus.node_ptr)
    trip = torch.tensor([[0, 1, 2], [3, 4, 5], [1, 0, 3], [2, 5, 4], [4, 2, 0], [5, 3, 1]], dtype=torch.int64)
    mask = _mask(G, nhid)
    loss, emb = model.native_step(cb, corpus.node_ptr, trip.to(cuda), margin, dropout_mask=mask.to(cuda), return_emb=True)
    grads = {k: p.grad.clone() for k, p in model.named_parameters()}
    res = {}
    for dt in (torch.float32, torch.float64):
        po = {k: v.clone().to(dt).requires_grad_(True) for k, v in params.items()}
        emb_o = R.sag_net_forward(po, torch.from_numpy(b["x"]).to(dt), torch.from_numpy(b["edge_index"]),
                                  torch.from_numpy(b["batch"]), 0.5, dropout_mask=mask.to(dt))
        loss_o, _, _ = R.triplet_margin_loss(emb_o[trip[:, 0]], emb_o[trip[:, 1]], emb_o[trip[:, 2]], margin)
        loss_o.backward()
        res[dt] = (emb_o.detach(), loss_o.detach(), {k: v.grad for k, v in po.items()})
    assert rel_err(emb, res[torch.float32][0]) <= TOL
    assert rel_err(loss, res[torch.float32][1]) <= TOL
    fwd_noise = max(rel_err(res[torch.float32][0], res[torch.float64][0]), 1e-7)
    for k in grads:
        grad_check(grads[k], res[torch.float32][2][k], res[torch.float64][2][k], TOL, k, fwd_noise)
    trainer = TripletTrainer(model, lr=1e-3)
    calls = _lib.launch_calls
    assert torch.isfinite(trainer.step(cb, None, corpus.node_ptr, trip.to(cuda)))
    assert _lib.launch_calls - calls == 1, "native path: one C-ABI call"


def test_out_of_range_label_on_the_native_entries_is_reported(cuda):
    from tsg import nn as tnn
    corpus = _corpus("DD", 8, 3, 2)
    cb = _compact(corpus, cuda)
    model, _ = _model(corpus, 32, 3, cuda)
    y = torch.from_numpy(corpus.y).to(cuda)
    tnn.check_fused_status()
    for bad in (3, -1):
        yb = y.clone(); yb[5] = bad
        loss = model.native_nll_step(cb, corpus.node_ptr, yb)
        assert torch.isfinite(loss)
        with pytest.raises(RuntimeError, match="label"):
            tnn.check_fused_status()
        model.native_classify(cb, corpus.node_ptr, yb)
        with pytest.raises(RuntimeError, match="label"):
            tnn.check_fused_status()
    model.native_nll_step(cb, corpus.node_ptr, y)
    model.native_classify(cb, corpus.node_ptr, y)
    tnn.check_fused_status()
