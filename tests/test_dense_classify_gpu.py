"""The dense encoders' supervised settings on the GPU (DenseClassifierTrainer, WaveClassifierTrainer): one step of every
encoder in every setting against the ATen composition (the model's forward, [softmax +] F.cross_entropy [+ link_loss],
backward, clip, Adam), base original at bench config 1's shape against run_config1's body; run_from_ids over many steps;
evaluate's independence of batch_graphs and its totals against oracle/dense_ref's graph-by-graph padded forward; a 2stg+
run continuing a stage-1 trainer's weights and Adam state; no trace in a second model."""
import copy

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import rel_err
from oracle import dense_ref as D
from tsg import eigen_synth, synth

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _table(max_nodes, F_, seed=777):
    return torch.from_numpy(np.random.default_rng(seed).normal(0.0, 2.0, (max_nodes, F_)).astype(np.float32))


def _model(kind, dev, final_dim="number_classes", max_nodes=1000, seed=777, F_=32, pred_hidden_dims=()):
    from tsg import dense, diffpool, gat
    torch.manual_seed(seed)
    if kind == "base":
        return dense.PackedGcnEncoder(32, 32, 32, 2, 2, bn=True, final_dim=final_dim,
                                      pred_hidden_dims=pred_hidden_dims).to(dev)
    if kind == "gat":
        return gat.PackedGatEncoder(32, 32, 32, 2, num_layers=3, num_heads=[2, 2], final_dim=final_dim).to(dev)
    if kind == "diffpool":
        return diffpool.PackedSoftPoolEncoder(max_nodes, 32, 32, 32, 2, 3, 32, assign_ratio=0.1,
                                              final_dim=final_dim).to(dev)
    return dense.PackedWaveEncoder(F_, 32, 32, 2, 2, num_pool_matrix=1, num_pool_final_matrix=1, pool_sizes=[10],
                                   pred_hidden_dims=[50]).to(dev)


def _setup(kind, shape, G, dev, seed=41, y=None):
    from tsg.feeder import DeviceCorpus
    corpus = synth.make_corpus(shape, G, seed=seed)
    if y is not None:
        corpus.y = np.asarray(y, np.int64)
    dc = DeviceCorpus(corpus, dev)
    if kind == "wave":
        dc.attach_eigen(eigen_synth.make_operands(corpus, 10, 1, 1))
    return corpus, dc


def _trainer(kind, model, dev, setting="original", **kw):
    from tsg.train import DenseClassifierTrainer, WaveClassifierTrainer
    if kind == "wave":
        return WaveClassifierTrainer(model, 1000, setting=setting, **kw)
    return DenseClassifierTrainer(model, _table(1000, 32).to(dev), 1000, setting=setting, **kw)


def _aten_logits(kind, model, batch, setting, linkpred=False):
    """the model's own forward (and, for linkpred, its readout's assignment) -> (logits, extra loss or None)"""
    if kind == "wave":
        args, kw = batch.readout_args()
        return model(*args, **kw), None
    if linkpred:
        out, aux = model.readout(batch.x, batch.csr, batch.graph_ptr, batch.has_pad, return_aux=True)
        return (model.pred_model(model.pre_pred_model(out)),
                model.link_loss(aux["s"], batch.csr, batch.graph_ptr, np.diff(batch.node_ptr_host)))
    a, b = model(batch.x, batch.csr, batch.graph_ptr, batch.max_nodes if kind == "gat" else batch.has_pad)
    return (b if setting == "original" else a), None          # 2stg+: element [0]


def _aten_step(kind, model, opt, batch, y, setting, softmax_first, clip, linkpred=False):
    """run_config1's body for the dense step: forward, [softmax +] cross_entropy [+ link loss], backward, clip, Adam"""
    logits, extra = _aten_logits(kind, model, batch, setting, linkpred)
    loss = F.cross_entropy(torch.softmax(logits, dim=1) if softmax_first else logits, y)
    if extra is not None:
        loss = loss + extra
    opt.zero_grad(set_to_none=True)
    loss.backward()
    if clip is not None:
        torch.nn.utils.clip_grad_norm_(model.parameters(), clip)
    opt.step()
    return loss.detach()


STEP_CASES = [
    ("base", "original", "number_classes", "PROTEINS", 1113, False),      # bench config 1: the whole corpus, one batch
    ("base", "2stg+", "pretrain", "PROTEINS", 200, False),
    ("gat", "original", "number_classes", "JANY", 60, False),
    ("gat", "2stg+", "output_dim", "JANY", 60, False),
    ("diffpool", "original", "number_classes", "DD", 40, False),
    ("diffpool", "original", "number_classes", "DD", 40, True),
    ("diffpool", "2stg+", "pretrain", "DD", 40, False),
    ("wave", "original", None, "DD", 40, False),
    ("wave", "2stg+", None, "DD", 40, False),
]


@pytest.mark.parametrize("kind,setting,final_dim,shape,G,linkpred", STEP_CASES)
def test_step_equals_the_aten_composition(cuda, kind, setting, final_dim, shape, G, linkpred):
    from tsg import nn as tnn
    corpus, dc = _setup(kind, shape, G, cuda, seed=777 if G == 1113 else 41)
    F_ = corpus.num_node_labels if kind == "wave" else 32
    ma = _model(kind, cuda, final_dim, F_=F_)
    mb = copy.deepcopy(ma)
    clip = None if kind == "wave" else 2.0
    ta = _trainer(kind, ma, cuda, setting, **({"linkpred": True} if linkpred else {}))
    assert ta.clip_norm == clip
    ob = torch.optim.Adam(mb.parameters(), lr=1e-3)
    ids = np.arange(G) if G == 1113 else np.random.default_rng(0).integers(0, G, G)
    for it in range(2):                                   # the second step runs on Adam's updated state
        if it:                                            # from the same parameters and Adam state on both sides
            mb.load_state_dict(ma.state_dict())
            ob.load_state_dict(ta.opt.state_dict())
        batch, y = ta._batch(dc, ta._check(dc, ids))
        p0 = [p.detach().clone() for p in ma.parameters()]
        st0 = copy.deepcopy(ta.opt.state_dict())
        la = ta.step(batch, y)
        lb = _aten_step(kind, mb, ob, batch, y, setting, ta.softmax_first, clip, linkpred)
        assert rel_err(la, lb) <= TOL, (it, float(la), float(lb))
        # Adam divides each entry by its own gradient history, so an entry whose gradient is small moves by about lr
        # whatever its last bits: the updated parameters are checked as Adam's update of this step's (clipped)
        # gradients, which are the ones compared with ATen's, and against ATen's parameters within Adam's bound
        ref = [q.clone().requires_grad_(True) for q in p0]
        for q, pa in zip(ref, ma.parameters()):
            q.grad = None if pa.grad is None else pa.grad.clone()
        oref = torch.optim.Adam(ref, lr=1e-3)
        oref.load_state_dict(st0)
        oref.step()
        for (k, pa), pb, q in zip(ma.named_parameters(), mb.parameters(), ref):
            if pb.grad is None:                           # heads outside the logits' path
                assert pa.grad is None, k
                assert torch.equal(pa, pb), k
                continue
            assert rel_err(pa.grad, pb.grad) <= TOL, (it, "grad", k, rel_err(pa.grad, pb.grad))
            assert rel_err(pa, q) <= 1e-6, (it, "param vs Adam of the step's gradients", k, rel_err(pa, q))
            assert float((pa - pb).detach().abs().max()) <= 2 * 1e-3 * 1.01, (it, "param vs ATen beyond Adam's bound", k)
    tnn.check_fused_status()


@pytest.mark.parametrize("kind,setting,final_dim", [("base", "original", "number_classes"), ("gat", "original", "number_classes"),
                                                    ("wave", "original", None)])
def test_run_from_ids_learns_a_separable_labelling(cuda, kind, setting, final_dim):
    """label = whether the graph has more nodes than the median: the readouts see the node count"""
    base = synth.make_corpus("PROTEINS", 240, seed=5)
    n = np.diff(base.node_ptr)
    corpus, dc = _setup(kind, "PROTEINS", 240, cuda, seed=5, y=(n > np.median(n)).astype(np.int64))
    F_ = corpus.num_node_labels if kind == "wave" else 32
    t = _trainer(kind, _model(kind, cuda, final_dim, F_=F_), cuda, setting, lr=1e-2)
    rng = np.random.default_rng(0)
    steps = [rng.integers(0, 240, 64) for _ in range(60)]
    losses = t.run_from_ids(dc, steps)
    assert len(losses) == 60 and all(np.isfinite(losses))
    assert np.mean(losses[-10:]) < 0.9 * np.mean(losses[:10]), (losses[:10], losses[-10:])
    acc, ce = t.evaluate(dc, np.arange(240))
    assert acc > 0.6 and np.isfinite(ce), (acc, ce)
    assert t.run_from_ids(dc, []) == []


# ------------------------------------------------------------------------------------------ evaluation
def _oracle_logits(kind, model, corpus, ids, table, max_nodes, setting):
    """graph by graph, padded to max_nodes: oracle/dense_ref's readout, then the head, on the CPU in fp32"""
    cs = lambda mods: [dict(weight=c.weight.detach().cpu(), bias=c.bias.detach().cpu()) for c in mods]
    if kind == "base":
        convs = cs(model.convs())
    elif kind == "gat":
        layers = [[dict(w=h.w.detach().cpu(), a=h.a.detach().cpu()) for h in layer.heads()] for layer in model.layers()]
    else:
        st = model._stack
        p = dict(conv=cs(st(model.conv_first, model.conv_block, model.conv_last)),
                 assign_conv=cs(st(model.assign_conv_first_modules[0], model.assign_conv_block_modules[0],
                                   model.assign_conv_last_modules[0])),
                 conv_after=cs(st(model.conv_first_after_pool[0], model.conv_block_after_pool[0],
                                  model.conv_last_after_pool[0])))
        p["assign_pred.weight"] = model.assign_pred_modules[0].weight.detach().cpu()
        p["assign_pred.bias"] = model.assign_pred_modules[0].bias.detach().cpu()
    head = copy.deepcopy(model).cpu()
    out = []
    with torch.no_grad():
        for g in ids:
            n = corpus.num_nodes(int(g))
            e0, e1 = corpus.edge_ptr[g], corpus.edge_ptr[g + 1]
            adj = torch.zeros(1, max_nodes, max_nodes)
            adj[0, torch.from_numpy(corpus.row[e0:e1]), torch.from_numpy(corpus.col[e0:e1])] = 1.0
            x = torch.zeros(1, max_nodes, table.size(1)); x[0, :n] = table[:n]
            if kind == "base":
                r = D.gcn_encoder_readout(x, adj, convs)
            elif kind == "gat":
                r = D.dgat_encoder_readout(x, adj, layers)
            else:
                r = D.soft_pool_readout(x, adj, [n], p)[0]
            if setting == "2stg+":
                out.append(r if kind == "gat" else head.map2_model(head.map_model(r)))
            else:
                out.append(head.pred_model(r) if kind == "gat" else head.pred_model(head.pre_pred_model(r)))
    return torch.cat(out)


@pytest.mark.parametrize("kind,setting,final_dim", [("base", "original", "number_classes"), ("base", "2stg+", "pretrain"),
                                                    ("gat", "original", "number_classes"), ("gat", "2stg+", "output_dim"),
                                                    ("diffpool", "original", "number_classes")])
def test_evaluate_against_the_oracle(cuda, kind, setting, final_dim):
    from tsg.train import DenseClassifierTrainer
    max_nodes = 64
    base = synth.make_corpus("PROTEINS", 120, seed=12)
    keep = [g for g in range(base.num_graphs) if 2 <= base.num_nodes(g) <= max_nodes and base.edge_ptr[g + 1] > base.edge_ptr[g]]
    sel = synth.select(base, keep[:48])
    from tsg.feeder import DeviceCorpus
    dc = DeviceCorpus(sel, cuda)
    table = _table(max_nodes, 32)
    model = _model(kind, cuda, final_dim, max_nodes=max_nodes)
    with torch.no_grad():                                   # non-zero biases: padded rows then carry a value
        for k, p in model.named_parameters():
            if k.endswith("bias"):
                p.copy_(torch.randn_like(p) * 0.2)
    t = DenseClassifierTrainer(model, table.to(cuda), max_nodes, setting=setting)
    ids = np.random.default_rng(0).permutation(sel.num_graphs)
    model.train()
    acc, ce = t.evaluate(dc, ids)
    assert model.training, "evaluate restores the training flag"
    z = _oracle_logits(kind, model, sel, ids, table, max_nodes, setting)
    y = torch.from_numpy(sel.y[ids])
    top2 = torch.topk(z, 2, dim=1).values
    assert bool(((top2[:, 0] - top2[:, 1]) > 1e-4).all()), "near-tie in the oracle's logits: pick another seed"
    assert acc == float((z.argmax(dim=1) == y).sum()) / len(ids)
    ref = F.cross_entropy(torch.softmax(z, dim=1) if setting == "2stg+" else z, y)
    assert rel_err(torch.tensor(ce), ref) <= TOL, (ce, float(ref))
    model.eval()
    for bg in (1, 7, 48):
        a2, c2 = t.evaluate(dc, ids, batch_graphs=bg)
        assert not model.training
        assert a2 == acc
        if kind == "gat":      # the padded-row term x_pad @ W is an ATen GEMM over the batch's graphs
            assert abs(c2 - ce) <= 1e-6 * max(abs(ce), 1.0), (bg, c2, ce)
        else:                  # per-graph kernels and one K16 call over all rows: independent of the batching
            assert c2 == ce, (bg, c2, ce)


def test_wave_evaluate_is_the_head_on_its_readouts(cuda):
    corpus, dc = _setup("wave", "DD", 40, cuda)
    model = _model("wave", cuda, F_=corpus.num_node_labels)
    t = _trainer("wave", model, cuda)
    ids = np.random.default_rng(2).permutation(40)
    acc, ce = t.evaluate(dc, ids)
    for bg in (1, 9):
        assert t.evaluate(dc, ids, batch_graphs=bg) == (acc, ce)
    with torch.no_grad():
        model.eval()
        z = model(*t.pack(dc, ids).readout_args()[0], **t.pack(dc, ids).readout_args()[1])
        model.train()
    y = torch.from_numpy(corpus.y[ids]).to(cuda)
    top2 = torch.topk(z, 2, dim=1).values
    assert bool(((top2[:, 0] - top2[:, 1]) > 1e-4).all()), "near-tie in the logits: pick another seed"
    assert acc == float((z.argmax(dim=1) == y).sum()) / len(ids)
    assert rel_err(torch.tensor(ce), F.cross_entropy(z, y)) <= TOL


def test_evaluate_reports_an_out_of_range_label(cuda):
    corpus, dc = _setup("base", "PROTEINS", 30, cuda)
    t = _trainer("base", _model("base", cuda), cuda)
    t.evaluate(dc, np.arange(30))
    dc.y[26] = 7                          # after the host check: K16 reads it clamped and sets status bit 8
    with pytest.raises(RuntimeError, match="label"):
        t.evaluate(dc, np.arange(30))


# ------------------------------------------------------------------------------------------ 2stg+ after stage 1
@pytest.mark.parametrize("kind", ["base", "gat", "diffpool", "wave"])
def test_2stg_plus_continues_stage_1(cuda, kind):
    from tsg.train import DenseTripletTrainer, WaveTripletTrainer
    corpus, dc = _setup(kind, "DD" if kind in ("diffpool", "wave") else "PROTEINS", 30, cuda)
    F_ = corpus.num_node_labels if kind == "wave" else 32
    model = _model(kind, cuda, {"base": "pretrain", "diffpool": "pretrain", "gat": "output_dim"}.get(kind), F_=F_)
    s1 = (WaveTripletTrainer(model, 1000) if kind == "wave"
          else DenseTripletTrainer(model, _table(1000, 32).to(cuda), 1000))
    trip = synth.sample_triplets(corpus.y, 8, seed=1)
    ids = np.concatenate([trip[:, 0], trip[:, 1], trip[:, 2]])
    tidx = torch.from_numpy(np.stack([np.arange(8), 8 + np.arange(8), 16 + np.arange(8)], 1).astype(np.int64)).pin_memory()
    s1.run_from_ids(dc, [(ids, tidx), (ids, tidx)])
    after1 = {k: v.clone() for k, v in model.state_dict().items()}
    fresh = _trainer(kind, model, cuda, "2stg+")
    for k, v in model.state_dict().items():
        assert torch.equal(v, after1[k]), k                  # building the trainer keeps the stage-1 weights
    assert fresh.opt is not s1.opt
    cont = _trainer(kind, model, cuda, "2stg+", optimizer=s1.opt)
    assert cont.opt is s1.opt
    p = model.conv_first.weight if kind != "gat" else model.conv_first.heads()[0].w
    assert int(s1.opt.state[p]["step"]) == 2
    cont.run_from_ids(dc, [np.arange(30)])
    assert int(s1.opt.state[p]["step"]) == 3                  # the stage-1 Adam state carries on
    assert not torch.equal(p, after1[[k for k, v in model.named_parameters() if v is p][0]])


def test_trainer_leaves_no_trace_in_a_second_model(cuda):
    """two trainers on deep copies of one model stay bitwise together through evaluate calls on one of them"""
    corpus, dc = _setup("base", "PROTEINS", 30, cuda)
    ta = _trainer("base", _model("base", cuda), cuda)
    tb = _trainer("base", copy.deepcopy(ta.model), cuda)
    ta.evaluate(dc, np.arange(30))
    ta.evaluate(dc, np.arange(10), batch_graphs=3)
    steps = [np.arange(20), np.arange(5, 30)]
    assert ta.run_from_ids(dc, steps) == tb.run_from_ids(dc, steps)
    for pa, pb in zip(ta.model.parameters(), tb.model.parameters()):
        assert torch.equal(pa, pb)
