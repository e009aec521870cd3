"""2stg for the dense encoders on the GPU: DeviceCorpus.pack_dense (K0d) against the host path bench.py's dense configs
take (synth.select -> synth.pack -> K1 build_csr(CSR_RAW)), equal array for array; its verification of the coalesced
promise; DenseTripletTrainer's step against the config-3/4 step on the host-assembled batch, bit for bit; embed against
oracle/dense_ref's per-graph forward on the padded wire format; evaluate against heads_ref's kNN and a hand-composed MLP."""
import copy

import numpy as np
import pytest
import torch

from conftest import rel_err
from oracle import dense_ref as D
from oracle import heads_ref as H
from tsg import synth

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _table(max_nodes, F, seed=777):
    return torch.from_numpy(np.random.default_rng(seed).normal(0.0, 2.0, (max_nodes, F)).astype(np.float32))


def _corpus_of(graphs, name="edge-cases", seed=0):
    """graphs: list of (n, row, col) with graph-local endpoints -> synth.Corpus"""
    n = np.array([g[0] for g in graphs], np.int64)
    e = np.array([len(g[1]) for g in graphs], np.int64)
    rng = np.random.default_rng(seed)
    return synth.Corpus(name, np.concatenate([[0], np.cumsum(n)]).astype(np.int64),
                        np.concatenate([[0], np.cumsum(e)]).astype(np.int64),
                        np.concatenate([np.asarray(g[1], np.int64) for g in graphs]),
                        np.concatenate([np.asarray(g[2], np.int64) for g in graphs]),
                        rng.integers(0, 3, int(n.sum())).astype(np.int32), rng.integers(0, 2, len(graphs)).astype(np.int64), 3)


def _edge_case_corpus(max_nodes, seed=5):
    """ordinary graphs plus: one node; nodes but no edges; three isolated trailing nodes; two isolated leading nodes and
    one in the middle; exactly max_nodes nodes"""
    base = synth.make_corpus("PROTEINS", 30, seed=seed)
    graphs = []
    for g in [g for g in range(base.num_graphs) if base.num_nodes(g) <= max_nodes // 2][:6]:
        e0, e1 = base.edge_ptr[g], base.edge_ptr[g + 1]
        graphs.append((base.num_nodes(g), base.row[e0:e1], base.col[e0:e1]))
    rng = np.random.default_rng(seed)
    graphs.append((1, [], []))
    graphs.append((5, [], []))
    r, c = synth._one_graph(rng, 9, 14)
    graphs.append((12, r, c))                                        # nodes 9, 10, 11 isolated at the end
    r, c = synth._one_graph(rng, 10, 15)
    shift = np.where(np.asarray(r) >= 5, 3, 2), np.where(np.asarray(c) >= 5, 3, 2)
    graphs.append((13, np.asarray(r) + shift[0], np.asarray(c) + shift[1]))   # 0, 1 and 7 isolated
    r, c = synth._one_graph(rng, max_nodes, 2 * max_nodes)
    graphs.append((max_nodes, r, c))
    return _corpus_of(graphs, seed=seed)


def _host_dense(corpus, ids, table, max_nodes, dev, want_eid=True):
    """bench.py::_dense_inputs with a given table: the host path pack_dense replaces"""
    from tsg import ops
    sel = synth.select(corpus, ids)
    n = np.diff(sel.node_ptr)
    local = np.concatenate([np.arange(k) for k in n])
    x = table[torch.from_numpy(local)].to(dev)
    ei = torch.from_numpy(synth.pack(sel, one_hot=False)["edge_index"]).to(dev)
    N = int(sel.node_ptr[-1])
    csr = ops.build_csr(ops.EdgeList.from_edge_index(ei), N, mode=ops.CSR_RAW, want_eid=want_eid)
    return x, csr, torch.from_numpy(sel.node_ptr).to(dev), torch.from_numpy(n < max_nodes).to(dev)


CSR_FIELDS = ("rowptr", "colidx", "val", "eid", "t_rowptr", "t_colidx", "t_val", "t_eid")


def _assert_same_batch(b, host, want_eid=True):
    x, csr, gptr, has_pad = host
    assert torch.equal(b.x, x)
    for f in CSR_FIELDS:
        if not want_eid and f in ("eid", "t_eid"):
            assert getattr(b.csr, f) is None
            continue
        assert torch.equal(getattr(b.csr, f), getattr(csr, f)), f
    assert b.csr.tile_ptr is None and not b.csr.tma_ok
    assert b.graph_ptr.dtype == torch.int64 and torch.equal(b.graph_ptr, gptr)
    assert torch.equal(b.has_pad, has_pad)


@pytest.mark.parametrize("shape,G", [("DD", 40), ("PROTEINS", 300), ("JANY", 30)])
@pytest.mark.parametrize("F", [32, 7])
def test_pack_dense_equals_the_host_path(cuda, shape, G, F):
    from tsg import nn as tnn
    from tsg.feeder import DeviceCorpus
    corpus = synth.make_corpus(shape, G, seed=31)
    dc = DeviceCorpus(corpus, cuda)
    assert dc.coalesced
    table = _table(1000, F)
    ids = np.random.default_rng(G).integers(0, G, 3 * G)                   # duplicates
    for want_eid in (True, False):
        b = dc.pack_dense(ids, table.to(cuda), 1000, want_eid=want_eid)
        _assert_same_batch(b, _host_dense(corpus, ids, table, 1000, cuda), want_eid)
        assert np.array_equal(b.node_ptr_host, synth.select(corpus, ids).node_ptr) and b.max_nodes == 1000
    tnn.check_fused_status()


@pytest.mark.parametrize("F", [32, 7])
def test_pack_dense_edge_cases(cuda, F):
    from tsg import nn as tnn
    from tsg.feeder import DeviceCorpus
    max_nodes = 64
    corpus = _edge_case_corpus(max_nodes)
    dc = DeviceCorpus(corpus, cuda)
    assert dc.coalesced
    table = _table(max_nodes, F)
    G = corpus.num_graphs
    for ids in (np.arange(G), np.arange(G)[::-1], np.array([G - 1]), np.array([7, 6, 0, 7]), np.array([8, 8]),
                np.array([6, 7, 8, 9, 6])):     # 6: one node, 7: no edges, 8: trailing isolated, 9: leading/middle
        # (K1 on the host side needs at least one edge in the batch)
        b = dc.pack_dense(ids, table.to(cuda), max_nodes, want_eid=True)
        _assert_same_batch(b, _host_dense(corpus, ids, table, max_nodes, cuda))
    assert not bool(dc.pack_dense([G - 1], table.to(cuda), max_nodes).has_pad[0])      # exactly max_nodes: no padding
    tnn.check_fused_status()


def test_pack_dense_general_path_for_lists_that_are_not_coalesced(cuda):
    """edges shuffled within each graph, a self loop and a one-way edge: K0 + K1 take it, with the same result"""
    from tsg import nn as tnn
    from tsg.feeder import DeviceCorpus
    c = synth.make_corpus("PROTEINS", 20, seed=9)
    rng = np.random.default_rng(1)
    graphs = []
    for g in range(c.num_graphs):
        e0, e1 = c.edge_ptr[g], c.edge_ptr[g + 1]
        p = rng.permutation(e1 - e0)
        r, q = list(c.row[e0:e1][p]), list(c.col[e0:e1][p])
        if g == 3:
            r.append(1); q.append(1)
        if g == 5:
            last = c.num_nodes(g) - 1
            r, q = [a for a, b in zip(r, q) if (a, b) != (last, 0)], [b for a, b in zip(r, q) if (a, b) != (last, 0)]
            if (0, last) not in set(zip(r, q)):
                r.append(0); q.append(last)                       # (0, last) listed, (last, 0) not
        graphs.append((c.num_nodes(g), r, q))
    corpus = _corpus_of(graphs, seed=2)
    dc = DeviceCorpus(corpus, cuda)
    assert not dc.coalesced
    table = _table(1000, 32)
    ids = rng.integers(0, 20, 50)
    for want_eid in (True, False):
        b = dc.pack_dense(ids, table.to(cuda), 1000, want_eid=want_eid)
        _assert_same_batch(b, _host_dense(corpus, ids, table, 1000, cuda), want_eid)
    tnn.check_fused_status()


@pytest.mark.parametrize("broken,bit,msg", [("unsorted", 2, "not sorted"), ("self_loop", 1, "self loop"),
                                            ("asymmetric", 4, "not symmetric")])
def test_pack_dense_reports_a_broken_promise(cuda, broken, bit, msg):
    from tsg import nn as tnn
    from tsg.feeder import DeviceCorpus
    c = synth.make_corpus("PROTEINS", 6, seed=3)
    row, col = c.row.copy(), c.col.copy()
    e0 = int(c.edge_ptr[2])
    if broken == "unsorted":
        row[e0], row[e0 + 1], col[e0], col[e0 + 1] = row[e0 + 1], row[e0], col[e0 + 1], col[e0]
    elif broken == "self_loop":
        col[e0] = row[e0]
    else:                                  # drop one direction of an edge: keep the list sorted, lose its partner
        keep = np.ones(row.shape[0], bool); keep[e0] = False
        ep = c.edge_ptr.copy(); ep[3:] -= 1
        row, col = row[keep], col[keep]
        c = synth.Corpus(c.name, c.node_ptr, ep, row, col, c.node_label, c.y, c.num_node_labels)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a.astype(np.int32))).to(cuda)
    dc = DeviceCorpus.from_device(t(c.node_label), t(row), t(col), c.node_ptr, c.edge_ptr, c.num_node_labels,
                                  coalesced=True)
    tnn.check_fused_status()
    b = dc.pack_dense(np.arange(6), _table(1000, 32).to(cuda), 1000, want_eid=True)
    torch.cuda.synchronize()
    assert int(tnn._status_word(cuda).item()) == bit
    assert int(b.csr.colidx.min()) >= 0 and int(b.csr.colidx.max()) < b.x.size(0)          # indices stay in range
    with pytest.raises(RuntimeError, match=msg):
        tnn.check_fused_status()


# ------------------------------------------------------------------------------------------ training
def _model(kind, dev, max_nodes=1000, seed=777):
    from tsg import dense, diffpool, gat
    torch.manual_seed(seed)
    if kind == "base":
        return dense.PackedGcnEncoder(32, 32, 32, 2, 2, bn=True).to(dev)
    if kind == "gat":
        return gat.PackedGatEncoder(32, 32, 32, 2, num_layers=3, num_heads=[2, 2]).to(dev)
    return diffpool.PackedSoftPoolEncoder(max_nodes, 32, 32, 32, 2, 3, 32, assign_ratio=0.1).to(dev)


STEP_CASES = [("base", "PROTEINS", 40), ("gat", "JANY", 10), ("diffpool", "DD", 10)]


def _triplet_ids(corpus, T, seed):
    trip = synth.sample_triplets(corpus.y, T, seed=seed)
    ids = np.concatenate([trip[:, 0], trip[:, 1], trip[:, 2]])
    tidx = np.stack([np.arange(T), T + np.arange(T), 2 * T + np.arange(T)], 1).astype(np.int64)
    return ids, torch.from_numpy(tidx).pin_memory()


def _bench_step(kind, model, opt, host, tr, max_nodes, clip=None):
    """bench.py run_config3 / run_config4's step on the host-assembled batch"""
    from tsg import ops
    x, csr, gptr, has_pad = host
    _, emb = model(x, csr, gptr, max_nodes if kind == "gat" else has_pad)
    loss, _, _ = ops.triplet_loss(emb, tr, 1.5)
    opt.zero_grad(set_to_none=True); loss.backward()
    if clip is not None:
        torch.nn.utils.clip_grad_norm_(model.parameters(), clip)
    opt.step()
    return loss.detach()


@pytest.mark.parametrize("kind,shape,T", STEP_CASES)
def test_step_from_ids_is_the_bench_step(cuda, kind, shape, T):
    from tsg.feeder import DeviceCorpus
    from tsg.train import DenseTripletTrainer
    corpus = synth.make_corpus(shape, 3 * T, seed=41)
    dc = DeviceCorpus(corpus, cuda)
    table = _table(1000, 32)
    ids, tr = _triplet_ids(corpus, T, 0)
    host = _host_dense(corpus, ids, table, 1000, cuda, want_eid=kind == "gat")
    for clip in (None, 2.0):
        ma, mb = _model(kind, cuda), _model(kind, cuda)
        ta = DenseTripletTrainer(ma, table.to(cuda), 1000, clip_norm=clip)
        ob = torch.optim.Adam(mb.parameters(), lr=1e-3)
        if clip is None:
            losses = ta.run_from_ids(dc, [(ids, tr)])
            la = torch.tensor(losses[0])
        else:
            la = ta.step(ta.pack(dc, ids), tr.to(cuda)).cpu()
        lb = _bench_step(kind, mb, ob, host, tr.to(cuda), 1000, clip).cpu()
        assert torch.equal(la, lb), (clip, float(la), float(lb))
        for (k, pa), pb in zip(ma.named_parameters(), mb.parameters()):
            if pb.grad is None:                            # heads outside the embedding's path (pred_model, ...)
                assert pa.grad is None, k
            else:
                assert torch.equal(pa.grad, pb.grad), (clip, "grad", k)
            assert torch.equal(pa, pb), (clip, "param", k)


def test_run_from_ids_trains_over_many_steps(cuda):
    from tsg.feeder import DeviceCorpus
    from tsg.train import DenseTripletTrainer
    corpus = synth.make_corpus("PROTEINS", 60, seed=42)
    dc = DeviceCorpus(corpus, cuda)
    ta = DenseTripletTrainer(_model("gat", cuda), _table(1000, 32).to(cuda), 1000)
    steps = [_triplet_ids(corpus, 20, s) for s in range(6)]
    losses = ta.run_from_ids(dc, steps)
    assert len(losses) == 6 and all(np.isfinite(losses))
    assert ta.run_from_ids(dc, []) == []


# ------------------------------------------------------------------------------------------ embeddings
def _oracle_embed(kind, model, corpus, ids, table, max_nodes):
    """per graph, padded to max_nodes: oracle/dense_ref's readout, then the model's map_model, on CPU in fp32"""
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
            out.append(r @ model.map_model.weight.detach().cpu().t() + model.map_model.bias.detach().cpu())
    return torch.cat(out)


@pytest.mark.parametrize("kind", ["base", "gat", "diffpool"])
def test_embed_matches_the_oracle(cuda, kind):
    from tsg import ops
    from tsg.feeder import DeviceCorpus
    from tsg.train import DenseTripletTrainer
    max_nodes = 64
    corpus = _edge_case_corpus(max_nodes, seed=8)
    extra = synth.make_corpus("PROTEINS", 40, seed=12)
    keep = [g for g in range(extra.num_graphs) if extra.num_nodes(g) <= max_nodes][:24]
    sel = synth.select(extra, keep)
    both = _corpus_of([(corpus.num_nodes(g), corpus.row[corpus.edge_ptr[g]:corpus.edge_ptr[g + 1]],
                        corpus.col[corpus.edge_ptr[g]:corpus.edge_ptr[g + 1]]) for g in range(corpus.num_graphs)] +
                      [(sel.num_nodes(g), sel.row[sel.edge_ptr[g]:sel.edge_ptr[g + 1]],
                        sel.col[sel.edge_ptr[g]:sel.edge_ptr[g + 1]]) for g in range(sel.num_graphs)], seed=3)
    dc = DeviceCorpus(both, cuda)
    table = _table(max_nodes, 32)
    ids = np.random.default_rng(0).permutation(both.num_graphs)
    for tc in ([False, True] if kind == "diffpool" else [True]):
        ops.USE_TCGEN05 = tc
        try:
            model = _model(kind, cuda, max_nodes=max_nodes)
            with torch.no_grad():                          # non-zero biases: padded rows then carry a value
                for k, p in model.named_parameters():
                    if k.endswith("bias"):
                        p.copy_(torch.randn_like(p) * 0.2)
            tt = DenseTripletTrainer(model, table.to(cuda), max_nodes)
            model.train()
            emb = tt.embed(dc, ids)
            assert model.training, "embed restores the training flag"
            ref = _oracle_embed(kind, model, both, ids, table, max_nodes)
            assert emb.shape == ref.shape
            assert rel_err(emb, ref) <= TOL, (kind, tc)
            model.eval()
            # a batch needs one edge: the split runs over the graphs that have edges
            sub = ids[np.diff(both.edge_ptr)[ids] > 0]
            whole = tt.embed(dc, sub, batch_graphs=len(sub))
            for bg in (1, 7):
                got = tt.embed(dc, sub, batch_graphs=bg)
                assert not model.training
                if kind == "gat":      # the padded-row term x_pad @ W is an ATen GEMM over the batch's graphs
                    assert rel_err(got, whole) <= 1e-6, (kind, tc, bg)
                else:                  # per-graph kernels, one head GEMM over all rows: independent of the batching
                    assert torch.equal(got, whole), (kind, tc, bg)
            dup = tt.embed(dc, np.concatenate([sub, sub[[3, 0, 3]]]))
            assert torch.equal(dup[len(sub):], dup[torch.tensor([3, 0, 3])])
        finally:
            ops.USE_TCGEN05 = True


# ------------------------------------------------------------------------------------------ scoring
def _boundary_is_clear(train, query, k):
    d = ((query[:, None, :].astype(np.float64) - train[None, :, :].astype(np.float64)) ** 2).sum(-1)
    s = np.sort(d, axis=1)
    if s.shape[1] <= k:
        return True
    gap = s[:, k] - s[:, k - 1]
    return bool(np.all((gap == 0) | (gap > 1e-5 * np.maximum(s[:, k], 1e-30))))


def _trainer(kind, shape, G, dev, seed=4, classes=3):
    from tsg.feeder import DeviceCorpus
    from tsg.train import DenseTripletTrainer
    corpus = synth.make_corpus(shape, G, seed=seed)
    if classes != 2:
        corpus.y = np.random.default_rng(seed).integers(0, classes, G).astype(np.int64)
    dc = DeviceCorpus(corpus, dev)
    return corpus, dc, DenseTripletTrainer(_model(kind, dev), _table(1000, 32).to(dev), 1000)


@pytest.mark.parametrize("kind,shape", [("base", "PROTEINS"), ("gat", "PROTEINS"), ("diffpool", "DD")])
def test_evaluate_knn_equals_the_oracle(cuda, kind, shape):
    corpus, dc, tt = _trainer(kind, shape, 60, cuda)
    perm = np.random.default_rng(1).permutation(60)
    tr_ids, ev_ids = perm[:45], perm[45:]
    for k in (1, 3, 8):
        acc = tt.evaluate(dc, tr_ids, ev_ids, head="knn", k=k, batch_graphs=16)
        tr = tt.embed(dc, tr_ids).cpu().numpy(); ev = tt.embed(dc, ev_ids).cpu().numpy()
        assert _boundary_is_clear(tr, ev, k), "near-tie in the embeddings' distances: pick another seed"
        pred = H.knn_predict(tr, corpus.y[tr_ids], ev, k)
        assert acc * len(ev_ids) == float((pred == corpus.y[ev_ids]).sum()), k
    assert tt.model.training


@pytest.mark.parametrize("kind", ["base", "gat", "diffpool"])
def test_evaluate_mlp_is_embed_plus_the_classifier(cuda, kind):
    from tsg import heads
    corpus, dc, tt = _trainer(kind, "PROTEINS" if kind != "diffpool" else "DD", 40, cuda)
    tr_ids, ev_ids = np.arange(30), np.arange(30, 40)
    rng = torch.get_rng_state()
    acc = tt.evaluate(dc, tr_ids, ev_ids, head="mlp", seed=11, mlp_epochs=2)
    assert torch.equal(torch.get_rng_state(), rng), "evaluate moved the RNG stream"
    emb_tr, emb_ev = tt.embed(dc, tr_ids), tt.embed(dc, ev_ids)
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(11)
        clf = heads.Mlp1Classifier(emb_tr.size(1), cuda, num_classes=3)
    y = lambda ids: torch.from_numpy(corpus.y[ids]).to(cuda)
    clf.fit(emb_tr, y(tr_ids)); clf.fit(emb_tr, y(tr_ids))
    assert acc == int(clf.score(emb_ev, y(ev_ids)).item()) / len(ev_ids)


def test_evaluate_reports_an_out_of_range_label(cuda):
    """labels are checked on the host against num_classes; one written into the device copy afterwards reaches K12,
    which reads it clamped and sets status bit 8"""
    from tsg import nn as tnn
    corpus, dc, tt = _trainer("base", "PROTEINS", 30, cuda)
    tr_ids, ev_ids = np.arange(24), np.arange(24, 30)
    tt.evaluate(dc, tr_ids, ev_ids, head="knn", num_classes=3)
    dc.y[26] = 7
    with pytest.raises(RuntimeError, match="label"):
        tt.evaluate(dc, tr_ids, ev_ids, head="knn", num_classes=3)
    tnn.check_fused_status()


def test_trainer_leaves_no_trace_in_a_second_model(cuda):
    """two trainers on deep copies of one model stay bitwise together through evaluate calls on one of them"""
    corpus, dc, ta = _trainer("base", "PROTEINS", 30, cuda, classes=2)
    from tsg.train import DenseTripletTrainer
    tb = DenseTripletTrainer(copy.deepcopy(ta.model), ta.table, 1000)
    ta.evaluate(dc, np.arange(20), np.arange(20, 30), head="mlp", seed=3)
    ta.evaluate(dc, np.arange(20), np.arange(20, 30))
    ids, tr = _triplet_ids(corpus, 10, 5)
    la, lb = ta.run_from_ids(dc, [(ids, tr)]), tb.run_from_ids(dc, [(ids, tr)])
    assert la == lb
    for pa, pb in zip(ta.model.parameters(), tb.model.parameters()):
        assert torch.equal(pa, pb)
