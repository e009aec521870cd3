"""2stg for the EigenGCN encoder on the GPU: DeviceCorpus.pack_eigen (K0e) against the host path (synth.select ->
synth.pack -> K1 build_csr(CSR_RAW), eigen_synth.pack_operands -> dense.build_rect_csr / build_csr(CSR_RAW,
edge_weight)), equal array for array; its verification of the adjacency and operand promises; WaveTripletTrainer's
step against bench config 5's step (model forward + triplet loss + Adam) on the host-assembled batch, bit for bit;
embed against oracle/dense_ref.wave_readout + mlp per graph on the padded wire format; evaluate against heads_ref's kNN
and a hand-composed MLP."""
import dataclasses

import numpy as np
import pytest
import torch

from conftest import rel_err
from oracle import dense_ref as D
from oracle import heads_ref as H
from tsg import eigen_synth, synth

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _corpus_of(graphs, seed=0, labels=3):
    """graphs: list of (n, row, col) with graph-local endpoints -> synth.Corpus"""
    n = np.array([g[0] for g in graphs], np.int64)
    e = np.array([len(g[1]) for g in graphs], np.int64)
    rng = np.random.default_rng(seed)
    return synth.Corpus("edge-cases", np.concatenate([[0], np.cumsum(n)]).astype(np.int64),
                        np.concatenate([[0], np.cumsum(e)]).astype(np.int64),
                        np.concatenate([np.asarray(g[1], np.int64) for g in graphs]),
                        np.concatenate([np.asarray(g[2], np.int64) for g in graphs]),
                        rng.integers(0, labels, int(n.sum())).astype(np.int32),
                        rng.integers(0, 2, len(graphs)).astype(np.int64), labels)


def _sym(pairs):
    """undirected pairs -> coalesced symmetric (row, col)"""
    r = [a for a, b in pairs] + [b for a, b in pairs]
    c = [b for a, b in pairs] + [a for a, b in pairs]
    o = np.lexsort((c, r))
    return np.asarray(r)[o], np.asarray(c)[o]


def _edge_case_corpus(max_nodes, seed=5):
    """ordinary graphs plus (pool_size 4): 6 one node; 7 nodes but no edges; 8 three isolated trailing nodes; 9 two
    isolated leading nodes and one in the middle; 10 exactly max_nodes nodes; 11 two clusters without an edge between
    them; 12 and 13 single clusters (no coarse entry)"""
    base = synth.make_corpus("PROTEINS", 30, seed=seed)
    graphs = []
    for g in [g for g in range(base.num_graphs) if base.num_nodes(g) <= max_nodes // 2][:6]:
        e0, e1 = base.edge_ptr[g], base.edge_ptr[g + 1]
        graphs.append((base.num_nodes(g), base.row[e0:e1], base.col[e0:e1]))
    rng = np.random.default_rng(seed)
    graphs.append((1, [], []))
    graphs.append((5, [], []))
    r, c = synth._one_graph(rng, 9, 14)
    graphs.append((12, r, c))
    r, c = synth._one_graph(rng, 10, 15)
    shift = np.where(np.asarray(r) >= 5, 3, 2), np.where(np.asarray(c) >= 5, 3, 2)
    graphs.append((13, np.asarray(r) + shift[0], np.asarray(c) + shift[1]))
    r, c = synth._one_graph(rng, max_nodes, 2 * max_nodes)
    graphs.append((max_nodes, r, c))
    graphs.append((8, *_sym([(0, 1), (1, 2), (2, 3), (0, 3), (4, 5), (5, 6), (6, 7)])))
    graphs.append((4, *_sym([(0, 1), (1, 2), (2, 3)])))
    graphs.append((3, *_sym([(0, 2), (1, 2)])))
    return _corpus_of(graphs, seed=seed)


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _host_eigen(corpus, op, ids, max_nodes, dev, J, Jf):
    """the host path pack_eigen replaces: synth.select / pack + K1 for x and the adjacency, eigen_synth.pack_operands +
    build_rect_csr / build_csr(CSR_RAW, edge_weight) for the pooling operators (as tests/test_feeder_gpu.py builds
    bench config 5's final pooling)"""
    from tsg import dense, ops
    sel = synth.select(corpus, ids)
    pk = synth.pack(sel)
    N, G = int(sel.node_ptr[-1]), len(ids)
    csr = ops.build_csr(ops.EdgeList.from_edge_index(_t(pk["edge_index"], dev)), N, mode=ops.CSR_RAW)
    po = eigen_synth.pack_operands(corpus, op, ids)
    NC = int(po["cluster_ptr"][-1])
    el = lambda s, d: ops.EdgeList(_t(s, dev), _t(d, dev), int(s.shape[0]))
    pool = [dense.build_rect_csr(el(s, d), _t(w, dev), NC, N) for s, d, w in po["pool"][:J]]
    s, d, w = po["coarse"]
    if s.shape[0]:
        coarse = ops.build_csr(el(s, d), NC, mode=ops.CSR_RAW, edge_weight=_t(w, dev))
    else:          # K1 takes no empty list: the empty RAW CSR by hand, with pack_eigen's one unreached zero slot
        z = torch.zeros(NC + 1, dtype=torch.int32, device=dev)
        e32, ef = torch.zeros(1, dtype=torch.int32, device=dev), torch.zeros(1, device=dev)
        coarse = ops.CSR(z, e32, ef, None, z, e32, ef, None, NC)
    final = [dense.build_rect_csr(el(s, d), _t(w, dev), G, NC) for s, d, w in po["final"][:Jf]]
    n, nc = np.diff(sel.node_ptr), np.diff(po["cluster_ptr"])
    has_pad = torch.from_numpy(np.stack([n < max_nodes, nc < max_nodes, np.full(G, max_nodes > 1)])).to(dev)
    return dict(x=_t(pk["x"], dev), csr=csr, graph_ptr=_t(sel.node_ptr, dev), pool=pool, coarse=coarse,
                cluster_ptr=_t(po["cluster_ptr"], dev), final=final, final_ptr=torch.arange(G + 1, device=dev),
                has_pad=has_pad)


CSR_FIELDS = ("rowptr", "colidx", "val", "eid", "t_rowptr", "t_colidx", "t_val", "t_eid", "num_nodes")


def _same_csr(a, b, what):
    for f in CSR_FIELDS:
        x, y = getattr(a, f), getattr(b, f)
        if x is None or y is None or isinstance(x, int):
            assert x == y, (what, f)
        else:
            assert x.dtype == y.dtype and torch.equal(x, y), (what, f)
    assert a.tile_ptr is None and not a.tma_ok


def _assert_same_batch(b, h):
    assert torch.equal(b.x, h["x"])
    _same_csr(b.csr, h["csr"], "adjacency")
    assert len(b.pool) == len(h["pool"]) and len(b.final) == len(h["final"])
    for j, (p, q) in enumerate(zip(b.pool, h["pool"])):
        _same_csr(p, q, f"pool {j}")
    _same_csr(b.coarse, h["coarse"], "coarse")
    for j, (p, q) in enumerate(zip(b.final, h["final"])):
        _same_csr(p, q, f"final {j}")
    for f in ("graph_ptr", "cluster_ptr", "final_ptr", "has_pad"):
        x, y = getattr(b, f), h[f]
        assert x.dtype == y.dtype and torch.equal(x, y), f


@pytest.mark.parametrize("shape,G,pool_size", [("DD", 40, 10), ("PROTEINS", 300, 4)])
@pytest.mark.parametrize("J,Jf", [(1, 1), (2, 0), (2, 1), (1, 0)])
def test_pack_eigen_equals_the_host_path(cuda, shape, G, pool_size, J, Jf):
    from tsg import nn as tnn
    from tsg.feeder import DeviceCorpus
    corpus = synth.make_corpus(shape, G, seed=31)
    op = eigen_synth.make_operands(corpus, pool_size, 2, 1)
    dc = DeviceCorpus(corpus, cuda)
    dc.attach_eigen(op)
    assert dc.coalesced
    ids = np.random.default_rng(G + J).integers(0, G, 3 * G)                  # duplicates
    b = dc.pack_eigen(ids, 1000, J, Jf)
    _assert_same_batch(b, _host_eigen(corpus, op, ids, 1000, cuda, J, Jf))
    assert np.array_equal(b.node_ptr_host, synth.select(corpus, ids).node_ptr) and b.max_nodes == 1000
    tnn.check_fused_status()


def test_pack_eigen_edge_cases(cuda):
    from tsg import nn as tnn
    from tsg.feeder import DeviceCorpus
    max_nodes = 64
    corpus = _edge_case_corpus(max_nodes)
    op = eigen_synth.make_operands(corpus, 4, 2, 1)
    assert np.diff(op.coarse_ptr)[11] == 0 and np.diff(op.cluster_ptr)[11] == 2
    dc = DeviceCorpus(corpus, cuda)
    dc.attach_eigen(op)
    G = corpus.num_graphs
    for ids in (np.arange(G), np.arange(G)[::-1], np.array([10]), np.array([7, 6, 0, 7]), np.array([8, 8]),
                np.array([6, 7, 8, 9, 6]), np.array([11, 12, 13, 12]), np.array([12]), np.array([6, 13, 7])):
        for J, Jf in ((2, 1), (1, 0)):
            b = dc.pack_eigen(ids, max_nodes, J, Jf)
            _assert_same_batch(b, _host_eigen(corpus, op, ids, max_nodes, cuda, J, Jf))
    b = dc.pack_eigen([10, 12], max_nodes)
    assert b.has_pad[0].tolist() == [False, True]                            # exactly max_nodes: no zero row
    assert b.coarse.colidx.numel() == np.diff(op.coarse_ptr)[10]
    tnn.check_fused_status()


def test_pack_eigen_general_path_for_lists_that_are_not_coalesced(cuda):
    """edges shuffled within each graph: K0 + K1 build the adjacency, K0e the rest, with the same result"""
    from tsg import nn as tnn
    from tsg.feeder import DeviceCorpus
    c = synth.make_corpus("PROTEINS", 20, seed=9)
    rng = np.random.default_rng(1)
    graphs = []
    for g in range(c.num_graphs):
        e0, e1 = c.edge_ptr[g], c.edge_ptr[g + 1]
        p = rng.permutation(e1 - e0)
        graphs.append((c.num_nodes(g), c.row[e0:e1][p], c.col[e0:e1][p]))
    corpus = _corpus_of(graphs, seed=2)
    op = eigen_synth.make_operands(corpus, 4, 2, 1)
    dc = DeviceCorpus(corpus, cuda)
    dc.attach_eigen(op)
    assert not dc.coalesced
    ids = rng.integers(0, 20, 50)
    _assert_same_batch(dc.pack_eigen(ids, 1000), _host_eigen(corpus, op, ids, 1000, cuda, 2, 1))
    tnn.check_fused_status()


@pytest.mark.parametrize("broken,bit,msg", [("cluster_id", 16, "EigenPooling operands"),
                                            ("coarse_unsorted", 16, "EigenPooling operands"),
                                            ("coarse_asymmetric", 16, "EigenPooling operands"),
                                            ("coarse_weight", 16, "EigenPooling operands"),
                                            ("adj_unsorted", 2, "not sorted"), ("adj_self_loop", 1, "self loop"),
                                            ("adj_asymmetric", 4, "not symmetric")])
def test_pack_eigen_reports_a_broken_promise(cuda, broken, bit, msg):
    from tsg import nn as tnn
    from tsg.feeder import DeviceCorpus
    c = synth.make_corpus("PROTEINS", 6, seed=3)
    op = eigen_synth.make_operands(c, 4, 1, 1)
    row, col = c.row.copy(), c.col.copy()
    e0, q0 = int(c.edge_ptr[2]), int(op.coarse_ptr[2])
    assert op.coarse_ptr[3] - q0 >= 2
    cl, qr, qc, qw = op.cluster_of.copy(), op.coarse_row.copy(), op.coarse_col.copy(), op.coarse_w.copy()
    if broken == "cluster_id":
        cl[int(c.node_ptr[2]) + 1] = op.cluster_ptr[3] - op.cluster_ptr[2]            # = nc of graph 2
    elif broken == "coarse_unsorted":
        qr[q0], qr[q0 + 1], qc[q0], qc[q0 + 1] = qr[q0 + 1], qr[q0], qc[q0 + 1], qc[q0]
    elif broken == "coarse_asymmetric":                 # drop one entry: the list stays sorted, loses a partner
        keep = np.ones(qr.shape[0], bool); keep[q0] = False
        qr, qc, qw = qr[keep], qc[keep], qw[keep]
        op = dataclasses.replace(op, coarse_ptr=np.concatenate([op.coarse_ptr[:3], op.coarse_ptr[3:] - 1]))
    elif broken == "coarse_weight":
        qw[q0] += 1.0
    elif broken == "adj_unsorted":
        row[e0], row[e0 + 1], col[e0], col[e0 + 1] = row[e0 + 1], row[e0], col[e0 + 1], col[e0]
    elif broken == "adj_self_loop":
        col[e0] = row[e0]
    else:                                  # drop one direction of an edge: keep the list sorted, lose its partner
        keep = np.ones(row.shape[0], bool); keep[e0] = False
        ep = c.edge_ptr.copy(); ep[3:] -= 1
        row, col = row[keep], col[keep]
        c = synth.Corpus(c.name, c.node_ptr, ep, row, col, c.node_label, c.y, c.num_node_labels)
    op = dataclasses.replace(op, cluster_of=cl, coarse_row=qr, coarse_col=qc, coarse_w=qw)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a.astype(np.int32))).to(cuda)
    dc = DeviceCorpus.from_device(t(c.node_label), t(row), t(col), c.node_ptr, c.edge_ptr, c.num_node_labels,
                                  coalesced=True)
    dc.attach_eigen(op)
    tnn.check_fused_status()
    b = dc.pack_eigen(np.arange(6), 1000)
    torch.cuda.synchronize()
    assert int(tnn._status_word(cuda).item()) == bit
    N, NC = b.x.size(0), int(b.cluster_ptr_host[-1])          # indices stay in range
    assert 0 <= int(b.csr.colidx.min()) and int(b.csr.colidx.max()) < N
    assert 0 <= int(b.pool[0].colidx.min()) and int(b.pool[0].colidx.max()) < N
    assert 0 <= int(b.pool[0].t_colidx.min()) and int(b.pool[0].t_colidx.max()) < NC
    assert 0 <= int(b.coarse.colidx.min()) and int(b.coarse.colidx.max()) < NC
    assert int(b.pool[0].rowptr[-1]) == N and (b.pool[0].rowptr.diff() >= 0).all()
    with pytest.raises(RuntimeError, match=msg):
        tnn.check_fused_status()


# ------------------------------------------------------------------------------------------ training
def _model(dev, F, J=1, Jf=1, seed=777):
    from tsg import dense
    torch.manual_seed(seed)
    return dense.PackedWaveEncoder(F, 32, 32, 2, 2, num_pool_matrix=J, num_pool_final_matrix=Jf, pool_sizes=[10],
                                   pred_hidden_dims=[50]).to(dev)


def _triplet_ids(corpus, T, seed):
    trip = synth.sample_triplets(corpus.y, T, seed=seed)
    ids = np.concatenate([trip[:, 0], trip[:, 1], trip[:, 2]])
    tidx = np.stack([np.arange(T), T + np.arange(T), 2 * T + np.arange(T)], 1).astype(np.int64)
    return ids, torch.from_numpy(tidx).pin_memory()


def _bench_step(model, opt, h, tr, clip=None):
    """bench.py Config5.step on the host-assembled batch: model forward, triplet loss, Adam (plus a manual clip)"""
    from tsg import ops
    emb = model(h["x"], h["csr"], h["graph_ptr"], [h["pool"], h["final"]], [h["coarse"]], [h["cluster_ptr"]],
                h["final_ptr"], has_pad=list(h["has_pad"]))
    loss, _, _ = ops.triplet_loss(emb, tr, 1.5)
    opt.zero_grad(set_to_none=True); loss.backward()
    if clip is not None:
        torch.nn.utils.clip_grad_norm_(model.parameters(), clip)
    opt.step()
    return loss.detach()


@pytest.mark.parametrize("shape,T,J,Jf", [("DD", 10, 1, 1), ("PROTEINS", 40, 2, 0)])
def test_step_from_ids_is_the_bench_step(cuda, shape, T, J, Jf):
    from tsg.feeder import DeviceCorpus
    from tsg.train import WaveTripletTrainer
    corpus = synth.make_corpus(shape, 3 * T, seed=41)
    op = eigen_synth.make_operands(corpus, 10, J, Jf)
    dc = DeviceCorpus(corpus, cuda)
    dc.attach_eigen(op)
    ids, tr = _triplet_ids(corpus, T, 0)
    h = _host_eigen(corpus, op, ids, 1000, cuda, J, Jf)
    F = corpus.num_node_labels
    for clip in (None, 2.0):
        ma, mb = _model(cuda, F, J, Jf), _model(cuda, F, J, Jf)
        ta = WaveTripletTrainer(ma, 1000, clip_norm=clip)
        ob = torch.optim.Adam(mb.parameters(), lr=1e-3)
        if clip is None:
            la = torch.tensor(ta.run_from_ids(dc, [(ids, tr)])[0])
        else:
            la = ta.step(ta.pack(dc, ids), tr.to(cuda)).cpu()
        lb = _bench_step(mb, ob, h, tr.to(cuda), clip).cpu()
        assert torch.equal(la, lb), (clip, float(la), float(lb))
        for (k, pa), pb in zip(ma.named_parameters(), mb.parameters()):
            assert pa.grad is not None and torch.equal(pa.grad, pb.grad), (clip, "grad", k)
            assert torch.equal(pa, pb), (clip, "param", k)


def test_without_has_pad_the_forward_is_bench_config_5s(cuda):
    """has_pad=None keeps the all-padded readout; with every graph padded, the flags change nothing"""
    from tsg.feeder import DeviceCorpus
    corpus = synth.make_corpus("DD", 12, seed=7)
    dc = DeviceCorpus(corpus, cuda)
    dc.attach_eigen(eigen_synth.make_operands(corpus, 10, 1, 1))
    b = dc.pack_eigen(np.arange(12), 1000)
    assert bool(b.has_pad.all())
    m = _model(cuda, corpus.num_node_labels)
    args, kw = b.readout_args()
    with torch.no_grad():
        assert torch.equal(m(*args), m(*args, **kw))
        assert torch.equal(m(*args), m.pred_model(m.readout(*args)))


def test_run_from_ids_trains_over_many_steps(cuda):
    from tsg.feeder import DeviceCorpus
    from tsg.train import WaveTripletTrainer
    corpus = synth.make_corpus("PROTEINS", 60, seed=42)
    dc = DeviceCorpus(corpus, cuda)
    dc.attach_eigen(eigen_synth.make_operands(corpus, 10, 1, 1))
    ta = WaveTripletTrainer(_model(cuda, corpus.num_node_labels), 1000)
    losses = ta.run_from_ids(dc, [_triplet_ids(corpus, 20, s) for s in range(6)])
    assert len(losses) == 6 and all(np.isfinite(losses))
    assert ta.run_from_ids(dc, []) == []


# ------------------------------------------------------------------------------------------ embeddings
def _oracle_embed(model, corpus, op, ids, max_nodes):
    """per graph, padded to max_nodes: oracle/dense_ref.wave_readout, then mlp with pred_model's layers, CPU fp32"""
    cs = lambda mods: [dict(weight=c.weight.detach().cpu(), bias=c.bias.detach().cpu()) for c in mods]
    p = dict(conv=cs([model.conv_first] + list(model.conv_block) + [model.conv_last]),
             conv_after=[cs([model.conv_first_after_pool[0]] + list(model.conv_block_after_pool[0]) +
                            [model.conv_last_after_pool[0]])])
    head = [dict(weight=l.weight.detach().cpu(), bias=l.bias.detach().cpu()) for l in model.pred_model
            if isinstance(l, torch.nn.Linear)]
    J, Jf, N = model.num_pool_matrix, model.num_pool_final_matrix, max_nodes
    out = []
    with torch.no_grad():
        for g in ids:
            n0, n = int(corpus.node_ptr[g]), corpus.num_nodes(int(g))
            e0, e1 = corpus.edge_ptr[g], corpus.edge_ptr[g + 1]
            c0, nc = int(op.cluster_ptr[g]), int(op.cluster_ptr[g + 1] - op.cluster_ptr[g])
            q0, q1 = int(op.coarse_ptr[g]), int(op.coarse_ptr[g + 1])
            adj = torch.zeros(1, N, N); adj[0, torch.from_numpy(corpus.row[e0:e1]), torch.from_numpy(corpus.col[e0:e1])] = 1
            x = torch.zeros(1, N, corpus.num_node_labels); x[0, torch.arange(n), torch.from_numpy(corpus.node_label[n0:n0 + n]).long()] = 1
            cl = torch.from_numpy(op.cluster_of[n0:n0 + n])
            P = []
            for j in range(J):
                m = torch.zeros(1, N, N); m[0, torch.arange(n), cl] = torch.from_numpy(op.pool_w[j][n0:n0 + n]); P.append(m)
            Pf = []
            for j in range(Jf):
                m = torch.zeros(1, N, N); m[0, :nc, 0] = torch.from_numpy(op.final_w[j][c0:c0 + nc]); Pf.append(m)
            ap = torch.zeros(1, N, N)
            ap[0, torch.from_numpy(op.coarse_row[q0:q1]), torch.from_numpy(op.coarse_col[q0:q1])] = torch.from_numpy(op.coarse_w[q0:q1])
            r = D.wave_readout(x, adj, [ap], [n], [[nc]], [P, Pf], p, num_pool_matrix=J, num_pool_final_matrix=Jf)
            out.append(D.mlp(r, head))
    return torch.cat(out)


@pytest.mark.parametrize("J,Jf", [(1, 1), (2, 1), (2, 0)])
def test_embed_matches_the_oracle(cuda, J, Jf):
    from tsg.feeder import DeviceCorpus
    from tsg.train import WaveTripletTrainer
    max_nodes = 64
    corpus = _edge_case_corpus(max_nodes, seed=8)
    op = eigen_synth.make_operands(corpus, 4, J, Jf)
    dc = DeviceCorpus(corpus, cuda)
    dc.attach_eigen(op)
    model = _model(cuda, corpus.num_node_labels, J, Jf)
    with torch.no_grad():                                  # non-zero biases: the padded rows' zero then matters
        for k, p in model.named_parameters():
            if k.endswith("bias"):
                p.copy_(torch.randn_like(p) * 0.2)
    tt = WaveTripletTrainer(model, max_nodes)
    ids = np.random.default_rng(0).permutation(corpus.num_graphs)
    model.train()
    emb = tt.embed(dc, ids)
    assert model.training, "embed restores the training flag"
    ref = _oracle_embed(model, corpus, op, ids, max_nodes)
    assert emb.shape == ref.shape and rel_err(emb, ref) <= TOL
    # one small graph alone: a single cluster, so an empty coarsened adjacency
    for g in (12, 13):
        assert rel_err(tt.embed(dc, [g]), _oracle_embed(model, corpus, op, [g], max_nodes)) <= TOL, g
    model.eval()
    sub = ids[np.diff(corpus.edge_ptr)[ids] > 0]            # a batch needs one edge: the split runs over those graphs
    whole = tt.embed(dc, sub, batch_graphs=len(sub))
    for bg in (1, 5):
        assert torch.equal(tt.embed(dc, sub, batch_graphs=bg), whole), bg
        assert not model.training
    dup = tt.embed(dc, np.concatenate([sub, sub[[3, 0, 3]]]))
    assert torch.equal(dup[len(sub):], dup[torch.tensor([3, 0, 3])])


# ------------------------------------------------------------------------------------------ scoring
def _boundary_is_clear(train, query, k):
    d = ((query[:, None, :].astype(np.float64) - train[None, :, :].astype(np.float64)) ** 2).sum(-1)
    s = np.sort(d, axis=1)
    if s.shape[1] <= k:
        return True
    gap = s[:, k] - s[:, k - 1]
    return bool(np.all((gap == 0) | (gap > 1e-5 * np.maximum(s[:, k], 1e-30))))


def _trainer(G, dev, seed=4, classes=3):
    from tsg.feeder import DeviceCorpus
    from tsg.train import WaveTripletTrainer
    corpus = synth.make_corpus("DD", G, seed=seed)
    corpus.y = np.random.default_rng(seed).integers(0, classes, G).astype(np.int64)
    dc = DeviceCorpus(corpus, dev)
    dc.attach_eigen(eigen_synth.make_operands(corpus, 10, 1, 1))
    return corpus, dc, WaveTripletTrainer(_model(dev, corpus.num_node_labels), 1000)


def test_evaluate_knn_equals_the_oracle(cuda):
    corpus, dc, tt = _trainer(60, cuda)
    perm = np.random.default_rng(1).permutation(60)
    tr_ids, ev_ids = perm[:45], perm[45:]
    for k in (1, 3, 8):
        acc = tt.evaluate(dc, tr_ids, ev_ids, head="knn", k=k, batch_graphs=16)
        tr = tt.embed(dc, tr_ids).cpu().numpy(); ev = tt.embed(dc, ev_ids).cpu().numpy()
        assert _boundary_is_clear(tr, ev, k), "near-tie in the embeddings' distances: pick another seed"
        pred = H.knn_predict(tr, corpus.y[tr_ids], ev, k)
        assert acc * len(ev_ids) == float((pred == corpus.y[ev_ids]).sum()), k
    assert tt.model.training


def test_evaluate_mlp_is_embed_plus_the_classifier(cuda):
    from tsg import heads
    corpus, dc, tt = _trainer(40, cuda)
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
