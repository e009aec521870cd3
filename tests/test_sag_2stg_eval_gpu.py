"""The 2stg evaluation on the GPU: TripletTrainer.embed against the float64-checked oracle forward, against
native_classify and against its own autograd-free fallback; TripletTrainer.evaluate against heads_ref's kNN and Adam loop
on the same embeddings; tsg_knn_classify against the oracle over class counts up to 1,024 and k up to 32 (exact ties
included); tsg_mlp1_predict's logits against the trainer's fmaf chain, bit for bit; and evaluate leaving the model, its
next training step and the RNG stream untouched."""
import numpy as np
import pytest
import torch

from conftest import rel_err
from oracle import heads_ref as H
from test_sag_classify_gpu import _compact, _corpus, _model
from test_sag_widths_gpu import _oracle, _same_selection
from tsg import synth

pytestmark = pytest.mark.gpu
TOL = 1e-5
FINAL_DIM = 16          # embedding width of the triplet models here (their "num_classes")

# (shape, G, nhid, seed): corpora whose fp32 and float64 oracles select the same nodes (tests/test_sag_widths_gpu.py)
EMBED_CASES = [("DD", 9, 32, 2041), ("PROTEINS", 48, 128, 13041)]


def _setup(shape, G, nhid, seed, dev, graph_classes=2, dropout=0.5):
    from tsg.feeder import DeviceCorpus
    from tsg.train import TripletTrainer
    corpus = _corpus(shape, G, graph_classes, seed)
    model, params = _model(corpus, nhid, FINAL_DIM, dev, dropout=dropout)
    return corpus, DeviceCorpus(corpus, dev), model, params, TripletTrainer(model)


@pytest.mark.parametrize("shape,G,nhid,seed", EMBED_CASES)
def test_embed_matches_the_oracle_and_native_classify(cuda, shape, G, nhid, seed):
    from tsg import nn as tnn
    corpus, dc, model, params, tt = _setup(shape, G, nhid, seed, cuda)
    model.train()
    cb = _compact(corpus, cuda)
    assert model.native_step_supported(cb, corpus.node_ptr)
    tnn.KEEP_ARENA = True
    try:
        emb = tt.embed(dc, np.arange(G))
        shape_, arena = tnn.LAST_ARENA
    finally:
        tnn.KEEP_ARENA = False
    assert model.training, "embed restores the training flag"
    perms = [tnn.sag_arena_view(shape_, arena, lvl, "perm").cpu() for lvl in range(3)]
    b = synth.pack(corpus)
    out32, aux32, _, _ = _oracle(params, b, torch.float32)
    out64, aux64, _, _ = _oracle(params, b, torch.float64)
    _same_selection(aux32, aux64, "eval forward")
    for lvl in range(3):
        assert torch.equal(perms[lvl], aux32["perm"][lvl]), f"perm level {lvl}"
    assert emb.shape == (G, FINAL_DIM) and emb.is_cuda
    assert rel_err(emb, out32) <= TOL
    # the same call the classification forward makes, bit for bit
    _, logp, _, _ = model.native_classify(cb, corpus.node_ptr)
    assert torch.equal(emb, logp)
    tnn.check_fused_status()


def test_embed_fallback_paths(cuda, monkeypatch):
    from tsg import nn as tnn
    shape, G, nhid, seed = EMBED_CASES[0]
    corpus, dc, model, params, tt = _setup(shape, G, nhid, seed, cuda)
    native = tt.embed(dc, np.arange(G))
    monkeypatch.setattr(tnn, "USE_NATIVE_STEP", False)            # what TSG_NATIVE_STEP=0 selects
    monkeypatch.setattr(model, "native_classify", lambda *a, **k: pytest.fail("native path taken"))
    model.train()
    fallback = tt.embed(dc, np.arange(G))
    assert model.training
    assert rel_err(fallback, native) <= TOL
    monkeypatch.undo()
    # a shape the native steps refuse (odd width): the no_grad forward, against the oracle
    corpus, dc, model, params, tt = _setup("DD", 7, 33, 12041, cuda)
    assert not model.native_step_supported(_compact(corpus, cuda), corpus.node_ptr)
    monkeypatch.setattr(model, "native_classify", lambda *a, **k: pytest.fail("native path taken"))
    emb = tt.embed(dc, np.arange(7))
    out32, aux32, _, _ = _oracle(params, synth.pack(corpus), torch.float32)
    _same_selection(aux32, _oracle(params, synth.pack(corpus), torch.float64)[1], "eval forward")
    assert rel_err(emb, out32) <= TOL


def test_embed_returns_rows_in_ids_order(cuda):
    shape, G, nhid, seed = EMBED_CASES[0]
    corpus, dc, model, params, tt = _setup(shape, G, nhid, seed, cuda)
    ref = tt.embed(dc, np.arange(G))
    ids = np.concatenate([np.random.default_rng(4).permutation(G), [3, 3, 0, 8, 3]])    # shuffled + duplicates
    got = tt.embed(dc, ids, batch_graphs=4)                                             # four packed batches
    assert got.shape == (ids.shape[0], FINAL_DIM)
    # a graph's embedding does not depend on the batch it is packed in (per-graph encoder, per-row head): bit for bit
    assert torch.equal(got, ref[torch.from_numpy(ids).to(cuda)])
    assert tt.embed(dc, np.zeros(0, np.int64)).shape == (0, FINAL_DIM)


def _boundary_is_clear(train, query, k):
    """No query has two train rows at nearly (but not exactly) equal float64 distance across its k-th neighbour: the
    fp32 kernel and the float64 oracle then pick the same neighbour set."""
    d = ((query[:, None, :].astype(np.float64) - train[None, :, :].astype(np.float64)) ** 2).sum(-1)
    s = np.sort(d, axis=1)
    if s.shape[1] <= k:
        return True
    gap = s[:, k] - s[:, k - 1]
    return bool(np.all((gap == 0) | (gap > 1e-5 * np.maximum(s[:, k], 1e-30))))


def test_evaluate_knn_equals_the_oracle_on_the_same_embeddings(cuda):
    corpus, dc, model, params, tt = _setup("PROTEINS", 60, 32, 5, cuda, graph_classes=3)
    perm = np.random.default_rng(1).permutation(60)
    tr_ids, ev_ids = perm[:48], perm[48:]
    for k in (1, 3, 8):
        acc = tt.evaluate(dc, tr_ids, ev_ids, head="knn", k=k, batch_graphs=16)
        tr = tt.embed(dc, tr_ids).cpu().numpy(); ev = tt.embed(dc, ev_ids).cpu().numpy()
        assert _boundary_is_clear(tr, ev, k), "near-tie in the embeddings' distances: pick another seed"
        pred = H.knn_predict(tr, corpus.y[tr_ids], ev, k)
        assert acc == float((pred == corpus.y[ev_ids]).sum()) / len(ev_ids), k
    assert model.training


# integer coordinates: every distance is exact in fp32 and float64, and many are equal -- the tie rules decide
@pytest.mark.parametrize("C", [2, 17, 40, 1024])
@pytest.mark.parametrize("k", [1, 3, 8, 32])
@pytest.mark.parametrize("M,Q", [(300, 77), (5, 9), (20, 0)])
def test_knn_classify_matches_the_oracle(cuda, C, k, M, Q):
    from tsg import heads
    rng = np.random.default_rng(C * 1000 + k * 10 + M)
    D = 4
    train = rng.integers(-2, 3, (M, D)).astype(np.float32)
    query = rng.integers(-2, 3, (Q, D)).astype(np.float32)
    labels = rng.integers(0, C, M); qlabels = rng.integers(0, C, Q)
    labels[: min(M, 3)] = C - 1                                     # the top class is used
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda)
    pred, correct = heads.knn_classify(t(train), t(labels), t(query), t(qlabels), k=k, num_classes=C)
    ref = H.knn_predict(train, labels, query, k) if Q else np.zeros(0, np.int64)
    assert np.array_equal(pred.cpu().numpy(), ref)
    assert int(correct.item()) == int((ref == qlabels).sum())
    pred2, none = heads.knn_classify(t(train), t(labels), t(query), k=k, num_classes=C)
    assert none is None and torch.equal(pred, pred2)


def test_knn_classify_at_the_default_shared_memory_boundary(cuda):
    """D + 64 k + C = 3,072 floats per warp: with the CTA's tallies the request is just past 48 KB and must opt in"""
    from tsg import heads
    rng = np.random.default_rng(7)
    D, k, C, M, Q = 64, 32, 960, 500, 300
    train = rng.integers(-1, 2, (M, D)).astype(np.float32)
    query = rng.integers(-1, 2, (Q, D)).astype(np.float32)
    labels = rng.integers(0, C, M); qlabels = rng.integers(0, C, Q)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda)
    pred, correct = heads.knn_classify(t(train), t(labels), t(query), t(qlabels), k=k, num_classes=C)
    ref = H.knn_predict(train, labels, query, k)
    assert np.array_equal(pred.cpu().numpy(), ref)
    assert int(correct.item()) == int((ref == qlabels).sum())


def test_knn_classify_reports_out_of_range_labels(cuda):
    from tsg import heads, nn as tnn
    rng = np.random.default_rng(0)
    train = torch.from_numpy(rng.normal(size=(30, 8)).astype(np.float32)).to(cuda)
    query = torch.from_numpy(rng.normal(size=(10, 8)).astype(np.float32)).to(cuda)
    labels = torch.from_numpy(rng.integers(0, 5, 30)).to(cuda); qlabels = torch.from_numpy(rng.integers(0, 5, 10)).to(cuda)
    tnn.check_fused_status()
    status = tnn._status_word(cuda)
    heads.knn_classify(train, labels, query, qlabels, k=30, num_classes=5, status=status)
    tnn.check_fused_status()
    for bad_train, bad_query in ((True, False), (False, True)):
        lb, qb = labels.clone(), qlabels.clone()
        if bad_train:
            lb[7] = 5                            # k = 30 = M: every train row votes, so the bad one is read
        else:
            qb[2] = -1
        status = tnn._status_word(cuda)
        heads.knn_classify(train, lb, query, qb, k=30, num_classes=5, status=status)
        with pytest.raises(RuntimeError, match="label"):
            tnn.check_fused_status()


def _fma(p_a, p_b, c):
    """fmaf(a, b, c) for float32 arrays, exactly: a * b is exact in float64, the sum's rounding error comes from TwoSum,
    and a float64 sum that lands on a float32 rounding midpoint is moved by the sign of that error."""
    p = p_a.astype(np.float64) * p_b.astype(np.float64)
    c64 = c.astype(np.float64)
    s = p + c64
    bp = s - c64
    e = (p - (s - bp)) + (c64 - bp)
    r = s.astype(np.float32)
    d = s - r.astype(np.float64)
    other = np.nextafter(r, np.where(d > 0, np.float32(np.inf), np.float32(-np.inf)).astype(np.float32))
    tie = (d != 0) & (np.abs(d) == np.abs(other.astype(np.float64) - r.astype(np.float64)) / 2)
    fix = tie & (np.sign(e) == np.sign(d))
    return np.where(fix, other, r).astype(np.float32)


def _trainer_forward(views, x, slope):
    """k_mlp1_train's forward: per unit, bias then one fmaf chain over the input index ascending; LeakyReLU in fp32."""
    w1, b1, w2, b2, w3, b3 = [v.cpu().numpy() for v in views]
    h = x.astype(np.float32)
    for i, (w, b) in enumerate(((w1, b1), (w2, b2), (w3, b3))):
        a = np.broadcast_to(b[None, :], (h.shape[0], b.shape[0])).astype(np.float32)
        for d in range(w.shape[1]):
            a = _fma(h[:, d:d + 1], w[None, :, d], a)
        h = a if i == 2 else np.where(a > 0, a, np.float32(slope) * a).astype(np.float32)
    return h


@pytest.mark.parametrize("D,C,Q", [(16, 2, 300), (128, 7, 2500), (32, 32, 65), (16, 40, 33), (16, 2, 1), (16, 3, 0)])
def test_mlp1_predict_is_the_trainers_forward(cuda, D, C, Q):
    from tsg import heads, nn as tnn
    torch.manual_seed(D + C)
    clf = heads.Mlp1Classifier(D, cuda, num_classes=C)
    g = torch.Generator().manual_seed(Q)
    trainable = C <= 32                                                 # tsg_mlp1_train's limit; the predictor has none
    if trainable:
        clf.fit(torch.randn(40, D, generator=g).to(cuda), torch.randint(0, C, (40,), generator=g).to(cuda))
    x = torch.randn(Q, D, generator=g)
    if Q > 3:
        x[3] = x[1]                                                     # two identical rows
    y = torch.randint(0, C, (Q,), generator=g)
    status = tnn._status_word(cuda)
    pred, logits, correct = heads.mlp1_predict(clf, x.to(cuda), y.to(cuda), want_logits=True, status=status)
    tnn.check_fused_status()
    assert torch.equal(logits.cpu(), torch.from_numpy(_trainer_forward(clf.views(), x.numpy(), clf.slope)))
    assert torch.equal(pred, logits.argmax(dim=1))
    assert int(correct.item()) == int((pred.cpu() == y).sum())
    assert torch.equal(clf.score(x.to(cuda), y.to(cuda)), correct)
    if Q and trainable:
        # the trainer's own loss at these parameters (lr 0: the parameters stay) is the cross-entropy of these logits
        still = heads.Mlp1Classifier(D, cuda, num_classes=C, lr=0.0)
        still.params.copy_(clf.params)
        losses = still.fit(x.to(cuda), y.to(cuda), want_losses=True)
        assert torch.equal(still.params, clf.params)
        ce = torch.nn.functional.cross_entropy(logits.double().cpu(), y, reduction="none")
        assert (losses.double().cpu() - ce).abs().max() <= 1e-5 * max(1.0, float(ce.abs().max()))


def test_mlp1_predict_argmax_ties_and_label_range(cuda):
    from tsg import heads, nn as tnn
    torch.manual_seed(0)
    clf = heads.Mlp1Classifier(8, cuda, num_classes=37)
    w1, b1, w2, b2, w3, b3 = clf.views()
    w3.zero_(); b3.zero_()
    b3[5] = 1.0; b3[36] = 1.0; b3[33] = 1.0                             # equal maxima owned by lanes 5, 4 and 1
    x = torch.randn(70, 8).to(cuda)
    pred, logits, _ = heads.mlp1_predict(clf, x, want_logits=True)
    assert torch.equal(pred, torch.full_like(pred, 5)) and torch.equal(pred, logits.argmax(dim=1))
    tnn.check_fused_status()
    y = torch.full((70,), 5, dtype=torch.int64, device=cuda)
    y[9] = 37
    status = tnn._status_word(cuda)
    assert int(clf.score(x, y, status=status).item()) == 69
    with pytest.raises(RuntimeError, match="label"):
        tnn.check_fused_status()


def test_evaluate_mlp_losses_match_the_reference_loop(cuda, monkeypatch):
    """one epoch of evaluate(head="mlp"): the Adam loop of evaluate_mlp on CPU torch (heads_ref.mlp1_train) from the same
    seeded initial weights, per-step losses to 1e-5; the accuracy is the trained classifier's count"""
    from tsg import heads
    corpus, dc, model, params, tt = _setup("PROTEINS", 30, 32, 8, cuda)
    perm = np.random.default_rng(2).permutation(30)
    tr_ids, ev_ids = perm[:24], perm[24:]
    recorded = []
    fit = heads.Mlp1Classifier.fit

    def recording_fit(self, emb, labels, want_losses=False):
        recorded.append((self.params.clone(), fit(self, emb, labels, want_losses=True)))
        return recorded[-1][1]
    monkeypatch.setattr(heads.Mlp1Classifier, "fit", recording_fit)
    acc = tt.evaluate(dc, tr_ids, ev_ids, head="mlp", seed=11)
    assert len(recorded) == 1
    emb_tr = tt.embed(dc, tr_ids).cpu(); emb_ev = tt.embed(dc, ev_ids).cpu()
    torch.manual_seed(11)
    ref_model = H.make_model(FINAL_DIM)
    ref_losses = H.mlp1_train(emb_tr, torch.from_numpy(corpus.y[tr_ids]), ref_model)
    assert rel_err(recorded[0][1], torch.tensor(ref_losses)) <= TOL
    # the accuracy: the same seeded classifier, trained the same way, scored by tsg_mlp1_predict
    monkeypatch.undo()
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(11)
        clf = heads.Mlp1Classifier(FINAL_DIM, cuda, num_classes=2)
    assert torch.equal(clf.params, recorded[0][0]), "initial weights drawn from `seed`"
    clf.fit(emb_tr.to(cuda), torch.from_numpy(corpus.y[tr_ids]).to(cuda))
    correct = clf.score(emb_ev.to(cuda), torch.from_numpy(corpus.y[ev_ids]).to(cuda))
    assert acc == int(correct.item()) / len(ev_ids)
    # two epochs continue the same classifier
    acc2 = tt.evaluate(dc, tr_ids, ev_ids, head="mlp", seed=11, mlp_epochs=2)
    clf.fit(emb_tr.to(cuda), torch.from_numpy(corpus.y[tr_ids]).to(cuda))
    assert acc2 == int(clf.score(emb_ev.to(cuda), torch.from_numpy(corpus.y[ev_ids]).to(cuda)).item()) / len(ev_ids)


def test_evaluate_has_no_side_effects(cuda):
    """training flag restored, CPU RNG stream untouched, and the next native triplet step bitwise what it is without
    the evaluate calls"""
    shape, G, nhid, seed = "PROTEINS", 24, 32, 6
    corpus, dc, model_a, params, ta = _setup(shape, G, nhid, seed, cuda)
    _, _, model_b, _, tb = _setup(shape, G, nhid, seed, cuda)
    tr_ids, ev_ids = np.arange(18), np.arange(18, 24)
    model_a.train()
    rng = torch.get_rng_state()
    ta.evaluate(dc, tr_ids, ev_ids, head="mlp", seed=3)
    ta.evaluate(dc, tr_ids, ev_ids, head="knn")
    assert model_a.training
    assert torch.equal(torch.get_rng_state(), rng), "evaluate moved the RNG stream"
    model_a.eval()
    ta.evaluate(dc, tr_ids, ev_ids)
    assert not model_a.training
    model_a.train()
    cb = _compact(corpus, cuda)
    trip = torch.from_numpy(np.stack([np.random.default_rng(i).permutation(G)[:3] for i in range(16)])).to(cuda)
    assert model_a.native_step_supported(cb, corpus.node_ptr)
    la, lb = ta.step(cb, None, corpus.node_ptr, trip), tb.step(cb, None, corpus.node_ptr, trip)
    assert torch.equal(la, lb)
    for (k, pa), pb in zip(model_a.named_parameters(), model_b.parameters()):
        assert torch.equal(pa.grad, pb.grad), k
        assert torch.equal(pa, pb), k
