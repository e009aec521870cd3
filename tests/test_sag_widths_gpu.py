"""The native SAGPool steps over the whole range of hidden widths and class counts they accept, against the float64
oracle.  tsg_sag_nll_step_compact, tsg_sag_triplet_step_compact, the two step halves and tsg_sag_classify_compact take
every even nhid and every class count C whose head fits shared memory (k14_sag_step.cu head_shape_ok); the bench and the
other tests run three widths.  Each row of ROWS is there for the branches it reaches (F4 = nhid / 4 float4 columns,
H2 = nhid / 2, "narrow" head = k_head_bwd's per-CTA gradient row, "wide" head = k_head_delta + K3's reductions):

  nhid, C    reaches
  2, 2       H2 = 1, F4 = 0: the scalar K2 (launch_spmm's non-float4 branch), gate_gather_fwd + readout_fwd and the
             non-fused level backward (k10_sag_exec.cu: H % 4 != 0)
  6, 3       H % 4 == 2: the non-fused forward (gate_gather + readout) and backward (gate_gather_bwd + relu_bwd_colsum of
             dscore + linear_bwd_weight(h, dsw) + relu_bwd_colsum_rank1); odd H2 in every head kernel
  48, 33     F4 = 12 < 16 lanes: the K2 dot epilogue (k2_spmm.cu fuse_dot) with idle lanes; C = 33: lane 0 of
             k_head_fwd / head_delta owns classes 0 and 32
  62, 31     H % 4 == 2, odd H2 = 31, C < 32 (lane 31 idle in the class loops)
  94, 27     narrow head at a width where C = 28 is wide
  94, 28     wide head: odd H2 = 47 and H = 94 put every tsg_linear_bwd_weight call of the head on K3's generic path
             (K or M not a multiple of 4)
  96, 7      narrow head, width a multiple of 4
  96, 8      wide head at the same width: K3's generic path for lin1 / lin2, its dense path for lin3
  94, 256    the largest C the wide head takes (head_shape_ok: C <= 256); 8 classes per lane
  100, 10    F4 = 25 on 32 lanes: the K2 dot epilogue with 7 idle lanes; wide head
  130, 65    nhid > 128 (label_spmm off) and H % 4 == 2; the largest C at this width; lin1's input 2H = 260 > 256
             columns in K3's weight gradient (M loop of k_linear_bwd_weight)
  132, 33    nhid > 128 with F4 = 33 > 32: K2 without the dot epilogue, and the fused gate_score_bwd /
             sag_conv_bwd_fused / gate_readout loop more than once over a row's float4 columns
  136, 2     the largest accepted width
  32, 1038   the largest C of the narrow head; 33 classes per lane

G in {1, 7, 9} across the rows, so that the head's batches of 8 graphs end short.  LARGE adds ~2,400 PROTEINS-shape
graphs (> 2 x 148 SMs x 8, TILE graphs repeated): every k_head_bwd CTA covers several batches of 8 graphs and k_head_fwd / k_head_delta
grid-stride; at nhid 32 (narrow) and 128 (wide).

Every row: the NLL step (injected dropout mask) against the fp32 oracle to 1e-5 (embeddings, loss) and against float64
through grad_check (18 gradients); every level's perm equal to the oracle's; the classification forward's pred / correct
exactly and nll_sum to 1e-5 against the eval-mode oracle; its log-probabilities bitwise equal to the step forward's
(native_forward, all-ones mask).  The triplet step on a subset.  FALLBACK shapes are refused by native_step_supported and
train / evaluate through autograd against the same oracle.  tests/test_sag_widths.py pins this table to the library's
workspace queries on the host."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import grad_check, rel_err
from oracle import pyg_ref as R
from test_sag_classify_gpu import _compact, _corpus, _mask, _model
from tsg import synth

pytestmark = pytest.mark.gpu
TOL = 1e-5

# (nhid, C, G, seed, head backward); seeds chosen so that the fp32 and float64 oracles select the same nodes (no near-tie)
ROWS = [
    (2, 2, 7, 2041, "narrow"),       # H2 = 1, F4 = 0, scalar K2 / gate / readout
    (6, 3, 9, 11041, "narrow"),      # % 4 == 2 encoder branches, odd H2
    (48, 33, 1, 1041, "narrow"),     # K2 dot epilogue with idle lanes, C = 33 (one lane owns two classes)
    (62, 31, 7, 11041, "narrow"),    # % 4 == 2, odd H2, C < 32
    (94, 27, 9, 11041, "narrow"),    # same H, narrow head ...
    (94, 28, 9, 11041, "wide"),      # ... then wide head; odd H2 = 47 in K3's generic path
    (96, 7, 7, 10041, "narrow"),     # the same switch at a width that is a multiple of 4
    (96, 8, 7, 10041, "wide"),
    (94, 256, 1, 1041, "wide"),      # largest C the wide head takes
    (100, 10, 9, 10041, "wide"),     # F4 = 25, wide head
    (130, 65, 7, 7041, "wide"),      # nhid > 128 and % 4 == 2, largest C at this width
    (132, 33, 9, 7041, "wide"),      # nhid > 128 with F4 = 33 > 32 in the fused gate / conv backward
    (136, 2, 1, 1041, "wide"),       # largest accepted width
    (32, 1038, 9, 2041, "narrow"),   # largest C of the narrow head
]
# (shape, G, nhid, C, seed, head backward): several batches of 8 graphs per k_head_bwd CTA, grid-stride head kernels
LARGE = [("PROTEINS", 2400, 32, 6, 21041, "narrow"), ("PROTEINS", 2400, 128, 6, 13041, "wide")]
TILE = 48       # graphs of the corpus a LARGE batch repeats
PAIRS = [(94, 27, 28), (96, 7, 8)]   # (nhid, C of the narrow row, C of the wide row)
TRIPLET = [(6, 3), (94, 28), (130, 65), (132, 33)]
# (nhid, C, G, seed): shapes the native steps refuse -- one class or two columns past the head's range, an odd width, and
# a classifier with hundreds of classes at nhid 128.  Through autograd, lin1's weight gradient at nhid > 128 has more
# than 256 input columns, and lin3's input gradient at C = 500 and 1039 is a K3 product too long for W's shared-memory
# slab in one pass (tsg_linear_fwd's K blocks)
FALLBACK = [(130, 66, 7, 7041), (138, 2, 7, 3041), (32, 1039, 7, 2041), (33, 2, 7, 12041), (128, 500, 7, 11041)]

_CASES = [pytest.param("DD", G, nhid, C, seed, id=f"nhid{nhid}-C{C}-G{G}") for nhid, C, G, seed, _ in ROWS] + \
         [pytest.param(shape, G, nhid, C, seed, id=f"{shape}-nhid{nhid}-C{C}-G{G}") for shape, G, nhid, C, seed, _ in LARGE]


def _batch(shape, G, C, seed):
    if G <= TILE:
        return _corpus(shape, G, C, seed)
    # 2,400 distinct PROTEINS-size graphs always hold some tie in the SAGPool scores: two nodes with the same label and
    # neighbourhood, equal in the oracle, which a different summation order splits by one ulp.  So a large batch
    # repeats TILE graphs without one
    corpus = synth.tile_corpus(_corpus(shape, TILE, C, seed), G)
    corpus.y = np.random.default_rng(seed).integers(0, C, G).astype(np.int64)
    return corpus


def _oracle(params, b, dt, mask=None, grads_of=None):
    """fp32 or float64 oracle forward (with the aux perms); `grads_of(emb)` -> a loss to differentiate."""
    po = {k: v.clone().to(dt).requires_grad_(grads_of is not None) for k, v in params.items()}
    emb, aux = R.sag_net_forward(po, torch.from_numpy(b["x"]).to(dt), torch.from_numpy(b["edge_index"]),
                                 torch.from_numpy(b["batch"]), 0.5, dropout_mask=None if mask is None else mask.to(dt),
                                 return_aux=True)
    if grads_of is None:
        return emb, aux, None, None
    loss = grads_of(emb)
    loss.backward()
    return emb.detach(), aux, loss.detach(), {k: v.grad for k, v in po.items()}


def _same_selection(aux32, aux64, what):
    for lvl in range(3):
        assert torch.equal(aux32["perm"][lvl], aux64["perm"][lvl]), (
            f"{what}: the fp32 and float64 oracles select different nodes at level {lvl}: this seed produced a near-tie "
            f"in the SAGPool scores, which says nothing about the kernels -- pick another seed")


def _check_step(grads, emb, loss, res, what):
    assert rel_err(emb, res[torch.float32][0]) <= TOL, what
    assert rel_err(loss, res[torch.float32][2]) <= TOL, what
    fwd_noise = max(rel_err(res[torch.float32][0], res[torch.float64][0]), 1e-7)
    assert len(grads) == 18
    for k in grads:
        grad_check(grads[k], res[torch.float32][3][k], res[torch.float64][3][k], TOL, f"{what} {k}", fwd_noise)


@pytest.mark.parametrize("shape,G,nhid,C,seed", _CASES)
def test_nll_step_and_classification_match_the_oracle(cuda, shape, G, nhid, C, seed):
    from tsg import nn as tnn
    corpus = _batch(shape, G, C, seed)
    b = synth.pack(corpus)
    cb = _compact(corpus, cuda)
    model, params = _model(corpus, nhid, C, cuda)
    model.train()
    y = torch.from_numpy(corpus.y)
    mask = _mask(G, nhid)
    assert model.native_step_supported(cb, corpus.node_ptr)
    tnn.KEEP_ARENA = True
    try:
        loss, emb = model.native_nll_step(cb, corpus.node_ptr, y.to(cuda), dropout_mask=mask.to(cuda), return_emb=True)
        shape_, arena = tnn.LAST_ARENA
    finally:
        tnn.KEEP_ARENA = False
    perms = [tnn.sag_arena_view(shape_, arena, lvl, "perm").cpu() for lvl in range(3)]
    grads = {k: p.grad.clone() for k, p in model.named_parameters()}
    tnn.check_fused_status()
    res = {dt: _oracle(params, b, dt, mask, lambda e: F.nll_loss(e, y)) for dt in (torch.float32, torch.float64)}
    _same_selection(res[torch.float32][1], res[torch.float64][1], "training forward")
    for lvl in range(3):
        assert torch.equal(perms[lvl], res[torch.float32][1]["perm"][lvl]), f"perm level {lvl}"
    _check_step(grads, emb, loss, res, "nll step")

    # classification: the eval-mode forward (no dropout), argmax, correct count and summed NLL
    pred, logp, correct, nll_sum = model.native_classify(cb, corpus.node_ptr, y.to(cuda))
    tnn.check_fused_status()
    out32, _, _, _ = _oracle(params, b, torch.float32)
    out64, _, _, _ = _oracle(params, b, torch.float64)
    pred_ref = out32.max(dim=1)[1]
    assert torch.equal(pred_ref, out64.max(dim=1)[1]), "near-tie between two classes in the oracle itself: pick another seed"
    assert rel_err(logp, out32) <= TOL
    assert torch.equal(pred.cpu(), pred_ref)
    assert int(correct.item()) == int((pred_ref == y).sum())
    nll_ref = float(F.nll_loss(out32.double(), y, reduction="sum"))
    assert abs(float(nll_sum.item()) - nll_ref) <= TOL * abs(nll_ref)
    # ... bitwise the step's forward (K10 + k_head_fwd) with every unit kept
    emb_fwd, _ = model.native_forward(cb, corpus.node_ptr, dropout_mask=torch.ones(G, nhid, device=cuda))
    assert torch.equal(logp, emb_fwd)


def _kernel_names(fn):
    """(fn(), names of the CUDA kernels it launched) -- from torch.profiler's device activity"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {e.name for e in prof.events()}


@pytest.mark.parametrize("nhid", [32, 64, 128])
def test_classification_equals_the_step_forward_with_and_without_k13(cuda, nhid):
    """At the widths the graph-resident kernels (K13) take, the classification forward's log-probabilities are bitwise
    those of the step's forward (K10 + the same head), with K13 on and off.  PROTEINS-size graphs (at most 93 nodes
    here), so that K13's per-graph working set fits shared memory at nhid 128 as well; the fused leg must have launched
    k_sag_fused_fwd and the other must not."""
    from tsg import _lib, nn as tnn
    G, C = 7, 2
    corpus = _corpus("PROTEINS", G, C, 1041)
    cb = _compact(corpus, cuda)
    model, _ = _model(corpus, nhid, C, cuda)
    y = torch.from_numpy(corpus.y).to(cuda)
    emb_fwd, _ = model.native_forward(cb, corpus.node_ptr, dropout_mask=torch.ones(G, nhid, device=cuda))
    out = {}
    for on in (0, 1):
        prev = _lib.lib.tsg_sag_set_fused(on)
        try:
            out[on], names = _kernel_names(lambda: model.native_classify(cb, corpus.node_ptr, y))
        finally:
            _lib.lib.tsg_sag_set_fused(prev)
        assert any("k_sag_fused_fwd" in n for n in names) == bool(on), (f"fused={on}", sorted(names))
    tnn.check_fused_status()
    for on in (0, 1):
        pred, logp, correct, nll_sum = out[on]
        assert torch.equal(logp, emb_fwd), f"fused={on}"
        assert torch.equal(pred, emb_fwd.max(dim=1)[1]), f"fused={on}"
    assert torch.equal(out[0][2], out[1][2]) and torch.equal(out[0][3], out[1][3])


@pytest.mark.parametrize("nhid,C", TRIPLET)
def test_triplet_step_matches_the_oracle(cuda, nhid, C):
    G, seed = next((r[2], r[3]) for r in ROWS if r[:2] == (nhid, C))
    margin = 50.0
    corpus = _corpus("DD", G, C, seed)
    b = synth.pack(corpus)
    cb = _compact(corpus, cuda)
    model, params = _model(corpus, nhid, C, cuda)
    model.train()
    assert G >= 3 and model.native_step_supported(cb, corpus.node_ptr)
    rng = np.random.default_rng(seed)
    trip = torch.from_numpy(np.stack([rng.permutation(G)[:3] for _ in range(2 * G)]).astype(np.int64))
    mask = _mask(G, nhid)
    loss, emb = model.native_step(cb, corpus.node_ptr, trip.to(cuda), margin, dropout_mask=mask.to(cuda), return_emb=True)
    grads = {k: p.grad.clone() for k, p in model.named_parameters()}

    def trip_loss(e):
        return R.triplet_margin_loss(e[trip[:, 0]], e[trip[:, 1]], e[trip[:, 2]], margin)[0]
    res = {dt: _oracle(params, b, dt, mask, trip_loss) for dt in (torch.float32, torch.float64)}
    _same_selection(res[torch.float32][1], res[torch.float64][1], "training forward")
    _check_step(grads, emb, loss, res, "triplet step")


@pytest.mark.parametrize("nhid,C,G,seed", FALLBACK)
def test_refused_shapes_train_and_evaluate_through_autograd(cuda, nhid, C, G, seed, monkeypatch):
    from tsg import nn as tnn
    from tsg.feeder import DeviceCorpus
    from tsg.train import ClassifierTrainer
    corpus = _corpus("DD", G, C, seed)
    b = synth.pack(corpus)
    cb = _compact(corpus, cuda)
    model, params = _model(corpus, nhid, C, cuda, dropout=0.0)
    assert not model.native_step_supported(cb, corpus.node_ptr)

    def native(*a, **k):
        raise AssertionError("a refused shape reached the native step")
    monkeypatch.setattr(model, "native_nll_step", native)
    monkeypatch.setattr(model, "native_classify", native)
    y = torch.from_numpy(corpus.y)
    trainer = ClassifierTrainer(model)
    # evaluate first: the step below moves the parameters
    acc, nll = trainer.evaluate(DeviceCorpus(corpus, cuda), np.arange(G), batch_graphs=4)
    out32, _, _, _ = _oracle(params, b, torch.float32)
    out64, _, _, _ = _oracle(params, b, torch.float64)
    pred_ref = out32.max(dim=1)[1]
    assert torch.equal(pred_ref, out64.max(dim=1)[1]), "near-tie between two classes in the oracle itself: pick another seed"
    assert round(acc * G) == int((pred_ref == y).sum())
    nll_ref = float(F.nll_loss(out32.double(), y))
    assert abs(nll - nll_ref) <= TOL * abs(nll_ref)
    loss = trainer.step(cb, None, corpus.node_ptr, y.to(cuda))
    tnn.check_fused_status()
    grads = {k: p.grad.clone() for k, p in model.named_parameters()}
    res = {dt: _oracle(params, b, dt, None, lambda e: F.nll_loss(e, y)) for dt in (torch.float32, torch.float64)}
    _same_selection(res[torch.float32][1], res[torch.float64][1], "training forward")
    assert rel_err(loss, res[torch.float32][2]) <= TOL
    fwd_noise = max(rel_err(res[torch.float32][0], res[torch.float64][0]), 1e-7)
    for k in grads:
        grad_check(grads[k], res[torch.float32][3][k], res[torch.float64][3][k], TOL, f"autograd {k}", fwd_noise)


@pytest.mark.parametrize("K,M", [(1039, 16), (700, 100), (513, 200), (456, 64)])
@pytest.mark.parametrize("transposed", [False, True])
def test_k3_linear_forward_blocks_a_long_k(cuda, K, M, transposed):
    """tsg_linear_fwd with an in_feat beyond W's shared-memory slab (blocks of K, one FMA chain per output carried
    through Y) against float64: the autograd head's input gradient of a layer with hundreds of classes"""
    from tsg import ops
    g = torch.Generator().manual_seed(K + M)
    x = torch.randn(300, K, generator=g)
    x[::3, ::5] = 0.0                                  # the kernel skips exact zeros: some rows and columns carry them
    w = torch.randn(M, K, generator=g) if transposed else torch.randn(K, M, generator=g)
    bias = torch.randn(M, generator=g)
    y = ops.linear_raw(x.to(cuda), w.to(cuda), bias.to(cuda), transposed=transposed)
    ref = x.double() @ (w.double().t() if transposed else w.double()) + bias.double()
    assert rel_err(y, ref) <= TOL
