"""K16 (tsg_pred_ce_fwd / _bwd, tsg_pred_classify) on the GPU: loss, logits and every gradient against ATen fp32 and a
float64 evaluation (conftest.grad_check at 1e-5) for the head shapes of the dense encoders' supervised settings at the
reference dims, at G in {1, 7, 3,504}; every layer bit for bit equal to tsg_linear_fwd; a row's logits independent of its
batch; run-to-run determinism; pred / correct against numpy's first-index argmax on the kernel's own logits; the label
range check through the status word."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import grad_check, rel_err

pytestmark = pytest.mark.gpu

# (name, D0, [(out, relu_after), ...], softmax_first): the logits table of DenseClassifierTrainer at the reference dims
HEADS = [
    ("base original 64-32-2", 64, [(32, False), (2, False)], False),          # pred_model(pre_pred_model(r))
    ("diffpool original 192-32-2", 192, [(32, False), (2, False)], False),
    ("base 2stg+ 96-32-2 softmax", 96, [(32, False), (2, False)], True),      # map2_model(map_model(r)), softmax first
    ("gat original 32-2", 32, [(2, False)], False),                           # pred_model(r)
    ("gat 2stg+ identity 32", 32, [], True),                                  # the readout itself, 32 classes
    ("eigen 192-50-relu-2", 192, [(50, True), (2, False)], False),            # pred_model with pred_hidden_dims=(50,)
    ("base pred_hidden_dims=(50,)", 64, [(50, True), (32, False), (50, True), (2, False)], False),
]
GS = [1, 7, 3504]


def _make(D0, spec, G, dev, seed=0, C=None):
    g = torch.Generator().manual_seed(seed)
    r = torch.randn(G, D0, generator=g)
    layers, inp = [], D0
    for out, relu in spec:
        w = torch.randn(out, inp, generator=g) / np.sqrt(inp)
        b = torch.randn(out, generator=g) * 0.1
        layers.append((w.to(dev), b.to(dev), relu))
        inp = out
    C = inp if C is None else C
    y = torch.randint(0, C, (G,), generator=g)
    return r.to(dev), layers, y.to(dev)


def _aten(r, layers, y, softmax_first, dtype):
    """the head as nn.Linear / ReLU / [softmax] / F.cross_entropy compose it, in `dtype`; -> loss, logits, grads"""
    r = r.detach().to(dtype).requires_grad_(True)
    ps = [(w.detach().to(dtype).requires_grad_(True), b.detach().to(dtype).requires_grad_(True), relu)
          for w, b, relu in layers]
    z = r
    for w, b, relu in ps:
        z = F.linear(z, w, b)
        if relu:
            z = F.relu(z)
    q = torch.softmax(z, dim=1) if softmax_first else z
    loss = F.cross_entropy(q, y)
    loss.backward()
    return loss.detach(), z.detach(), r.grad, [(w.grad, b.grad) for w, b, _ in ps]


def _k16(r, layers, y, softmax_first):
    from tsg import ops
    r = r.detach().clone().requires_grad_(True)
    ps = [(w.detach().clone().requires_grad_(True), b.detach().clone().requires_grad_(True), relu) for w, b, relu in layers]
    loss = ops.pred_ce(r, ps, y, softmax_first)
    loss.backward()
    return loss.detach(), r.grad, [(w.grad, b.grad) for w, b, _ in ps]


@pytest.mark.parametrize("G", GS)
@pytest.mark.parametrize("name,D0,spec,softmax_first", HEADS, ids=[h[0] for h in HEADS])
def test_pred_ce_matches_aten_and_float64(cuda, name, D0, spec, softmax_first, G):
    from tsg import nn as tnn, ops
    r, layers, y = _make(D0, spec, G, cuda, seed=G)
    loss, dr, dps = _k16(r, layers, y, softmax_first)
    l32, z32, dr32, g32 = _aten(r, layers, y, softmax_first, torch.float32)
    l64, z64, dr64, g64 = _aten(r, layers, y, softmax_first, torch.float64)
    tnn.check_fused_status()
    assert rel_err(loss, l32) <= 1e-5 or rel_err(loss, l64) <= 1e-5, (float(loss), float(l32), float(l64))
    _, logits, _, _ = ops.pred_classify(r, layers, y, softmax_first, want_logits=True)
    assert rel_err(logits, z32) <= 1e-5
    grad_check(dr, dr32, dr64, name=f"{name} G={G} dr")
    for l, ((dw, db), (w32, b32), (w64, b64)) in enumerate(zip(dps, g32, g64)):
        grad_check(dw, w32, w64, name=f"{name} G={G} dW{l}")
        grad_check(db, b32, b64, name=f"{name} G={G} db{l}")


def _linear_fwd_chain(x, w, b):
    """tsg_linear_fwd(x, w, b, w_transposed=1): one fmaf chain per unit.  Its GEMV-shaped kernel for out <= 4 splits a
    row over lanes (a different summation order), so there the input goes in at a 4-byte offset, which that kernel does
    not take: the call then runs the row kernel, the chain K16 documents."""
    from tsg import ops
    if w.size(0) <= 4 and x.size(1) % 4 == 0 and x.size(1) <= 128:
        buf = torch.empty(x.numel() + 1, dtype=x.dtype, device=x.device)
        xm = buf[1:].view_as(x)
        xm.copy_(x)
        x = xm
    return ops.linear_raw(x, w, b, transposed=True)


@pytest.mark.parametrize("name,D0,spec,softmax_first", HEADS, ids=[h[0] for h in HEADS])
def test_every_layer_is_tsg_linear_fwd_bit_for_bit(cuda, name, D0, spec, softmax_first):
    from tsg import ops
    r, layers, y = _make(D0, spec, 3504, cuda, seed=5)
    _, logits, _, _ = ops.pred_classify(r, layers, y, softmax_first, want_logits=True)
    a = r
    for l, (w, b, relu) in enumerate(layers):
        _, one, _, _ = ops.pred_classify(a, [(w, b, relu)], None, False, want_logits=True)      # K16, this layer alone
        ref = _linear_fwd_chain(a, w, b)
        if relu:
            ref = torch.clamp_min(ref, 0.0)
        assert torch.equal(one, ref), (name, l)
        a = ref
    assert torch.equal(logits, a), name


@pytest.mark.parametrize("name,D0,spec,softmax_first", HEADS, ids=[h[0] for h in HEADS])
def test_a_rows_logits_do_not_depend_on_its_batch(cuda, name, D0, spec, softmax_first):
    from tsg import ops
    r, layers, y = _make(D0, spec, 3504, cuda, seed=9)
    _, whole, _, _ = ops.pred_classify(r, layers, y, softmax_first, want_logits=True)
    perm = torch.randperm(3504, generator=torch.Generator().manual_seed(1)).to(cuda)
    _, shuffled, _, _ = ops.pred_classify(r[perm], layers, y[perm], softmax_first, want_logits=True)
    assert torch.equal(shuffled, whole[perm])
    for i in (0, 1234, 3503):
        _, alone, _, _ = ops.pred_classify(r[i:i + 1], layers, None, softmax_first, want_logits=True)
        assert torch.equal(alone[0], whole[i]), i
    # the training forward computes the same logits
    loss_a, _, _ = _k16(r, layers, y, softmax_first)
    _, _, _, ce_sum = ops.pred_classify(r, layers, y, softmax_first)
    assert rel_err(loss_a, ce_sum / 3504) <= 1e-6


@pytest.mark.parametrize("name,D0,spec,softmax_first", HEADS, ids=[h[0] for h in HEADS])
def test_two_runs_are_bitwise_equal(cuda, name, D0, spec, softmax_first):
    r, layers, y = _make(D0, spec, 3504, cuda, seed=3)
    la, dra, ga = _k16(r, layers, y, softmax_first)
    lb, drb, gb = _k16(r, layers, y, softmax_first)
    assert torch.equal(la, lb) and torch.equal(dra, drb)
    for (wa, ba), (wb, bb) in zip(ga, gb):
        assert torch.equal(wa, wb) and torch.equal(ba, bb)


def test_backward_scales_with_the_upstream_gradient(cuda):
    from tsg import ops
    r, layers, y = _make(64, [(32, False), (2, False)], 7, cuda, seed=2)
    r1 = r.clone().requires_grad_(True)
    (3.0 * ops.pred_ce(r1, layers, y)).backward()
    _, dr, _ = _k16(r, layers, y, False)
    assert rel_err(r1.grad, 3.0 * dr) <= 1e-6


@pytest.mark.parametrize("name,D0,spec,softmax_first", HEADS, ids=[h[0] for h in HEADS])
def test_pred_and_correct_are_the_first_index_argmax(cuda, name, D0, spec, softmax_first):
    from tsg import nn as tnn, ops
    G = 3504
    r, layers, y = _make(D0, spec, G, cuda, seed=11)
    if layers:                           # ties: the last layer's units 0 and 1 equal for every row
        w, b, relu = layers[-1]
        w, b = w.clone(), b.clone()
        w[1], b[1] = w[0], b[0]
        layers = layers[:-1] + [(w, b, relu)]
    else:                                # identity head: rows with a repeated maximum
        r[::3, 5] = r[::3].max(dim=1).values + 1.0
        r[::3, 9] = r[::3, 5]
    pred, logits, correct, ce_sum = ops.pred_classify(r, layers, y, softmax_first, want_logits=True)
    z = logits.cpu().numpy()
    ref = np.argmax(z, axis=1)
    assert (z[np.arange(G), ref] == z.max(axis=1)).all()
    ties = (z == z.max(axis=1, keepdims=True)).sum(axis=1) > 1
    assert ties.sum() > G // 10, "the case has no ties"
    assert np.array_equal(pred.cpu().numpy(), ref)
    assert int(correct.item()) == int((ref == y.cpu().numpy()).sum())
    _, _, _, ce_ref = ops.pred_classify(r, layers, y, softmax_first)
    assert torch.equal(ce_sum, ce_ref)
    p, _, c0, s0 = ops.pred_classify(r, layers, None, softmax_first)
    assert torch.equal(p, pred) and c0 is None and s0 is None
    tnn.check_fused_status()


@pytest.mark.parametrize("bad", [2, -1, 7])
def test_an_out_of_range_label_raises_through_the_status_word(cuda, bad):
    from tsg import nn as tnn, ops
    tnn.check_fused_status()
    r, layers, y = _make(64, [(32, False), (2, False)], 7, cuda, seed=1)
    y = y.clone()
    y[4] = bad
    loss = ops.pred_ce(r, layers, y)
    assert bool(torch.isfinite(loss))                                 # read clamped
    with pytest.raises(RuntimeError, match="label"):
        tnn.check_fused_status()
    ops.pred_classify(r, layers, y)
    with pytest.raises(RuntimeError, match="label"):
        tnn.check_fused_status()
    ops.pred_classify(r, layers, y.clamp(0, 1))
    tnn.check_fused_status()
