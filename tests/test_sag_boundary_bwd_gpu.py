"""tsg_sag_boundary_bwd (a pooled SAGPool level's conv input and weight gradients and the readout gradient of the level
below, in one pass; K3) against the sequence it replaces -- tsg_linear_fwd(transposed), tsg_readout_bwd(MAX|MEAN|ACCUM)
and tsg_linear_bwd_weight -- BIT FOR BIT (the header promises it, the sign of zero included), and the executor that
uses it against the op-by-op path."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
READOUT_MAX, READOUT_MEAN, READOUT_ACCUM = 1, 2, 8


def _case(sizes, H, seed, dev, dz_pad=0):
    rng = np.random.default_rng(seed)
    sizes = np.asarray(sizes, np.int64)
    G, gptr = len(sizes), np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    N = int(gptr[-1])
    dxw = rng.standard_normal((N, H)).astype(np.float32)
    dxw[rng.random((N, H)) < 0.1] = -0.0                      # negative zeros: dX's "+ 0.f" must turn them into +0
    dxw[rng.random(N) < 0.05] = -0.0                           # whole rows of them
    x = rng.standard_normal((N, H)).astype(np.float32)
    x[rng.random((N, H)) < 0.3] = 0.0                          # gated ReLU rows
    W = (rng.standard_normal((H, H)) / np.sqrt(H)).astype(np.float32)
    dz = rng.standard_normal((G, 2 * H + dz_pad)).astype(np.float32)
    dz[rng.random((G, 2 * H + dz_pad)) < 0.05] = -0.0
    am = np.full((G, H), -1, np.int32)                         # empty graphs keep -1
    for g in range(G):
        if sizes[g] == 0:
            continue
        am[g] = gptr[g] + rng.integers(0, sizes[g], H)
        if g % 3 == 0:
            am[g, : H // 2] = gptr[g]                          # one row the argmax of several columns
        if g % 5 == 1:
            am[g, rng.random(H) < 0.3] = -1
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    return dict(dxw=t(dxw), x=t(x), W=t(W), dz=t(dz), am=t(am), gptr=t(gptr), G=G, N=N, H=H, ds=2 * H + dz_pad)


def _sequence(c):
    from tsg import _lib
    dev, N, H, G = c["dxw"].device, c["N"], c["H"], c["G"]
    dxg = torch.full((N, H), float("nan"), device=dev)
    dW = torch.full((H, H), float("nan"), device=dev)
    ws = _lib.workspace(_lib.lib.tsg_linear_bwd_weight_workspace_bytes(H, H), dev)
    s = _lib.stream_ptr()
    _lib.call("tsg_linear_fwd", _lib.ptr(c["dxw"]), _lib.ptr(c["W"]), None, _lib.ptr(dxg), N, H, H, 1, 0, s)
    _lib.call("tsg_readout_bwd", _lib.ptr(c["dz"]), c["ds"], _lib.ptr(c["am"]), _lib.ptr(c["gptr"]), G, N, H,
              READOUT_MAX | READOUT_MEAN | READOUT_ACCUM, _lib.ptr(dxg), s)
    _lib.call("tsg_linear_bwd_weight", _lib.ptr(c["x"]), _lib.ptr(c["dxw"]), _lib.ptr(dW), None, N, H, H, _lib.ptr(ws), ws.numel(), s)
    return dxg, dW


def _boundary(c, H=None):
    from tsg import _lib
    dev, N, G = c["dxw"].device, c["N"], c["G"]
    H = c["H"] if H is None else H
    dxg = torch.full((N, c["H"]), float("nan"), device=dev)
    dW = torch.full((c["H"], c["H"]), float("nan"), device=dev)
    ws = _lib.workspace(_lib.lib.tsg_linear_bwd_weight_workspace_bytes(c["H"], c["H"]), dev)
    _lib.call("tsg_sag_boundary_bwd", _lib.ptr(c["dxw"]), _lib.ptr(c["x"]), _lib.ptr(c["W"]), _lib.ptr(c["dz"]), c["ds"],
              _lib.ptr(c["am"]), _lib.ptr(c["gptr"]), G, N, H, _lib.ptr(dxg), _lib.ptr(dW), _lib.ptr(ws), ws.numel(),
              _lib.stream_ptr())
    return dxg, dW


def _bitwise(a, b):
    return torch.equal(a.view(torch.int32), b.view(torch.int32))


def _sizes(N, seed):
    """ragged graphs summing to N, with empty and one-row graphs among them"""
    rng = np.random.default_rng(seed)
    out, left = [], N
    while left > 0:
        s = int(min(left, rng.choice([0, 1, 1, 2, 37, 70, 140, 300])))
        out.append(s); left -= s
    return out + [0]


ROWS = {
    "one": [1],
    "below_grid": [0, 1, 5, 0, 70, 1, 40, 0, 50, 1],           # 169 rows: fewer than the 296 CTAs
    "ragged": None,                                             # 12,345 rows (not a multiple of 128)
    "level2": None,                                             # about bench's level 2
}


@pytest.mark.parametrize("H", [8, 12, 16, 32, 64])
@pytest.mark.parametrize("rows", list(ROWS))
def test_bit_identical_to_the_sequence(cuda, H, rows):
    sizes = {"ragged": lambda: _sizes(12345, 1), "level2": lambda: _sizes(243_000, 2)}.get(rows, lambda: ROWS[rows])()
    c = _case(sizes, H, 7, cuda, dz_pad=4 if rows == "ragged" else 0)
    ref_dxg, ref_dW = _sequence(c)
    dxg, dW = _boundary(c)
    torch.cuda.synchronize()
    assert _bitwise(dxg, ref_dxg), (H, rows)
    assert _bitwise(dW, ref_dW), (H, rows)


@pytest.mark.parametrize("H", [12, 32])
def test_two_runs_identical(cuda, H):
    c = _case(_sizes(50_000, 4), H, 9, cuda)
    a, b = _boundary(c), _boundary(c)
    assert _bitwise(a[0], b[0]) and _bitwise(a[1], b[1])


@pytest.mark.parametrize("H", [4, 6, 10, 68, 130])
def test_out_of_envelope_widths_refused(cuda, H):
    c = _case([3, 2], 8, 1, cuda)
    with pytest.raises(RuntimeError, match="sag_boundary_bwd"):
        _boundary(c, H=H)


@pytest.mark.parametrize("shape,G,nhid", [("DD", 12, 8), ("PROTEINS", 50, 12), ("DD", 6, 64)])
def test_executor_matches_op_by_op(cuda, shape, G, nhid):
    """the executor (boundary passes at levels 2 and 1) against the op-by-op path, as test_sag_exec_gpu does at other
    widths: conv gradients bit for bit, the score layer within its fixed-order summation distance"""
    from tsg import nn as tnn, synth
    c = synth.make_corpus(shape, G, seed=5)
    b = synth.pack(c)
    x = torch.from_numpy(b["x"]).to(cuda)
    ei = torch.from_numpy(b["edge_index"]).to(cuda)
    torch.manual_seed(3)
    model = tnn.PackedSAGNet(c.num_node_labels, nhid, 8, 0.5, 0.0).to(cuda)
    cot = torch.randn(G, 8, generator=torch.Generator().manual_seed(1)).to(cuda)
    res = {}
    try:
        for use in (False, True):
            tnn.USE_EXECUTOR = use
            model.zero_grad(set_to_none=True)
            out = model(x, ei, b["node_ptr"])
            (out * cot).sum().backward()
            res[use] = (out.detach().clone(), {k: p.grad.detach().clone() for k, p in model.named_parameters()})
    finally:
        tnn.USE_EXECUTOR = True
    assert torch.equal(res[True][0], res[False][0])
    for k in res[False][1]:
        if k.endswith("score_layer.weight") or k.endswith("score_layer.bias"):
            scale = float(res[False][1][k].abs().max()) + 1e-12
            assert float((res[True][1][k] - res[False][1][k]).abs().max()) <= 2e-5 * scale, k
        else:
            assert _bitwise(res[True][1][k], res[False][1][k]), k
