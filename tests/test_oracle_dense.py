"""oracle/dense_ref.py (restatement) against fixtures produced by the REAL reference modules
(oracle/make_golden.py imports /root/reference/Code/*/encoders*.py).  This is what pins the dense half
of the oracle; tolerance 2e-6 relative covers summation-order differences of identical fp32 math."""
import torch

from conftest import rel_err
from golden_util import clone_req, conv_names, convs, gat_layers, load
from oracle import dense_ref as D

PIN = 2e-6


def test_base_encoder_matches_reference():
    d = load("dense_base.npz")
    N, Fi, H, O, L = [int(v) for v in d["dims"]]
    names = conv_names("conv_first", "conv_block", "conv_last", L)
    for gi in range(3):
        cs = clone_req(convs(d, "conv_first", "conv_block", "conv_last"))
        out = D.gcn_encoder_readout(d[f"g{gi}/x"], d[f"g{gi}/adj"], cs)
        assert rel_err(out, d[f"g{gi}/readout"]) <= PIN
        yp = torch.nn.functional.linear(out, d["param/map_model.weight"], d["param/map_model.bias"])
        assert rel_err(yp, d[f"g{gi}/ypred"]) <= PIN
        (out * d["cot"]).sum().backward()
        for c, nm in zip(cs, names):
            assert rel_err(c["weight"].grad, d[f"g{gi}/grad/{nm}.weight"]) <= 5e-6, (gi, nm)
            assert rel_err(c["bias"].grad, d[f"g{gi}/grad/{nm}.bias"]) <= 5e-6, (gi, nm)


def test_gcn_forward_matches_reference():
    d = load("dense_gcn_forward.npz")
    N, Fi, H, O, L = [int(v) for v in d["dims"]]
    cs = clone_req(convs(d, "conv_first", "conv_block", "conv_last"))
    z = D.gcn_forward(d["x"], d["adj"], cs, True, D.construct_mask(N, [d["n"]]))
    assert rel_err(z, d["z"]) <= PIN
    (z * d["cot"]).sum().backward()
    for c, nm in zip(cs, conv_names("conv_first", "conv_block", "conv_last", L)):
        assert rel_err(c["weight"].grad, d[f"grad/{nm}.weight"]) <= 5e-6
        assert rel_err(c["bias"].grad, d[f"grad/{nm}.bias"]) <= 5e-6


def test_gat_matches_reference():
    d = load("dense_gat.npz")
    layers = gat_layers(d)
    req = [[dict(w=h["w"].clone().requires_grad_(True), a=h["a"].clone().requires_grad_(True)) for h in hs]
           for _, hs in layers]
    head0 = D.dgat_head(d["x"], d["adj"], req[0][0]["w"], req[0][0]["a"], concat=True)
    assert rel_err(head0, d["head0"]) <= PIN
    out = D.dgat_encoder_readout(d["x"], d["adj"], req)
    assert rel_err(out, d["readout"]) <= PIN
    (out * d["cot"]).sum().backward()
    for (lname, hs), rq in zip(layers, req):
        for h, r in enumerate(rq):
            assert rel_err(r["w"].grad, d[f"grad/{lname}.attention_{h}.w"]) <= 1e-5, (lname, h)
            assert rel_err(r["a"].grad, d[f"grad/{lname}.attention_{h}.a"]) <= 1e-5, (lname, h)


def _diffpool_params(d, req=False):
    p = dict(conv=convs(d, "conv_first", "conv_block", "conv_last"),
             assign_conv=convs(d, "assign_conv_first_modules.0", "assign_conv_block_modules.0", "assign_conv_last_modules.0"),
             conv_after=convs(d, "conv_first_after_pool.0", "conv_block_after_pool.0", "conv_last_after_pool.0"))
    p["assign_pred.weight"] = d["param/assign_pred_modules.0.weight"]
    p["assign_pred.bias"] = d["param/assign_pred_modules.0.bias"]
    if req:
        for k in ("conv", "assign_conv", "conv_after"):
            p[k] = clone_req(p[k])
        p["assign_pred.weight"] = p["assign_pred.weight"].clone().requires_grad_(True)
        p["assign_pred.bias"] = p["assign_pred.bias"].clone().requires_grad_(True)
    return p


def test_diffpool_matches_reference():
    d = load("dense_diffpool.npz")
    p = _diffpool_params(d, req=True)
    out, aux = D.soft_pool_readout(d["x"], d["adj"], [d["n"]], p)
    assert rel_err(aux["s"], d["assign"]) <= PIN
    assert rel_err(out, d["readout"]) <= PIN
    (out * d["cot"]).sum().backward()
    N, Fi, H, O, L = [int(v) for v in d["dims"]]
    for key, (f, b, l) in dict(conv=("conv_first", "conv_block", "conv_last"),
                               assign_conv=("assign_conv_first_modules.0", "assign_conv_block_modules.0", "assign_conv_last_modules.0"),
                               conv_after=("conv_first_after_pool.0", "conv_block_after_pool.0", "conv_last_after_pool.0")).items():
        for c, nm in zip(p[key], conv_names(f, b, l, L)):
            assert rel_err(c["weight"].grad, d[f"grad/{nm}.weight"]) <= 1e-5, nm
    assert rel_err(p["assign_pred.weight"].grad, d["grad/assign_pred_modules.0.weight"]) <= 1e-5


def test_eigen_matches_reference():
    d = load("dense_eigen.npz")
    N, Fi, H, O, L = [int(v) for v in d["dims"]]
    p = dict(conv=clone_req(convs(d, "conv_first", "conv_block", "conv_last")),
             conv_after=[clone_req(convs(d, "conv_first_after_pool.0", "conv_block_after_pool.0", "conv_last_after_pool.0"))])
    pm = [[d["P0"][None], d["P1"][None]], [d["Pf"][None]]]
    out = D.wave_readout(d["x"], d["adj"], [d["adj_pool"][None]], [d["n"]], [[d["nc"]]], pm, p,
                         num_pool_matrix=2, num_pool_final_matrix=1)
    head = [dict(weight=d["param/pred_model.0.weight"], bias=d["param/pred_model.0.bias"]),
            dict(weight=d["param/pred_model.2.weight"], bias=d["param/pred_model.2.bias"])]
    y = D.mlp(out, head)
    assert rel_err(y, d["y"]) <= PIN
    (y * d["cot"]).sum().backward()
    for c, nm in zip(p["conv"], conv_names("conv_first", "conv_block", "conv_last", L)):
        assert rel_err(c["weight"].grad, d[f"grad/{nm}.weight"]) <= 1e-5, nm
    for c, nm in zip(p["conv_after"][0], conv_names("conv_first_after_pool.0", "conv_block_after_pool.0", "conv_last_after_pool.0", L)):
        assert rel_err(c["weight"].grad, d[f"grad/{nm}.weight"]) <= 1e-5, nm


def test_gcn_cross_check_dense():
    """PyG-style GCNConv (oracle/pyg_ref.py, unpinned upstream) against the reference's importable
    dense formulation: D^-1/2 (A+I) D^-1/2 X W + b == GraphConv(add_self=False, normalise off) on the
    pre-normalised dense adjacency with self loops."""
    from oracle import pyg_ref as R
    from tsg import synth
    c = synth.make_corpus("PROTEINS", 3, seed=5); b = synth.pack(c)
    x = torch.randn(b["x"].shape[0], 6, generator=torch.Generator().manual_seed(0))
    ei = torch.from_numpy(b["edge_index"]); n = x.size(0)
    w = torch.randn(6, 4, generator=torch.Generator().manual_seed(1)); bias = torch.randn(4)
    out = R.gcn_conv(x, ei, w, bias)
    A = torch.zeros(n, n); A[ei[1], ei[0]] = 1.0; A = A + torch.eye(n)
    dis = A.sum(1).pow(-0.5)
    An = dis.view(-1, 1) * A * dis.view(1, -1)
    ref = D.graph_conv(x[None], An[None], w, bias, normalize_embedding=False)[0]
    assert rel_err(out, ref) <= 1e-5


# ---------------------------------------------------------------- BASELINE-dimension fixtures (configs 3, 4, 5)
def test_gat_cfg3_matches_reference():
    """Config 3 dims: n = 203-ish JAN.Y-shape graph, N = 1000, heads [2,2], widths 32 -> 64 -> 64 -> 32."""
    from golden_util import dense_adj, padded
    d = load("dense_gat_cfg3.npz")
    N = int(d["dims"][0])
    layers = gat_layers(d)
    req = [[dict(w=h["w"].clone().requires_grad_(True), a=h["a"].clone().requires_grad_(True)) for h in hs]
           for _, hs in layers]
    out = D.dgat_encoder_readout(padded(d["x"], N), dense_adj(d["ei"], N), req)
    assert rel_err(out, d["readout"]) <= PIN
    (out * d["cot"]).sum().backward()
    for (lname, hs), rq in zip(layers, req):
        for h, r in enumerate(rq):
            assert rel_err(r["w"].grad, d[f"grad/{lname}.attention_{h}.w"]) <= 1e-5, (lname, h)
            assert rel_err(r["a"].grad, d[f"grad/{lname}.attention_{h}.a"]) <= 1e-5, (lname, h)


# Config 4's assignment tower: its weight gradients are ill-conditioned in fp32.  The fixture (the original project's
# fp32 result) sits 4.9e-5 to 7.8e-5 from their float64 value, and the fp32 oracle lands up to 1.7e-4 from the fixture
# depending on the host BLAS's summation order (one thread; 4e-6 where it sums like the machine that made the fixture).
# Both bounds below are against the fixture: the float64 oracle must reproduce it to within its own fp32 noise (host
# independent), the fp32 oracle to within that noise plus the host's.
ASSIGN_TOWER = ("assign_conv_first_modules.0", "assign_conv_block_modules.0.0", "assign_conv_last_modules.0",
                "assign_pred_modules.0")
ASSIGN_FP64_VS_FIXTURE = 1e-4
ASSIGN_FP32_VS_FIXTURE = 3e-4


def test_diffpool_cfg4_matches_reference():
    """Config 4 dims: N = 1000 -> K = 100, D = 96, Linear(164 -> 100), DD-shape graph.  Every weight gradient of the
    fp32 oracle AND of its float64 evaluation against the fixture: 1e-5, the assignment tower at the bounds above."""
    from golden_util import dense_adj, padded
    d = load("dense_diffpool_cfg4.npz")
    N, Fi, H, O, L = [int(v) for v in d["dims"]]
    n = int(d["n"])
    x, adj = padded(d["x"], N), dense_adj(d["ei"], N)
    p = _diffpool_params(d, req=True)
    out, aux = D.soft_pool_readout(x, adj, [n], p)
    assert aux["s"].shape[-1] == 100 and out.shape[-1] == 192
    assert rel_err(aux["s"][0, :n], d["assign"]) <= PIN
    assert rel_err(out, d["readout"]) <= PIN
    (out * d["cot"]).sum().backward()
    d64 = {k: v.double() if torch.is_tensor(v) and v.is_floating_point() else v for k, v in d.items()}
    p64 = _diffpool_params(d64, req=True)
    o64, _ = D.soft_pool_readout(x.double(), adj.double(), [n], p64)
    (o64 * d64["cot"]).sum().backward()
    grads = {"assign_pred_modules.0": (p["assign_pred.weight"].grad, p64["assign_pred.weight"].grad)}
    for key, (f, b, l) in dict(conv=("conv_first", "conv_block", "conv_last"),
                               assign_conv=("assign_conv_first_modules.0", "assign_conv_block_modules.0", "assign_conv_last_modules.0"),
                               conv_after=("conv_first_after_pool.0", "conv_block_after_pool.0", "conv_last_after_pool.0")).items():
        for c, c64, nm in zip(p[key], p64[key], conv_names(f, b, l, L)):
            grads[nm] = (c["weight"].grad, c64["weight"].grad)
    assert len(grads) == 3 * L + 1 and set(ASSIGN_TOWER) <= set(grads)
    for nm, (g32, g64) in grads.items():
        fixture = d[f"grad/{nm}.weight"]
        tower = nm in ASSIGN_TOWER
        assert rel_err(g64, fixture) <= (ASSIGN_FP64_VS_FIXTURE if tower else 1e-5), ("float64", nm)
        assert rel_err(g32, fixture) <= (ASSIGN_FP32_VS_FIXTURE if tower else 1e-5), ("fp32", nm)


def test_eigen_cfg5_matches_reference():
    """Config 5 dims: 89 one-hot labels, L = 2, D = 64, 27 clusters of <= 10 nodes, pred 192 -> 50 -> 2."""
    from golden_util import eigen_cfg5_operands
    d = load("dense_eigen_cfg5.npz")
    N, Fi, H, O, L = [int(v) for v in d["dims"]]
    x, adj, ap, P, Pf = eigen_cfg5_operands(d)
    p = dict(conv=clone_req(convs(d, "conv_first", "conv_block", "conv_last")),
             conv_after=[clone_req(convs(d, "conv_first_after_pool.0", "conv_block_after_pool.0", "conv_last_after_pool.0"))])
    out = D.wave_readout(x, adj, [ap], [int(d["n"])], [[int(d["nc"])]], [[P], [Pf]], p, num_pool_matrix=1, num_pool_final_matrix=1)
    head = [dict(weight=d["param/pred_model.0.weight"], bias=d["param/pred_model.0.bias"]),
            dict(weight=d["param/pred_model.2.weight"], bias=d["param/pred_model.2.bias"])]
    y = D.mlp(out, head)
    assert out.shape[-1] == 192
    assert rel_err(y, d["y"]) <= PIN
    (y * d["cot"]).sum().backward()
    for c, nm in zip(p["conv"], conv_names("conv_first", "conv_block", "conv_last", L)):
        assert rel_err(c["weight"].grad, d[f"grad/{nm}.weight"]) <= 1e-5, nm
    for c, nm in zip(p["conv_after"][0], conv_names("conv_first_after_pool.0", "conv_block_after_pool.0", "conv_last_after_pool.0", L)):
        assert rel_err(c["weight"].grad, d[f"grad/{nm}.weight"]) <= 1e-5, nm


def test_linkpred_loss_matches_reference():
    """encoders.py:416-440 run for real (two upstream defects papered over by the generator, see golden_linkpred)."""
    d = load("dense_linkpred.npz")
    s = d["assign"].clone().requires_grad_(True)
    l = D.link_pred_loss(s, d["adj"], [int(d["n"])])
    l.backward()
    assert abs(float(l) - float(d["link_loss"])) <= PIN * abs(float(d["link_loss"]))
    assert rel_err(s.grad, d["dassign"]) <= 5e-6
