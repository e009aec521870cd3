"""DeviceCorpus.build_eigen (K17 + K11) against the host operands of tsg.eigen_synth: the integer arrays and coarse
weights exactly; every stored eigenvector either equal to the host's (simple eigenvalue) or, where the host's eigenvalue
is repeated, a unit vector of the same eigenspace that keeps the sign and repeat rules.  Edge cases, device-side
refusals, determinism and chunk independence, a from_device shard, and the trainers on a device build against the same
operands read back and attached from the host."""
import numpy as np
import pytest
import torch

from conftest import rel_err
from test_eigen_2stg_gpu import _corpus_of, _model, _oracle_embed, _sym, _triplet_ids
from tsg import eigen_synth, synth
from tsg.eigen_synth import EigenOperands

pytestmark = pytest.mark.gpu
TOL = 1e-5
FINAL_MAX = 112


def _read_back(dc) -> EigenOperands:
    op = dc.eigen
    h = lambda t: t.cpu().numpy()
    return EigenOperands(h(op["cluster_ptr"]), h(op["cluster_of"]).astype(np.int64), [w for w in h(op["pool_w"])],
                         h(op["coarse_ptr"]), h(op["coarse_row"]).astype(np.int64), h(op["coarse_col"]).astype(np.int64),
                         h(op["coarse_w"]), [w for w in h(op["final_w"])][:op["Jf"]])


def _lap(adj):
    a = np.asarray(adj, np.float64)
    return np.diag(a.sum(1)) - a


class Tally:
    def __init__(self):
        self.simple = self.degenerate = 0

    def check(self, lap, host, dev, what):
        """host / dev: [J, m] vectors over the same node order; the rule of DeviceCorpus.build_eigen"""
        w, _ = np.linalg.eigh(lap)
        m = lap.shape[0]
        scale = max(1.0, float(np.abs(lap).sum(1).max()))
        for j in range(host.shape[0]):
            r = min(j, m - 1)
            hv, dv = host[j].astype(np.float64), dev[j].astype(np.float64)
            gaps = np.abs(np.delete(w, r) - w[r])
            if gaps.size == 0 or gaps.min() > 1e-6 * scale:
                self.simple += 1
                if abs(hv[0]) < 1e-6:                     # the sign rule cannot decide on a zero first entry
                    err = min(np.abs(dv - hv).max(), np.abs(dv + hv).max())
                else:
                    err = np.abs(dv - hv).max()
                assert err <= TOL, (what, j, err)
            else:
                self.degenerate += 1
                assert abs(np.linalg.norm(dv) - 1.0) <= TOL, (what, j, "norm")
                assert np.linalg.norm(lap @ dv - w[r] * dv) <= TOL * scale, (what, j, "eigenspace")
                assert dv[0] >= 0, (what, j, "sign")
            if j >= m:
                assert np.array_equal(dev[j], dev[m - 1]), (what, j, "repeat")


def _members(op, g, n0, n, order):
    cl = op.cluster_of[n0:n0 + n]
    nc = int(op.cluster_ptr[g + 1] - op.cluster_ptr[g])
    o = np.arange(n) if order is None else order[n0:n0 + n]
    mem = o[np.argsort(cl[o], kind="stable")]
    starts = np.searchsorted(cl[mem], np.arange(nc + 1))
    return [mem[starts[k]:starts[k + 1]] for k in range(nc)]


def _check(corpus, ref, dev_op, J, Jf, order, tally):
    """integers exact, vectors by the rule; ref may carry more vectors than J / Jf"""
    for k in ("cluster_ptr", "cluster_of", "coarse_ptr", "coarse_row", "coarse_col"):
        assert np.array_equal(getattr(ref, k), getattr(dev_op, k)), k
    assert np.array_equal(ref.coarse_w, dev_op.coarse_w)
    assert len(dev_op.pool_w) == J and len(dev_op.final_w) == Jf
    for g in range(corpus.num_graphs):
        n0, n = int(corpus.node_ptr[g]), corpus.num_nodes(g)
        e0, e1 = corpus.edge_ptr[g], corpus.edge_ptr[g + 1]
        adj = np.zeros((n, n)); adj[corpus.row[e0:e1], corpus.col[e0:e1]] = 1
        for k, mem in enumerate(_members(ref, g, n0, n, order)):
            if mem.size == 0:
                continue
            host = np.stack([ref.pool_w[j][n0 + mem] for j in range(J)])
            dev = np.stack([dev_op.pool_w[j][n0 + mem] for j in range(J)])
            tally.check(_lap(adj[np.ix_(mem, mem)]), host, dev, ("pool", g, k))
        if Jf:
            c0, c1 = int(ref.cluster_ptr[g]), int(ref.cluster_ptr[g + 1])
            q0, q1 = int(ref.coarse_ptr[g]), int(ref.coarse_ptr[g + 1])
            ca = np.zeros((c1 - c0, c1 - c0)); ca[ref.coarse_row[q0:q1], ref.coarse_col[q0:q1]] = 1
            host = np.stack([ref.final_w[j][c0:c1] for j in range(Jf)])
            dev = np.stack([dev_op.final_w[j][c0:c1] for j in range(Jf)])
            tally.check(_lap(ca), host, dev, ("final", g))


def _labels(corpus, pool_size, seed):
    """a clustering of our own: a random permutation of every graph cut into chunks of pool_size"""
    rng = np.random.default_rng(seed)
    return np.concatenate([rng.permutation(corpus.num_nodes(g)) // pool_size for g in range(corpus.num_graphs)])


@pytest.mark.parametrize("user", [False, True])
@pytest.mark.parametrize("pool_size", [1, 10, 32])
@pytest.mark.parametrize("shape,G", [("DD", 10), ("PROTEINS", 40)])
def test_build_matches_the_host_operands(cuda, shape, G, pool_size, user):
    from tsg.feeder import DeviceCorpus
    corpus = synth.make_corpus(shape, G, seed=31)
    if user:
        labels = _labels(corpus, pool_size, 3)
        ref, order = eigen_synth.operands_from_clusters(corpus, labels, 2, 2), None
    else:
        labels = None
        ref = eigen_synth.make_operands(corpus, pool_size, 2, 2)
        order = eigen_synth.bfs_clusters(corpus, pool_size)[1]
    dc = DeviceCorpus(corpus, cuda)
    tally = Tally()
    full = None
    for J in (2, 1):
        for Jf in (2, 1, 0):
            fb = dc.build_eigen(pool_size, J, Jf, cluster_of=labels)
            op = _read_back(dc)
            assert fb == (int((np.diff(ref.cluster_ptr) > FINAL_MAX).sum()) if Jf else 0)
            if full is None:
                full = op
                _check(corpus, ref, op, J, Jf, order, tally)
            else:                                         # fewer vectors: the leading ones of the full build
                for k in ("cluster_ptr", "cluster_of", "coarse_ptr", "coarse_row", "coarse_col", "coarse_w"):
                    assert np.array_equal(getattr(full, k), getattr(op, k)), k
                for j in range(J):
                    assert np.array_equal(full.pool_w[j], op.pool_w[j]), ("pool", j)
                for j in range(Jf):
                    assert np.array_equal(full.final_w[j], op.final_w[j]), ("final", j)
    assert tally.simple > 0
    if pool_size > 1:
        assert tally.degenerate > 0


def _edge_cases():
    """1 node; 5 nodes without edges; two components plus two isolated nodes; a single cluster (n <= pool_size 4);
    600 nodes (150 clusters: above the final-pooling cap); ordinary PROTEINS graphs"""
    rng = np.random.default_rng(2)
    graphs = [(1, [], []), (5, [], [])]
    r1, c1 = synth._one_graph(rng, 6, 8)
    r2, c2 = synth._one_graph(rng, 5, 6)
    pairs = [(a, b) for a, b in zip(r1, c1) if a < b] + [(a + 7, b + 7) for a, b in zip(r2, c2) if a < b]
    graphs.append((14,) + _sym(pairs))
    graphs.append((4,) + _sym([(0, 1), (1, 2), (2, 3)]))
    r, c = synth._one_graph(rng, 600, 900)
    graphs.append((600, r, c))
    base = synth.make_corpus("PROTEINS", 6, seed=9)
    for g in range(base.num_graphs):
        e0, e1 = base.edge_ptr[g], base.edge_ptr[g + 1]
        graphs.append((base.num_nodes(g), base.row[e0:e1], base.col[e0:e1]))
    return _corpus_of(graphs)


def test_edge_cases(cuda):
    from tsg.feeder import DeviceCorpus
    corpus = _edge_cases()
    assert synth.is_coalesced_symmetric(corpus)
    dc = DeviceCorpus(corpus, cuda)
    tally = Tally()
    ref = eigen_synth.make_operands(corpus, 4, 2, 2)
    assert dc.build_eigen(4, 2, 2) == 1                   # the 600-node graph's final pooling comes from the host
    op = _read_back(dc)
    _check(corpus, ref, op, 2, 2, eigen_synth.bfs_clusters(corpus, 4)[1], tally)
    assert np.diff(op.cluster_ptr)[[0, 1, 3]].tolist() == [1, 2, 1] and op.coarse_ptr[4] == op.coarse_ptr[3]
    assert op.final_w[0][int(op.cluster_ptr[0])] == 1.0
    # labels of our own with an empty cluster (graph 2: ids 0, 2, 3 used of 0 .. 3)
    labels = _labels(corpus, 3, 7)
    n0 = int(corpus.node_ptr[2])
    labels[n0:n0 + 14] = np.repeat([0, 2, 3, 0], [4, 4, 4, 2])
    ref = eigen_synth.operands_from_clusters(corpus, labels, 1, 1)
    fb = dc.build_eigen(10, 1, 1, cluster_of=torch.from_numpy(labels).to(cuda))
    assert fb == int((np.diff(ref.cluster_ptr) > FINAL_MAX).sum()) and fb >= 1
    _check(corpus, ref, _read_back(dc), 1, 1, None, tally)
    assert tally.simple > 0 and tally.degenerate > 0


def test_device_side_refusals_attach_nothing(cuda):
    from tsg.feeder import DeviceCorpus
    corpus = synth.make_corpus("PROTEINS", 8, seed=3)
    big = int(np.argmax(np.diff(corpus.node_ptr)))
    assert corpus.num_nodes(big) > 32
    labels = _labels(corpus, 4, 0)
    dc = DeviceCorpus(corpus, cuda)
    over = labels.copy(); over[corpus.node_ptr[big]:corpus.node_ptr[big + 1]] = 0
    with pytest.raises(ValueError, match=f"graph {big} has a cluster of more than 32"):
        dc.build_eigen(cluster_of=over)
    out = labels.copy(); out[corpus.node_ptr[5]] = corpus.num_nodes(5)
    with pytest.raises(ValueError, match="graph 5 has a cluster id outside"):
        dc.build_eigen(cluster_of=out)
    assert "eigen" not in dc.__dict__
    assert dc.build_eigen(cluster_of=labels) == 0 and "eigen" in dc.__dict__


def _arrays(dc):
    return {k: v.cpu().clone() for k, v in dc.eigen.items() if isinstance(v, torch.Tensor)}


def test_deterministic_and_independent_of_the_chunk_size(cuda):
    from tsg.feeder import DeviceCorpus
    corpus = synth.make_corpus("DD", 24, seed=5)
    dc = DeviceCorpus(corpus, cuda)
    for labels in (None, _labels(corpus, 10, 1)):
        dc.build_eigen(10, 2, 2, cluster_of=labels)
        a = _arrays(dc)
        for chunk in (1 << 24, 1, 3000):
            dc.build_eigen(10, 2, 2, cluster_of=labels, chunk_size=chunk)
            b = _arrays(dc)
            for k in a:
                assert torch.equal(a[k], b[k]), (chunk, k)


def test_from_device_shard_equals_the_base_build_per_tile(cuda):
    """a shard assembled on the GPU as bench.Config5 does (owned = rank::world of a tiled id space, one K0 gather)"""
    from tsg.feeder import DeviceCorpus
    base = synth.make_corpus("DD", 30, seed=777)
    owned = np.arange(1, 200, 2, dtype=np.int64)
    bseq = owned % base.num_graphs
    base_dc = DeviceCorpus(base, cuda)
    cb, nptr = base_dc.pack_compact(bseq)
    _, _, eptr = base_dc.offsets(bseq)
    shard = DeviceCorpus.from_device(cb.label, cb.row, cb.col, nptr, eptr, base.num_node_labels, base_dc.coalesced)
    assert base_dc.build_eigen(10, 1, 1) == 0 and shard.build_eigen(10, 1, 1, chunk_size=20000) == 0
    b, s = _read_back(base_dc), _read_back(shard)
    sel = synth.select(synth.Corpus("", base.node_ptr, b.coarse_ptr, b.coarse_row, b.coarse_col,
                                    b.cluster_of.astype(np.int32), base.y, 1), bseq)
    assert np.array_equal(sel.edge_ptr, s.coarse_ptr) and np.array_equal(sel.row, s.coarse_row)
    assert np.array_equal(sel.col, s.coarse_col) and np.array_equal(sel.node_label, s.cluster_of)
    nidx = synth._ragged_arange(base.node_ptr[bseq], np.diff(base.node_ptr)[bseq])
    cidx = synth._ragged_arange(b.cluster_ptr[bseq], np.diff(b.cluster_ptr)[bseq])
    qidx = synth._ragged_arange(b.coarse_ptr[bseq], np.diff(b.coarse_ptr)[bseq])
    assert np.array_equal(np.diff(s.cluster_ptr), np.diff(b.cluster_ptr)[bseq])
    assert np.array_equal(b.pool_w[0][nidx], s.pool_w[0]) and np.array_equal(b.final_w[0][cidx], s.final_w[0])
    assert np.array_equal(b.coarse_w[qidx], s.coarse_w)


def test_trainers_on_a_device_build_equal_the_read_back_operands(cuda):
    from tsg import nn as tnn
    from tsg.feeder import DeviceCorpus
    from tsg.train import WaveClassifierTrainer, WaveTripletTrainer
    corpus = synth.make_corpus("DD", 30, seed=11)
    dev_dc, host_dc = DeviceCorpus(corpus, cuda), DeviceCorpus(corpus, cuda)
    dev_dc.build_eigen(10, 2, 1)
    op = _read_back(dev_dc)
    host_dc.attach_eigen(op)
    for k in ("cluster_ptr", "coarse_ptr", "cluster_of", "coarse_row", "coarse_col", "coarse_w", "pool_w", "final_w"):
        a, b = dev_dc.eigen[k], host_dc.eigen[k]
        assert a.dtype == b.dtype and a.shape == b.shape and torch.equal(a, b), k
    for k in ("nc", "ncoarse"):
        assert np.array_equal(dev_dc.eigen[k], host_dc.eigen[k]) and dev_dc.eigen[k].dtype == host_dc.eigen[k].dtype
    dev_dc.pack_eigen(np.arange(30), 1000)
    torch.cuda.synchronize()
    tnn.check_fused_status()
    F = corpus.num_node_labels
    ids, tr = _triplet_ids(corpus, 10, 0)
    ma, mb = _model(cuda, F, 2, 1), _model(cuda, F, 2, 1)
    ta, tb = WaveTripletTrainer(ma, 1000), WaveTripletTrainer(mb, 1000)
    la = ta.step(ta.pack(dev_dc, ids), tr.to(cuda)).cpu()
    lb = tb.step(tb.pack(host_dc, ids), tr.to(cuda)).cpu()
    assert torch.equal(la, lb)
    for (k, pa), pb in zip(ma.named_parameters(), mb.parameters()):
        assert torch.equal(pa, pb), ("triplet", k)
    ca, cb = _model(cuda, F, 2, 1), _model(cuda, F, 2, 1)
    sa, sb = WaveClassifierTrainer(ca, 1000), WaveClassifierTrainer(cb, 1000)
    y = torch.from_numpy(corpus.y[ids]).to(cuda)
    la, lb = sa.step(sa.pack(dev_dc, ids), y).cpu(), sb.step(sb.pack(host_dc, ids), y).cpu()
    assert torch.equal(la, lb)
    for (k, pa), pb in zip(ca.named_parameters(), cb.parameters()):
        assert torch.equal(pa, pb), ("classifier", k)
    emb = ta.embed(dev_dc, np.arange(30))
    assert rel_err(emb, _oracle_embed(ma, corpus, op, np.arange(30), 1000)) <= TOL
