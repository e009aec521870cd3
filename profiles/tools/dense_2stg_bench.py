"""Speed of 2stg for the dense encoders from an HBM-resident corpus: batch assembly, training steps, embed, evaluate.

Configs (bench.py's shapes, corpora seeded 777, the N(0, 2^2) feature table [1000, 32] of bench.py::_dense_inputs):
  base      PackedGcnEncoder(32,32,32,2,L=2,bn)                 PROTEINS-shape 1,113 graphs, 371 triplets = 1,113 per step
  gat       PackedGatEncoder(32,32,32,2,L=3,heads [2,2])        JAN.Y-shape 744 graphs, 744 triplets = 3x744 per step
  diffpool  PackedSoftPoolEncoder(1000,32,32,32,2,L=3,32,0.1)   DD-shape 1,168 graphs, 1,168 triplets = 3x1,168 per step
Per config, in one process, each phase is timed in turn, round after round (device events around `--steps` calls,
warm-up first; a call's host work is inside the window):
  assemble_host_ms   bench.py::_dense_inputs for the step's ids: synth.select + synth.pack on the CPU, the H2D copies,
                     K1 build_csr(CSR_RAW) (the host path; eids for GAT)
  assemble_dense_ms  DeviceCorpus.pack_dense for the same ids (one staged upload + K0d)
  step_prebuilt_ms   DenseTripletTrainer.step on one batch assembled once (bench.py configs 3/4's formulation)
  run_from_ids_ms    DenseTripletTrainer.run_from_ids per step (ids + triplets from the host, pack_dense every step)
  embed_ms           DenseTripletTrainer.embed of the whole corpus
  evaluate_knn_ms / evaluate_mlp_ms   evaluate on a seeded 80/20 split (k = 3; one MLP epoch)
clip_norm=None throughout (bench's step).  Prints one JSON line with the card's name and power limit, read in the same
run.

    python profiles/tools/dense_2stg_bench.py [--steps 10] [--warmup 3] [--rounds 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "two-stage-gnn_b200"), os.path.join(ROOT, "profiles", "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

from classify_bench import card, timed  # noqa: E402


def _model(kind, dev):
    from tsg import dense, diffpool, gat
    torch.manual_seed(777)
    if kind == "base":
        return dense.PackedGcnEncoder(32, 32, 32, 2, 2, bn=True).to(dev)
    if kind == "gat":
        return gat.PackedGatEncoder(32, 32, 32, 2, num_layers=3, num_heads=[2, 2]).to(dev)
    return diffpool.PackedSoftPoolEncoder(1000, 32, 32, 32, 2, 3, 32, assign_ratio=0.1).to(dev)


CONFIGS = [("base", "PROTEINS", 1113, 371), ("gat", "JANY", 744, 744), ("diffpool", "DD", 1168, 1168)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if a.steps < 1 or a.rounds < 1:
        raise SystemExit("--steps and --rounds must be at least 1")
    assert torch.cuda.is_available(), "dense_2stg_bench measures the GPU; there is no CPU fallback"
    import bench
    from tsg import _lib, nn as tnn, synth
    from tsg.feeder import DeviceCorpus
    from tsg.train import DenseTripletTrainer

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    _lib.init_device()
    table = torch.from_numpy(np.random.default_rng(777).normal(0.0, 2.0, (1000, 32)).astype(np.float32)).to(dev)
    res = {}
    for kind, shape, G, T in CONFIGS:
        corpus = synth.make_corpus(shape, G, seed=777)
        dc = DeviceCorpus(corpus, dev)
        trip = synth.sample_triplets(corpus.y, T, seed=0)
        ids = np.concatenate([trip[:, 0], trip[:, 1], trip[:, 2]])
        tr_host = torch.from_numpy(np.stack([np.arange(T), T + np.arange(T), 2 * T + np.arange(T)], 1)
                                   .astype(np.int64)).pin_memory()
        tr = tr_host.to(dev)
        tt = DenseTripletTrainer(_model(kind, dev), table, 1000, clip_norm=None)
        batch = tt.pack(dc, ids)
        perm = np.random.default_rng(0).permutation(G)
        n_train = int(round(0.8 * G))
        train_ids, eval_ids = perm[:n_train], perm[n_train:]
        all_ids = np.arange(G)
        K = a.steps

        def run_ids(i):
            tt.run_from_ids(dc, [(ids, tr_host)] * K)

        variants = {
            "assemble_host_ms": (lambda i: bench._dense_inputs(corpus, ids, dev, want_eid=kind == "gat"), K),
            "assemble_dense_ms": (lambda i: tt.pack(dc, ids), K),
            "step_prebuilt_ms": (lambda i: tt.step(batch, tr), K),
            "run_from_ids_ms": (run_ids, 1),
            "embed_ms": (lambda i: tt._embed(dc, all_ids, 4096), K),
            "evaluate_knn_ms": (lambda i: tt.evaluate(dc, train_ids, eval_ids, head="knn"), K),
            "evaluate_mlp_ms": (lambda i: tt.evaluate(dc, train_ids, eval_ids, head="mlp"), K),
        }
        for fn, n in variants.values():
            timed(fn, min(n, a.warmup) if n > 1 else 1)
        samples = {k: [] for k in variants}
        for _ in range(a.rounds):
            for k, (fn, n) in variants.items():
                ms = timed(fn, n)
                samples[k].append(ms / K if n == 1 else ms)
        tnn.check_fused_status()
        r = {k: float(np.median(v)) for k, v in samples.items()}
        r["samples_ms"] = {k: [round(x, 4) for x in v] for k, v in samples.items()}
        N, E = int(batch.node_ptr_host[-1]), int(batch.csr.colidx.numel())
        r.update(graphs_per_step=int(ids.shape[0]), nodes_per_step=N, directed_edges_per_step=E,
                 corpus_graphs=G, train_graphs=len(train_ids), eval_graphs=len(eval_ids),
                 assembly_speedup=r["assemble_host_ms"] / r["assemble_dense_ms"],
                 step_graphs_per_s=ids.shape[0] / (r["run_from_ids_ms"] * 1e-3),
                 accuracy={"knn": tt.evaluate(dc, train_ids, eval_ids, head="knn"),
                           "mlp": tt.evaluate(dc, train_ids, eval_ids, head="mlp")})
        res[kind] = r
        del tt, batch, dc
        torch.cuda.empty_cache()

    name, plim = card()
    line = {"workload": "2stg of the dense encoders from an HBM-resident corpus (untrained models, clip_norm=None): "
                        "base PROTEINS 1113 graphs / 371 triplets per step, GAT JAN.Y 744 / 744, DiffPool DD 1168 / 1168; "
                        "embed = whole corpus, evaluate = seeded 80/20 split, kNN k=3, one MLP epoch",
            "gpu": name, "power_limit_w": plim, "steps": a.steps, "warmup": a.warmup, "rounds": a.rounds,
            "unix_time": int(time.time()), **res}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
