"""Speed of 2stg for the EigenGCN encoder from an HBM-resident corpus: batch assembly, training steps, embed, evaluate.

Workload: bench.py's config-5 model, PackedWaveEncoder(89,32,32,2,L=2,num_pool_matrix=1,num_pool_final_matrix=1,
pool_sizes [10],pred_hidden [50]), on the 1,168-graph DD-shape corpus (seed 777) with its synthetic EigenPooling operands
(eigen_synth.make_operands, pool_size 10), 1,168 triplets = 3x1,168 graphs per step.  Each phase is timed in turn, round
after round (device events around `--steps` calls, warm-up first; a call's host work is inside the window):
  assemble_config5_ms  bench.Config5.assemble + eigenpool.build (K11) for the step's ids: today's config-5 path
  assemble_eigen_ms    DeviceCorpus.pack_eigen for the same ids (one staged upload + K0e)
  step_prebuilt_ms     WaveTripletTrainer.step on one batch assembled once
  run_from_ids_ms      WaveTripletTrainer.run_from_ids per step (ids + triplets from the host, pack_eigen every step)
  embed_ms             WaveTripletTrainer.embed of the whole corpus
  evaluate_knn_ms / evaluate_mlp_ms   evaluate on a seeded 80/20 split (k = 3; one MLP epoch)
Medians over the rounds.  Prints one JSON line with the card's name and power limit, read in the same run.

    python profiles/tools/eigen_2stg_bench.py [--steps 10] [--warmup 3] [--rounds 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import importlib.util
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


def _bench_module():
    """bench.py as a module, imported as tests/test_feeder_gpu.py does (its argument parser sees no arguments)"""
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    argv, sys.argv = sys.argv, ["bench.py"]
    try:
        spec.loader.exec_module(mod)
    finally:
        sys.argv = argv
    return mod


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if a.steps < 1 or a.rounds < 1:
        raise SystemExit("--steps and --rounds must be at least 1")
    assert torch.cuda.is_available(), "eigen_2stg_bench measures the GPU; there is no CPU fallback"
    bench = _bench_module()
    from tsg import _lib, dense, eigenpool, nn as tnn, synth
    from tsg.feeder import DeviceCorpus
    from tsg.train import WaveTripletTrainer

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    _lib.init_device()
    G = T = 1168
    c5 = bench.Config5(dev, num_graphs=G, base_graphs=G)       # one rank: the shard is the base corpus, id for id
    corpus, op = c5.base, c5.opnd
    dc = DeviceCorpus(corpus, dev)
    dc.attach_eigen(op)
    trip = synth.sample_triplets(corpus.y, T, seed=0)
    ids = np.concatenate([trip[:, 0], trip[:, 1], trip[:, 2]])
    tr_host = torch.from_numpy(np.stack([np.arange(T), T + np.arange(T), 2 * T + np.arange(T)], 1)
                               .astype(np.int64)).pin_memory()
    tr = tr_host.to(dev)
    torch.manual_seed(777)
    model = dense.PackedWaveEncoder(corpus.num_node_labels, 32, 32, 2, 2, num_pool_matrix=1, num_pool_final_matrix=1,
                                    pool_sizes=[10], pred_hidden_dims=[50]).to(dev)
    tt = WaveTripletTrainer(model, 1000)
    batch = tt.pack(dc, ids)
    perm = np.random.default_rng(0).permutation(G)
    n_train = int(round(0.8 * G))
    train_ids, eval_ids = perm[:n_train], perm[n_train:]
    all_ids = np.arange(G)
    K = a.steps

    def assemble_config5(i):
        b = c5.assemble(ids)
        return eigenpool.build(b["csr_adj"], b["el"], b["cl"], b["NC"], 1)

    def run_ids(i):
        tt.run_from_ids(dc, [(ids, tr_host)] * K)

    variants = {
        "assemble_config5_ms": (assemble_config5, K),
        "assemble_eigen_ms": (lambda i: tt.pack(dc, ids), K),
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
    r.update(graphs_per_step=int(ids.shape[0]), nodes_per_step=int(batch.node_ptr_host[-1]),
             directed_edges_per_step=int(batch.csr.colidx.numel()), clusters_per_step=int(batch.cluster_ptr_host[-1]),
             coarse_entries_per_step=int(batch.coarse.rowptr[-1]), corpus_graphs=G, train_graphs=len(train_ids),
             eval_graphs=len(eval_ids), assembly_speedup=r["assemble_config5_ms"] / r["assemble_eigen_ms"],
             step_graphs_per_s=ids.shape[0] / (r["run_from_ids_ms"] * 1e-3),
             accuracy={"knn": tt.evaluate(dc, train_ids, eval_ids, head="knn"),
                       "mlp": tt.evaluate(dc, train_ids, eval_ids, head="mlp")})
    name, plim = card()
    line = {"workload": "2stg of the EigenGCN encoder from an HBM-resident corpus (untrained bench config-5 model, "
                        "clip_norm=None): DD 1168 graphs, pool_size 10, 1168 triplets per step; embed = whole corpus, "
                        "evaluate = seeded 80/20 split, kNN k=3, one MLP epoch",
            "gpu": name, "power_limit_w": plim, "steps": a.steps, "warmup": a.warmup, "rounds": a.rounds,
            "unix_time": int(time.time()), "eigen": r}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
