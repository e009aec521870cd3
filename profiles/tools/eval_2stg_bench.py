"""Speed of the 2stg evaluation: TripletTrainer.embed, then the stage-2 kNN and one MLP epoch, on bench.py's corpus.

Corpus: bench.py's 1,168-graph DD-shape corpus (seed 777), resident in HBM, split 80/20 by a seeded permutation
(934 train graphs, 234 eval graphs).  For nhid 32 and 128 (final_dim --final-dim, an untrained triplet model: the
phases do not depend on the weights), in one process, each phase is timed in turn, round after round (device events,
warm-up first):
  embed_ms        TripletTrainer.embed of the train ids and of the eval ids (packed batches, eval mode)
  knn_ms          tsg_knn_classify of the eval embeddings against the train embeddings, k = 3, with the correct count
  mlp_epoch_ms    Mlp1Classifier: one epoch over the train embeddings (tsg_mlp1_train), then tsg_mlp1_predict's count
  evaluate_knn_ms / evaluate_mlp_ms   the whole TripletTrainer.evaluate call (includes its one device-to-host read)
Prints one JSON line with the card's name and power limit, read in the same run.

    python profiles/tools/eval_2stg_bench.py [--steps 20] [--warmup 3] [--rounds 3] [--out FILE]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--final-dim", type=int, default=32)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if a.steps < 1 or a.rounds < 1:
        raise SystemExit("--steps and --rounds must be at least 1")
    assert torch.cuda.is_available(), "eval_2stg_bench measures the GPU; there is no CPU fallback"
    from tsg import _lib, heads, nn as tnn, synth
    from tsg.feeder import DeviceCorpus
    from tsg.train import TripletTrainer

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    _lib.init_device()
    corpus = synth.make_corpus("DD", 1168, seed=777)
    dc = DeviceCorpus(corpus, dev)
    perm = np.random.default_rng(0).permutation(corpus.num_graphs)
    n_train = int(round(0.8 * corpus.num_graphs))
    train_ids, eval_ids = perm[:n_train], perm[n_train:]
    C = int(corpus.y.max()) + 1
    ytr = dc.y[torch.from_numpy(train_ids).to(dev)]
    yev = dc.y[torch.from_numpy(eval_ids).to(dev)]
    status = tnn._status_word(dev)

    res = {}
    for nhid in (32, 128):
        torch.manual_seed(0)
        model = tnn.PackedSAGNet(corpus.num_node_labels, nhid, a.final_dim, 0.5, 0.5).to(dev)
        tt = TripletTrainer(model)
        cb, nptr = dc.pack_compact(train_ids[:8])
        assert model.native_step_supported(cb, nptr), f"nhid {nhid}: native classification forward unavailable"
        emb = {"train": tt.embed(dc, train_ids), "eval": tt.embed(dc, eval_ids)}

        def embed(i):
            tt._embed(dc, train_ids, 4096)
            tt._embed(dc, eval_ids, 4096)

        def knn(i):
            heads.knn_classify(emb["train"], ytr, emb["eval"], yev, k=3, num_classes=C, status=status)

        def mlp(i):
            with torch.random.fork_rng(devices=[]):
                torch.manual_seed(0)
                clf = heads.Mlp1Classifier(a.final_dim, dev, num_classes=C)
            clf.fit(emb["train"], ytr)
            clf.score(emb["eval"], yev, status=status)

        def eval_knn(i):
            tt.evaluate(dc, train_ids, eval_ids, head="knn")

        def eval_mlp(i):
            tt.evaluate(dc, train_ids, eval_ids, head="mlp")

        variants = {"embed_ms": embed, "knn_ms": knn, "mlp_epoch_ms": mlp, "evaluate_knn_ms": eval_knn,
                    "evaluate_mlp_ms": eval_mlp}
        for fn in variants.values():
            timed(fn, a.warmup)
        samples = {k: [] for k in variants}
        for _ in range(a.rounds):
            for k, fn in variants.items():
                samples[k].append(timed(fn, a.steps))
        tnn.check_fused_status()
        r = {k: float(np.median(v)) for k, v in samples.items()}
        r["samples_ms"] = {k: [round(x, 4) for x in v] for k, v in samples.items()}
        r["embed_graphs_per_s"] = corpus.num_graphs / (r["embed_ms"] * 1e-3)
        r["accuracy"] = {"knn": tt.evaluate(dc, train_ids, eval_ids, head="knn"),
                         "mlp": tt.evaluate(dc, train_ids, eval_ids, head="mlp")}
        res[f"nhid{nhid}"] = r

    name, plim = card()
    line = {"workload": f"2stg evaluation of an untrained PackedSAGNet(89, nhid, final_dim {a.final_dim}, ratio 0.5): "
                        f"DD-shape corpus 1168 graphs, {len(train_ids)} train / {len(eval_ids)} eval, kNN k=3, one MLP "
                        f"epoch (in -> 64 -> 32 -> {C})",
            "gpu": name, "power_limit_w": plim, "steps": a.steps, "warmup": a.warmup, "rounds": a.rounds,
            "unix_time": int(time.time()), **res}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
