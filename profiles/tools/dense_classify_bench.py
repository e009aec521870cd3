"""Speed of the dense encoders' supervised settings (DenseClassifierTrainer / WaveClassifierTrainer, K16 head + loss).

Workloads (the bench configs' models and corpora, every graph of the corpus in one prebuilt packed batch, as config 1):
  base      GcnEncoderGraph(32,32,32,2,L=2,bn), PROTEINS-shape 1,113 graphs (bench config 1)
  gat       DGATEncoderGraph(32,32,32,2,L=3,heads [2,2]), JAN.Y-shape 744 graphs (config 3)
  diffpool  SoftPoolingGcnEncoder(1000,32,32,32,2,L=3,assign 32, ratio 0.1), DD-shape 1,168 graphs (config 4)
  eigen     WavePoolingGcnEncoder(89,32,32,2,L=2,J=1,Jf=1,pool 10,pred_hidden [50]), DD-shape 1,168 graphs (config 5)
For each and each setting (original, 2stg+), in one process, round after round (device events, every variant warmed up
first):
  step_k16_ms    trainer.step on the prebuilt batch: readout, K16 head + cross-entropy, backward, clip, Adam
  step_aten_ms   the same step with the head and the loss composed in ATen here (F.linear / ReLU / [softmax] /
                 F.cross_entropy), alternated with the K16 step
  run_from_ids_ms  trainer.run_from_ids per step, the whole corpus's ids each step (batch assembled on the GPU)
  evaluate_ms    trainer.evaluate over the whole corpus
Each figure is the median over the rounds, with the rounds' min and max.  Kernels per step (K16 and ATen steps) are
counted from torch.profiler in a separate pass after the timing.  Prints one JSON line with the card's name and power
limit, read in the same run.

    python profiles/tools/dense_classify_bench.py [--steps 10] [--warmup 3] [--rounds 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "two-stage-gnn_b200"), os.path.join(ROOT, "profiles", "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

from classify_bench import card, timed          # noqa: E402


def _workloads(dev):
    from tsg import dense, diffpool, eigen_synth, gat, synth
    from tsg.feeder import DeviceCorpus
    table = torch.from_numpy(np.random.default_rng(777).normal(0.0, 2.0, (1000, 32)).astype(np.float32)).to(dev)

    def corpus(shape, G, eigen=False):
        c = synth.make_corpus(shape, G, seed=777)
        dc = DeviceCorpus(c, dev)
        if eigen:
            dc.attach_eigen(eigen_synth.make_operands(c, pool_size=10, num_pool_matrix=1, num_pool_final_matrix=1))
        return c, dc

    return [
        ("base", lambda fd: dense.PackedGcnEncoder(32, 32, 32, 2, 2, bn=True, final_dim=fd), ("number_classes", "pretrain"),
         corpus("PROTEINS", 1113)),
        ("gat", lambda fd: gat.PackedGatEncoder(32, 32, 32, 2, num_layers=3, num_heads=[2, 2], final_dim=fd),
         ("number_classes", "output_dim"), corpus("JANY", 744)),
        ("diffpool", lambda fd: diffpool.PackedSoftPoolEncoder(1000, 32, 32, 32, 2, 3, 32, assign_ratio=0.1, final_dim=fd),
         ("number_classes", "pretrain"), corpus("DD", 1168)),
        ("eigen", lambda fd: dense.PackedWaveEncoder(89, 32, 32, 2, 2, num_pool_matrix=1, num_pool_final_matrix=1,
                                                     pool_sizes=[10], pred_hidden_dims=[50]), (None, None),
         corpus("DD", 1168, eigen=True)),
    ], table


def _aten_step(t, batch, y):
    """trainer.step with the head and the loss composed in ATen"""
    t.model.train()
    z = t._readout(batch)
    for w, b, relu in t._layers():
        z = F.linear(z, w, b)
        if relu:
            z = F.relu(z)
    loss = F.cross_entropy(torch.softmax(z, dim=1) if t.softmax_first else z, y)
    t.opt.zero_grad(set_to_none=True)
    loss.backward()
    if t.clip_norm is not None:
        torch.nn.utils.clip_grad_norm_(list(t.model.parameters()), t.clip_norm)
    t.opt.step()
    return loss.detach()


def _kernels(fn):
    """kernels one call of fn() runs on the device (torch.profiler, CUDA activity; copies and memsets not counted)"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    return sum(1 for n in names if "memcpy" not in n.lower() and "memset" not in n.lower())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "dense_classify_bench measures the GPU; there is no CPU fallback"
    from tsg import _lib, nn as tnn
    from tsg.train import DenseClassifierTrainer, WaveClassifierTrainer

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    _lib.init_device()
    workloads, table = _workloads(dev)
    res = {}
    for kind, make, final_dims, (corpus, dc) in workloads:
        ids = np.arange(corpus.num_graphs)
        for setting, fd in zip(("original", "2stg+"), final_dims):
            torch.manual_seed(0)
            model = make(fd).to(dev)
            t = (WaveClassifierTrainer(model, 1000, setting=setting) if kind == "eigen"
                 else DenseClassifierTrainer(model, table, 1000, setting=setting))
            batch, y = t._batch(dc, t._check(dc, ids))
            variants = {
                "step_k16_ms": lambda i: t.step(batch, y),
                "step_aten_ms": lambda i: _aten_step(t, batch, y),
                "run_from_ids_ms": lambda i: t.run_from_ids(dc, [ids]),
                "evaluate_ms": lambda i: t.evaluate(dc, ids),
            }
            for fn in variants.values():
                timed(fn, a.warmup)
            samples = {k: [] for k in variants}
            for _ in range(a.rounds):
                for k, fn in variants.items():
                    samples[k].append(timed(fn, a.steps))
            tnn.check_fused_status()
            r = {k: {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v))}
                 for k, v in samples.items()}
            r["graphs_per_step"] = int(ids.shape[0])
            r["k16_vs_aten_step"] = r["step_aten_ms"]["median"] / r["step_k16_ms"]["median"]
            r["kernels_per_step_k16"] = _kernels(lambda: t.step(batch, y))
            r["kernels_per_step_aten"] = _kernels(lambda: _aten_step(t, batch, y))
            acc, ce = t.evaluate(dc, ids)
            r["final_eval"] = {"accuracy": acc, "mean_ce": ce}
            res[f"{kind}_{setting}"] = r
            print(kind, setting, json.dumps(r), file=sys.stderr, flush=True)

    name, plim = card()
    line = {"workload": "dense encoders' supervised settings (original / 2stg+), whole corpus as one packed batch: "
                        "base PROTEINS 1113, GAT JAN.Y 744, DiffPool DD 1168, EigenGCN DD 1168 pool 10",
            "gpu": name, "power_limit_w": plim, "steps": a.steps, "warmup": a.warmup, "rounds": a.rounds,
            "unix_time": int(time.time()), **res}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
