"""Speed of the supervised ("original") setting against the 2stg step, on bench.py's headline batch.

Batch: as bench.py's `value` -- a compact DD-shape batch of 3,504 graphs (the ids of 1,168 sampled triplets) assembled
once in HBM from the 1,168-graph corpus, two such batches alternating.  For nhid 32 and nhid 128, in one process, the
variants are timed in turn, round after round (device events, warm-up first):
  (a) ClassifierTrainer.step, native (tsg_sag_nll_step_compact, C = 2 graph classes)
  (b) the same step through autograd (what TSG_NATIVE_STEP=0 selects)
  (c) TripletTrainer.step on the same batch (the 2stg step, final_dim --final-dim)
  (d) ClassifierTrainer.evaluate over the whole corpus, in graphs/s
Prints one JSON line with the card's name and power limit, read in the same run.  Kernel times are not taken here:
use torch.profiler in a separate run.

    python profiles/tools/classify_bench.py [--steps 20] [--warmup 5] [--rounds 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "two-stage-gnn_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)


def card():
    """(name, power limit in W) of cuda:0, read now."""
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return name, float(out.splitlines()[0])
    except Exception:
        return name, None


def timed(fn, steps):
    """ms per call of fn() over `steps` calls, between two device events."""
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    for i in range(steps):
        fn(i)
    e.record()
    e.synchronize()
    return s.elapsed_time(e) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--final-dim", type=int, default=32)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if a.steps < 20:
        raise SystemExit("--steps must be at least 20")
    assert torch.cuda.is_available(), "classify_bench measures the GPU; there is no CPU fallback"
    from tsg import _lib, nn as tnn, synth
    from tsg.feeder import DeviceCorpus
    from tsg.train import ClassifierTrainer, TripletTrainer

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    _lib.init_device()
    corpus = synth.make_corpus("DD", 1168, seed=777)
    dc = DeviceCorpus(corpus, dev)
    T = 1168
    tidx = torch.from_numpy(np.stack([np.arange(T), T + np.arange(T), 2 * T + np.arange(T)], 1).astype(np.int64)).to(dev)
    batches = []
    for b in range(2):
        trip = synth.sample_triplets(corpus.y, T, seed=b)
        ids = np.concatenate([trip[:, 0], trip[:, 1], trip[:, 2]])
        cb, nptr = dc.pack_compact(ids)
        batches.append((cb, nptr, dc.y[torch.from_numpy(ids).to(dev)]))
    torch.cuda.synchronize()
    C = int(corpus.y.max()) + 1
    all_ids = np.arange(corpus.num_graphs)

    res = {}
    for nhid in (32, 128):
        torch.manual_seed(0)
        sup = tnn.PackedSAGNet(corpus.num_node_labels, nhid, C, 0.5, 0.5).to(dev)
        trip_m = tnn.PackedSAGNet(corpus.num_node_labels, nhid, a.final_dim, 0.5, 0.5).to(dev)
        ct, tt = ClassifierTrainer(sup), TripletTrainer(trip_m)
        assert sup.native_step_supported(batches[0][0], batches[0][1]), f"nhid {nhid}: native supervised step unavailable"
        assert trip_m.native_step_supported(batches[0][0], batches[0][1]), f"nhid {nhid}: native triplet step unavailable"

        def native(i):
            cb, nptr, y = batches[i % 2]
            ct.step(cb, None, nptr, y)

        def autograd(i):
            tnn.USE_NATIVE_STEP = False
            try:
                native(i)
            finally:
                tnn.USE_NATIVE_STEP = True

        def triplet(i):
            cb, nptr, _ = batches[i % 2]
            tt.step(cb, None, nptr, tidx)

        def evaluate(i):
            ct.evaluate(dc, all_ids, batch_graphs=4096)

        variants = {"nll_native_ms": native, "nll_autograd_ms": autograd, "triplet_native_ms": triplet,
                    "evaluate_ms": evaluate}
        calls = _lib.launch_calls
        native(0)
        launches_per_step = _lib.launch_calls - calls
        for fn in variants.values():
            timed(fn, a.warmup)
        samples = {k: [] for k in variants}
        for _ in range(a.rounds):
            for k, fn in variants.items():
                samples[k].append(timed(fn, a.steps))
        tnn.check_fused_status()
        r = {k: float(np.median(v)) for k, v in samples.items()}
        r["samples_ms"] = {k: [round(x, 4) for x in v] for k, v in samples.items()}
        r["nll_native_graphs_per_s"] = 3 * T / (r["nll_native_ms"] * 1e-3)
        r["triplet_native_graphs_per_s"] = 3 * T / (r["triplet_native_ms"] * 1e-3)
        r["evaluate_graphs_per_s"] = corpus.num_graphs / (r["evaluate_ms"] * 1e-3)
        r["nll_vs_triplet"] = r["nll_native_ms"] / r["triplet_native_ms"]
        r["native_speedup_vs_autograd"] = r["nll_autograd_ms"] / r["nll_native_ms"]
        r["libtsg_calls_per_native_step"] = launches_per_step
        acc, nll = ct.evaluate(dc, all_ids)
        r["final_eval"] = {"accuracy": acc, "mean_nll": nll}
        res[f"nhid{nhid}"] = r

    name, plim = card()
    line = {"workload": f"SAGPool supervised step vs 2stg step, DD-shape corpus 1168 graphs, 3504-graph compact batch "
                        f"(2 alternating), Net(89, nhid, C={C} | final_dim {a.final_dim}, ratio 0.5, dropout 0.5)",
            "gpu": name, "power_limit_w": plim, "steps": a.steps, "warmup": a.warmup, "rounds": a.rounds,
            "unix_time": int(time.time()), **res}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
