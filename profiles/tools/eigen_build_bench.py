"""Time to build a corpus's EigenPooling operands: the host loop against DeviceCorpus.build_eigen.

Workloads (pool_size 10, J = Jf = 1, BFS clusters):
  host_make_operands_ms   eigen_synth.make_operands on the 1,168-graph DD-shape corpus (seed 777), host clock
  device_build_ms         DeviceCorpus.build_eigen on the same corpus (device events; includes its one count read)
  shard_build_ms          build_eigen on a `--shard-graphs` from_device shard, assembled as bench.Config5 assembles
                          its shard (the base corpus tiled, one K0 gather on the GPU)
Medians over `--rounds` rounds after one warm-up build.  The device build is also checked against the host operands
(integer arrays equal) and the shard's per-graph counts against the base build's, tile by tile.  Prints one JSON line
with the card's name and power limit, read in the same run.

    python profiles/tools/eigen_build_bench.py [--rounds 3] [--shard-graphs 1000000] [--out FILE]
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

from classify_bench import card  # noqa: E402


def device_ms(fn):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    out = fn()
    e.record()
    e.synchronize()
    return s.elapsed_time(e), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--shard-graphs", type=int, default=1_000_000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from tsg import eigen_synth, synth
    from tsg.feeder import DeviceCorpus
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    name, power = card()
    base = synth.make_corpus("DD", 1168, seed=777)
    host_ms = []
    for _ in range(a.rounds):
        t0 = time.perf_counter()
        ref = eigen_synth.make_operands(base, 10, 1, 1)
        host_ms.append((time.perf_counter() - t0) * 1e3)
    dc = DeviceCorpus(base, dev)
    dc.build_eigen(10, 1, 1)
    dev_ms = [device_ms(lambda: dc.build_eigen(10, 1, 1))[0] for _ in range(a.rounds)]
    for k in ("cluster_ptr", "cluster_of", "coarse_ptr", "coarse_row", "coarse_col", "coarse_w"):
        assert np.array_equal(dc.eigen[k].cpu().numpy(), getattr(ref, k)), k
    base_nc, base_nq = dc.eigen["nc"], dc.eigen["ncoarse"]

    bseq = np.arange(a.shard_graphs, dtype=np.int64) % base.num_graphs          # rank 0 of world 1, as Config5
    cb, nptr = dc.pack_compact(bseq)
    _, _, eptr = dc.offsets(bseq)
    shard = DeviceCorpus.from_device(cb.label, cb.row, cb.col, nptr, eptr, base.num_node_labels, dc.coalesced)
    del cb
    shard_ms, fallback = [], None
    for r in range(a.rounds + 1):
        ms, fallback = device_ms(lambda: shard.build_eigen(10, 1, 1))
        if r:
            shard_ms.append(ms)
        shard.eigen = None
    shard.build_eigen(10, 1, 1)
    assert np.array_equal(shard.eigen["nc"], base_nc[bseq]) and np.array_equal(shard.eigen["ncoarse"], base_nq[bseq])
    med = lambda v: float(np.median(v))
    out = dict(tool="eigen_build_bench", gpu=name, power_limit_w=power, pool_size=10, J=1, Jf=1, rounds=a.rounds,
               base_graphs=base.num_graphs, base_nodes=int(base.node_ptr[-1]), base_edges=int(base.edge_ptr[-1]),
               host_make_operands_ms=med(host_ms), device_build_ms=med(dev_ms),
               host_over_device=med(host_ms) / med(dev_ms), shard_graphs=a.shard_graphs,
               shard_nodes=int(nptr[-1]), shard_edges=int(eptr[-1]), shard_build_ms=med(shard_ms),
               shard_clusters=int(shard.eigen["nc"].sum()), shard_coarse_entries=int(shard.eigen["ncoarse"].sum()),
               shard_host_fallback_graphs=int(fallback), peak_mem_gb=torch.cuda.max_memory_allocated() / 2 ** 30,
               host_ms=host_ms, device_ms=dev_ms, shard_ms=shard_ms)
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
