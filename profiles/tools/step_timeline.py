"""Kernel timeline of bench.py's `value` step (the HBM-resident compact SAGPool triplet step) under torch.profiler.

Same corpus, seeds, batches, model and trainer as bench.py's `value`: two alternating compact batches of 3,504 graphs,
PackedSAGNet(89, 32, 32, 0.5, 0.5), TripletTrainer.step (one native tsg_sag_triplet_step_compact call, then Adam).
After --warmup steps, --steps steps are enqueued back to back (no synchronisation between them, as in bench.py) under
the profiler with CUDA activities.  The GPU activities are cut into steps after each fused-Adam kernel, the last
launch of a step; for every profiled step the line reports the kernel count, the sum of kernel durations, the sum
of idle gaps between consecutive GPU activities (kernels, memsets, copies) and the wall time from the first start
to the last end.  The step with the median wall time is written out in full: each activity's name, start (us from
the step's first start) and duration.

    python profiles/tools/step_timeline.py --out-dir DIR [--steps 5] [--warmup 10] [--tag NAME]

Writes DIR/step_timeline[_TAG].json; the Chrome trace stays in DIR only with --keep-trace.  The card's name, power
limit and maximum SM clock are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "two-stage-gnn_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np
import torch


def card():
    """nvidia-smi's name, power limit and maximum SM clock of the visible card, read now."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out
    except Exception as ex:
        return f"nvidia-smi unavailable: {ex}"


def gpu_activities(trace_path):
    """[(name, kind, ts_us, dur_us)] of the trace's device activities on the compute stream, in start order."""
    with open(trace_path) as f:
        ev = json.load(f)["traceEvents"]
    kinds = {"kernel": "kernel", "gpu_memset": "memset", "gpu_memcpy": "memcpy"}
    acts = [(e["name"], kinds[e["cat"]], float(e["ts"]), float(e.get("dur", 0.0)))
            for e in ev if e.get("ph") == "X" and e.get("cat") in kinds]
    acts.sort(key=lambda a: a[2])
    return acts


def split_steps(acts):
    """Cut after every fused-Adam kernel (the last launch of TripletTrainer.step)."""
    steps, cur = [], []
    for a in acts:
        cur.append(a)
        if a[1] == "kernel" and "FusedOptimizerTensorListMetadata" in a[0]:
            steps.append(cur)
            cur = []
    return steps


def summarize(step):
    t0 = step[0][2]
    end = max(a[2] + a[3] for a in step)
    kern = [a for a in step if a[1] == "kernel"]
    gaps, last_end = 0.0, step[0][2] + step[0][3]
    for a in step[1:]:
        gaps += max(0.0, a[2] - last_end)
        last_end = max(last_end, a[2] + a[3])
    return {"kernels": len(kern), "other_activities": len(step) - len(kern),
            "kernel_time_us": round(sum(a[3] for a in kern), 3), "gap_sum_us": round(gaps, 3),
            "wall_us": round(end - t0, 3),
            "kernels_under_6us": sum(1 for a in kern if a[3] < 6.0),
            "kernels_under_6us_time_us": round(sum(a[3] for a in kern if a[3] < 6.0), 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", required=True)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--tag", default="")
    ap.add_argument("--keep-trace", action="store_true")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "step_timeline traces the GPU; there is no CPU fallback"
    import bench
    from tsg import _lib, nn as tnn, ops
    from tsg.train import TripletTrainer

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    assert _lib.lib.tsg_check_device() == 0, _lib.last_error()
    ba = argparse.Namespace(corpus=1168, triplets=1168, nhid=32, final_dim=32)
    corpus, batches, compact, _ = bench.make_step_batches(ba, 0, num_batches=2)
    torch.manual_seed(777)
    model = tnn.PackedSAGNet(corpus.num_node_labels, ba.nhid, ba.final_dim, 0.5, 0.5).to(dev)
    trainer = TripletTrainer(model, lr=5e-4, weight_decay=1e-4, margin=1.5)
    t = lambda v: (torch.from_numpy(v) if isinstance(v, np.ndarray) else v).to(dev)
    dev_compact = [(ops.CompactBatch(t(c["label"]), t(c["row"]), t(c["col"]), t(c["node_ptr"]), t(c["edge_ptr"]),
                                     corpus.num_node_labels, int(np.diff(c["edge_ptr"]).max()), c["coalesced"]),
                    c["node_ptr"], b["triplets"].to(dev)) for c, b in zip(compact, batches)]

    def step(i):
        cb, nptr, trip = dev_compact[i % 2]
        trainer.step(cb, None, nptr, trip)

    for i in range(a.warmup):
        step(i)
    torch.cuda.synchronize()
    k0 = _lib.kernel_launches
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for i in range(a.steps):
            step(a.warmup + i)
        torch.cuda.synchronize()
    libtsg_launches = (_lib.kernel_launches - k0) / a.steps
    os.makedirs(a.out_dir, exist_ok=True)
    suffix = f"_{a.tag}" if a.tag else ""
    trace = os.path.join(a.out_dir, f"step_timeline{suffix}.pt.trace.json")
    prof.export_chrome_trace(trace)
    steps = split_steps(gpu_activities(trace))
    if not a.keep_trace:
        os.remove(trace)
    assert len(steps) == a.steps, f"found {len(steps)} steps in the trace, expected {a.steps}"
    sums = [summarize(s) for s in steps]
    mid = sorted(range(len(steps)), key=lambda k: sums[k]["wall_us"])[len(steps) // 2]
    s = steps[mid]
    t0 = s[0][2]
    out = {"workload": bench.workload_name(argparse.Namespace(corpus=1168, triplets=1168, nhid=32, final_dim=32)),
           "card": card(), "torch": torch.__version__, "profiled_steps": a.steps, "warmup": a.warmup,
           "libtsg_kernel_launches_per_step": libtsg_launches,
           "steps": sums, "median_step_index": mid, "median_step": sums[mid],
           "timeline": [{"name": n, "kind": k, "start_us": round(ts - t0, 3), "dur_us": round(d, 3)} for n, k, ts, d in s]}
    path = os.path.join(a.out_dir, f"step_timeline{suffix}.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"out": path, "card": out["card"], "median_step": sums[mid],
                      "wall_us_all": [x["wall_us"] for x in sums]}))


if __name__ == "__main__":
    main()
