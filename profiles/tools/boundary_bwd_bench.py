"""A/B of the SAGPool backward's level boundary: tsg_sag_boundary_bwd (one pass + the dW fold) against the sequence
it replaces in the executor -- tsg_linear_fwd(dxw, W^T) -> tsg_readout_bwd(MAX|MEAN|ACCUM) and
tsg_linear_bwd_weight(x, dxw) -- at the row counts of bench.py's `value` step at levels 1 and 2 (the DD-shape corpus
of 1,168 graphs, 3 x 1,168 graphs packed, ratio 0.5: level l keeps ceil(n / 2) rows of each graph of level l - 1).

Each timed call is preceded by bench.py's KernelTimer L2 flush (a 256 MB write, then a 256 MB read), timed with CUDA
events on the launching stream; the arms alternate call by call and the medians are reported.  Both arms' outputs
are compared bit for bit first.  The card's name, power limit and maximum SM clock are read in the same run.

    python profiles/tools/boundary_bwd_bench.py --out DIR/boundary_bwd_ab.json [--reps 50] [--nhid 32]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "two-stage-gnn_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np
import torch

READOUT_MAX, READOUT_MEAN, READOUT_ACCUM = 1, 2, 8


def level_sizes(node_ptr, levels=2):
    """per-graph row counts of levels 1 .. levels: top-k keeps ceil(0.5 n) rows of every graph"""
    n = np.diff(np.asarray(node_ptr, np.int64))
    out = []
    for _ in range(levels):
        n = (n + 1) // 2
        out.append(n.copy())
    return out


def operands(sizes, H, dev, seed):
    rng = np.random.default_rng(seed)
    G = len(sizes)
    gptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    N = int(gptr[-1])
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    am = np.where(sizes[:, None] > 0, gptr[:-1, None] + rng.integers(0, np.maximum(sizes, 1)[:, None], (G, H)), -1)
    return dict(dxw=t(rng.standard_normal((N, H)).astype(np.float32)), x=t(rng.standard_normal((N, H)).astype(np.float32)),
                W=t((rng.standard_normal((H, H)) / np.sqrt(H)).astype(np.float32)),
                dz=t(rng.standard_normal((G, 2 * H)).astype(np.float32)), am=t(am.astype(np.int32)), gptr=t(gptr),
                G=G, N=N, H=H)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warm", type=int, default=5)
    ap.add_argument("--nhid", type=int, default=32)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "boundary_bwd_bench times the GPU; there is no CPU fallback"
    import bench
    from step_timeline import card
    from tsg import _lib

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    assert _lib.lib.tsg_check_device() == 0, _lib.last_error()
    ba = argparse.Namespace(corpus=1168, triplets=1168, nhid=a.nhid, final_dim=32)
    _, _, compact, _ = bench.make_step_batches(ba, 0, num_batches=1)
    flush = bench.KernelTimer(dev)
    H = a.nhid
    s = lambda: _lib.stream_ptr()
    res = {"workload": bench.workload_name(ba), "card": card(), "torch": torch.__version__, "reps": a.reps,
           "timing": "CUDA events around one call, L2 flushed before each (bench.py KernelTimer), arms alternating; median",
           "levels": {}}
    for lvl, sizes in zip((1, 2), level_sizes(compact[0]["node_ptr"])):
        c = operands(sizes, H, dev, 100 + lvl)
        N, G = c["N"], c["G"]
        ws = _lib.workspace(_lib.lib.tsg_linear_bwd_weight_workspace_bytes(H, H), dev)
        out = {k: (torch.empty(N, H, device=dev), torch.empty(H, H, device=dev)) for k in ("sequence", "boundary")}
        P = _lib.ptr

        def sequence():
            dxg, dW = out["sequence"]
            _lib.call("tsg_linear_fwd", P(c["dxw"]), P(c["W"]), None, P(dxg), N, H, H, 1, 0, s())
            _lib.call("tsg_readout_bwd", P(c["dz"]), 2 * H, P(c["am"]), P(c["gptr"]), G, N, H,
                      READOUT_MAX | READOUT_MEAN | READOUT_ACCUM, P(dxg), s())
            _lib.call("tsg_linear_bwd_weight", P(c["x"]), P(c["dxw"]), P(dW), None, N, H, H, P(ws), ws.numel(), s())

        def boundary():
            dxg, dW = out["boundary"]
            _lib.call("tsg_sag_boundary_bwd", P(c["dxw"]), P(c["x"]), P(c["W"]), P(c["dz"]), 2 * H, P(c["am"]), P(c["gptr"]),
                      G, N, H, P(dxg), P(dW), P(ws), ws.numel(), s())

        arms = {"sequence": sequence, "boundary": boundary}
        sequence(); boundary(); torch.cuda.synchronize()
        same = all(torch.equal(out["sequence"][i].view(torch.int32), out["boundary"][i].view(torch.int32)) for i in range(2))
        durs = {k: [] for k in arms}
        for it in range(a.warm + a.reps):
            for k, fn in arms.items():
                flush.flush.zero_()
                flush.flush_r.sum()
                st, en = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                st.record(); fn(); en.record()
                torch.cuda.synchronize()
                if it >= a.warm:
                    durs[k].append(st.elapsed_time(en) * 1e3)
        med = {k: statistics.median(v) for k, v in durs.items()}
        # one pass needs dxw, x and dxg once each (+ W, dz, argmax, graph_ptr, the partials: < 1 %)
        alg_bytes = 3 * N * H * 4
        res["levels"][f"l{lvl}"] = {
            "rows": N, "graphs": G, "hidden": H, "bit_identical": bool(same),
            "median_us": {k: round(v, 2) for k, v in med.items()},
            "spread_us": {k: [round(min(v), 2), round(max(v), 2)] for k, v in durs.items()},
            "speedup": round(med["sequence"] / med["boundary"], 3),
            "boundary_gbs_of_3NH": round(alg_bytes / (med["boundary"] * 1e-6) / 1e9, 1)}
        print(f"level {lvl}: N={N} G={G} H={H} bit_identical={same} sequence {med['sequence']:.1f} us, "
              f"boundary {med['boundary']:.1f} us", flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(res["card"])


if __name__ == "__main__":
    main()
