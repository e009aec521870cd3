#!/usr/bin/env python
"""bench.py -- train graphs/sec (fwd+bwd+optimizer) on synthetic graphs of the dataset shapes BASELINE.json names.

Headline workload (BASELINE.json configs[1]): Code/sag `Net(89, nhid=32, final_dim=32, ratio=0.5, dropout=0.5)`
(the run_examples.txt command), 2stg triplet step over the 1,168-graph DD-shape corpus: every graph is the anchor of
one triplet, so one step = 1,168 triplets = 3,504 graph forward+backward passes packed into ONE block-diagonal batch
(~0.97 M nodes, ~4.9 M directed edges), MarginRankingLoss(1.5), backward, Adam.  Per rank (weak scaling): each rank
owns its own corpus shard and step batch; one all-reduce per step carries the weighted gradients and the loss (NCCL).

  python bench.py [--gpus N] [--steps K] [--warmup W]          our arm
  python bench.py --impl reference ...                         reference CPU arm (oracle port, B=1 as shipped)

One JSON line on stdout (rank 0):
  value      graphs/s of the step with its inputs resident in HBM (compact form: node labels + graph-local int32
             endpoints -- what the dataset stores; `value_pyg_wire` = the same step on fp32 one-hot x / int64 edge_index)
  e2e        the same metric through the public API with HOST inputs every step: TripletTrainer.run_from_ids against the
             HBM-resident corpus -- per step the host computes the packed offsets of the sampled graphs, uploads ids +
             offsets + triplets from pinned memory, the GPU assembles the batch (K0), runs the step, the loss comes back.
             Nothing is pre-packed or cached across steps.  `e2e_host_batches` = pre-packed pinned compact host batches
             (43 MB H2D per step), `e2e_fp32_wire` = the PyG wire format from the host (PCIe bound).
  roofline   the dominant kernel timed alone with CUDA events (L2 flushed between launches): algorithmic bytes / time
             against MEASURED_PEAKS.json
  cpu_baseline  the oracle port of the reference path on this box's host cores (B=1 as shipped), plus math-only and
             1-thread figures
  configs    BASELINE configs 1, 3, 4, 5 on the same GPU: value, ms_per_step, roofline of their dominant kernel, CPU
             baselines (as shipped / math only)
  value_allgather (N > 1)  the step with the embeddings all-gathered so triplets may cross ranks (north_star's
             formulation); config5_dp (N > 1) the EigenGCN step data-parallel on the sharded 1 M-graph corpus
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "two-stage-gnn_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np
import torch
import torch.distributed as dist

METRIC = "train graphs/sec (fwd+bwd)"
UNIT = "graphs/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="tsg", choices=["tsg", "reference"])
    ap.add_argument("--corpus", type=int, default=1168, help="graphs in the DD-shape corpus (per rank)")
    ap.add_argument("--triplets", type=int, default=1168, help="triplets per step (per rank)")
    ap.add_argument("--nhid", type=int, default=32)
    ap.add_argument("--final-dim", type=int, default=32)
    ap.add_argument("--ref-triplets", type=int, default=8, help="triplets per reference-arm step")
    ap.add_argument("--cpu-baseline-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--configs", default="1,3,4,5", help="other BASELINE configs to run at N=1 ('' = none)")
    ap.add_argument("--config-steps", type=int, default=8)
    ap.add_argument("--corpus5", type=int, default=1_000_000, help="graphs in the config-5 corpus (whole job, N > 1)")
    ap.add_argument("--breakdown", action="store_true", help="print per-entry-point device time shares to stderr")
    ap.add_argument("--profile-step", default="", choices=["", "dense", "compact"],
                    help="run only warmup + steps of the device-resident step in that input form and exit without a JSON "
                         "line (the command profiles/ launch lists are taken with under ncu)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps of `value`, write what the last of them computed -- the loss it returned, "
                         "every parameter's gradient and every parameter after the optimiser step -- as float32 "
                         "DIR/<name>.npy (inputs and initial parameters are seeded: equal arguments give equal inputs; "
                         "git ignores bench_outputs/)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


def dump_outputs(out_dir, loss, model):
    """DIR/loss.npy, DIR/grad.<parameter>.npy, DIR/param.<parameter>.npy (float32, ~70 KB at the default widths)."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss}
    for k, p in model.named_parameters():
        arrays[f"grad.{k}"] = p.grad
        arrays[f"param.{k}"] = p
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def workload_name(a):
    return (f"SAGPool 2stg triplet step, DD-shape corpus {a.corpus} graphs, {a.triplets} triplets/step "
            f"(3x{a.triplets} graphs packed), Net(89,{a.nhid},{a.final_dim},ratio 0.5,dropout 0.5)")


# ------------------------------------------------------------------------------------------ data
def make_step_batches(a, rank: int, num_batches: int):
    from tsg import synth
    corpus = synth.make_corpus("DD", a.corpus, seed=777 + 1_000_003 * rank)
    coalesced = synth.is_coalesced_symmetric(corpus)     # TUDataset form (checked once; the kernels re-verify per graph)
    out, compact, id_lists = [], [], []
    T = a.triplets
    tidx = np.stack([np.arange(T), T + np.arange(T), 2 * T + np.arange(T)], 1).astype(np.int64)
    for b in range(num_batches):
        trip = synth.sample_triplets(corpus.y, T, seed=1000 * rank + b)
        ids = np.concatenate([trip[:, 0], trip[:, 1], trip[:, 2]])
        id_lists.append(ids)
        pk = synth.pack(corpus, ids)
        out.append(dict(x=torch.from_numpy(pk["x"]).pin_memory(),
                        edge_index=torch.from_numpy(pk["edge_index"]).pin_memory(),
                        node_ptr=pk["node_ptr"], triplets=torch.from_numpy(tidx).pin_memory()))
        sel = synth.select(corpus, ids)
        compact.append(dict(label=torch.from_numpy(sel.node_label.astype(np.int32)).pin_memory(),
                            row=torch.from_numpy(sel.row.astype(np.int32)).pin_memory(),
                            col=torch.from_numpy(sel.col.astype(np.int32)).pin_memory(),
                            node_ptr=sel.node_ptr.copy(), edge_ptr=sel.edge_ptr.copy(),
                            triplets=torch.from_numpy(tidx).pin_memory(), coalesced=coalesced))
    return corpus, out, compact, id_lists


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    def __init__(self, index: int, period: float = 0.2):
        super().__init__(daemon=True)
        self.index, self.period, self.samples, self.reasons, self.max_mhz = index, period, [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    NAMES = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
             0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
             0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def run(self):
        if not self.ok:
            return
        while not self._stop_evt.is_set():
            try:
                self.samples.append(int(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                r = int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                for bit, name in self.NAMES.items():
                    if r & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(self.period)

    def finish(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


class KernelTimer:
    """One kernel (or one C-ABI entry point) alone: L2 flushed before every launch, CUDA events on the launching
    stream, mean of `reps` after `warm` warm-ups.  The flush is a 256 MB WRITE (evicts the kernel's operands) followed
    by a 256 MB READ of another buffer (evicts the write's dirty lines: without it their write-back to DRAM runs
    concurrently with the timed kernel and is charged to it -- round 1's figure carried that)."""

    def __init__(self, dev):
        self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)      # > 126 MB L2
        self.flush_r = torch.zeros(64 * 1024 * 1024, dtype=torch.float32, device=dev)   # 256 MB, read only

    def __call__(self, fn, reps=10, warm=3):
        durs = []
        for it in range(warm + reps):
            self.flush.zero_()
            self.flush_r.sum()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(); fn(); e.record()
            torch.cuda.synchronize()
            if it >= warm:
                durs.append(s.elapsed_time(e))
        return sum(durs) / len(durs)


def roofline_block(kernel, alg_bytes, ms, peaks, flops=None, traffic=None, note=None):
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = alg_bytes / (ms * 1e-3) / 1e9
    out = {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
           "peak_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)",
           "algorithmic_bytes_per_launch": int(alg_bytes), "avg_launch_ms": ms, "traffic": traffic,
           "frac_of_nominal_8TBs": achieved / 8000.0}
    if flops is not None:
        out["tflops"] = flops / (ms * 1e-3) / 1e12
    if note:
        out["note"] = note
    return out


def committed_traffic(tag: str, sources):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from a COMMITTED `ncu --set full` capture (profiles/),
    valid only while the kernel source it was taken from is unchanged (sha1 recorded beside it); else None."""
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", tag)))
        h = hashlib.sha1()
        for s in sources:
            h.update(open(os.path.join(ROOT, "two-stage-gnn_b200", "csrc", s), "rb").read())
        if tj.get("source_sha1") == h.hexdigest():
            return int(tj["dram_bytes_read"] + tj["dram_bytes_write"]), f"profiles/{tag} (ncu --set full, same kernel source)"
    except Exception:
        pass
    return None, None


# ------------------------------------------------------------------------------------------ CPU reference (SAGPool)
class CpuReference:
    """The reference's stage-1 loop (Code/sag/train_triplet.py:203-214) on the host cores through the
    oracle port: per triplet three SINGLE-graph forwards (the scripts' effective batch size),
    pairwise distances, MarginRankingLoss, backward, Adam step."""

    def __init__(self, a, n_graphs: int = 64, threads: int | None = None):
        from oracle import pyg_ref as R
        from tsg import synth
        self.R, self.a = R, a
        torch.set_num_threads(threads or os.cpu_count() or 1)
        n_graphs = min(a.corpus, n_graphs)
        corpus = synth.make_corpus("DD", n_graphs, seed=777)
        self.corpus = corpus
        self.graphs = []
        for g in range(n_graphs):
            pk = synth.pack(corpus, [g])
            self.graphs.append((torch.from_numpy(pk["x"]), torch.from_numpy(pk["edge_index"]),
                                torch.zeros(pk["x"].shape[0], dtype=torch.long)))
        self.trip = synth.sample_triplets(corpus.y, 4096, seed=0)
        self.params = {k: v.clone().requires_grad_(True)
                       for k, v in R.init_sag_params(corpus.num_node_labels, a.nhid, a.final_dim, 777).items()}
        self.opt = torch.optim.Adam(list(self.params.values()), lr=5e-4, weight_decay=1e-4)
        self.gen = torch.Generator().manual_seed(0)
        self.t = 0

    def triplet(self):
        R, a = self.R, self.a
        embs = []
        for gid in self.trip[self.t % len(self.trip)]:
            x, ei, batch = self.graphs[int(gid)]
            mask = (torch.rand(1, a.nhid, generator=self.gen) >= 0.5).float() * 2.0     # dropout p=0.5
            embs.append(R.sag_net_forward(self.params, x, ei, batch, 0.5, dropout_mask=mask))
        loss, _, _ = R.triplet_margin_loss(embs[0], embs[1], embs[2], 1.5)
        self.opt.zero_grad(); loss.backward(); self.opt.step()
        self.t += 1

    def packed_step(self, T: int):
        """math-only variant: the SAME arithmetic on ONE packed batch of 3T graphs (what the GPU arm runs), tensors
        pre-built -- the batching the reference operators support but its scripts never use."""
        from tsg import synth
        R = self.R
        if not hasattr(self, "_packed") or self._packed[0] != T:
            trip = self.trip[:T] % self.corpus.num_graphs
            ids = np.concatenate([trip[:, 0], trip[:, 1], trip[:, 2]])
            pk = synth.pack(self.corpus, ids)
            self._packed = (T, torch.from_numpy(pk["x"]), torch.from_numpy(pk["edge_index"]), torch.from_numpy(pk["batch"]))
        _, x, ei, batch = self._packed
        mask = (torch.rand(3 * T, self.a.nhid, generator=self.gen) >= 0.5).float() * 2.0
        emb = R.sag_net_forward(self.params, x, ei, batch, 0.5, dropout_mask=mask)
        loss, _, _ = R.triplet_margin_loss(emb[:T], emb[T:2 * T], emb[2 * T:], 1.5)
        self.opt.zero_grad(); loss.backward(); self.opt.step()

    def rate(self, seconds: float, max_triplets: int):
        self.triplet()   # warm-up
        done, t0 = 0, time.perf_counter()
        while done < max_triplets and (time.perf_counter() - t0) < seconds:
            self.triplet(); done += 1
        el = time.perf_counter() - t0
        return 3 * done / el, 3 * done, el

    def rate_packed(self, seconds: float, T: int = 16):
        self.packed_step(T)
        done, t0 = 0, time.perf_counter()
        while (time.perf_counter() - t0) < seconds:
            self.packed_step(T); done += 1
        el = time.perf_counter() - t0
        return 3 * T * done / el, 3 * T * done, el


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    ref = CpuReference(a)
    # thread calibration (outside the timed region): the reference's B=1 forwards on ~269-node graphs can be FASTER on one
    # thread than on all of them (intra-op pool wake-ups); the arm runs with whichever is faster on this box
    cal = {}
    for th in sorted({cores, 1}, reverse=True):
        torch.set_num_threads(th)
        ref.triplet()
        t0 = time.perf_counter()
        for _ in range(3):
            ref.triplet()
        cal[th] = time.perf_counter() - t0
    use = min(cal, key=cal.get)
    torch.set_num_threads(use)
    for _ in range(max(a.warmup, 0)):
        ref.triplet()
    t0 = time.perf_counter()
    for s in range(a.steps):
        for _ in range(a.ref_triplets):
            ref.triplet()
    el = time.perf_counter() - t0
    graphs = 3 * a.ref_triplets * a.steps
    rate = graphs / el
    sample = (f"{a.ref_triplets} triplets/step x 3 single-graph forwards (B=1 as shipped), DD-shape, oracle port "
              f"of PyG ops under torch CPU, {use} thread(s) (calibrated: " +
              ", ".join(f"{th} thr {3 * 3 / v:.0f} graphs/s" for th, v in cal.items()) + f"; box has {cores} cores)")
    cores = use
    line = {"metric": METRIC, "value": rate, "unit": UNIT, "impl": "reference", "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": 1000 * el / max(a.steps, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(a), "reference_step": sample},
            "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ other configs (N = 1)
def _timed_steps(fn, steps, warmup):
    for i in range(warmup):
        fn(i)
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for i in range(steps):
        last = fn(i)
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / steps, float(last)


def _triplet_batch(corpus, seed):
    from tsg import synth
    T = corpus.num_graphs
    trip = synth.sample_triplets(corpus.y, T, seed=seed)
    ids = np.concatenate([trip[:, 0], trip[:, 1], trip[:, 2]])
    tidx = np.stack([np.arange(T), T + np.arange(T), 2 * T + np.arange(T)], 1).astype(np.int64)
    return ids, tidx


def _dense_inputs(corpus, ids, dev, feat_dim=32, max_nodes=1000, want_eid=False):
    """packed x (rows of the shared N(0, 2^2) feature table, Code/sage+gat+diffpool/train_triplet.py:379-385), the RAW
    0/1 CSR of the packed adjacency, graph offsets and the has-padded-rows flags."""
    from tsg import ops, synth
    sel = synth.select(corpus, ids)
    n = np.diff(sel.node_ptr)
    table = torch.from_numpy(np.random.default_rng(777).normal(0.0, 2.0, (max_nodes, feat_dim)).astype(np.float32))
    local = np.concatenate([np.arange(k) for k in n])
    x = table[torch.from_numpy(local)].to(dev)
    pk = synth.pack(sel, one_hot=False)
    ei = torch.from_numpy(pk["edge_index"]).to(dev)
    N = int(sel.node_ptr[-1])
    csr = ops.build_csr(ops.EdgeList.from_edge_index(ei), N, mode=ops.CSR_RAW, want_eid=want_eid)
    gptr = torch.from_numpy(sel.node_ptr).to(dev)
    has_pad = torch.from_numpy(n < max_nodes).to(dev)
    return x, csr, gptr, has_pad, N, int(ei.size(1)), sel, table


class _CpuDense:
    """CPU legs of the dense configs: the oracle port of the reference modules (oracle/dense_ref.py, pinned to fixtures
    generated by the real modules) driven the way the reference scripts drive them -- ONE graph per forward.
    as_shipped: zero-padded to --max-nodes = 1000 including the per-graph host marshaling the scripts perform
    (`torch.Tensor([ndarray])`, tripletnet.py:18-33; the DataLoader's numpy padding + collate for `train.py`);
    math_only: tensors pre-built, padded tight to the graph."""

    def __init__(self, corpus, table, kind, seconds):
        from oracle import dense_ref as D
        self.D, self.corpus, self.table, self.kind, self.seconds = D, corpus, table, kind, seconds
        torch.set_num_threads(os.cpu_count() or 1)
        g = torch.Generator().manual_seed(777)
        rnd = lambda *s: (torch.randn(*s, generator=g) * 0.2).requires_grad_(True)
        conv = lambda i, o: dict(weight=rnd(i, o), bias=torch.zeros(o, requires_grad=True))
        if kind == "base":          # GcnEncoderGraph(32,32,32,2,L=2): conv_first, conv_last, pred head 64 -> 32 -> 2
            self.p = dict(conv=[conv(32, 32), conv(32, 32)], head=[rnd(32, 64), rnd(2, 32)])
        elif kind == "gat":         # heads [2,2], L=3: 32 -> 64 -> 64 -> 32
            head = lambda i, o: dict(w=rnd(i, o), a=rnd(2 * o, 1))
            self.p = dict(layers=[[head(32, 32), head(32, 32)], [head(64, 32), head(64, 32)], [head(64, 32), head(64, 32)]],
                          head=[rnd(32, 32)])
        elif kind == "diffpool":    # N=1000 -> K=100, D=96
            self.p = dict(conv=[conv(32, 32), conv(32, 32), conv(32, 32)],
                          assign_conv=[conv(32, 32), conv(32, 32), conv(32, 100)],
                          conv_after=[conv(96, 32), conv(32, 32), conv(32, 32)], head=[rnd(32, 192)])
            self.p["assign_pred.weight"] = rnd(100, 164); self.p["assign_pred.bias"] = torch.zeros(100, requires_grad=True)
        leaves = []

        def walk(o):
            if torch.is_tensor(o):
                leaves.append(o)
            elif isinstance(o, dict):
                [walk(v) for v in o.values()]
            elif isinstance(o, (list, tuple)):
                [walk(v) for v in o]
        walk(self.p)
        self.opt = torch.optim.Adam(leaves, lr=1e-3)

    def _graph(self, g, N, marshal):
        c = self.corpus
        n = c.num_nodes(g)
        e0, e1 = int(c.edge_ptr[g]), int(c.edge_ptr[g + 1])
        N = max(N, n)
        adj = np.zeros((N, N), np.float32); adj[c.row[e0:e1], c.col[e0:e1]] = 1.0
        feats = np.zeros((N, 32), np.float32); feats[:n] = self.table[:n].numpy()
        if marshal == "triplet":          # tripletnet.py:18-19
            return torch.Tensor([adj]), torch.Tensor([feats]), n
        return torch.from_numpy(adj)[None], torch.from_numpy(feats)[None], n

    def _embed(self, adj, x, n):
        D, p = self.D, self.p
        if self.kind == "base":
            r = D.gcn_encoder_readout(x, adj, p["conv"])
            return torch.relu(r @ p["head"][0].t()) @ p["head"][1].t()
        if self.kind == "gat":
            return D.dgat_encoder_readout(x, adj, p["layers"]) @ p["head"][0].t()
        r, _ = D.soft_pool_readout(x, adj, [n], p)
        return r @ p["head"][0].t()

    def run(self, as_shipped: bool):
        c = self.corpus
        N = 1000 if as_shipped else 0
        marshal = ("triplet" if self.kind != "base" else "loader") if as_shipped else None
        pre = None if as_shipped else [self._graph(g, 0, None) for g in range(min(c.num_graphs, 24))]
        done, t0, g = 0, time.perf_counter(), 0
        budget = self.seconds
        while True:
            if self.kind == "base":           # original setting: cross-entropy per graph (train.py:85-130)
                adj, x, n = self._graph(g % c.num_graphs, N, marshal) if as_shipped else pre[g % len(pre)]
                logits = self._embed(adj, x, n)
                loss = torch.nn.functional.cross_entropy(logits, torch.tensor([int(c.y[g % c.num_graphs])]))
                g += 1; done += 1
            else:                              # 2stg triplet: three single-graph forwards (tripletnet.py:36-38)
                embs = []
                for k in range(3):
                    adj, x, n = self._graph((g + k) % c.num_graphs, N, marshal) if as_shipped else pre[(g + k) % len(pre)]
                    embs.append(self._embed(adj, x, n))
                dp = torch.nn.functional.pairwise_distance(embs[0], embs[1], 2)
                dn = torch.nn.functional.pairwise_distance(embs[0], embs[2], 2)
                loss = torch.clamp(dp - dn + 1.5, min=0).mean()
                g += 3; done += 3
            self.opt.zero_grad(); loss.backward(); self.opt.step()
            if done >= 3 and time.perf_counter() - t0 >= budget:
                break
        el = time.perf_counter() - t0
        return done / el, done, el


def _best_of_threads(run, seconds):
    """A CPU leg under all host threads AND under one thread (single 39-269 node graphs are far below the size where
    torch's intra-op pool pays for itself: its wake-up latency alone can exceed the arithmetic); the FASTER one is the
    baseline, with the thread count it used."""
    cores = os.cpu_count() or 1
    res = {}
    for th in sorted({cores, 1}, reverse=True):
        torch.set_num_threads(th)
        res[th] = run(seconds / 2.0)
    torch.set_num_threads(cores)
    best = max(res, key=lambda th: res[th][0])
    return best, res


def _cpu_block(corpus, table, kind, seconds):
    cpu = _CpuDense(corpus, table, kind, seconds)

    def leg(as_shipped):
        def run(sec):
            cpu.seconds = sec
            return cpu.run(as_shipped)
        return _best_of_threads(run, seconds)
    bs, rs = leg(True)
    bm, rm = leg(False)
    fmt = lambda res: ", ".join(f"{th} thread(s): {r[0]:.1f} graphs/s ({r[1]} graphs in {r[2]:.1f} s)" for th, r in res.items())
    return {"value": rs[bs][0], "unit": UNIT, "cores": bs, "kind": "port",
            "sample": "as shipped: single-graph fwd+bwd+Adam, B=1, zero-padded to --max-nodes=1000, host marshaling included "
                      f"(oracle/dense_ref.py port of the reference module); {fmt(rs)}; faster one reported",
            "math_only": {"value": rm[bm][0], "unit": UNIT, "cores": bm,
                          "sample": f"tensors pre-built, padded tight to the graph; {fmt(rm)}; faster one reported"}}


def run_config1(a, dev, kt, peaks, cpu):
    from tsg import dense, ops, synth
    corpus = synth.make_corpus("PROTEINS", 1113, seed=777)
    ids = np.arange(corpus.num_graphs)
    x, csr, gptr, has_pad, N, E, sel, table = _dense_inputs(corpus, ids, dev)
    y = torch.from_numpy(corpus.y).to(dev)
    torch.manual_seed(777)
    model = dense.PackedGcnEncoder(32, 32, 32, 2, 2, bn=True, final_dim="number_classes").to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, capturable=True)

    def body():
        _, logits = model(x, csr, gptr, has_pad)
        loss = torch.nn.functional.cross_entropy(logits, y)
        opt.zero_grad(set_to_none=False); loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 2.0)          # train.py clip 2.0
        opt.step()
        return loss.detach()
    ms_eager, _ = _timed_steps(lambda i: body(), a.config_steps, 3)
    # the original setting trains on the SAME packed corpus every epoch: the step is captured once into a CUDA graph
    from tsg.train import CapturedStep
    cap = CapturedStep(body)
    ms, loss = _timed_steps(lambda i: cap.replay(), max(a.config_steps, 20), 3)
    kms = kt(lambda: ops.spmm_raw(csr.rowptr, csr.colidx, csr.val, x))
    alg = 4 * 2 * N * 32 + 4 * (N + 1) + 4 * E          # SURVEY 8d config 1: unweighted 0/1 adjacency
    out = {"workload": "GraphSAGE original setting (cross-entropy, clip 2.0, Adam 1e-3), PROTEINS-shape, 1,113 graphs = one "
                       "packed batch, GcnEncoderGraph(32,32,32,2,L=2,bn,final_dim=number_classes)",
           "value": corpus.num_graphs / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "graphs_per_step": corpus.num_graphs,
           "nodes_per_step": N, "directed_edges_per_step": E, "loss": loss,
           "step": "captured once into a CUDA graph (tsg.train.CapturedStep) and replayed: the batch is the whole corpus, its shape never changes",
           "eager": {"value": corpus.num_graphs / (ms_eager / 1e3), "ms_per_step": ms_eager,
                     "note": "same step enqueued launch by launch from Python (launch bound: ~200 launches for 43 k nodes)"},
           "roofline": roofline_block(f"k_spmm_g RAW (adj @ x, N={N}, nnz={E}, F=32)", alg, kms, peaks,
                                      note="43 k nodes per launch: 12 MB moved, launch / latency bound by size")}
    if cpu:
        out["cpu_baseline"] = _cpu_block(corpus, table, "base", 3.0)
    return out


def run_config3(a, dev, kt, peaks, cpu):
    from tsg import gat, ops, synth
    from tsg.gat import _GatAggregate
    corpus = synth.make_corpus("JANY", 744, seed=777)
    ids, tidx = _triplet_batch(corpus, 0)
    x, csr, gptr, has_pad, N, E, sel, table = _dense_inputs(corpus, ids, dev, want_eid=True)
    tr = torch.from_numpy(tidx).to(dev)
    torch.manual_seed(777)
    model = gat.PackedGatEncoder(32, 32, 32, 2, num_layers=3, num_heads=[2, 2]).to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)

    def step(i):
        _, emb = model(x, csr, gptr, 1000)
        loss, _, _ = ops.triplet_loss(emb, tr, 1.5)
        opt.zero_grad(set_to_none=True); loss.backward(); opt.step()
        return loss.detach()
    ms, loss = _timed_steps(step, a.config_steps, 3)
    Hd, Fo = 2, 32
    h = torch.randn(N, Hd * Fo, device=dev); s1 = torch.randn(N, Hd, device=dev); s2 = torch.randn(N, Hd, device=dev)
    with torch.no_grad():
        kms = kt(lambda: _GatAggregate.apply(h, s1, s2, csr, Hd, Fo, 0.2))
    # SURVEY 8d config 3, per head: 4 n F (h in) + 4 n F (h' out) + 4 (n + 1) + 4 E per orientation (both are read)
    alg = Hd * (4 * N * Fo * 2) + 2 * (4 * (N + 1) + 4 * E) + 4 * N * Hd * 2
    out = {"workload": f"GAT 2stg+ stage-1 triplet step, JAN.Y-shape, 3x{corpus.num_graphs} graphs packed, "
                       "DGATEncoderGraph(32,32,32,2,L=3,heads [2,2]) -> widths 32/64/64/32, N = 1000 semantics",
           "value": ids.shape[0] / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "graphs_per_step": int(ids.shape[0]),
           "nodes_per_step": N, "directed_edges_per_step": E, "loss": loss,
           "roofline": roofline_block(f"tsg_gat_fwd (k_gat_colstats + k_gat_aggregate, 2 heads x 32, N={N}, E={E})", alg, kms, peaks)}
    if cpu:
        out["cpu_baseline"] = _cpu_block(corpus, table, "gat", 3.0)
    return out


def run_config4(a, dev, kt, peaks, cpu):
    from tsg import diffpool, ops, synth
    corpus = synth.make_corpus("DD", 1168, seed=777)
    ids, tidx = _triplet_batch(corpus, 0)
    x, csr, gptr, has_pad, N, E, sel, table = _dense_inputs(corpus, ids, dev)
    tr = torch.from_numpy(tidx).to(dev)
    torch.manual_seed(777)
    model = diffpool.PackedSoftPoolEncoder(1000, 32, 32, 32, 2, 3, 32, assign_ratio=0.1).to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)

    def step(i):
        _, emb = model(x, csr, gptr, has_pad)
        loss, _, _ = ops.triplet_loss(emb, tr, 1.5)
        opt.zero_grad(set_to_none=True); loss.backward(); opt.step()
        return loss.detach()
    ms, loss = _timed_steps(step, a.config_steps, 3)
    K, D = 100, 96
    G = int(ids.shape[0])
    # dominant kernel of the step (profiles/r02f_launches_diffpool_step.csv): the row-local product d[Z | AS] = S dC of the
    # contraction's backward on tcgen05 -- per graph [n_g, K] x [K, D + K]
    s = torch.softmax(torch.randn(N, K, device=dev), dim=1); dc = torch.randn(G, K, D + K, device=dev)
    kms = kt(lambda: ops.seg_linear_raw(s, dc, gptr, False, tensor_cores=True))
    alg = 4 * (N * K + N * (D + K) + G * K * (D + K))
    flops = 2.0 * N * K * (D + K)
    rf = roofline_block(f"k_seg_linear_tc (tcgen05 3xTF32, Y[r,:] = S[r,:] dC_g, K={K}, D+K={D + K}, {G} graphs)", alg, kms, peaks,
                        flops=flops, note="HBM bound by arithmetic intensity (%.1f flop/B); tflops = useful fp32 flops, the "
                                          "tensor pipe issues 3 TF32 MMAs per product; bound in practice by the SIMT hi/lo split "
                                          "(profiles/r02f_k7_seg_linear_tc.md)" % (flops / alg))
    out = {"workload": f"DiffPool 2stg triplet step, DD-shape, 3x{corpus.num_graphs} graphs packed, "
                       "SoftPoolingGcnEncoder(N=1000,32,32,32,2,L=3,assign_ratio=0.1): K=100, D=96",
           "value": G / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "graphs_per_step": G, "nodes_per_step": N,
           "directed_edges_per_step": E, "loss": loss, "tensor_cores": bool(ops.USE_TCGEN05), "roofline": rf}
    if cpu:
        out["cpu_baseline"] = _cpu_block(corpus, table, "diffpool", 3.0)
    return out


class Config5:
    """EigenGCN 2stg+ stage-1 triplet step against an HBM-RESIDENT corpus of `num_graphs` DD-shape graphs (BASELINE
    config 5: 1 M graphs), sharded graph_id % world.  The corpus is the 1,168-graph DD-shape base corpus tiled to
    `num_graphs` ids (SURVEY 8d); this rank's shard is materialised IN HBM by one K0 gather from the base (compact form:
    node labels, graph-local int32 endpoints, per-node cluster labels, per-cluster final-pooling weights; 13 GB for 1 M
    graphs on one GPU).  A step: the host samples 3T graph ids of the shard (anchor / positive / negative by label) and
    computes their packed offsets; the GPU gathers the batch from the resident corpus, expands it (K0), builds the RAW CSR
    (K1), the pooling operators P^T and the coarsened adjacency (K11), trains WavePoolingGcnEncoder + triplet loss + Adam.
    Nothing about a batch is cached between steps."""

    def __init__(self, dev, num_graphs, rank=0, world=1, base_graphs=1168):
        from tsg import dense, eigen_synth, synth
        from tsg.feeder import DeviceCorpus, DeviceRagged
        self.dev, self.rank, self.world, self.num_graphs = dev, rank, world, num_graphs
        base = synth.make_corpus("DD", base_graphs, seed=777)
        opnd = eigen_synth.make_operands(base, pool_size=10, num_pool_matrix=1, num_pool_final_matrix=1)
        self.base, self.opnd = base, opnd
        owned = np.arange(rank, num_graphs, world, dtype=np.int64)
        bseq = owned % base.num_graphs                       # corpus id -> base graph
        self.owned, self.y = owned, base.y[bseq]
        base_dc = DeviceCorpus(base, dev)
        cb, nptr = base_dc.pack_compact(bseq)                # the shard, assembled on the GPU
        _, _, eptr = base_dc.offsets(bseq)
        self.corpus = DeviceCorpus.from_device(cb.label, cb.row, cb.col, nptr, eptr, base.num_node_labels, base_dc.coalesced)
        t = lambda v, dt: torch.from_numpy(np.ascontiguousarray(v.astype(dt))).to(dev)
        cl_base = DeviceRagged(base.node_ptr, t(opnd.cluster_of, np.int32))
        fw_base = DeviceRagged(opnd.cluster_ptr, t(opnd.final_w[0], np.float32))
        cl_vals, _ = cl_base.gather(bseq)
        fw_vals, cptr = fw_base.gather(bseq)
        self.cluster = DeviceRagged(nptr, cl_vals)
        self.final_w = DeviceRagged(cptr, fw_vals)
        self.nc = np.diff(cptr).astype(np.int64)
        self.resident_bytes = int(cb.label.numel() * 4 + cb.row.numel() * 8 + cl_vals.numel() * 4 + fw_vals.numel() * 4
                                  + 3 * 8 * (owned.shape[0] + 1))
        torch.manual_seed(777)
        self.model = dense.PackedWaveEncoder(base.num_node_labels, 32, 32, 2, 2, num_pool_matrix=1, num_pool_final_matrix=1,
                                             pool_sizes=[10], pred_hidden_dims=[50]).to(dev)
        self.opt = torch.optim.Adam(self.model.parameters(), lr=1e-3)

    def sample(self, seed, T):
        """host sampler: local shard indices of T anchors, positives (same label) and negatives (other label)"""
        rng = np.random.default_rng(10_000 * self.rank + seed)
        M = self.owned.shape[0]
        pool = {k: np.nonzero(self.y == k)[0] for k in (0, 1)}
        anchors = rng.integers(0, M, T)
        ya = self.y[anchors]
        pos = np.where(ya == 1, pool[1][rng.integers(0, len(pool[1]), T)], pool[0][rng.integers(0, len(pool[0]), T)])
        neg = np.where(ya == 1, pool[0][rng.integers(0, len(pool[0]), T)], pool[1][rng.integers(0, len(pool[1]), T)])
        return np.concatenate([anchors, pos, neg]).astype(np.int64)

    def assemble(self, ids):
        """3T shard indices -> device operands of the step (everything on the GPU from the resident corpus)."""
        from tsg import dense, ops
        dev = self.dev
        cb, nptr = self.corpus.pack_compact(ids)
        x, ei = cb.expand()                                   # K0: one-hot x [N, 89], int64 edge_index
        N, E, G = int(nptr[-1]), int(ei.size(1)), ids.shape[0]
        el = ops.EdgeList.from_edge_index(ei)
        csr_adj = ops.build_csr(el, N, mode=ops.CSR_RAW)
        cl_local, _ = self.cluster.gather(ids)
        fw, cptr = self.final_w.gather(ids)
        NC = int(cptr[-1])
        nc = np.diff(cptr)
        small = torch.from_numpy(np.concatenate([cptr[:-1], np.diff(nptr), nc, cptr])).pin_memory().to(dev, non_blocking=True)
        coff, n_dev, nc_dev, cptr_dev = small[:G], small[G:2 * G], small[2 * G:3 * G], small[3 * G:]
        cl = (cl_local + torch.repeat_interleave(coff, n_dev, output_size=N).to(torch.int32)).contiguous()
        fsrc = torch.arange(NC, device=dev, dtype=torch.int64)
        fdst = torch.repeat_interleave(torch.arange(G, device=dev, dtype=torch.int64), nc_dev, output_size=NC)
        final = [dense.build_rect_csr(ops.EdgeList(fsrc, fdst, NC), fw, G, NC)]
        T = G // 3
        tidx = torch.from_numpy(np.stack([np.arange(T), T + np.arange(T), 2 * T + np.arange(T)], 1).astype(np.int64)).pin_memory().to(dev, non_blocking=True)
        return dict(x=x, el=el, csr_adj=csr_adj, cl=cl, NC=NC, G=G, N=N, E=E, final=final, gptr=cb.node_ptr, cptr=cptr_dev,
                    fptr=torch.arange(G + 1, device=dev, dtype=torch.int64), tr=tidx)

    def step(self, b, group=None):
        from tsg import eigenpool, ops
        from tsg.train import all_reduce_grads_and_loss
        built = eigenpool.build(b["csr_adj"], b["el"], b["cl"], b["NC"], 1)       # K11: P_0^T + coarsened adjacency
        emb = self.model(b["x"], b["csr_adj"], b["gptr"], [[built["pool"][0]], b["final"]], [built["coarse"]],
                         [b["cptr"]], b["fptr"])
        loss, _, _ = ops.triplet_loss(emb, b["tr"], 1.5)
        self.opt.zero_grad(set_to_none=True); loss.backward()
        if self.world > 1:
            loss = all_reduce_grads_and_loss(list(self.model.parameters()), loss, int(b["tr"].size(0)), group)
        self.opt.step()
        return loss.detach()

    def step_from_ids(self, ids, group=None):
        return self.step(self.assemble(ids), group)


def run_config5(a, dev, kt, peaks, cpu):
    from tsg import eigenpool, ops
    c5 = Config5(dev, a.corpus5)
    T = 1168
    id_lists = [c5.sample(s, T) for s in range(4)]
    ms, loss = _timed_steps(lambda i: c5.step_from_ids(id_lists[i % 4]), a.config_steps, 3)
    b = c5.assemble(id_lists[0])
    ms_dev, _ = _timed_steps(lambda i: c5.step(b), a.config_steps, 2)
    built = eigenpool.build(b["csr_adj"], b["el"], b["cl"], b["NC"], 1)
    P = built["pool"][0]
    D = 64
    z = torch.randn(b["N"], D, device=dev)
    kms = kt(lambda: ops.spmm_raw(P.rowptr, P.colidx, P.val, z))
    alg = 4 * (b["N"] * D + b["NC"] * D) + 8 * b["N"]          # SURVEY 8d config 5
    out = {"workload": f"EigenGCN 2stg+ stage-1 triplet step against an HBM-resident corpus of {a.corpus5:,} DD-shape graphs "
                       f"({c5.resident_bytes / 1e9:.1f} GB on this GPU), 3x{T} graphs per step gathered by id on the GPU, "
                       "WavePoolingGcnEncoder(89,32,32,2,L=2,num_pool_matrix=1,num_pool_final_matrix=1,pool_sizes [10],"
                       "pred_hidden [50]); CSR + pooling operators (K11) built on the GPU every step",
           "value": b["G"] / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "graphs_per_step": b["G"], "nodes_per_step": b["N"],
           "directed_edges_per_step": b["E"], "clusters_per_step": b["NC"], "loss": loss, "corpus_graphs": a.corpus5,
           "corpus_resident_bytes": c5.resident_bytes,
           "value_batch_resident": {"value": b["G"] / (ms_dev / 1e3), "ms_per_step": ms_dev,
                                    "note": "same step on one batch already assembled in HBM (no gather / expand / CSR build)"},
           "roofline": roofline_block(f"k_spmm_g on P^T (eigen pooling, N={b['N']}, clusters={b['NC']}, D={D})", alg, kms, peaks)}
    if cpu:
        out["cpu_baseline"] = _cpu_wave(c5, 3.0)
    del c5
    return out


def _cpu_wave(c5, seconds):
    """Reference WavePoolingGcnEncoder path on the host (oracle/dense_ref.py port), B = 1: as shipped (N = 1000 padded
    operands incl. ~10 `torch.Tensor([ndarray])` conversions per graph, eigengcn/tripletnet.py:19-56) / math only."""
    from oracle import dense_ref as D
    from tsg import eigen_synth, synth
    torch.set_num_threads(os.cpu_count() or 1)
    base, opnd = c5.base, c5.opnd
    g = torch.Generator().manual_seed(777)
    rnd = lambda *s: (torch.randn(*s, generator=g) * 0.2).requires_grad_(True)
    conv = lambda i, o: dict(weight=rnd(i, o), bias=torch.zeros(o, requires_grad=True))
    p = dict(conv=[conv(89, 32), conv(32, 32)], conv_after=[[conv(64, 32), conv(32, 32)]])
    head = [dict(weight=rnd(50, 192), bias=torch.zeros(50, requires_grad=True)), dict(weight=rnd(2, 50), bias=torch.zeros(2, requires_grad=True))]
    leaves = [c[k] for cs in (p["conv"], p["conv_after"][0]) for c in cs for k in ("weight", "bias")] + [h[k] for h in head for k in ("weight", "bias")]
    opt = torch.optim.Adam(leaves, lr=1e-3)

    def operands(gi, N):
        n = base.num_nodes(gi); n0 = int(base.node_ptr[gi]); e0, e1 = int(base.edge_ptr[gi]), int(base.edge_ptr[gi + 1])
        N = max(N, n)
        nc = int(opnd.cluster_ptr[gi + 1] - opnd.cluster_ptr[gi])
        adj = np.zeros((N, N), np.float32); adj[base.row[e0:e1], base.col[e0:e1]] = 1.0
        x = np.zeros((N, 89), np.float32); x[np.arange(n), base.node_label[n0:n0 + n]] = 1.0
        P = np.zeros((N, N), np.float32); P[np.arange(n), opnd.cluster_of[n0:n0 + n]] = opnd.pool_w[0][n0:n0 + n]
        c0, c1 = int(opnd.coarse_ptr[gi]), int(opnd.coarse_ptr[gi + 1])
        ap = np.zeros((N, N), np.float32); ap[opnd.coarse_row[c0:c1], opnd.coarse_col[c0:c1]] = opnd.coarse_w[c0:c1]
        k0 = int(opnd.cluster_ptr[gi])
        Pf = np.zeros((N, N), np.float32); Pf[:nc, 0] = opnd.final_w[0][k0:k0 + nc]
        return adj, x, P, ap, Pf, n, nc

    def embed(ops_, marshal):
        adj, x, P, ap, Pf, n, nc = ops_
        cv = (lambda v: torch.Tensor([v])) if marshal else (lambda v: v)
        adj, x, P, ap, Pf = cv(adj), cv(x), cv(P), cv(ap), cv(Pf)
        r = D.wave_readout(x, adj, [ap], [n], [[nc]], [[P], [Pf]], p, num_pool_matrix=1, num_pool_final_matrix=1)
        return D.mlp(r, head)

    def run(as_shipped, seconds):
        pre = None if as_shipped else [tuple(torch.from_numpy(v)[None] if isinstance(v, np.ndarray) else v for v in operands(gi, 0))
                                       for gi in range(12)]
        done, t0, gi = 0, time.perf_counter(), 0
        while True:
            embs = [embed(operands((gi + k) % base.num_graphs, 1000), True) if as_shipped else embed(pre[(gi + k) % 12], False)
                    for k in range(3)]
            dp = torch.nn.functional.pairwise_distance(embs[0], embs[1], 2)
            dn = torch.nn.functional.pairwise_distance(embs[0], embs[2], 2)
            loss = torch.clamp(dp - dn + 1.5, min=0).mean()
            opt.zero_grad(); loss.backward(); opt.step()
            gi += 3; done += 3
            if time.perf_counter() - t0 >= seconds:
                break
        el = time.perf_counter() - t0
        return done / el, done, el
    bs, rs = _best_of_threads(lambda sec: run(True, sec), seconds)
    bm, rm = _best_of_threads(lambda sec: run(False, sec), seconds)
    fmt = lambda res: ", ".join(f"{th} thread(s): {r[0]:.1f} graphs/s ({r[1]} graphs in {r[2]:.1f} s)" for th, r in res.items())
    return {"value": rs[bs][0], "unit": UNIT, "cores": bs, "kind": "port",
            "sample": "as shipped: single-graph fwd+bwd+Adam, B=1, N=1000 padded adjacency / pooling / coarsened operands with the "
                      f"per-graph torch.Tensor([ndarray]) marshaling (oracle/dense_ref.py port); {fmt(rs)}; faster one reported",
            "math_only": {"value": rm[bm][0], "unit": UNIT, "cores": bm,
                          "sample": f"tensors pre-built, tight padding; {fmt(rm)}; faster one reported"}}


# ------------------------------------------------------------------------------------------ our arm
def main():
    a = parse()
    if a.impl == "reference":
        run_reference(a)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: tsg has no CPU path")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    # stdout carries exactly ONE JSON line: keep a private copy of the real stdout for it and point fd 1 at stderr,
    # so nothing else (NCCL's C-level "NCCL version ..." banner, library chatter) can land there
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    # each rank keeps to its own share of the host cores (8 processes on one box otherwise fight over every core
    # with their intra-op pools: the enqueue thread is what matters here)
    ncpu = os.cpu_count() or 1
    if world > 1:
        per = max(1, ncpu // world)
        try:
            os.sched_setaffinity(0, set(range(local_rank * per, min(ncpu, (local_rank + 1) * per))))
        except Exception:
            pass
        torch.set_num_threads(max(1, min(per, 4)))
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from tsg import _lib, nn as tnn, ops
    from tsg.feeder import DeviceCorpus
    from tsg.train import TripletTrainer
    assert _lib.lib.tsg_check_device() == 0, _lib.last_error()
    peaks = load_peaks()
    kt = KernelTimer(dev)

    corpus, batches, compact, id_lists = make_step_batches(a, rank, num_batches=2)
    dev_batches = [dict(x=b["x"].to(dev), edge_index=b["edge_index"].to(dev), node_ptr=b["node_ptr"],
                        triplets=b["triplets"].to(dev)) for b in batches]
    torch.manual_seed(777)
    model = tnn.PackedSAGNet(corpus.num_node_labels, a.nhid, a.final_dim, 0.5, 0.5).to(dev)
    if world > 1:
        for p in model.parameters():
            dist.broadcast(p.data, 0)
    trainer = TripletTrainer(model, lr=5e-4, weight_decay=1e-4, margin=1.5)
    graphs_per_step = 3 * a.triplets

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(steps):
            fn(i)
        e.record()
        barrier()
        ms = torch.tensor([s.elapsed_time(e)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    rate = lambda ms: world * graphs_per_step * a.steps / (ms / 1000.0)
    t = lambda v: (torch.from_numpy(v) if isinstance(v, np.ndarray) else v).to(dev)
    dev_compact = [(ops.CompactBatch(t(c["label"]), t(c["row"]), t(c["col"]), t(c["node_ptr"]), t(c["edge_ptr"]),
                                     corpus.num_node_labels, int(np.diff(c["edge_ptr"]).max()), c["coalesced"]),
                    c["node_ptr"], b["triplets"]) for c, b in zip(compact, dev_batches)]

    def step_wire(i):
        b = dev_batches[i % len(dev_batches)]
        trainer.step(b["x"], b["edge_index"], b["node_ptr"], b["triplets"])

    last_loss = [None]

    def step_resident(i):
        cb, nptr, trip = dev_compact[i % len(dev_compact)]
        last_loss[0] = trainer.step(cb, None, nptr, trip)

    if a.profile_step:
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for i in range(a.warmup + a.steps):
            if i == a.warmup:
                ev[0].record()
            (step_resident if a.profile_step == "compact" else step_wire)(i)
        ev[1].record()
        torch.cuda.synchronize()
        print(f"[profile-step] {a.profile_step}: {ev[0].elapsed_time(ev[1]) / max(a.steps, 1):.4f} ms/step over {a.steps} steps",
              file=sys.stderr)
        os.close(json_fd)
        return

    # ---- device-resident throughput (value): the compact input form resident in HBM
    W = max(a.warmup, 3)
    for i in range(W):
        step_resident(i)
    cvd = [v for v in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if v.strip().isdigit()]
    sampler = ClockSampler(int(cvd[local_rank]) if local_rank < len(cvd) else local_rank)
    sampler.start()
    k0 = _lib.kernel_launches
    ms = timed(step_resident, a.steps)
    launches = _lib.kernel_launches - k0
    clocks = sampler.finish()
    value = rate(ms)
    if a.dump_outputs and rank == 0:
        # before anything else runs the model: gradients and parameters are those of the last timed step
        dump_outputs(a.dump_outputs, last_loss[0], model)

    # ---- the same step on the PyG wire format resident in HBM (fp32 one-hot x, int64 edge_index)
    for i in range(3):
        step_wire(i)
    ms_wire = timed(step_wire, a.steps)

    # ---- end to end (headline): HBM-resident corpus, per step ids + offsets + triplets from the host, batch assembled
    #      on the GPU, loss read back; host-side offset computation, staging and level planning are INSIDE the timed loop
    dcorp = DeviceCorpus(corpus, dev)
    trip_pinned = batches[0]["triplets"]

    def run_ids(steps):
        return trainer.run_from_ids(dcorp, ((id_lists[i % len(id_lists)], trip_pinned) for i in range(steps)))

    run_ids(3)
    ms_e2e = timed(lambda i: run_ids(a.steps) if i == 0 else None, 1)
    ids_h2d = 8 * (graphs_per_step + 2 * (graphs_per_step + 1)) + trip_pinned.numel() * 8 + 4 * 8 * (graphs_per_step + 1)

    # ---- end to end from pre-packed pinned COMPACT host batches (43 MB H2D per step)
    def run_compact(steps):
        return trainer.run_from_host_compact((compact[i % len(compact)] for i in range(steps)), dev, corpus.num_node_labels)

    run_compact(2)
    ms_e2e_host = timed(lambda i: run_compact(a.steps) if i == 0 else None, 1)
    c0 = compact[0]
    h2d_compact = (c0["label"].numel() * 4 + c0["row"].numel() * 8 + c0["triplets"].numel() * 8 + 8 * (3 * (graphs_per_step + 1)))

    # ---- end to end on the PyG wire format from the host (what Batch.to(device) moves): PCIe bound
    def run_wire(steps):
        return trainer.run_from_host((batches[i % len(batches)] for i in range(steps)), dev)

    run_wire(2)
    ms_e2e_wire = timed(lambda i: run_wire(a.steps) if i == 0 else None, 1)
    b0 = batches[0]
    h2d_wire = b0["x"].numel() * 4 + b0["edge_index"].numel() * 8 + b0["triplets"].numel() * 8 + 4 * 8 * (graphs_per_step + 1)

    # ---- N > 1: the all-gather formulation (embeddings of every rank gathered, triplets may cross ranks)
    value_allgather = None
    if world > 1:
        # global triplets, identical on every rank: anchors = every rank's first T graphs, positive / negative drawn from
        # the graphs of ALL ranks by label (seeded), so most of them live on another GPU
        glob_trip = []
        M = graphs_per_step
        for bi in range(len(id_lists)):
            ys = [None] * world
            dist.all_gather_object(ys, corpus.y[id_lists[bi]].astype(np.int64))
            yg = np.concatenate(ys)                                   # label of gathered row r * M + i
            rng = np.random.default_rng(4242 + bi)
            pools = {k: np.nonzero(yg == k)[0] for k in (0, 1)}
            anchors = np.concatenate([r * M + np.arange(a.triplets) for r in range(world)])
            ya = yg[anchors]
            pos = np.array([pools[int(v)][rng.integers(0, len(pools[int(v)]))] for v in ya])
            neg = np.array([pools[1 - int(v)][rng.integers(0, len(pools[1 - int(v)]))] for v in ya])
            glob_trip.append(torch.from_numpy(np.stack([anchors, pos, neg], 1).astype(np.int64)).to(dev))

        def step_allgather(i):
            cb, nptr, _ = dev_compact[i % len(dev_compact)]
            trainer.step_allgather(cb, None, nptr, glob_trip[i % len(glob_trip)])
        for i in range(3):
            step_allgather(i)
        ms_ag = timed(step_allgather, a.steps)
        value_allgather = {"value": rate(ms_ag), "unit": UNIT, "ms_per_step": ms_ag / a.steps,
                           "note": "embeddings [3T, D] of every rank all-gathered (NCCL), global triplet loss evaluated on every "
                                   "rank over triplets whose positives / negatives live on OTHER ranks, gradient all-reduce"}

    # ---- roofline of the dominant kernel: level-1 aggregation (K2 SpMM, F = nhid), timed alone
    b = dev_batches[0]
    N = int(b["node_ptr"][-1]); E = int(b["edge_index"].size(1)); Fh = a.nhid
    csr = ops.build_csr(ops.EdgeList.from_edge_index(b["edge_index"]), N)
    H = torch.randn(N, Fh, device=dev)
    bias = torch.zeros(Fh, device=dev)
    spmm_ms = kt(lambda: ops.spmm_raw(csr.rowptr, csr.colidx, csr.val, H, bias, relu=True))
    nnz = E + N
    alg_bytes = 4 * (N * Fh + N * Fh) + 4 * (N + 1) + 8 * nnz       # SURVEY 8d: H once, Y once, CSR once
    traffic, traffic_src = committed_traffic("r02_spmm_g_traffic.json", ["k2_spmm.cu"])
    roofline = roofline_block(f"k_spmm_g (level-1 GCN aggregation, N={N}, nnz={nnz}, F={Fh})", alg_bytes, spmm_ms, peaks,
                              traffic=traffic)
    roofline["traffic_source"] = traffic_src
    step_bytes = getattr(trainer, "last_step_compulsory_bytes", None)

    # ---- optional per-entry-point breakdown (device time shares; not part of any reported number)
    if a.breakdown and rank == 0:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(10):
            step_resident(i)
        t1 = time.perf_counter()
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        print(f"[breakdown] host enqueue {1e2 * (t1 - t0):.3f} ms/step, drained after {1e3 * (t2 - t1):.3f} ms "
              f"(enqueue ~ step time => launch bound)", file=sys.stderr)
        step_resident(0)
        _lib.profile = {}
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(); step_resident(0); e.record(); torch.cuda.synchronize()
        total = s.elapsed_time(e)
        prof = _lib.profile
        rows = sorted(((sum(x.elapsed_time(y) for x, y in v), k, len(v)) for k, v in prof.items()), reverse=True)
        _lib.profile = None
        print(f"[breakdown] one step {total:.3f} ms", file=sys.stderr)
        for tt, k, n in rows:
            print(f"[breakdown] {k:28s} calls={n:3d} {tt:8.3f} ms  {100 * tt / total:5.1f}%", file=sys.stderr)

    # ---- the other BASELINE configs (rank 0, N = 1) and, at N > 1, config 5 data-parallel on the sharded corpus
    want_cpu = rank == 0 and world == 1 and not a.no_cpu_baseline
    configs = {}
    if world == 1:
        fns = {"1": run_config1, "3": run_config3, "4": run_config4, "5": run_config5}
        for c in [c.strip() for c in a.configs.split(",") if c.strip()]:
            try:
                configs[c] = fns[c](a, dev, kt, peaks, want_cpu)
            except Exception as ex:      # a failing side config must not cost the headline line
                configs[c] = {"error": f"{type(ex).__name__}: {ex}"}
            torch.cuda.empty_cache()
    config5_dp = None
    if world > 1 and "5" in a.configs:
        c5 = Config5(dev, a.corpus5, rank, world)
        for p in c5.model.parameters():
            dist.broadcast(p.data, 0)
        T5 = 1168
        ids5 = [c5.sample(s, T5) for s in range(4)]
        for i in range(3):
            c5.step_from_ids(ids5[i % 4])
        ms5 = timed(lambda i: c5.step_from_ids(ids5[i % 4]), a.config_steps)
        config5_dp = {"value": world * 3 * T5 * a.config_steps / (ms5 / 1e3), "unit": UNIT, "ms_per_step": ms5 / a.config_steps,
                      "corpus_graphs": a.corpus5, "graphs_owned_per_rank": int(c5.owned.shape[0]),
                      "corpus_resident_bytes_per_rank": c5.resident_bytes,
                      "sharding": "graph_id % world", "graphs_per_step_per_gpu": 3 * T5,
                      "note": "EigenGCN (config 5) stage-1 triplet step, data-parallel: each rank holds its shard of the corpus in HBM, "
                              "samples triplets among the graphs it owns, gathers the batch by id on the GPU, one all-reduce per step"}
        del c5

    # ---- CPU baselines (rank 0, N=1 only)
    cpu_baseline = None
    if want_cpu:
        sec = a.cpu_baseline_seconds
        cores = os.cpu_count() or 1
        ref = CpuReference(a)
        best, res = _best_of_threads(lambda s_: ref.rate(s_, 10_000), sec * 0.7)
        bestp, resp = _best_of_threads(lambda s_: ref.rate_packed(s_), sec * 0.3)
        fmt = lambda r: ", ".join(f"{th} thread(s): {v[0]:.1f} graphs/s ({v[1]} graphs in {v[2]:.1f} s)" for th, v in r.items())
        cpu_baseline = {"value": res[best][0], "unit": UNIT, "cores": best, "kind": "port",
                        "sample": "as shipped: three single-graph forwards per triplet (B=1), MarginRankingLoss, backward, Adam step "
                                  f"each; oracle port of the PyG ops under torch CPU; {fmt(res)}; faster one reported",
                        "all_threads": {"value": res[cores][0], "cores": cores}, "one_thread": {"value": res[1][0], "cores": 1},
                        "math_only": {"value": resp[bestp][0], "unit": UNIT, "cores": bestp,
                                      "sample": "the GPU arm's formulation on the CPU: packed batches of 48 graphs (16 triplets), "
                                                f"tensors pre-built; {fmt(resp)}; faster one reported"}}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps,
                "warmup": W, "ms_per_step": ms / a.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": workload_name(a), "graphs_per_step_per_gpu": graphs_per_step,
                           "nodes_per_step": N, "directed_edges_per_step": E,
                           "kernel_timer_l2_policy": "L2 flushed before every timed kernel launch: 256 MB write, then 256 MB read of another buffer",
                           "l2_policy": "inputs larger than L2 where dense (x alone is %.0f MB); 2 alternating batches of different "
                                        "graphs; every step streams ~4 GB of intermediates through the 126 MB L2" % (N * corpus.num_node_labels * 4 / 1e6),
                           "parallelism": f"dp{world}: shard by graph; one all-reduce per step carrying [T_r * grads, T_r * loss, T_r]",
                           "input_form": "value / e2e: node labels + graph-local int32 endpoints (what the dataset stores); "
                                         "value_pyg_wire / e2e_fp32_wire: fp32 one-hot x + int64 edge_index; identical forward results "
                                         "(tests/test_compact_gpu.py)"},
                "e2e": {"value": rate(ms_e2e), "unit": UNIT, "ms_per_step": ms_e2e / a.steps,
                        "h2d_bytes_per_step": int(ids_h2d), "d2h_bytes_per_step": 4,
                        "api": "TripletTrainer.run_from_ids(DeviceCorpus, (graph ids, triplets) per step): corpus resident in HBM; "
                               "per step the host computes packed offsets, uploads ids + offsets + triplets from pinned memory, K0 "
                               "gathers the compact batch on the GPU, step, loss read back; nothing pre-packed or cached"},
                "e2e_host_batches": {"value": rate(ms_e2e_host), "unit": UNIT, "ms_per_step": ms_e2e_host / a.steps,
                                     "h2d_bytes_per_step": int(h2d_compact), "d2h_bytes_per_step": 4,
                                     "api": "TripletTrainer.run_from_host_compact: PRE-PACKED pinned host batches (labels i32, local "
                                            "edge lists i32, offsets, triplets), copy-stream double buffering; host-side batch assembly "
                                            "is outside the timed region"},
                "e2e_fp32_wire": {"value": rate(ms_e2e_wire), "unit": UNIT, "ms_per_step": ms_e2e_wire / a.steps,
                                  "h2d_bytes_per_step": int(h2d_wire), "d2h_bytes_per_step": 4,
                                  "api": "TripletTrainer.run_from_host: pre-packed pinned x[f32 N,89] / edge_index[i64 2,E] / triplets "
                                         "(the tensors PyG's Batch.to(device) moves): PCIe bound"},
                "value_pyg_wire": {"value": rate(ms_wire), "unit": UNIT, "ms_per_step": ms_wire / a.steps,
                                   "note": "device-resident step on fp32 one-hot x + int64 edge_index (round 1's `value`)"},
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
                "cpu_baseline": cpu_baseline, "configs": configs}
        if step_bytes:
            line["step_hbm"] = {"compulsory_bytes_per_step": int(step_bytes),
                                "achieved_gbs": step_bytes / (ms / a.steps * 1e-3) / 1e9,
                                "frac_of_measured_peak": step_bytes / (ms / a.steps * 1e-3) / 1e9 / float(peaks.get("hbm_gbs", 6650.0))}
        if value_allgather:
            line["value_allgather"] = value_allgather
        if config5_dp:
            line["config5_dp"] = config5_dp
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    os.close(json_fd)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
