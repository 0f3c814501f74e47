#!/usr/bin/env python
"""Cost of the evaluation features on the bench's DLRM (Criteo cardinalities capped at 10 M rows,
D = 128, B = 65 536): one JSON line per measurement, the card's name and power limit in each.

  * rtf_auc_update alone (CUDA events over 200 back-to-back launches after warm-up) at
    n = 65 536 and 4 194 304, uniform predictions and predictions clustered in two buckets;
    GB/s at 8 B per element against the B200's 7.7 TB/s.  The 4 194 304 case cycles through 8
    input pairs (256 MB > the 126 MB L2) so each launch reads from HBM.
  * the DLRM training step (CUDA-graph replay, as bench.py) without and with metrics=[AUC()],
    two graphs of the same trainer, alternated, 3 runs each.
  * DLRMTrainer.evaluate throughput, eager and with cuda_graph=True, alternated, 3 runs each.

    python tools/time_eval.py [--out FILE.jsonl]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch

import bench
import recommend_tf2_b200 as pkg
from recommend_tf2_b200 import _lib as L
from recommend_tf2_b200.core import StepGraph

HBM_GBS = 7700.0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.splitlines()
    name, power = [s.strip() for s in q[torch.cuda.current_device()].split(",")]
    return {"gpu": name, "power_limit": power}


def time_auc_update(n, kind, iters=200):
    bufs = 8 if n * 8 * 8 > 126e6 else 1
    g = torch.Generator(device="cuda").manual_seed(n)
    ps, ys = [], []
    for _ in range(bufs):
        if kind == "uniform":
            p = torch.rand(n, device="cuda", generator=g)
        else:       # a trained model near its base rate: two buckets
            p = torch.where(torch.rand(n, device="cuda", generator=g) < 0.7, 0.03, 0.04)
        ps.append(p.float())
        ys.append((torch.rand(n, device="cuda", generator=g) < 0.25).float())
    m = pkg.metrics.AUC()
    m.build("cuda")
    fn, st = L.lib().rtf_auc_update, L.current_stream_ptr()
    args = [(p.data_ptr(), y.data_ptr(), n, 200, m.counts.data_ptr(), m.err.data_ptr(), st)
            for p, y in zip(ps, ys)]
    for i in range(10):
        L.check(fn(*args[i % bufs]), "rtf_auc_update")
    torch.cuda.synchronize()
    per = []
    for _ in range(3):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(20_000_000)        # the host enqueues every launch before the first runs
        a.record()
        for i in range(iters):
            fn(*args[i % bufs])
        b.record()
        torch.cuda.synchronize()
        per.append(a.elapsed_time(b) / iters)
    m.check()
    us = statistics.median(per) * 1e3
    gbs = 8.0 * n / (us * 1e-6) / 1e9
    return {"what": "rtf_auc_update", "n": n, "preds": kind, "T": 200, "launches": iters,
            "us_per_call": round(us, 3), "us_runs": [round(x * 1e3, 3) for x in per],
            "GBps": round(gbs, 1), "frac_hbm_7700": round(gbs / HBM_GBS, 3),
            "source": "HBM (8 input pairs cycled)" if bufs > 1 else "L2-resident input"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--eval-batches", type=int, default=16)
    a = ap.parse_args()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(1234)
    info = card()
    lines = []

    def emit(d):
        d.update(info)
        lines.append(d)
        print(json.dumps(d), flush=True)

    for n in (65536, 4194304):
        for kind in ("uniform", "clustered"):
            emit(time_auc_update(n, kind))

    B = a.batch
    fc = pkg.criteo_feature_columns(bench.EMBED_DIM, rows=bench.CRITEO_ROWS)
    model = pkg.DLRM(fc, bench.BOT_MLP, bench.TOP_MLP, interaction="dot", seed=1234)
    tr = pkg.DLRMTrainer(model, lr=1e-3, cuda_graph=True)
    host = bench.make_batches(a.steps + a.eval_batches, B, bench.CRITEO_ROWS, "uniform", seed=1000)
    dev = [tuple(t.cuda() for t in b) for b in host]
    train, ev = dev[:a.steps], dev[a.steps:]

    # two graphs of one trainer: captured without and with the metric update in the step body
    auc = pkg.metrics.AUC()
    graphs = {}
    for label, metrics in (("no_metrics", []), ("auc", [auc])):
        tr.metrics = metrics
        tr.graph = StepGraph(tr._body, tr._advance)
        for i in range(5):
            tr.step(*train[i])
        graphs[label] = tr.graph
    runs = {k: [] for k in graphs}
    for _ in range(3):
        for label, g in graphs.items():
            tr.graph = g
            for i in range(3):
                tr.step(*train[i])
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for b in train:
                tr.step(*b)
            e1.record()
            torch.cuda.synchronize()
            runs[label].append(e0.elapsed_time(e1) / len(train))
    for label, ms in runs.items():
        emit({"what": "DLRM train step (CUDA-graph replay)", "metrics": label, "batch": B,
              "steps_per_run": len(train), "ms_runs": [round(x, 3) for x in ms],
              "ms_median": round(statistics.median(ms), 3)})
    auc.check()

    # evaluate: eager and graph evaluators of the same trainer, alternated
    tr.metrics = [pkg.metrics.AUC()]
    evaluators = {}
    for graph in (False, True):
        tr.cuda_graph, tr._evaluator = graph, None
        tr.evaluate(ev)                          # warm-up (and the capture)
        evaluators[graph] = tr._evaluator
    res = {False: [], True: []}
    out = {}
    for _ in range(3):
        for graph, e in evaluators.items():
            tr._evaluator = e
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out[graph] = tr.evaluate(ev)         # ends with a host sync
            res[graph].append(len(ev) * B / (time.perf_counter() - t0))
    assert out[False] == out[True], (out[False], out[True])
    for graph, sps in res.items():
        emit({"what": "DLRMTrainer.evaluate", "cuda_graph": graph, "batch": B,
              "batches_per_run": len(ev), "samples_per_s_runs": [round(x) for x in sps],
              "samples_per_s_median": round(statistics.median(sps)), "result": out[graph]})

    if a.out:
        with open(a.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
