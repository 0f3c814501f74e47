#!/usr/bin/env python
"""fp32-fed vs plane-fed dense GEMM (csrc/dense_gemm.cuh vs csrc/dense_gemm_planes.cuh) at every
GEMM shape the DLRM bench step launches: top MLP 480-1024-1024-512-256 and bottom MLP 512-256-128
at M = 65 536, each as nn (forward), nt (dgrad) and tn (wgrad, split-K as core._wgrad_splits
picks).  The planes are split before the timed region; the split pass (rtf_split_bf16x3) of each
operand is timed on its own.  Both kernels run on the same operands, alternated in rounds of
`--iters` launches between CUDA events (operands > 126 MB L2 for M = 65 536 x K >= 480), and the
median over `--rounds` rounds is reported.  The outputs are checked bit-identical first.

One JSON line per shape and layout, the card's name and power limit in each.

    python tools/time_dense_planes.py [--out profiles/r4_dense_planes.jsonl]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch

import recommend_tf2_b200  # noqa: F401  (loads librtf_b200)
from recommend_tf2_b200 import core

M = 65536
LAYERS = [("top", 480, 1024), ("top", 1024, 1024), ("top", 1024, 512), ("top", 512, 256),
          ("bottom", 512, 256), ("bottom", 256, 128)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.splitlines()
    name, power = [s.strip() for s in q[torch.cuda.current_device()].split(",")]
    return {"gpu": name, "power_limit": power}


def timed(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    info = card()
    rows = []
    for mlp, K, N in LAYERS:
        x = torch.randn(M, K, device="cuda")
        w = torch.randn(K, N, device="cuda") * K ** -0.5
        b = torch.randn(N, device="cuda")
        g = torch.randn(M, N, device="cuda") * 1e-3
        xp, wp, gp = core.split_planes(x), core.split_planes(w), core.split_planes(g)
        splits = core._wgrad_splits(M, K, N)
        cases = {
            "nn": (lambda: core.dense_gemm("nn", x, w, b, True),
                   lambda: core.dense_gemm_planes("nn", xp, wp, b, True), 2.0 * M * K * N),
            "nt": (lambda: core.dense_gemm("nt", g, w),
                   lambda: core.dense_gemm_planes("nt", gp, wp), 2.0 * M * K * N),
            "tn": (lambda: core.dense_gemm("tn", x, g, splits=splits),
                   lambda: core.dense_gemm_planes("tn", xp, gp, splits=splits), 2.0 * M * K * N),
        }
        split_ms = {}
        for name, t in (("x", x), ("g", g)):
            core.split_planes(t)
            split_ms[name] = statistics.median(
                timed(lambda: core.split_planes(t), args.iters) for _ in range(args.rounds))
        for layout, (f32, planes, flop) in cases.items():
            same = torch.equal(f32(), planes())
            for _ in range(2):
                timed(f32, 2), timed(planes, 2)
            t32, tpl = [], []
            for _ in range(args.rounds):
                t32.append(timed(f32, args.iters))
                tpl.append(timed(planes, args.iters))
            m32, mpl = statistics.median(t32), statistics.median(tpl)
            row = dict(info, mlp=mlp, M=M, K=K, N=N, layout=layout,
                       splits=splits if layout == "tn" else 1, bit_identical=same,
                       fp32_fed_ms=round(m32, 4), planes_ms=round(mpl, 4),
                       fp32_fed_ms_runs=[round(v, 4) for v in t32],
                       planes_ms_runs=[round(v, 4) for v in tpl],
                       speedup=round(m32 / mpl, 3),
                       fp32_fed_tflops=round(flop / m32 / 1e9, 1),
                       planes_tflops=round(flop / mpl / 1e9, 1),
                       split_x_ms=round(split_ms["x"], 4), split_g_ms=round(split_ms["g"], 4),
                       split_x_gbs=round(10.0 * M * K / split_ms["x"] / 1e6, 1),
                       split_g_gbs=round(10.0 * M * N / split_ms["g"] / 1e6, 1))
            rows.append(row)
            print(json.dumps(row), flush=True)
        del x, w, g, xp, wp, gp
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
