#!/usr/bin/env python
"""bench.py — DLRM training throughput on synthetic Criteo-shaped data (BASELINE.json configs[1]).

    python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
    python bench.py --impl reference --gpus N ...          # the reference op sequence on host cores

A step = one full training pass of the hot path over one batch: bottom MLP, fused embedding
gather + pairwise-dot interaction (K1+K4), top MLP, Keras BCE, backward (K4 bwd), deterministic
embedding backward with in-place sparse Adam (K2), dense Adam.  Prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# Criteo-Kaggle cardinalities capped at 10 M rows (SURVEY.md §8d)
CRITEO_ROWS = [min(n, 10_000_000) for n in (
    1460, 583, 10131227, 2202608, 305, 24, 12517, 633, 3, 93145, 5683, 8351593, 3194, 27, 14992,
    5461306, 10, 5652, 2173, 4, 7046547, 18, 15, 286181, 105, 142572)]
EMBED_DIM = 128
N_DENSE = 13
BOT_MLP = (512, 256, 128)
TOP_MLP = (1024, 1024, 512, 256)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="dlrm",
                    choices=["dlrm", "fm", "din", "autoint", "sasrec", "youtubednn"],
                    help="dlrm = BASELINE.json's metric config (configs[1], default); the others are "
                         "configs[0], [2], [3], [4] (bench_workloads.py): same contract line each")
    ap.add_argument("--batch", type=int, default=65536, help="samples per GPU per step")
    ap.add_argument("--ids", default="uniform", choices=["uniform", "zipf"])
    ap.add_argument("--cpu-batch", type=int, default=2048)
    ap.add_argument("--cpu-row-cap", type=int, default=1_000_000)
    ap.add_argument("--mlp-gemm", default="bf16x6", choices=["bf16x6", "bf16x9", "native"],
                    help="dense-MLP GEMMs: librtf_b200's tcgen05 GEMM (fp32 split into 3 bf16 terms, 6 "
                         "products, fp32-accurate), cuBLAS 12.9 FP32 emulation (BF16x9), or SGEMM")
    ap.add_argument("--pad-to", type=int, default=8, help="round the interaction width up (479 -> 480)")
    ap.add_argument("--exchange", default="peer", choices=["peer", "p2p", "nccl"],
                    help="multi-GPU row exchange: 'peer' = tables sharded table-wise + row-wise, rows "
                         "pulled / gradients pushed over NVLink inside K4; 'p2p' = table-wise, pooled rows "
                         "pulled from the owners' K1 output; 'nccl' = table-wise, NCCL all-to-all")
    ap.add_argument("--row-wise-min-rows", type=int, default=5_000_000)
    ap.add_argument("--replicate-max-rows", type=int, default=-1,
                    help="peer exchange: tables up to this many rows are replicated on every GPU "
                         "(local lookups, one dense gradient all-reduce); 0 = shard everything; "
                         "-1 = 16384 from 4 GPUs up (at 2 GPUs half the rows are local anyway and "
                         "sharding everything measured 2 %% faster)")
    ap.add_argument("--peer-gather", default="owner", choices=["owner", "direct"],
                    help="peer exchange: rows gathered by their holders (K1) and pulled by sample, or "
                         "pulled straight from the remote table shards")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pipeline", action="store_true",
                    help="multi-GPU: do not hand the next batch's ids to the step (no pipelining of the "
                         "embedding exchange behind the previous step)")
    ap.add_argument("--no-parity-check", action="store_true",
                    help="skip the untimed sharded-vs-single-GPU self-check run before a multi-GPU measurement")
    ap.add_argument("--no-kernel-timing", action="store_true")
    ap.add_argument("--cuda-graph", default="auto", choices=["auto", "on", "off"],
                    help="replay the training step from a CUDA graph (core.StepGraph). auto = on for "
                         "single-GPU dlrm and the launch-bound workloads (fm, din, autoint, youtubednn), "
                         "off for sasrec and for multi-GPU runs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the loss of the last one and the model parameters "
                         "and buffers it left (large embedding tables as a fixed sample of updated rows; "
                         "no optimizer state) to DIR/<name>.npy, so that two builds can be compared "
                         "output for output (single process only)")
    return ap.parse_args()


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


DUMP_ROWS = 512                 # rows kept of a table larger than DUMP_TABLE_ROWS
DUMP_TABLE_ROWS = 4096
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, loss, model):
    """--dump-outputs: `loss` (what the last timed step returned) and the parameters and buffers
    that step left in `model`, one DIR/<name>.npy per float tensor (float64 stays float64, the rest
    is written as float32).  Optimizer state (Adam moments) is not written.  Of a 2-D tensor with
    more than DUMP_TABLE_ROWS rows (an embedding table) only DUMP_ROWS rows are kept, listed in
    DIR/<name>.rows.npy and drawn with a fixed seed among the rows the table's sparse optimizer has
    updated (non-zero first moment), so that they carry what training computed; a table without
    optimizer state is sampled over all its rows."""
    import zlib

    import numpy as np
    import torch
    from recommend_tf2_b200.embedding import EmbeddingTables
    params = dict(model.named_parameters())
    updated = {}
    for mname, mod in model.named_modules():
        if isinstance(mod, EmbeddingTables):
            for i, m1 in enumerate(mod.state1):
                if m1 is not None:
                    updated[f"{mname}.weights.{i}".lstrip(".")] = m1.ne(0).any(1).nonzero()[:, 0]
    if not set(updated) <= set(params):
        raise RuntimeError(f"--dump-outputs: tables {sorted(set(updated) - set(params))} not among the "
                           "model's parameters")
    out = {"loss": loss}
    for name, t in list(params.items()) + list(model.named_buffers()):
        if not t.is_floating_point():
            continue
        if t.dim() == 2 and t.shape[0] > DUMP_TABLE_ROWS:
            rng = np.random.default_rng(zlib.crc32(name.encode()))
            cand = updated[name].cpu().numpy() if len(updated.get(name, ())) else np.arange(t.shape[0])
            rows = np.sort(cand[rng.choice(len(cand), min(DUMP_ROWS, len(cand)), replace=False)])
            rows = torch.from_numpy(rows).long()
            out[name + ".rows"] = rows.double()
            t = t[rows.to(t.device)]
        out[name] = t
    arrays = {k: v.detach().to("cpu", torch.float64 if v.dtype == torch.float64 else torch.float32).numpy()
              for k, v in out.items()}
    nbytes = sum(v.nbytes for v in arrays.values())
    if nbytes > DUMP_MAX_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {nbytes} bytes (limit {DUMP_MAX_BYTES})")
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def make_batches(n, B, rows, ids_kind, seed):
    """Synthetic Criteo-shaped batches in pinned host memory: dense U[0,1) (B,13) f32, sparse
    (B,26) i32 (uniform or Zipf(1.05) mod N_t), labels Bernoulli(0.25)."""
    import numpy as np
    import torch
    from recommend_tf2_b200.data import synthetic_criteo_batch
    rng = np.random.default_rng(seed)
    return [tuple(torch.from_numpy(a) for a in synthetic_criteo_batch(rng, B, rows, ids_kind))
            for _ in range(n)]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms from before the warm-up (the tool
    needs ~0.2 s to start) to the end of the timed region; the summary uses the samples whose
    timestamps fall inside the timed region, or — when the region is shorter than the sampling
    period — all samples taken under load (warm-up + timed), and says which."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc = None
        self.t_load = time.time()
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            pass

    def stop(self, t0=None, t1=None):
        import datetime
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []
        for line in out.splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm_mhz, sm_max = float(parts[1]), float(parts[2])
            except ValueError:
                continue
            try:
                ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except ValueError:
                ts = float("inf")      # unknown format: counts as "under load", never as "inside"
            rows.append((ts, sm_mhz, sm_max,
                         [nm for nm, v in zip(names, parts[4:8]) if v.lower().startswith("active")]))
        inside = [r for r in rows if t0 is not None and t0 <= r[0] <= t1]
        window = "timed region"
        if not inside:
            inside = [r for r in rows if r[0] >= self.t_load + 0.05] or rows
            window = "warm-up + timed region (timed region shorter than the sampling period)"
        sm = [r[1] for r in inside]
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(r[2] for r in inside) if inside else None,
                "reasons": sorted({x for r in inside for x in r[3]}), "samples": len(sm),
                "window": window}


def cpu_reference_run(args, steps, warmup):
    """The reference op sequence on host cores (oracle/dlrm_ref.py), bounded sample."""
    import torch
    from oracle import dlrm_ref
    rows = [min(r, args.cpu_row_cap) for r in CRITEO_ROWS]
    batches = make_batches(warmup + steps, args.cpu_batch, rows, args.ids, seed=1)
    batches = [(d, s, y) for d, s, y in batches]
    sps, threads, sec_step = dlrm_ref.time_cpu_train(rows, EMBED_DIM, BOT_MLP, TOP_MLP, batches,
                                                     warmup=warmup, threads=os.cpu_count())
    sample = (f"{steps} steps x {args.cpu_batch} samples, tables capped at {args.cpu_row_cap} rows "
              f"(host RAM), sparse-row Adam; torch-CPU restatement of the reference op sequence, "
              f"not TensorFlow")
    return {"value": sps, "unit": "samples/s", "cores": threads, "kind": "port", "sample": sample,
            "ms_per_step": sec_step * 1e3}


def bench_config(args, world):
    return {"workload": "dlrm_criteo_synthetic", "tables": len(CRITEO_ROWS),
            "rows_total": sum(CRITEO_ROWS), "embed_dim": EMBED_DIM, "bot_mlp": list(BOT_MLP),
            "top_mlp": list(TOP_MLP), "interaction": "dot", "batch_per_gpu": args.batch,
            "global_batch": args.batch * world, "ids": args.ids,
            "optimizer": "adam (sparse rows fused in K2, dense MLP rtf_dense_adam)",
            "cuda_graph": ("step replayed from one CUDA graph (batch copied into static buffers, Adam "
                           "step size read from a device scalar)"
                           if world == 1 and args.cuda_graph != "off" else "off (eager launches)"),
            "l2_flush": "inputs larger than L2: 17.2 GB of tables, distinct batch every step",
            "parallelism": "single" if world == 1 else
            f"tables sharded over {world} GPUs ({args.exchange} row exchange"
            + (f"/{args.peer_gather} gather, row-wise >= {args.row_wise_min_rows} rows, "
               f"replicated <= {args.replicate_max_rows} rows" if args.exchange == "peer" else "")
            + ") + dp MLP"
            + ("" if (world == 1 or args.no_pipeline) else
               "; exchange of batch n+1 (ids, holder gather, NVLink pull) pipelined behind step n")}


def reference_config(args):
    """The config the CPU arm ACTUALLY runs: same model, a bounded batch and tables capped to fit
    host RAM (the GPU arm's config is repeated under "gpu_arm_config" for the comparison)."""
    rows = [min(r, args.cpu_row_cap) for r in CRITEO_ROWS]
    return {"workload": "dlrm_criteo_synthetic", "tables": len(rows), "rows_total": sum(rows),
            "row_cap": args.cpu_row_cap, "embed_dim": EMBED_DIM, "bot_mlp": list(BOT_MLP),
            "top_mlp": list(TOP_MLP), "interaction": "dot", "batch_per_gpu": args.cpu_batch,
            "global_batch": args.cpu_batch, "ids": args.ids,
            "optimizer": "adam (sparse rows for the tables, dense for the MLP)",
            "parallelism": "host cores, one process", "same_config": False,
            "differs_from_gpu_arm": "batch (bounded sample) and table rows capped at row_cap "
                                    "(host RAM); identical model, dims, id distribution"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    r = cpu_reference_run(args, args.steps, max(args.warmup, 1))
    line = {"metric": "DLRM train samples/sec", "value": r["value"], "unit": "samples/s",
            "impl": "reference", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(reference_config(args), gpu_arm_config=bench_config(args, world)),
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def embed_bwd_launches(rows, n_tables):
    row_bits = max(1, (max(rows) - 1).bit_length())
    table_bits = max(1, n_tables.bit_length())
    total = row_bits + table_bits
    passes = (total + 9) // 10
    return 1 + passes * 5 + 3 + 3   # keys + passes*(hist + 3 scan + scatter) + seg scan + A/B/C


def time_kernels(pkg, model, dev_batches, peaks_gbs):
    """Per-kernel CUDA-event timing of the hot-path launches on the bench's own batches."""
    import torch
    from recommend_tf2_b200 import _lib as L
    ts = model.embed_layers
    F, D = len(ts.weights), EMBED_DIM
    cols = pkg.dot_out_cols(F + 1, D, model.pad_to)
    res = {}

    def timed(fn, n, warm=3):
        for i in range(warm):          # untimed: clocks, caches and lazy inits settle per kernel
            fn(i % n)
        torch.cuda.synchronize()
        evs = []
        for i in range(n):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            # keep the stream busy while the host enqueues, so the events bracket device time
            # only (not the Python/ctypes launch latency of an idle stream)
            torch.cuda._sleep(600_000)
            a.record()
            fn(i)
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        return statistics.median(a.elapsed_time(b) for a, b in evs)

    n = len(dev_batches)
    B = dev_batches[0][1].shape[0]
    dense_rows = [torch.randn(B, D, device="cuda") for _ in range(2)]
    gout = torch.randn(B, cols, device="cuda")
    gemb = torch.randn(B, F * D, device="cuda")
    tables = list(ts.weights)

    # K1 standalone (the "embedding-lookup HBM GB/s" half of the metric)
    out = torch.empty(B, F * D, device="cuda")
    ms = timed(lambda i: pkg.embed_fwd(tables, dev_batches[i][1], "BF", None, out=out), n)
    by = B * F * (4 + D * 4 + D * 4)
    res["embed_fwd_vec(K1)"] = (ms, by)
    # fused K1+K4 forward / backward
    with torch.no_grad():
        ms = timed(lambda i: pkg.embed_dot(ts, dev_batches[i][1], dense_rows[i % 2], pad_to=model.pad_to), n)
    by = B * (F * (4 + D * 4) + D * 4 + cols * 4)
    res["dot_fwd_kernel(K1+K4)"] = (ms, by)
    import ctypes as C
    from recommend_tf2_b200.embedding import _ptr_array
    rows_arr = L.host_array(C.c_int64, [int(t.shape[0]) for t in tables])
    gdense = torch.empty(B, D, device="cuda")

    def bwd(i):
        ids = dev_batches[i][1]
        L.check(L.lib().rtf_embed_dot_bwd(_ptr_array(tables), rows_arr, F, D, ids.data_ptr(), 0, B,
                                          ids.stride(0), ids.stride(1), dense_rows[i % 2].data_ptr(), D,
                                          gout.data_ptr(), cols, gdense.data_ptr(), D, gemb.data_ptr(),
                                          F * D, L.current_stream_ptr()), "rtf_embed_dot_bwd")
    ms = timed(bwd, n)
    by = B * (F * (4 + D * 4) + D * 4 + cols * 4 + D * 4 + F * D * 4)
    res["dot_bwd_kernel(K4 bwd)"] = (ms, by)
    # K2 pipeline with Adam (whole call: keys + radix sort + segments + reduce/update)
    opt = ts.optimizer.struct_for_step(max(ts.optimizer.step, 1))
    uniq = []
    for i in range(n):
        ids = dev_batches[i][1].long()
        keys = ids + (torch.arange(F, device="cuda").view(1, F) << 32)
        uniq.append(int(torch.unique(keys).numel()))

    # K2 as the training step runs it: the id-only half (keys, sort, segments, work items) on the
    # side stream behind the dense MLP, the gradient half = ONE launch (seg_apply) timed here
    prepared = {}

    def k2_prepare(i):
        prepared[i] = ts.prepare_backward(dev_batches[i][1], list(range(F)))
        torch.cuda.current_stream().wait_event(prepared[i]["ev"])

    for i in range(n):
        k2_prepare(i)
    ms = timed(lambda i: ts.apply_prepared(prepared[i], gemb), n)
    by = B * F * D * 4 + statistics.mean(uniq) * 6 * D * 4
    res["seg_apply(K2: segment reduce + sparse Adam)"] = (ms, by)

    def k2(i):      # the whole pipeline on one stream (keys + sort + segments + work items + apply)
        pkg.embed_bwd(ts.wlist(), list(range(F)), dev_batches[i][1], gemb, "BF", None,
                      opt=opt, state1=ts.state1, state2=ts.state2)
    ms = timed(k2, n)
    by = B * F * (4 + D * 4) + statistics.mean(uniq) * 6 * D * 4
    res["embed_bwd(K2 pipeline: keys+sort+segments+apply, 24 launches)"] = (ms, by)
    out = {}
    for k, (ms, by) in res.items():
        gbs = by / (ms * 1e-3) / 1e9
        out[k] = {"ms": round(ms, 4), "algorithmic_bytes": int(by), "gbs": round(gbs, 1),
                  "frac_hbm": round(gbs / peaks_gbs, 4)}
    return out


def time_dense_gemm(pkg, peaks):
    """The dense-MLP GEMM (60 % of the step, SURVEY f2) against ITS roofline: fp32-equivalent
    TFLOP/s of the 65 536 x 1024 x 1024 layer (forward / dgrad / wgrad) over the measured
    sustained bf16 tensor peak divided by 6 — the kernel issues 6 bf16 products per fp32 product."""
    import torch
    from recommend_tf2_b200 import core
    M, N, K = 65536, 1024, 1024
    x = torch.randn(M, K, device="cuda")
    w = torch.randn(K, N, device="cuda") * 0.03
    b = torch.zeros(N, device="cuda")
    g = torch.randn(M, N, device="cuda")
    peak = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0)) / 6.0
    out = {}

    def timed(fn, n=6):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        evs = []
        for _ in range(n):
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a_.record()
            fn()
            b_.record()
            evs.append((a_, b_))
        torch.cuda.synchronize()
        return statistics.median(p.elapsed_time(q) for p, q in evs)

    for name, fn in (("fwd (nn, bias+ReLU)", lambda: core.dense_gemm("nn", x, w, b, True)),
                     ("dgrad (nt)", lambda: core.dense_gemm("nt", g, w)),
                     ("wgrad (tn, split-K)", lambda: core._wgrad(x, g))):
        ms = timed(fn)
        tf = 2.0 * M * N * K / (ms * 1e-3) / 1e12
        out[name] = {"ms": round(ms, 4), "tflops_fp32_equiv": round(tf, 1), "frac": round(tf / peak, 4)}
    worst = min(out.values(), key=lambda v: v["frac"])
    return {"kernel": "rtf_dense_gemm_* (tcgen05 2-SM, fp32 split into 3 bf16 terms, 6 products; CUTLASS "
                      "collective instantiated in csrc/dense_gemm.cuh)",
            "bound": "tensor", "unit": "TFLOP/s", "peak": round(peak, 1),
            "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained / 6 (fp32-equivalent ceiling)",
            "shape": [M, N, K], "achieved": worst["tflops_fp32_equiv"], "frac": worst["frac"],
            "by_layout": out}


def count_own_launches(trainer, batch):
    """Kernels of librtf_b200.so launched by ONE training step on this rank (CUPTI via
    torch.profiler, on an extra untimed step): the hand-written rtf:: kernels and the tcgen05
    dense GEMMs instantiated in csrc/dense_gemm_*.cu.  None if the profiler is unavailable."""
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            trainer.step(*batch)
            torch.cuda.synchronize()
        n = 0
        for ev in prof.events():
            name = ev.name
            # (the GEMM's name may come back mangled: _ZN7cutlass13device_kernelI...FastF32...)
            if "rtf::" in name or "N3rtf" in name or ("device_kernel" in name and "FastF32" in name):
                n += 1
        return n or None
    except Exception:
        return None


CUDA_LIB = "/usr/local/cuda/lib64"


def preload_cublas_fp32_emulation():
    """The dense MLPs either side of the hot path are plain library GEMMs (SURVEY f2).  The
    image's cuBLAS 12.9 can run fp32 GEMMs as 9 BF16 tensor-core products of a 3-way split
    (CUBLAS_COMPUTE_32F_EMULATED_16BFX9) — fp32-accurate (measured error vs fp64 below native
    SGEMM's, tools/probe_cublas_emulation.py) at ~2.4x the SGEMM rate.  torch bundles cuBLAS
    12.8, so the 12.9 libraries are loaded first (same SONAME => torch binds to them) and the
    emulation is switched on through cuBLAS's own environment variable.  Must run before
    `import torch`.  Returns a description for the JSON line."""
    import ctypes
    libs = [os.path.join(CUDA_LIB, n) for n in ("libcublasLt.so.12", "libcublas.so.12")]
    if "torch" in sys.modules or not all(os.path.exists(p) for p in libs):
        return "native fp32 SGEMM (cuBLAS bundled with torch)"
    os.environ["CUBLAS_EMULATE_SINGLE_PRECISION"] = "1"
    for p in libs:
        ctypes.CDLL(p, mode=ctypes.RTLD_GLOBAL)
    return "cuBLAS 12.9 FP32 emulation BF16x9 (fp32-accurate), fp32 in/out"


def run_b200(args):
    gemm_desc = "native fp32 SGEMM (cuBLAS bundled with torch)"
    if args.mlp_gemm == "bf16x9":
        gemm_desc = preload_cublas_fp32_emulation()
    elif args.mlp_gemm == "bf16x6":
        gemm_desc = ("librtf_b200 tcgen05 GEMM: fp32 operands split into 3 bf16 terms, 6 products "
                     "(fp32-accurate, ~2e-7 vs fp64), fp32 in/out; 13-wide first layer and 1-wide "
                     "last layer on cuBLAS SGEMM")
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 path has no CPU fallback "
                         "(use --impl reference for the host baseline)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.backends.cuda.matmul.allow_tf32 = False   # fp32 parity with the reference (1e-5)
    torch.backends.cudnn.allow_tf32 = False
    # the MLP weights come from torch's default CUDA generator, which torch seeds at random in every
    # process: seeded here, runs with the same arguments start from the same model
    torch.manual_seed(1234)

    import recommend_tf2_b200 as pkg
    pkg.lib()
    from recommend_tf2_b200 import core as _core
    _core.set_dense_gemm("bf16x6" if args.mlp_gemm == "bf16x6" else "library")
    peaks, peak_src = load_peaks()

    B = args.batch
    K, W = args.steps, max(args.warmup, 3)
    parity = None
    fc = pkg.criteo_feature_columns(EMBED_DIM, rows=CRITEO_ROWS)
    if world == 1:
        model = pkg.DLRM(fc, BOT_MLP, TOP_MLP, interaction="dot", seed=1234, pad_to=args.pad_to)
        # the step is replayed from one CUDA graph: the GPU is the bound at this batch size, but the
        # host needs 4-5 ms per 7.7 ms step to enqueue it eagerly and measured 8-14 ms on a busy box
        # (the step then runs at the host's pace); a replay costs it ~0.1 ms
        use_graph = args.cuda_graph != "off"
        trainer = pkg.DLRMTrainer(model, lr=1e-3, cuda_graph=use_graph)
    else:
        from recommend_tf2_b200.sharded import (PeerShardedDLRM, ShardedDLRM, ShardedDLRMTrainer,
                                                all_ranks_ok, parity_self_check)
        # untimed: sharded == single-GPU replica on this very world, for the exchange mode measured
        # (row-wise + table-wise + replicated tables forced; plus the all-sharded placement when
        # the measured config replicates nothing)
        if not args.no_parity_check:
            checks = [parity_self_check(args.exchange, args.peer_gather, 70)]
            if args.exchange == "peer" and args.replicate_max_rows == 0:
                checks.append(parity_self_check(args.exchange, args.peer_gather, 0))
            parity = {"world": world, "modes": [m for c in checks for m in c["modes"]],
                      "steps": checks[0]["steps"],
                      "max_rel_err": max(c["max_rel_err"] for c in checks),
                      "max_rel_err_state": max(c["max_rel_err_state"] for c in checks),
                      "tol": 1e-5, "tol_state": 1e-4, "ok": all(c["ok"] for c in checks),
                      "what": "sharded vs single-GPU replica on every rank: predictions + loss (tol), "
                              "table shards, Adam moments, MLP weights after 3 steps (tol_state)"}
        if args.exchange == "peer":
            model, ok = None, True
            try:
                model = PeerShardedDLRM(fc, BOT_MLP, TOP_MLP, seed=1234, pad_to=args.pad_to,
                                        row_wise_min_rows=args.row_wise_min_rows, gather=args.peer_gather,
                                        replicate_max_rows=args.replicate_max_rows)
            except Exception as e:   # no NVLink peer mapping on this box: NCCL all-to-all, table-wise
                sys.stderr.write(f"bench.py: peer exchange unavailable ({e!r}); using --exchange nccl\n")
                ok = False
            if not all_ranks_ok(ok, torch.device("cuda", local_rank)):   # the fallback is collective
                del model
                args.exchange = "nccl"
                model = ShardedDLRM(fc, BOT_MLP, TOP_MLP, seed=1234, pad_to=args.pad_to, exchange="nccl")
        else:
            model = ShardedDLRM(fc, BOT_MLP, TOP_MLP, seed=1234, pad_to=args.pad_to, exchange=args.exchange)
        trainer = ShardedDLRMTrainer(model, lr=1e-3)

    host = make_batches(W + K, B, CRITEO_ROWS, args.ids, seed=1000 + rank)
    host = [tuple(t.pin_memory() for t in b) for b in host]
    dev = [tuple(t.cuda(non_blocking=True) for t in b) for b in host]
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing (value)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    # multi-GPU: the NEXT batch's sparse ids are handed to the step (a prefetching feeder has
    # them): its embedding exchange is pipelined behind the current step (sharded.py prefetch)
    pipelined = world > 1 and not args.no_pipeline
    nxt = (lambda i: {"next_sparse": dev[i + 1][1]} if pipelined and i + 1 < len(dev) else {})
    graphed = world == 1 and trainer.graph is not None
    if graphed:             # the eager steps and the capture happen before the W warm-up steps
        for i in range(4):
            trainer.step(*dev[i % W])
        assert trainer.graph.graph is not None
    for i in range(W):
        trainer.step(*dev[i], **nxt(i))
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_start = time.time()
    e0.record()
    for i in range(W, W + K):
        last_loss = trainer.step(*dev[i], **nxt(i))
    e1.record()
    host_ms = (time.time() - t_start) * 1e3 / K     # host enqueue time (the CPU runs ahead of the GPU)
    barrier()
    t_end = time.time()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop(t_start, t_end) if sampler else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_loss, model)

    # ---- end to end: pinned host batches in, loss out, every step, inside the timed region
    loss_host = torch.zeros(K, dtype=torch.float32).pin_memory()
    for _ in pkg.DeviceFeeder(host[:2]):     # untimed: lets the allocator cache the staging slots
        pass
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    # the public input path: pinned host batches -> DeviceFeeder (copy stream, one step ahead)
    feeder = pkg.DeviceFeeder(host[W:W + K])
    for i, (d, s, y) in enumerate(feeder):
        if pipelined:
            nb = feeder.peek_next()
            loss = trainer.step(d, s, y, next_sparse=None if nb is None else nb[1])
        else:
            loss = trainer.step(d, s, y)
        loss_host[i].copy_(loss, non_blocking=True)
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    model.embed_layers.check_ids()

    t = torch.tensor([ms_total, ms_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e = float(t[0]), float(t[1])
    h2d = sum(x.numel() * x.element_size() for x in host[0])

    if rank == 0:
        kernels = None
        roof = None
        roof_compute = None
        if not args.no_kernel_timing and world == 1:
            kernels = time_kernels(pkg, model, dev[W:W + min(K, 8)], peaks["hbm_gbs"])
            # DRAM traffic per launch: from the committed `ncu --set full` capture of the same
            # kernels on the same workload (profiles/r2_ncu_traffic.json) — NOT measured in this
            # run; the entry names its source so a stale capture is visible
            traffic, tsrc = {}, None
            tpath = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")
            if os.path.exists(tpath) and B == 65536 and args.ids == "uniform":
                with open(tpath) as f:
                    tj = json.load(f)
                traffic = {k: int(v["traffic_bytes"]) for k, v in tj["kernels"].items()}
                tsrc = tj.get("source")
            for k, v in kernels.items():
                v["traffic_bytes_ncu"] = traffic.get(k)
                # DRAM-side rate: tables smaller than L2 (11 of the 26) are served from L2, so the
                # algorithmic rate of a gather can exceed the HBM peak while the DRAM rate does not
                v["dram_gbs_ncu_traffic"] = (round(traffic[k] / (v["ms"] * 1e-3) / 1e9, 1)
                                             if k in traffic else None)
            # the dominant SINGLE kernel of the embedding path inside the training step (K1 alone
            # and the multi-launch K2 pipeline are reported under "kernels" but are not step kernels)
            in_step = {k: v for k, v in kernels.items() if not k.startswith(("embed_fwd_vec", "embed_bwd("))}
            top = max(in_step.items(), key=lambda kv: kv[1]["ms"])
            roof = {"kernel": top[0], "bound": "hbm", "achieved": top[1]["gbs"],
                    "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": top[1]["frac_hbm"],
                    "traffic": traffic.get(top[0]), "traffic_source": tsrc, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": top[1]["algorithmic_bytes"],
                    "ms_per_launch": top[1]["ms"]}
            path_ms = sum(v["ms"] for v in in_step.values())
            path_by = sum(v["algorithmic_bytes"] for v in in_step.values())
            roof["embedding_path_in_step"] = {
                "kernels": list(in_step), "ms": round(path_ms, 4), "algorithmic_bytes": int(path_by),
                "gbs": round(path_by / (path_ms * 1e-3) / 1e9, 1),
                "frac_hbm": round(path_by / (path_ms * 1e-3) / 1e9 / peaks["hbm_gbs"], 4)}
            roof_compute = time_dense_gemm(pkg, peaks)
        cpu = None
        if not args.no_cpu_baseline and world == 1:     # reported on rank 0 at N=1 only
            cpu = cpu_reference_run(args, steps=3, warmup=1)
            cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
        # (one extra step: single-process only — a sharded step is a collective on every rank)
        per_step = count_own_launches(trainer, dev[W]) if world == 1 else None
        if per_step is None:   # profiler unavailable: count from the known launch structure
            if world == 1:     # fused gather+dot fwd, its bwd, K2 pipeline
                per_step = 2 + embed_bwd_launches(CRITEO_ROWS, len(CRITEO_ROWS))
            elif args.exchange == "peer":
                lay = model.layout
                mine = [lay.local_rows(0, t) for t in lay.shard_fields[0]]
                per_step = 2 + (args.peer_gather == "owner") + embed_bwd_launches(mine, max(len(mine), 1))
                if lay.rep_fields:       # replicated tables: local K1 + reduce-only K2
                    rep = [lay.rows[t] for t in lay.rep_fields]
                    per_step += 1 + embed_bwd_launches(rep, len(rep))
            else:
                mine = [CRITEO_ROWS[t] for t in model.layout.slots[0]]
                per_step = 3 + embed_bwd_launches(mine, len(mine))
            if args.mlp_gemm == "bf16x6":
                per_step += 7 * 3          # fwd, dgrad, wgrad of the 7 hidden Dense layers
            per_step += 7 * 2              # fused ReLU-mask + bias-gradient, two stages
        per_step *= world
        line = {"metric": "DLRM train samples/sec", "value": B * world * K / (ms_total * 1e-3),
                "unit": "samples/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": dict(bench_config(args, world), mlp_gemm=gemm_desc,
                               interaction_cols=pkg.dot_out_cols(len(CRITEO_ROWS) + 1, EMBED_DIM, args.pad_to)),
                "clocks": clocks,
                "e2e": {"value": B * world * K / (ms_e2e * 1e-3), "unit": "samples/s",
                        "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                        "ms_per_step": ms_e2e / K},
                "host_enqueue_ms_per_step": round(host_ms, 3),
                "gpu_launches": per_step * K, "roofline": roof, "roofline_compute": roof_compute,
                "kernels": kernels,
                "cpu_baseline": cpu, "final_loss": float(loss_host[-1])}
        if parity is not None:
            line["parity_check"] = parity
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    if parity is not None and not parity["ok"]:
        sys.stderr.write(f"bench.py: multi-GPU parity check FAILED: {parity}\n")
        sys.exit(3)


def run_workload_reference(args):
    """--impl reference for a non-DLRM workload: its CPU port on the host cores."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import bench_workloads as BW
    wl = BW.WORKLOADS[args.workload]()
    r = BW.run_cpu(wl, steps=args.steps, warmup=max(args.warmup, 1))
    cfg = dict(wl.config(), batch_per_gpu=wl.cpu_batch, global_batch=wl.cpu_batch,
               parallelism="host cores, one process", same_config=wl.cpu_batch == wl.batch)
    line = {"metric": wl.metric, "value": r["value"], "unit": "samples/s", "impl": "reference",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": cfg,
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def run_workload(args):
    """A non-DLRM BASELINE config through the same protocol: W warm-up steps, K timed steps on
    device-resident batches (value), K steps from pinned host batches through DeviceFeeder with the
    loss read back every step (e2e), the model's dominant hot-path kernel against its roofline,
    the CPU port beside it.  N > 1 = N independent replicas (these paths do not shard)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    import bench_workloads as BW

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 path has no CPU fallback "
                         "(use --impl reference for the host baseline)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.manual_seed(1234)     # same model from run to run (see run_b200)
    import recommend_tf2_b200 as pkg
    pkg.lib()
    peaks, peak_src = load_peaks()
    wl = BW.WORKLOADS[args.workload]()
    B = wl.batch
    K, W = args.steps, max(args.warmup, 3)
    wl.cuda_graph = wl.graphable and (args.cuda_graph == "on" or
                                      (args.cuda_graph == "auto" and args.workload in GRAPH_AUTO))
    st = wl.build(pkg)
    rng = np.random.default_rng(1000 + rank)
    host = [tuple(torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in wl.host_batch(rng, B))
            for _ in range(W + K)]
    dev = [tuple(t.cuda(non_blocking=True) for t in b) for b in host]
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if wl.cuda_graph:       # the eager steps + the capture happen before the W warm-up steps
        for i in range(4):
            st.step(*dev[i % W])
        assert st.trainer.graph.graph is not None
    sampler = ClockSampler(local_rank) if rank == 0 else None
    for i in range(W):
        st.step(*dev[i])
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_start = time.time()
    e0.record()
    for i in range(W, W + K):
        last_loss = st.step(*dev[i])
    e1.record()
    barrier()
    t_end = time.time()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop(t_start, t_end) if sampler else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_loss, st.model)

    loss_host = torch.zeros(K, dtype=torch.float32).pin_memory()
    for _ in pkg.DeviceFeeder(host[:2]):
        pass
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for i, b in enumerate(pkg.DeviceFeeder(host[W:W + K])):
        loss_host[i].copy_(st.step(*b), non_blocking=True)
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    for ts in st.trainer.tables:
        ts.check_ids()
    t = torch.tensor([ms_total, ms_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e = float(t[0]), float(t[1])
    h2d = sum(x.numel() * x.element_size() for x in host[0])
    if rank == 0:
        roof = None
        if not args.no_kernel_timing:
            roof = wl.roofline(pkg, st, dev[W:W + min(K, 6)], peaks)
            if roof is not None:
                roof.setdefault("peak_source", peak_src)
        cpu = None
        if not args.no_cpu_baseline:
            cpu = BW.run_cpu(wl, steps=3, warmup=1)
            cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
        per_step = count_own_launches(_StepShim(st), dev[W])
        line = {"metric": wl.metric, "value": B * world * K / (ms_total * 1e-3), "unit": "samples/s",
                "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_total / K,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": dict(wl.config(), global_batch=B * world,
                               l2_flush="distinct batch every step over tables larger than L2"
                               if args.workload != "fm" else "distinct batch every step (17 GB-class tables)",
                               parallelism="single" if world == 1 else f"{world} independent replicas "
                               "(this path does not shard)"),
                "clocks": clocks,
                "e2e": {"value": B * world * K / (ms_e2e * 1e-3), "unit": "samples/s",
                        "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / K},
                "gpu_launches": (per_step or 0) * K * world, "roofline": roof, "cpu_baseline": cpu,
                "final_loss": float(loss_host[-1])}
        line["config"]["cuda_graph"] = (
            "step replayed from one CUDA graph (inputs copied into static buffers, Adam step size "
            "read from a device scalar)" if wl.cuda_graph else "off (eager launches)")
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


GRAPH_AUTO = ("fm", "din", "autoint", "youtubednn")


class _StepShim:
    def __init__(self, st):
        self.st = st

    def step(self, *b):
        return self.st.step(*b)


def main():
    args = parse_args()
    if args.dump_outputs and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        raise SystemExit("bench.py: --dump-outputs runs in a single process (--gpus 1)")
    if args.workload != "dlrm":
        return run_workload_reference(args) if args.impl == "reference" else run_workload(args)
    if args.replicate_max_rows < 0:     # same resolved config for both arms
        world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
        args.replicate_max_rows = 16384 if world >= 4 else 0
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
