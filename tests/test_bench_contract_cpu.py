"""bench.py's reference arm (the CPU restatement of the reference op sequence, timed on the host
cores) runs without a GPU and prints the contract's JSON line."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                          "--steps", "1", "--warmup", "1", "--cpu-batch", "256", "--cpu-row-cap", "20000"],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    r = json.loads(lines[0])
    assert r["impl"] == "reference" and r["metric"] == "DLRM train samples/sec"
    assert r["unit"] == "samples/s" and r["higher_is_better"] is True and r["value"] > 0
    assert r["config"]["workload"] == "dlrm_criteo_synthetic" and r["config"]["embed_dim"] == 128
    cb = r["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == r["value"] and cb["sample"]
    assert r["e2e"] == {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0}
    assert r["vs_baseline"] is None and r["dtype"] == "f32" and r["data"] == "synthetic"


def test_b200_arm_refuses_to_run_without_cuda():
    """No CPU fallback: without a CUDA device the product arm exits with an error."""
    import torch
    if torch.cuda.is_available():
        return
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert res.returncode != 0
    assert "no CUDA device" in (res.stderr + res.stdout)


def test_dump_outputs_writes_loss_state_and_sampled_table_rows(tmp_path):
    """--dump-outputs: the loss, every float parameter / buffer as .npy (float64 kept, the rest
    float32), tables above DUMP_TABLE_ROWS rows as a seeded sample of the rows their sparse
    optimizer has updated (all rows without optimizer state), the same files for the same state."""
    import numpy as np
    import torch
    import bench
    from recommend_tf2_b200.embedding import EmbeddingTables, SparseOptimizer

    n = bench.DUMP_TABLE_ROWS + 1000
    m = torch.nn.Module()
    m.emb = EmbeddingTables([n, 50], [4, 4], device="cpu", optimizer=SparseOptimizer("adam"))
    m.plain = EmbeddingTables([n], [4], device="cpu")
    m.dense = torch.nn.Linear(4, 3).double()
    updated = torch.randperm(n)[:3000]
    m.emb.state1[0][updated] = 1e-3
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), torch.tensor(0.25, dtype=torch.bfloat16), m)
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")}
    assert sorted(got) == ["dense.bias", "dense.weight", "emb.weights.0", "emb.weights.0.rows", "emb.weights.1",
                           "loss", "plain.weights.0", "plain.weights.0.rows"]
    assert got["loss"] == 0.25 and got["loss"].dtype == np.float32 and got["dense.weight"].dtype == np.float64
    rows = got["emb.weights.0.rows"].astype(np.int64)
    assert len(rows) == bench.DUMP_ROWS and np.isin(rows, updated.numpy()).all()
    np.testing.assert_array_equal(got["emb.weights.0"], m.emb.weights[0].detach().numpy()[rows])
    np.testing.assert_array_equal(got["emb.weights.1"], m.emb.weights[1].detach().numpy())
    assert len(got["plain.weights.0.rows"]) == bench.DUMP_ROWS
    for f in os.listdir(tmp_path / "a"):
        np.testing.assert_array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))


def _profile_lines():
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r2_bench_*.json"))):
        text = open(path).read().strip()
        try:
            rec = json.loads(text)
        except json.JSONDecodeError:
            rec = json.loads(text.splitlines()[-1])
        yield os.path.basename(path), rec


def test_committed_bench_lines_are_self_consistent():
    """The bench lines committed as evidence under profiles/ carry every key of the contract and
    their derived numbers agree with each other (value = batch / step time, roofline.frac =
    achieved / peak against the measured peak, e2e with its copy sizes, clocks without thermal
    throttling, the multi-GPU lines with a green parity self-check)."""
    seen = 0
    for name, r in _profile_lines():
        seen += 1
        assert r["unit"] == "samples/s" and r["higher_is_better"] is True and r["scaling"] == "weak", name
        assert r["dtype"] == "f32" and r["data"] == "synthetic" and r["vs_baseline"] is None, name
        assert r["config"]["workload"], name
        if r.get("impl") == "reference":
            assert r["cpu_baseline"]["kind"] == "port" and r["config"].get("same_config") is False, name
            continue
        gb = r["config"]["global_batch"]
        assert abs(r["value"] - gb / (r["ms_per_step"] * 1e-3)) <= 1e-3 * r["value"], name
        assert r["steps"] >= 1 and r["warmup"] >= 3 and r["gpu_launches"] > 0, name
        e = r["e2e"]
        assert e["value"] > 0 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0, name
        assert e["value"] != r["value"], name
        rf = r["roofline"]
        if r["n_gpus"] == 1:        # kernel timings are taken on the single-GPU run only
            assert rf["bound"] in ("hbm", "tensor", "fp32_fma") and rf["peak"] > 0, name
            assert abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 2e-3, name
            assert 0 < rf["frac"] < 1.2, name
        bad = {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
        assert not bad & set(r["clocks"]["reasons"]), name
        if r["n_gpus"] > 1:
            pc = r["parity_check"]
            assert pc["ok"] is True and pc["world"] == r["n_gpus"] and pc["max_rel_err"] <= pc["tol"], name
        else:
            assert r["cpu_baseline"]["value"] > 0 and r["cpu_baseline"]["cores"] >= 1, name
    assert seen >= 10
