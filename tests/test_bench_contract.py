"""CPU test of bench.py's contract: the reference arm prints exactly one JSON line with the agreed keys."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, LENS_BENCH_CPU_SECONDS="2")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "1", "--streams", "8", "--queries", "2", "--places", "200"],
                         capture_output=True, text=True, env=env, timeout=300)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "query_timesteps_per_sec" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]


def test_config_table_matches_baseline_json():
    """--config k names BASELINE.json configs[k-1]; the default line is config 3 (the largest single-GPU
    configuration), strong-scaled over the ranks; weak-scaled configurations keep their per-GPU size."""
    sys.path.insert(0, ROOT)
    import argparse
    import bench
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert len(base["configs"]) == 5 and sorted(bench.CONFIGS) == [1, 2, 3, 4, 5]
    args = argparse.Namespace(config=3, streams=None, queries=None, places=None, seq_len=None, events=None)
    c1 = bench.resolve(args, world=1)
    assert (c1["places"], c1["streams_per_gpu"], c1["queries"], c1["seq_len"]) == (10000, 65536, 10, 10)
    assert "10k-place" in base["configs"][2] and "64k" in base["configs"][2]
    c8 = bench.resolve(args, world=8)
    assert c8["scaling"] == "strong" and c8["streams_per_gpu"] == 8192 and c8["streams_total"] == 65536
    w = bench.workload_config(c8, 8)
    assert w["workload"].startswith("config3") and w["streams_total"] == 65536 and "model" not in w
    c5 = bench.resolve(args, config=5, world=8)
    assert c5["scaling"] == "weak" and c5["streams_per_gpu"] == 1024 and c5["places"] == 100000
    c4 = bench.resolve(args, config=4, world=8)
    assert c4["events"] == 10 ** 9 and "places" not in c4
    over = argparse.Namespace(config=3, streams=64, queries=None, places=500, seq_len=None, events=None)
    co = bench.resolve(over, world=1)
    assert co["overridden"] and "overridden" in bench.workload_config(co, 1)["workload"]


def test_steps_must_be_positive():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"],
                         capture_output=True, text=True, timeout=120)
    assert res.returncode == 2 and "--steps must be at least 1" in res.stderr


def test_dump_outputs_writes_a_seeded_row_sample_within_budget(tmp_path):
    """--dump-outputs: float32 / float64 files, the same rows of every per-stream array, the byte budget kept,
    the whole array when it fits, and the same sample from call to call."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    g = torch.Generator().manual_seed(0)
    B, Q, P, N = 300, 3, 40, 5
    arrays = dict(S=torch.randint(0, 60, (B, Q, P), generator=g).float(),
                  top_val=torch.rand((B, Q - 1, N), generator=g),
                  top_idx=torch.randint(-1, P, (B, Q - 1, N), generator=g, dtype=torch.int32),
                  hits=torch.tensor([5, 9, 11], dtype=torch.int64), n_valid=torch.tensor([17], dtype=torch.int64))
    budget = 100_000
    per_row = Q * P * 4 + (Q - 1) * N * (4 + 8) + 8
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays, budget=budget)
    got = {n: np.load(tmp_path / "a" / (n + ".npy")) for n in list(arrays) + ["sample_rows"]}
    for n, a in got.items():
        assert np.array_equal(a, np.load(tmp_path / "b" / (n + ".npy"))), n
    assert got["S"].dtype == got["top_val"].dtype == np.float32
    assert got["top_idx"].dtype == got["hits"].dtype == got["sample_rows"].dtype == np.float64
    rows = got["sample_rows"].astype(np.int64)
    assert len(rows) == (budget - 4 * 8) // per_row < B
    assert np.all(np.diff(rows) > 0) and rows[0] >= 0 and rows[-1] < B
    for n in ("S", "top_val", "top_idx"):
        assert np.array_equal(got[n], arrays[n].numpy()[rows]), n
    assert np.array_equal(got["hits"], [5, 9, 11]) and np.array_equal(got["n_valid"], [17])
    assert sum(a.nbytes for a in got.values()) <= budget
    bench.dump_outputs(str(tmp_path / "whole"), arrays)
    assert np.array_equal(np.load(tmp_path / "whole" / "sample_rows.npy"), np.arange(B))
    assert np.array_equal(np.load(tmp_path / "whole" / "S.npy"), arrays["S"].numpy())
