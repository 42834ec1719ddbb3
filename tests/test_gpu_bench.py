"""GPU test of bench.py's own arm: one JSON line with the contract's keys on a small override of config 2."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_line_has_the_contract_keys():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "2", "--streams", "130", "--queries", "3",
                          "--places", "600", "--steps", "2", "--warmup", "3", "--extras", "1", "--cpu-seconds", "1"],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, res.stdout[-2000:]
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "rooflines", "clocks",
              "cpu_baseline", "extras"):
        assert k in d, k
    assert d["metric"] == "query_timesteps_per_sec" and d["value"] > 0 and d["vs_baseline"] is None
    assert d["steps"] == 2 and d["warmup"] == 3 and d["n_gpus"] == 1 and d["gpu_launches"] > 0
    assert "overridden" in d["config"]["workload"] and "model" not in d["config"]
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 130 * 3 * 80 * 80 and e["d2h_bytes_per_step"] > 0
    r = d["roofline"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in r, k
    assert r["bound"] == "tensor" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    kinds = [x["kernel"][:2] for x in d["rooflines"]]
    assert kinds == ["K2", "K3", "K4"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] > 0
    assert d["extras"]["config1_latency"]["us_per_step"] > 0
    assert set(("sm_mhz", "sm_max_mhz", "reasons")) <= set(d["clocks"])


def test_dump_outputs_repeat_and_match_the_oracle(tmp_path):
    """--dump-outputs: two runs with the same arguments write the same arrays, and every stream's top-N lists are
    the oracle's sequence matching + top-N of that stream's dumped spike counts."""
    import numpy as np
    from oracle import oracle as O
    B, Q, P, L = 70, 3, 600, 2
    argv = [sys.executable, os.path.join(ROOT, "bench.py"), "--config", "2", "--streams", str(B), "--queries", str(Q),
            "--places", str(P), "--seq-len", str(L), "--steps", "2", "--warmup", "3", "--no-extras", "--no-cpu-baseline"]
    for run in ("a", "b"):
        res = subprocess.run(argv + ["--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-3000:]
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == ["S.npy", "hits.npy", "n_valid.npy", "overflow.npy", "sample_rows.npy", "top_idx.npy", "top_val.npy"]
    a = {n[:-4]: np.load(tmp_path / "a" / n) for n in names}
    for n, x in a.items():
        assert x.dtype in (np.float32, np.float64) and np.array_equal(x, np.load(tmp_path / "b" / (n + ".npy"))), n
    assert np.array_equal(a["sample_rows"], np.arange(B)) and a["S"].shape == (B, Q, P)
    assert a["overflow"][0] == 0 and 0 < a["n_valid"][0] and np.all(a["hits"] <= a["n_valid"][0])
    for b in range(B):
        idx, val = O.topk(O.seqmatch(a["S"][b], L), 25)
        assert np.array_equal(a["top_idx"][b], idx) and np.array_equal(a["top_val"][b], val), b
