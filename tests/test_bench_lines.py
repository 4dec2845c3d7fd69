"""The bench contract, checked on CPU against the lines committed under profiles/ (what `bench.py` printed on B200s):
every key the driver reads is there, and the numbers that are functions of each other agree."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROFILES = os.path.join(ROOT, "profiles")
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "roofline", "e2e", "gpu_launches", "clocks"}


def _load(name):
    with open(os.path.join(PROFILES, name)) as f:
        return json.loads(f.read().strip().splitlines()[-1])


@pytest.mark.parametrize("name,gpus", [("r2_bench_1gpu.json", 1), ("r2_bench_2gpu.json", 2), ("r2_bench_8gpu.json", 8)])
def test_committed_bench_line_follows_the_contract(name, gpus):
    d = _load(name)
    assert BASE_KEYS <= set(d), BASE_KEYS - set(d)
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert base["metric"].startswith("drone-substeps/sec")         # the headline metric of BASELINE.json ...
    assert d["metric"] == "drone_substeps_per_sec" and d["unit"] == "drone-substeps/s"   # ... under this name and unit
    assert d["n_gpus"] == gpus and d["scaling"] == "weak" and d["higher_is_better"] is True and d["data"] == "synthetic"
    assert d["vs_baseline"] is None                       # BASELINE.md publishes no number for this metric
    cfg = d["config"]
    assert "workload" in cfg and "model" not in cfg
    # value = units all ranks processed / max-over-ranks time
    units = gpus * cfg["envs_per_gpu"] * cfg["drones_per_env"] * cfg["substeps_per_step"]
    assert d["value"] == pytest.approx(units / (d["ms_per_step"] * 1e-3), rel=1e-6)
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s"
    assert r["frac"] == pytest.approx(r["achieved"] / r["peak"], rel=1e-9)
    assert 0.5 < r["frac"] < 1.0
    assert r["achieved"] == pytest.approx(r["algorithmic_bytes_per_launch"] / (d["ms_per_step"] * 1e-3) / 1e9, rel=1e-3)
    assert "traffic_source" in r                          # the static ncu figure is labelled as such
    e = d["e2e"]
    assert e["unit"] == d["unit"] and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0
    assert e["value"] < d["value"]                        # host copies inside the timed region
    assert d["gpu_launches"] >= d["steps"]
    c = d["clocks"]
    assert c["sm_mhz"] > 0.9 * c["sm_max_mhz"]
    assert not ({"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(c["reasons"]))
    if gpus == 1:
        cb = d["cpu_baseline"]
        assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] > 0 and "sample" in cb
    m = d["mappo"]
    assert m["train_step_ms"] == pytest.approx(m["rollout_ms"] + m["returns_ms"] + m["update_ms"], rel=0.05)
    if gpus > 1:                                          # the trainer's collective is this library's own kernel
        assert m["gradient_allreduce_impl"].startswith("peer-memory kernel")
        assert m["collectives_per_train_step"]["kl_pair_allreduce"] == 0
        assert m["gradient_allreduce_us"] < m["nccl_same_sizes_us"]


def test_committed_reference_arm_line():
    d = _load("r2_bench_reference.json")
    assert d["impl"] == "reference" and d["dtype"] == "f64"
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["kind"] == "port"
    ours = _load("r2_bench_1gpu.json")
    assert d["metric"] == ours["metric"] and d["unit"] == ours["unit"] and d["higher_is_better"] == ours["higher_is_better"]


def test_bench_cli_defaults():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--dump-outputs"):
        assert flag in out.stdout


def test_bench_rejects_a_run_without_timed_steps():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                         timeout=120)
    assert out.returncode == 2 and "--steps must be at least 1" in out.stderr


def test_dumped_outputs_are_a_fixed_sample_under_64_mb(tmp_path):
    import bench
    N, M, D = 65536, 4, 72                                   # the default workload: obs (N, M, D), three (N,) arrays
    rows = bench.dump_rows(N, M * D + 3)
    assert np.array_equal(rows, bench.dump_rows(N, M * D + 3))
    assert np.all(np.diff(rows) > 0) and rows[0] >= 0 and rows[-1] < N and len(rows) > N // 2
    assert np.array_equal(bench.dump_rows(1000, M * D + 3), np.arange(1000))
    n = len(rows)
    bench.write_outputs(str(tmp_path / "out"), {"obs": np.zeros((n, M, D), np.float32), "reward": np.zeros(n, np.float32),
                                                "terminated": np.zeros(n, np.float32), "truncated": np.zeros(n, np.float32)})
    files = sorted(os.listdir(tmp_path / "out"))
    assert files == ["obs.npy", "reward.npy", "terminated.npy", "truncated.npy"]
    assert sum(os.path.getsize(tmp_path / "out" / f) for f in files) <= 64_000_000
