"""bench.py contract (CPU side): the reference arm must print exactly one JSON line on stdout with the keys the
driver reads, on the same metric/unit as our arm, and BASELINE.json's metric must be the one bench.py reports."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    line = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["dtype"] == "f64" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["e2e"]["value"] == line["value"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    sys.path.insert(0, ROOT)
    import bench
    cfg = bench.CONFIGS["metric"]
    assert line["metric"] == bench.metric_name(cfg) and line["unit"] == bench.UNIT
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert "N=300, E=10, H=40, fp64" in base["metric"] and "N=300, E=10, H=40, fp64" in line["metric"]
    assert cfg["N"] == 300 and cfg["Ds"] == 10 and cfg["H"] == 40
    # the driver checks steps x ms_per_step against its own clock: they must be the run's real figures
    assert line["steps"] == 1 and line["ms_per_step"] > 0
    assert abs(line["value"] - line["rollout_steps_per_bench_step"] / (line["ms_per_step"] * 1e-3)) < 1e-6 * line["value"]
    # same workload string as our arm prints for this config
    assert line["config"]["workload"] == bench.workload_string(cfg, cfg["R"])
    # every BASELINE.json config has a bench shape
    assert {"metric", "test_cascade", "inverted_pendulum", "inv_double_pendulum", "smgpr", "swimmer"} <= set(bench.CONFIGS)


def test_dump_outputs_writes_float64_and_samples_above_the_limit(tmp_path, monkeypatch):
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    ids = np.arange(10, 20)
    arrays = {"traj": np.random.RandomState(1).rand(10, 3, 4), "reward": np.arange(10.0)}
    bench.dump_outputs(str(tmp_path / "all"), ids, arrays)
    for name, a in arrays.items():
        got = np.load(tmp_path / "all" / (name + ".npy"))
        assert got.dtype == np.float64 and np.array_equal(got, a)
    assert np.array_equal(np.load(tmp_path / "all" / "restarts.npy"), ids)
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 8 * 13 * 4)            # room for 4 of the 10 restarts
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), ids, arrays)
    rows = np.load(tmp_path / "s1" / "restarts.npy")
    assert len(rows) == 4 and np.array_equal(rows, np.load(tmp_path / "s2" / "restarts.npy"))   # fixed sample
    assert np.array_equal(np.load(tmp_path / "s1" / "reward.npy"), rows - 10)
    assert np.array_equal(np.load(tmp_path / "s1" / "traj.npy"), arrays["traj"][(rows - 10).astype(int)])
    assert sum(f.stat().st_size for f in (tmp_path / "s1").iterdir()) < 2 * 8 * 13 * 4 + 3 * 256   # + .npy headers
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode != 0 and "--dump-outputs" in out.stderr
