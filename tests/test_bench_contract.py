"""CPU-side checks of bench.py's output contract (no GPU): the reference arm's JSON line and the clock sampler.

The product arm needs a B200 and is exercised by the driver; what can be pinned here is that the reference arm
(`--impl reference`, which times the reference's C graph builder from oracle/_ref plus the CPU restatement) prints one
JSON line with every key the driver reads, and that the nvidia-smi sampler keeps only rows inside the timed window.
"""
import json
import os
import stat
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    env = dict(os.environ, OMP_NUM_THREADS="4")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["unit"] == "atoms/s" and d["higher_is_better"] is True and d["value"] > 0
    assert "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e2e = d["e2e"]
    assert e2e["value"] == d["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_reference_arm_other_ranks_do_no_work():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    t0 = time.time()
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == "", (out.stdout, out.stderr[-500:])
    assert time.time() - t0 < 120


def test_dump_outputs_keeps_a_fixed_sample_under_the_cap(tmp_path, monkeypatch):
    import numpy as np
    import torch

    sys.path.insert(0, ROOT)
    import importlib

    bench = importlib.import_module("bench")
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 16)
    f = np.arange(3 * 10000, dtype=np.float32).reshape(-1, 3)  # 120 kB of forces, row k = (3k, 3k+1, 3k+2)
    arrays = {"resident_energy": np.float64(-1.5), "energy": torch.tensor(-1.5, dtype=torch.float64),
              "forces": torch.from_numpy(f), "stress": torch.zeros(3, 3), "n": np.arange(4)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    got = {k: np.load(tmp_path / "a" / f"{k}.npy") for k in arrays}
    assert all(v.dtype in (np.float32, np.float64) for v in got.values())
    assert sum(v.nbytes for v in got.values()) <= 1 << 16
    rows = got["forces"]
    assert rows.dtype == np.float32 and 0 < len(rows) < len(f)
    assert np.array_equal(rows, f[(rows[:, 0] / 3).astype(np.int64)]) and np.all(np.diff(rows[:, 0]) > 0)
    assert np.array_equal(rows, np.load(tmp_path / "b" / "forces.npy"))
    assert float(got["energy"]) == -1.5 and got["stress"].shape == (3, 3) and np.array_equal(got["n"], np.arange(4))


def test_clock_sampler_windows(tmp_path, monkeypatch):
    fake = tmp_path / "nvidia-smi"
    fake.write_text("#!/bin/bash\nsleep 0.2\nwhile true; do echo '0, 1965, 1965, 500.1, 0x0, Not Active, Not Active, "
                    "Not Active, Active'; sleep 0.05; done\n")
    fake.chmod(fake.stat().st_mode | stat.S_IEXEC)
    monkeypatch.setenv("PATH", f"{tmp_path}:{os.environ['PATH']}")
    sys.path.insert(0, ROOT)
    import importlib

    bench = importlib.import_module("bench")
    s = bench.ClockSampler(0)
    s.start()
    assert s.rows, "start() must wait for the first row (NVML start-up stays outside the timed region)"
    t0 = time.perf_counter()
    time.sleep(1.0)  # ~20 rows at the 50 ms cadence; generous so that a loaded CI host still sees >= 2
    t1 = time.perf_counter()
    c = s.stop([("timed", t0, t1), ("e2e", t1, t1 + 1)])
    assert c["window"] == "timed" and c["samples"] >= 2
    assert c["sm_mhz"] == 1965.0 and c["sm_max_mhz"] == 1965.0 and c["reasons"] == ["sw_power_cap"]
    # a window that caught nothing falls back to the next one (also under load) and says so
    s = bench.ClockSampler(0)
    s.start()
    t0 = time.perf_counter()
    t2 = time.perf_counter()
    time.sleep(1.0)
    t3 = time.perf_counter()
    c = s.stop([("timed", t0, t0), ("e2e", t2, t3)])
    assert c["window"] == "timed+e2e" and c["samples"] >= 2
