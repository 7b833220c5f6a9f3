"""Host-side pieces of bench.py that can be checked without a GPU: the nvidia-smi clock sampler (fed by a stand-in
`nvidia-smi` script) and the workload table."""
import importlib.util
import os
import stat
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_clock_sampler_counts_only_samples_of_the_timed_region(tmp_path, monkeypatch):
    fake = tmp_path / "nvidia-smi"
    fake.write_text("#!/bin/bash\nsleep 0.1\nwhile true; do echo '1965, 1965, 450.1, Not Active, Not Active, Not Active, Active'; sleep 0.1; done\n")
    fake.chmod(fake.stat().st_mode | stat.S_IEXEC)
    monkeypatch.setenv("PATH", str(tmp_path) + os.pathsep + os.environ["PATH"])
    b = _bench()
    c = b.ClockSampler(0)
    time.sleep(0.45)                 # "warm-up": samples arrive but must not be counted
    before = len(c.rows)
    c.mark_start()
    time.sleep(0.35)
    r = c.stop()
    assert before >= 2
    assert 1 <= r["samples"] <= 5 and r["samples"] < before + 5
    assert r["sm_mhz"] == 1965.0 and r["reasons"] == ["sw_power_cap"] and "note" not in r
    # a timed region shorter than the sampling period falls back to the last warm-up sample and says so
    c = b.ClockSampler(0)
    time.sleep(0.45)
    c.mark_start()
    r = c.stop()
    assert r["samples"] == 1 and "note" in r


def test_default_workload_is_baseline_config_3():
    b = _bench()
    shape, kshape, _, degrees, inc, snr = b.WORKLOADS["cfg3"]
    assert shape == (512, 1024, 1024) and kshape == (128, 128, 128) and len(degrees) == 6 and inc == 5 and snr == 25.0
    assert b.workload_config("cfg3")["workload"].startswith("BASELINE config 3")


def test_dump_outputs_keeps_small_arrays_and_samples_large_ones_reproducibly(tmp_path, monkeypatch):
    import numpy as np
    b = _bench()
    monkeypatch.setattr(b, "DUMP_BYTES", 4096)          # two arrays: 512 floats each at most
    small = np.arange(4 * 8 * 8, dtype=np.float32).reshape(4, 8, 8)
    large = np.arange(10000, dtype=np.float64).reshape(10, 1000)
    b.dump_outputs(str(tmp_path / "a"), {"small": small, "large": large})
    b.dump_outputs(str(tmp_path / "b"), {"small": small, "large": large})
    assert sorted(os.listdir(tmp_path / "a")) == ["large.npy", "small.npy"]
    s, l_ = np.load(tmp_path / "a" / "small.npy"), np.load(tmp_path / "a" / "large.npy")
    assert s.dtype == l_.dtype == np.float32 and np.array_equal(s, small)
    # the sample is values at sorted distinct flat indices (arange: value == index), the same in every run
    assert l_.shape == (512,) and np.all(np.diff(l_) > 0) and l_[0] >= 0 and l_[-1] < large.size
    assert np.array_equal(l_, np.load(tmp_path / "b" / "large.npy"))
    assert sum(os.path.getsize(p) for p in (tmp_path / "a").iterdir()) <= 4096 + 2 * 128      # + the .npy headers


def test_reference_arm_prints_the_config_it_runs_and_ignores_omp_num_threads():
    """VERDICT r1: the reference arm printed the full-size config while running a sub-volume, and ran on ONE core under
    torchrun (OMP_NUM_THREADS=1).  It now runs the workload it prints, on every processor of the process."""
    import json
    import subprocess
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="2", LOCAL_RANK="0")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "small", "--gpus", "2", "--steps", "5",
                        "--warmup", "3"], capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    b = _bench()
    shape, kshape, _, _, inc, snr = b.WORKLOADS["small"]
    assert line["impl"] == "reference" and line["steps_effective"] == 1
    assert line["config"]["volume_xyz"] == [shape[2], shape[1], shape[0]] and line["config"]["psf_xyz"] == [kshape[2], kshape[1], kshape[0]]
    assert line["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0)) and line["cpu_baseline"]["kind"] == "port"
    assert f"{shape[2]}x{shape[1]}x{shape[0]}" in line["cpu_baseline"]["sample"]
    assert line["value"] == line["e2e"]["value"] == line["cpu_baseline"]["value"] > 0
    # the other ranks print nothing and exit 0
    env["RANK"] = "1"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "small", "--gpus", "2"],
                       capture_output=True, text=True, env=env, timeout=60)
    assert r.returncode == 0 and r.stdout.strip() == ""
