"""bench.py on the GPU: --steps sets the timed steps, and --dump-outputs writes what the timed calls returned."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_are_what_the_timed_view_calls_return(tmp_path):
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "small", "--steps", "2", "--warmup", "1", "--no-cpu",
                        "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])

    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    import mvsim_b200 as mv
    shape, kshape, sigma, degrees, inc, snr = b.WORKLOADS["small"]
    nv = len(degrees)
    # the timed loop ran 2 steps: one fused z pass per view and step; the e2e arm timed 2 steps (per caller when pipelined)
    assert line["steps"] == 2 and line["value"] > 0 and line["stages"]["fft_zfused"]["launches"] == 2 * nv, line["stages"]
    assert line["e2e"]["steps"] == 2 * (line["e2e"]["callers"] if line["e2e"]["mode_key"] == "pipelined" else 1), line["e2e"]
    assert sorted(os.listdir(out)) == sorted([f"acquired_view{v}.npy" for v in range(nv)] + [f"psf_view{v}.npy" for v in range(nv)])
    gt = b.make_ground_truth(shape)
    for v, psf in enumerate(b.make_psfs(kshape, sigma, nv)):
        acq = mv.SimulateMultiViewDataset.simulateView(gt, psf, degrees[v], inc=inc, poissonSNR=snr, rnd=464232194, stream=v)
        got = np.load(out / f"acquired_view{v}.npy")
        assert got.dtype == np.float32 and got.shape == acq.shape
        # the timed steps normalise an already normalised PSF again: intensities may differ by an ulp, which flips a count rarely
        assert np.mean(got == acq) >= 0.999, v
        assert rel_err(np.load(out / f"psf_view{v}.npy"), psf) <= 1e-6


def test_dump_outputs_of_the_slab_workload_is_a_fixed_sample_of_the_convolved_slab(tmp_path):
    runs = []
    for d in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg5small", "--steps", "1", "--warmup", "1",
                            "--dump-outputs", str(tmp_path / d)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        assert os.listdir(tmp_path / d) == ["convolved_slab_rank0.npy"]
        runs.append(np.load(tmp_path / d / "convolved_slab_rank0.npy"))
    # 256x512x512 voxels on one rank: sampled down to the 60 MiB budget, the same voxels and values in both runs
    assert runs[0].dtype == np.float32 and runs[0].shape == ((60 << 20) // 4,)
    assert np.isfinite(runs[0]).all() and runs[0].max() > 0 and np.array_equal(runs[0], runs[1])
