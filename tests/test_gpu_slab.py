"""Largest-single-volume path on the GPU: SlabConvolution against the plain convolution (one GPU), overlap-save
y blocks at real size, and -- when the box has >= 2 GPUs -- the NCCL all-to-all run under torchrun."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import gaussian_psf, rel_err

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def mv():
    import mvsim_b200
    return mvsim_b200


def _slab_single(mv, vol, psf):
    import torch
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        ctx = mv.Context(0, cuda_stream=stream.cuda_stream)
        sc = mv.SlabConvolution(ctx, vol.shape, psf.shape)
        img = torch.from_numpy(vol).cuda()
        k = torch.from_numpy(psf).cuda()
        out = torch.empty_like(img)
        sc.convolve(img, k, out)
        stream.synchronize()
        res = out.cpu().numpy()
        nb = sc.y_blocks
        sc.close()
        ctx.close()
    return res, nb


def test_slab_plan_on_one_gpu_equals_plain_convolution(mv, oracle):
    rng = np.random.default_rng(21)
    vol = rng.random((24, 40, 56), dtype=np.float32)
    psf = rng.random((5, 7, 9), dtype=np.float32)
    oracle.norm_image(psf)
    got, nb = _slab_single(mv, vol, psf)
    ref = mv.SimulateMultiViewDataset.convolve(vol, psf.copy())
    assert nb == 1 and np.array_equal(got, ref)
    assert rel_err(got, oracle.convolve(vol, psf.copy(), "direct")) <= 1e-5


def test_y_lines_beyond_the_size_table_use_overlap_save_blocks(mv):
    # Y + KY - 1 = 1720 > 1600: two blocks; sparse kernel so the expected value is a 3-tap sum
    rng = np.random.default_rng(22)
    vol = rng.random((6, 1700, 24), dtype=np.float32)
    psf = np.zeros((3, 21, 5), dtype=np.float32)
    taps = [((0, 0, 0), 0.5), ((2, 20, 4), 0.3), ((1, 10, 2), 0.2)]
    for t, w in taps:
        psf[t] = w
    got, nb = _slab_single(mv, vol, psf)
    assert nb == 2
    plain = mv.SimulateMultiViewDataset.convolve(vol, psf.copy())
    assert rel_err(plain, got) <= 1e-6

    def mir(i, n):
        p = 2 * (n - 1); j = i % p
        return p - j if j >= n else j
    for (z, y, x) in [(0, 0, 0), (5, 1699, 23), (3, 849, 11), (3, 850, 11), (3, 851, 12), (2, 1690, 1)]:
        exp = sum(w * vol[mir(z - (t[0] - 1), 6), mir(y - (t[1] - 10), 1700), mir(x - (t[2] - 2), 24)] for t, w in taps)
        assert got[z, y, x] == pytest.approx(exp, rel=2e-5)


def _run_slab_workers(tmp_path, mode, world, shared, shape="32x72x118", kshape="9x7x11"):
    out = tmp_path / f"slab_{mode}_{world}_{int(shared)}.json"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(29700 + (os.getpid() + world + 7 * shared + 3 * (mode == "p2p")) % 200), os.path.join(HERE, "slab_worker.py"),
           shape, kshape, str(out), mode, "shared" if shared else "own"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(out.read_text())


@pytest.mark.parametrize("world", [2, 4])
@pytest.mark.parametrize("mode", ["p2p", "nccl"])
def test_multi_rank_slab_convolution_on_one_shared_gpu(tmp_path, mode, world):
    """The decomposed path on the 1-GPU box: `world` processes share GPU 0.  p2p: the peers' exchange buffers are mapped with
    CUDA IPC and the y / z kernels store straight into them (the product's default mode, same kernels as over NVLink);
    nccl: the all-to-all layout, staged through host memory by gloo because NCCL refuses two ranks on one device.  The
    result must be bit-identical to the undecomposed convolution (reference convolve, S/SimulateMultiViewDataset.java:253-264)."""
    d = _run_slab_workers(tmp_path, mode, world, shared=True)
    assert d["world"] == world and d["p2p"] == (mode == "p2p") and d["shared_gpu"] and d["identical"], d


def test_multi_rank_slab_convolution_with_overlap_save_blocks_on_one_shared_gpu(tmp_path):
    """y lines beyond the size table (1700 + 21 - 1 > 1600): two overlap-save blocks, two buffer sets in flight."""
    d = _run_slab_workers(tmp_path, "p2p", 2, shared=True, shape="8x1700x56", kshape="3x21x5")      # X + KX - 1 = 60 -> 32 complex columns = 4 kx tiles
    assert d["y_blocks"] == 2 and d["identical"], d


@pytest.mark.parametrize("mode", ["p2p", "nccl"])
def test_slab_convolution_with_one_kx_tile_per_rank_matches_single_gpu(tmp_path, mode):
    """Four ranks and four kx tiles (X + KX - 1 = 62 -> 32 complex columns): every rank owns exactly one tile of the z pass.  On a
    machine with four GPUs every rank has its own (p2p: exchanges fused into the kernels as NVLink peer stores; nccl: two
    all_to_all_single per y block); with fewer the ranks share GPU 0 (CUDA IPC; NCCL's layout staged through gloo).  The result
    must be bit-identical to the undecomposed convolution."""
    import torch
    shared = torch.cuda.device_count() < 4
    d = _run_slab_workers(tmp_path, mode, 4, shared=shared, shape="40x56x52", kshape="9x7x11")
    assert d["world"] == 4 and d["p2p"] == (mode == "p2p") and d["shared_gpu"] == shared and d["identical"], d


@pytest.mark.parametrize("world,inc", [(2, 3), (4, 5)])
def test_whole_view_of_a_slab_decomposed_volume_equals_the_undecomposed_view(tmp_path, world, inc):
    """SlabView on `world` ranks sharing GPU 0: rotate + attenuate per slab on the whole ground truth, decomposed convolution,
    adjustImage with an all-gather of the per-rank sums (S/Tools.java:143-147), extractSlices + Poisson keyed by global voxel
    indices -- against mvsim_simulate_view of the same volume (loop body S/SimulateMultiViewDataset.java:570-585)."""
    out = tmp_path / f"view_{world}.json"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(29900 + (os.getpid() + world) % 90), os.path.join(HERE, "slab_view_worker.py"), "40x56x52", "9x7x11", str(out),      # X + KX - 1 = 62 -> 32 complex columns = 4 kx tiles
           str(inc), "shared"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads(out.read_text())
    assert d["world"] == world and d["clean"]["shape_ok"] and d["noisy"]["shape_ok"]
    assert d["clean"]["conv_max_rel_err"] <= 1e-6 and d["clean"]["max_rel_err"] <= 1e-6, d
    # the Poisson draw of a voxel depends on (seed, stream, GLOBAL voxel index) only; the intensities agree to ~1 ulp, so all but a
    # handful of counts are identical
    assert d["noisy"]["identical_fraction"] >= 0.999, d
