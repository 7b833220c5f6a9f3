"""Worker of tests/test_gpu_fft_sizes.py for the process-wide knobs (MVSIM_H_MATERIALIZE, MVSIM_NO_TMA are read once per process):
runs the stand-alone sweep of fft_cases.cases() through SimulateMultiViewDataset.convolve and the whole-view call at every z length
of the built range (inc 3 and 5), and writes the outputs to one .npz for the parent to compare with its references."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

import fft_cases  # noqa: E402
import mvsim_b200 as mv  # noqa: E402


def main():
    out_path = sys.argv[1]
    S = mv.SimulateMultiViewDataset
    ctx = mv.Context(0)
    res = {}
    for case in fft_cases.cases():
        vol, psf = case.arrays()
        res["conv_" + case.id] = S.convolve(vol, psf, ctx=ctx)
    for n in fft_cases.whole_view_lengths():
        case = fft_cases.whole_view_case(n)
        vol, psf = case.arrays()
        for inc in (3, 5):
            res[f"view_{case.id}_{inc}"] = S.simulateView(vol, psf.copy(), 0, inc=inc, poissonSNR=-1.0, ctx=ctx, strict_reference=False)
    ctx.close()
    np.savez(out_path, **res)


if __name__ == "__main__":
    main()
