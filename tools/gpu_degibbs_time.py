"""Timing and effect of Gibbs-ringing removal on the GPU (batched.degibbs, csrc/met2_degibbs.cu): CUDA-event medians on
the 96 x 96 x 60 x 32 ellipsoid phantom (masked like the orchestrator) and on a 256 x 256 x 60 x 32 volume, FP64
operations counted from the kernels, the NumPy restatement's time per 96 x 96 slice on one core (bitwise checked
against the device), and the MWF error (spline + X2-I) with and without unringing on the ringing block phantom of
tests/test_gpu_degibbs.py.  Prints one JSON line and, given a path as the first argument, writes the record there.
Needs a CUDA device."""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

import degibbs_oracle as O  # noqa: E402
from multicomponent_t2_toolbox_b200 import batched  # noqa: E402
from multicomponent_t2_toolbox_b200.phantom import make_phantom  # noqa: E402
from test_gpu_degibbs import mwf_mae_with_and_without_degibbs, tables  # noqa: E402

FP64_PEAK_TFLOPS = 34.0     # profiles/r01_fp64_peak_microbench.json (DFMA counted as 2)


def ev_times(fn, reps=11):
    """CUDA-event times (ms) of `reps` calls of fn(), after one warm-up call."""
    fn()
    out = []
    for _ in range(reps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1))
    return out


def flops_per_slice(n0, n1, nsh=O.NSH, minW=O.MINW, maxW=O.MAXW):
    """FP64 operations of one n0 x n1 slice, counted from the kernels (useful work only: the padded positions of the
    last thread row are not counted).  Split: rows of real input 4 per term, complex columns / rows 8 per term, the real
    part 4 per term, G0 4 and v0 / v1 2 per element.  Unringing of a line of length n: 2 per term of the 2 nsh + 1
    convolutions of n terms, the two TVs 4 (maxW - minW + 1) per position and shift, the two convolutions at the chosen
    shift and the interpolation 4 n + 5 per position.  The final sum 1 per element.  The 4 n per position of the
    recomputed convolutions (about 4 % of the total) is work of this implementation, which recomputes y at the chosen
    shift instead of keeping every y_q; the definition itself does not need it."""
    split = 4 * n0 * n1 * n1 + 8 * n1 * n0 * n0 + 4 * n0 * n1 + 8 * n0 * n1 * n1 + 4 * n1 * n0 * n0 + 2 * n0 * n1
    W = maxW - minW + 1
    nq = 2 * nsh + 1

    def unring(n, lines):
        return lines * (nq * (2 * n * n + 4 * W * n) + n * (4 * n + 5))

    return split + unring(n0, n1) + unring(n1, n0) + n0 * n1


def main():
    assert torch.cuda.is_available(), "gpu_degibbs_time.py needs a CUDA device"
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().split("\n")[0]
    res = {"gpu": q, "nsh": O.NSH, "minW": O.MINW, "maxW": O.MAXW, "fp64_peak_TFLOPs_measured_dfma": FP64_PEAK_TFLOPS}
    ph = make_phantom((96, 96, 60), seed=2, fa_mode="b1", mask_mode="ellipsoid", backend="gpu")
    host = ph["data"] * ph["mask"][..., None]
    host[host < 0.0] = 0.0
    host = np.ascontiguousarray(host)
    rng = np.random.default_rng(0)
    vols = {"96x96x60x32": torch.as_tensor(host).cuda(),
            "256x256x60x32": (100.0 + 10.0 * torch.randn(256, 256, 60, 32, dtype=torch.float64,
                                                          generator=torch.Generator().manual_seed(1))).cuda()}
    for name, d in vols.items():
        n0, n1, nz, nt = d.shape
        ms = ev_times(lambda: batched.degibbs(d))
        fl = flops_per_slice(n0, n1) * nz * nt
        med = float(np.median(ms))
        res[name] = {"ms_median": med, "ms_min_max": [float(min(ms)), float(max(ms))], "fp64_flop": fl,
                     "achieved_TFLOPs": fl / (med * 1e-3) / 1e12,
                     "share_of_measured_fp64_dfma_peak": fl / (med * 1e-3) / 1e12 / FP64_PEAK_TFLOPS}
        del d
    out = batched.degibbs(vols["96x96x60x32"]).cpu().numpy()
    z, t = rng.integers(0, 60, 4), rng.integers(0, 32, 4)
    t0 = time.perf_counter()
    ref = O.degibbs(np.ascontiguousarray(host[:, :, z, t]), tables(96), tables(96))
    res["numpy_restatement_s_per_96x96_slice_1core"] = (time.perf_counter() - t0) / 4
    assert np.array_equal(out[:, :, z, t], ref)
    res["ringing_block_phantom_mwf_mae"] = mwf_mae_with_and_without_degibbs()
    print(json.dumps(res))
    if out_path:
        with open(out_path, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
