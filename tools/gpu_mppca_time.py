"""Timing and accuracy of MP-PCA denoising on the GPU (batched.mppca_denoise, csrc/met2_mppca.cu) on the 96 x 96 x 60 x 32
ellipsoid phantom masked like the orchestrator: CUDA-event median, FP64 operations counted from the code (with the
Jacobi sweep counts of the NumPy restatement, which is bitwise equal to the kernel, on a fixed sample of voxels), the
restatement's host time per voxel, the MWF error (spline + X2-I) after no denoising, NESMA and MP-PCA on a white phantom
and on the block phantom of tests/test_gpu_spatial.py, and the sigma map against the phantom's per-voxel sigma.  Prints
one JSON line and, given a path as the first argument, writes the record there.  Needs a CUDA device."""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))     # test_gpu_spatial imports met2_oracle
import torch  # noqa: E402

import mppca_oracle as O  # noqa: E402
from multicomponent_t2_toolbox_b200 import batched, pipeline  # noqa: E402
from multicomponent_t2_toolbox_b200.phantom import make_phantom  # noqa: E402
from test_gpu_spatial import block_phantom  # noqa: E402

TE = 10.0 * np.arange(1, 33)
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


def flops_per_voxel(N, M, sweeps, n_signal):
    """FP64 operations of one voxel, counted from mppca_kernel: mean (M adds, 1 division per echo); covariance (per
    sample: N subtractions, N^2 multiply-adds); per Jacobi round: rotation parameters of N indices (<= 12 operations
    each: theta 3, t 5, c 3, s 1, the skip test 2) and, per entry of A (three rotations of 3 operations) and of V (one),
    12 operations on N^2 entries; the trace N adds; MP (8 per component); reconstruction 2 N^2 per signal component."""
    Np = N + (N & 1)
    rounds = (Np - 1) * sweeps
    return (M * N + N) + (M * N + 2 * M * N * N) + N + rounds * (12 * N + 12 * N * N) + 8 * N + 4 * N * n_signal


def mwf_mae(data, mask, truth, region):
    res = {}
    for name in ("None", "NESMA", "MPPCA"):
        d = data
        if name == "NESMA":
            d = batched.nesma_filter(data, mask).cpu().numpy()
        elif name == "MPPCA":
            d = batched.mppca_denoise(data, mask)[0].cpu().numpy()
        vol = pipeline.recon_arrays(d, mask, TE, 1000.0, "X2", "I", "spline", premasked=True)
        res[name] = float(np.abs(vol["MWF"] - truth)[region].mean())
    return res


def main():
    assert torch.cuda.is_available(), "gpu_mppca_time.py needs a CUDA device"
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().split("\n")[0]
    shape = (96, 96, 60)
    ph = make_phantom(shape, seed=2, fa_mode="b1", mask_mode="ellipsoid", backend="gpu")
    host = ph["data"] * ph["mask"][..., None]
    host[host < 0.0] = 0.0
    host = np.ascontiguousarray(host)
    data = torch.as_tensor(host).cuda()
    mask = torch.as_tensor(ph["mask"]).cuda()
    nt = data.shape[3]
    res = {"gpu": q, "shape": list(shape) + [nt], "masked_voxels": int(ph["mask"].sum()), "patch_radius": 2}
    ms = ev_times(lambda: batched.mppca_denoise(data, mask))
    res["mppca_ms_median"] = float(np.median(ms))
    res["mppca_ms_min_max"] = [float(min(ms)), float(max(ms))]
    den, sigma, nsig = batched.mppca_denoise(data, mask)
    nsig_h = nsig.cpu().numpy()
    m = ph["mask"] == 1
    res["n_signal_histogram"] = np.bincount(nsig_h[m].ravel()).tolist()
    # sweeps from the restatement on a fixed sample (bitwise equal to the kernel, so the same sweep counts)
    rng = np.random.default_rng(0)
    centres = np.argwhere(m)
    sample = centres[np.sort(rng.choice(len(centres), 256, replace=False))]
    t0 = time.perf_counter()
    r = O.mppca_batch(host, sample, 2)
    res["numpy_restatement_ms_per_voxel_1core"] = (time.perf_counter() - t0) * 1e3 / len(sample)
    assert np.array_equal(r["out"], den.cpu().numpy()[sample[:, 0], sample[:, 1], sample[:, 2]])
    res["sweeps_mean"] = float(r["sweeps"].mean())
    res["sweeps_max"] = int(r["sweeps"].max())
    res["sweep_cap_reached"] = int(r["capped"].sum())
    fl = flops_per_voxel(nt, 125, res["sweeps_mean"], float(nsig_h[m].mean()))
    res["fp64_flop_per_voxel"] = fl
    res["fp64_flop_total"] = fl * res["masked_voxels"]
    res["achieved_TFLOPs"] = res["fp64_flop_total"] / (res["mppca_ms_median"] * 1e-3) / 1e12
    res["share_of_measured_fp64_peak"] = res["achieved_TFLOPs"] / FP64_PEAK_TFLOPS
    # sigma map against the phantom's sigma = S0 / SNR of the noiseless signal (first echo)
    from multicomponent_t2_toolbox_b200.phantom import epg_signal_batch  # noqa: F401
    small = make_phantom((24, 24, 8), seed=1, fa_mode="b1")
    tr = small["truth"]
    V = tr["mwf"].size
    T1 = np.full(V, 1000.0)
    from multicomponent_t2_toolbox_b200.phantom import epg_signal_batch as epg
    s0 = (tr["mwf"].ravel() * epg(32, 10.0, T1, tr["t2m"].ravel(), tr["fa"].ravel())[:, 0]
          + tr["iewf"].ravel() * epg(32, 10.0, T1, tr["t2ie"].ravel(), tr["fa"].ravel())[:, 0]
          + tr["fwf"].ravel() * epg(32, 10.0, T1, np.full(V, 2000.0), tr["fa"].ravel())[:, 0])
    s0 *= 1000.0 * (1.0 - np.exp(-1.0))
    sig_true = (s0 / tr["snr"].ravel()).reshape(tr["mwf"].shape)
    _, sg, _ = batched.mppca_denoise(small["data"], small["mask"])
    ratio = sg.cpu().numpy() / sig_true
    res["white_phantom_sigma_over_true"] = {"median": float(np.median(ratio)),
                                           "quartiles": [float(np.percentile(ratio, 25)), float(np.percentile(ratio, 75))],
                                           "true_sigma_median": float(np.median(sig_true))}
    res["white_phantom_mwf_mae"] = mwf_mae(small["data"], small["mask"], tr["mwf"], np.ones(tr["mwf"].shape, bool))
    bd, bm, btruth, interior = block_phantom()
    res["block_phantom_mwf_mae_inside_blocks"] = mwf_mae(bd, bm, btruth, interior)
    res["block_phantom_mwf_mae_whole"] = mwf_mae(bd, bm, btruth, np.ones(btruth.shape, bool))
    print(json.dumps(res))
    if out_path:
        with open(out_path, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
