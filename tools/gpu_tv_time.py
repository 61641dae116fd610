"""Timing of Step 1 with --denoise TV on the GPU (batched.noise_sigma, batched.tv_denoise) on the 96 x 96 x 60 x 32
phantom masked like the orchestrator, with the NumPy restatement's time per iteration on the host beside it.  Prints
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
import torch  # noqa: E402

import tv_oracle as T  # noqa: E402
from multicomponent_t2_toolbox_b200 import batched  # noqa: E402
from multicomponent_t2_toolbox_b200.phantom import make_phantom  # noqa: E402


def ev_time(fn, reps=5):
    """Best of `reps` CUDA-event timings (ms) of fn(), after one warm-up call."""
    fn()
    best = 1e30
    for _ in range(reps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return r, best


def main():
    assert torch.cuda.is_available(), "gpu_tv_time.py needs a CUDA device"
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().split("\n")[0]
    shape = (96, 96, 60)
    ph = make_phantom(shape, seed=2, fa_mode="b1", mask_mode="ellipsoid", backend="gpu")
    host = ph["data"] * ph["mask"][..., None]
    host[host < 0.0] = 0.0
    data = torch.as_tensor(np.ascontiguousarray(host)).cuda()
    nt = data.shape[3]
    N = int(np.prod(shape))
    res = {"gpu": q, "shape": list(shape) + [nt]}
    sigma, ms = ev_time(lambda: batched.noise_sigma(data))
    res["noise_sigma_ms"] = ms
    w = 2.0 * sigma
    (den, iters), ms = ev_time(lambda: batched.tv_denoise(data, weight=w))
    res["tv_denoise_ms"] = ms
    (_, _), ms_all = ev_time(lambda: batched.tv_denoise(data))
    res["tv_denoise_with_sigma_ms"] = ms_all
    it = iters.cpu().numpy()
    res["iterations_per_echo"] = it.tolist()
    res["echo_iterations_total"] = int(it.sum())
    # bytes per voxel and echo-iteration the kernels move, counted from the code: (a) image, p (nd = 3), out, d^2;
    # (b) out, p read + written, |g|; partial sums: d^2 and |g| read again.  Neighbour reads are counted once.
    per_voxel = 8 * ((1 + 3 + 1 + 1) + (1 + 3 + 3 + 1) + 2)
    res["bytes_per_echo_iteration"] = per_voxel * N
    res["bytes_per_iteration_all_echoes"] = per_voxel * N * nt
    res["bytes_total"] = per_voxel * N * int(it.sum())
    res["achieved_TBps"] = res["bytes_total"] / (ms * 1e-3) / 1e12
    res["ms_per_echo_iteration"] = ms / float(it.sum())
    # host: the restatement on echo 0, single core, a few iterations
    vol = host[..., 0]
    wt = float(w[0].cpu())
    t0 = time.perf_counter()
    T.denoise_tv_chambolle(vol, wt, max_num_iter=5)
    res["numpy_restatement_ms_per_iteration_1core"] = (time.perf_counter() - t0) * 1e3 / 5
    res["numpy_restatement_estimated_s_for_this_volume"] = res["numpy_restatement_ms_per_iteration_1core"] * it.sum() / 1e3
    print(json.dumps(res))
    if out_path:
        with open(out_path, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
