"""Timing of the three-pool parametric fit (Met2Plan.param_fit) on the config-2 phantom (96 x 96 x 60 x 32, 552 960
voxels, spline FA + X2-I point fit, seeded): CUDA-event times of the point fit and of param_fit (median of 7 after a
warm-up), the iteration histogram, the share of voxels at max_iter and at a bound, and the MWF errors of
tests/test_gpu_param.py's phantom.  Prints one JSON line and, given a path as the first argument, writes the record
there.  Needs a CUDA device."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

from multicomponent_t2_toolbox_b200 import batched, pipeline  # noqa: E402
from multicomponent_t2_toolbox_b200.phantom import make_phantom  # noqa: E402
from test_gpu_param import phantom_mae  # noqa: E402


def event():
    e = torch.cuda.Event(enable_timing=True)
    e.record()
    return e


def main():
    assert torch.cuda.is_available(), "gpu_param_time.py needs a CUDA device"
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().split("\n")
    res = {"gpus": q, "volume": "config-2 phantom 96x96x60x32, seed 2, b1 FA, full mask",
           "method": "spline FA + X2-I point fit, then param_fit", "settings": batched.PARAM_DEFAULTS}
    ph = make_phantom((96, 96, 60), seed=2, fa_mode="b1", backend="gpu")
    _, sig_h = pipeline.masked_voxel_list(ph["data"], ph["mask"])
    res["voxels"] = int(sig_h.shape[0])
    plan = batched.Met2Plan(32, 10.0, 1000.0, reg_method="X2", reg_matrix="I", FA_method="spline")
    sig = torch.as_tensor(sig_h).cuda()
    fa, t2 = plan.fit(sig[:4096])                                  # warm-up
    plan.param_fit(sig[:4096], fa["fa_deg"], t2["fsol"], t2["status"])
    torch.cuda.synchronize()
    point, param = [], []
    for _ in range(7):
        e0 = event()
        fa, t2 = plan.fit(sig)
        e1 = event()
        pf = plan.param_fit(sig, fa["fa_deg"], t2["fsol"], t2["status"])
        e2 = event()
        torch.cuda.synchronize()
        point.append(e0.elapsed_time(e1))
        param.append(e1.elapsed_time(e2))
    res["point_fit_ms"] = point
    res["param_fit_ms"] = param
    res["point_fit_ms_median"] = float(np.median(point))
    res["param_fit_ms_median"] = float(np.median(param))
    res["param_over_point"] = res["param_fit_ms_median"] / res["point_fit_ms_median"]
    st = pf["status"].cpu().numpy()
    it = pf["iters"].cpu().numpy()
    fitted = (st & (batched.ST_SKIPPED | batched.ST_NONFINITE)) == 0
    mi = batched.PARAM_DEFAULTS["max_iter"]
    edges = [0, 5, 10, 20, 40, 80, 160, 320, 640, 1280, mi]
    res["iters_histogram"] = {"edges": edges, "counts": np.histogram(it[fitted], bins=edges + [mi + 1])[0].tolist()}
    res["iters_mean"] = float(it[fitted].mean())
    res["iters_median"] = float(np.median(it[fitted]))
    res["share_at_max_iter"] = float(np.mean((st[fitted] & batched.ST_ITMAX) != 0))
    res["share_at_bound"] = float(np.mean((st[fitted] & batched.ST_AT_BOUND) != 0))
    print(json.dumps(res), flush=True)
    x2, par = phantom_mae()
    res["phantom"] = "make_phantom((24, 24, 8), seed=5, fa_mode='b1'), SNR 50-150, MWF MAE against truth"
    res["mwf_mae_x2_i"], res["mwf_mae_3pool"] = x2, par
    print(json.dumps(res))
    if out_path:
        with open(out_path, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
