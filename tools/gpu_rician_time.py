"""Timing of the Rician-likelihood fit (Met2Plan.rician_fit) on the config-2 phantom (96 x 96 x 60 x 32, 552 960
voxels, spline FA + X2-I point fit, seeded, SNR 20-40 and 50-150, sigma = the phantom's true noise SD): CUDA-event
times of the point fit, of the lambda refit under REG_IS_LAMBDA and of rician_fit (median of 5 after a warm-up), the
distribution of MM iterations, and the bias table of tests/test_gpu_rician.py.  Prints one JSON line and, given a path
as the first argument, writes the record there.  Needs a CUDA device."""
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
from test_gpu_rician import bias_table  # noqa: E402


def event():
    e = torch.cuda.Event(enable_timing=True)
    e.record()
    return e


def main():
    assert torch.cuda.is_available(), "gpu_rician_time.py needs a CUDA device"
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().split("\n")
    res = {"gpus": q, "volume": "config-2 phantom 96x96x60x32, seed 2, b1 FA, full mask",
           "method": "spline FA + X2-I point fit, lambda refit (REG_IS_LAMBDA), then rician_fit",
           "settings": batched.RICIAN_DEFAULTS, "runs": {}}
    plan = batched.Met2Plan(32, 10.0, 1000.0, reg_method="X2", reg_matrix="I", FA_method="spline")
    for snr in ((20.0, 40.0), (50.0, 150.0)):
        ph = make_phantom((96, 96, 60), seed=2, fa_mode="b1", backend="gpu", snr_range=snr)
        flat, sig_h = pipeline.masked_voxel_list(ph["data"], ph["mask"])
        res["voxels"] = int(sig_h.shape[0])
        sig = torch.as_tensor(sig_h).cuda()
        sigma = torch.as_tensor(ph["truth"]["sigma"].reshape(-1)[flat]).cuda()
        fa, t2 = plan.fit(sig[:4096])                                  # warm-up
        lam = plan.t2_fit(sig[:4096], fa["fa_index"], flags=batched.REG_IS_LAMBDA)["reg"]
        plan.rician_fit(sig[:4096], fa["fa_index"], lam, sigma[:4096], t2["fsol"], t2["status"])
        torch.cuda.synchronize()
        point, refit, rician = [], [], []
        for _ in range(5):
            e0 = event()
            fa, t2 = plan.fit(sig)
            e1 = event()
            lam = plan.t2_fit(sig, fa["fa_index"], flags=batched.REG_IS_LAMBDA)["reg"]
            e2 = event()
            rf = plan.rician_fit(sig, fa["fa_index"], lam, sigma, t2["fsol"], t2["status"])
            e3 = event()
            torch.cuda.synchronize()
            point.append(e0.elapsed_time(e1))
            refit.append(e1.elapsed_time(e2))
            rician.append(e2.elapsed_time(e3))
        st = rf["status"].cpu().numpy()
        it = rf["iters"].cpu().numpy()
        fitted = (st & batched.ST_SKIPPED) == 0
        r = {"point_fit_ms": point, "lambda_refit_ms": refit, "rician_fit_ms": rician,
             "point_fit_ms_median": float(np.median(point)), "lambda_refit_ms_median": float(np.median(refit)),
             "rician_fit_ms_median": float(np.median(rician)),
             "iters_median": float(np.median(it[fitted])), "iters_mean": float(it[fitted].mean()),
             "iters_p90": float(np.percentile(it[fitted], 90)), "iters_p99": float(np.percentile(it[fitted], 99)),
             "iters_max": int(it[fitted].max()),
             "share_mm_cap": float(np.mean((st[fitted] & batched.ST_MM_CAP) != 0)),
             "share_itmax": float(np.mean((st[fitted] & batched.ST_ITMAX) != 0))}
        r["stage_over_point"] = (r["lambda_refit_ms_median"] + r["rician_fit_ms_median"]) / r["point_fit_ms_median"]
        res["runs"]["snr_%g_%g" % snr] = r
        print(json.dumps(r), flush=True)
    res["bias_table"] = {"phantom": "make_phantom((14, 14, 4), seed=3, fa_mode='b1'), 784 voxels, recon_arrays with "
                                    "spline FA", "rows": bias_table()}
    print(json.dumps(res))
    if out_path:
        with open(out_path, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
