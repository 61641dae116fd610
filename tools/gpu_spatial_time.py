"""Timing of the spatially regularised fit (Met2Plan.spatial_fit) on the config-2 phantom (96 x 96 x 60 x 32, 552 960
voxels, spline FA + X2-I, seeded): CUDA-event times of the point fit, the lambda fit (t2_fit with
MET2_T2_FLAG_REG_IS_LAMBDA), every half-sweep of 10 sweeps and the output kernel, and J after every sweep; then the
MWF error on the block phantom of tests/test_gpu_spatial.py over a decade grid of mu.  Prints one JSON line and, given
a path as the first argument, writes the record there.  Needs a CUDA device."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import torch  # noqa: E402

from multicomponent_t2_toolbox_b200 import _lib, batched, pipeline  # noqa: E402
from multicomponent_t2_toolbox_b200.batched import _ptr, _stream  # noqa: E402
from multicomponent_t2_toolbox_b200.phantom import make_phantom  # noqa: E402
from test_gpu_spatial import MU_VALUE_CHECK, mwf_mae, objective  # noqa: E402

MU_GRID = (0.0, 1e-4, 1e-3, 1e-2, 1e-1, 1.0, 10.0)


def event():
    e = torch.cuda.Event(enable_timing=True)
    e.record()
    return e


def main():
    assert torch.cuda.is_available(), "gpu_spatial_time.py needs a CUDA device"
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().split("\n")
    res = {"gpus": q, "volume": "config-2 phantom 96x96x60x32, seed 2, b1 FA, full mask", "method": "spline FA + X2-I",
           "mu": MU_VALUE_CHECK}
    ph = make_phantom((96, 96, 60), seed=2, fa_mode="b1", backend="gpu")
    shape = ph["data"].shape[:3]
    flat, sig_h = pipeline.masked_voxel_list(ph["data"], np.ones(shape))
    V = sig_h.shape[0]
    res["voxels"] = V
    plan = batched.Met2Plan(32, 10.0, 1000.0, reg_method="X2", reg_matrix="I", FA_method="spline")
    sig = torch.as_tensor(sig_h).cuda()
    plan.fit(sig[:4096])                                            # warm-up
    torch.cuda.synchronize()
    e0 = event()
    fa_out, t2 = plan.fit(sig)
    e1 = event()
    lam = plan.t2_fit(sig, fa_out["fa_index"], flags=batched.REG_IS_LAMBDA)["reg"]
    e2 = event()
    torch.cuda.synchronize()
    res["point_fit_ms"] = e0.elapsed_time(e1)
    res["lambda_fit_ms"] = e1.elapsed_time(e2)
    fa = fa_out["fa_index"]
    fitted = ((t2["status"] & batched.ST_SKIPPED) == 0).cpu().numpy()
    nbr, colours = pipeline.spatial_neighbours(flat, shape, fitted)
    d_nbr, d_col = torch.as_tensor(nbr).cuda(), [torch.as_tensor(c).cuda() for c in colours]
    mu = MU_VALUE_CHECK
    x = torch.where(torch.as_tensor(fitted).cuda()[:, None], t2["fsol"] / sig[:, :1], 0.0).contiguous()
    st = t2["status"].clone()
    plan.spatial_half_sweep(sig, fa, lam, x.clone(), d_nbr, d_col[0][:4096], mu, st.clone())   # warm-up
    J = [objective(plan, sig, fa, lam, x, nbr, fitted, mu)]
    half_ms = []
    for _ in range(10):
        for vox in d_col:
            torch.cuda.synchronize()
            a = event()
            plan.spatial_half_sweep(sig, fa, lam, x, d_nbr, vox, mu, st)
            b = event()
            torch.cuda.synchronize()
            half_ms.append(a.elapsed_time(b))
        J.append(objective(plan, sig, fa, lam, x, nbr, fitted, mu))
    out = {k: torch.empty_like(t2[k]) for k in ("fsol", "est_signal", "maps")}
    a = event()
    _lib.check(plan.lib.met2_spatial_finish(
        _ptr(sig), _ptr(fa), _ptr(st), _ptr(x), V, plan.nTE, plan.npc, plan.dict_hr.nA, _ptr(plan.dict_hr.dicT),
        _ptr(plan.logT2), _ptr(plan.comp), _ptr(out["fsol"]), _ptr(out["est_signal"]), _ptr(out["maps"]), _stream()),
        "met2_spatial_finish")
    b = event()
    torch.cuda.synchronize()
    res["half_sweep_ms"] = half_ms
    res["half_sweep_ms_median"] = float(np.median(half_ms))
    res["finish_ms"] = a.elapsed_time(b)
    res["ten_sweeps_ms"] = float(np.sum(half_ms)) + res["finish_ms"]
    res["ten_sweeps_over_point_fit"] = res["ten_sweeps_ms"] / res["point_fit_ms"]
    res["J_per_sweep"] = J
    res["itmax_voxels"] = int(((st & batched.ST_ITMAX) != 0).sum())
    torch.cuda.synchronize()
    e0 = event()
    sp = plan.spatial_fit(sig, fa, lam, t2["fsol"], nbr, colours, mu, 10, status=t2["status"])
    e1 = event()
    torch.cuda.synchronize()
    res["spatial_fit_10_sweeps_ms"] = e0.elapsed_time(e1)
    res["spatial_fit_same_as_loop"] = bool(torch.equal(sp["x"], x) and torch.equal(sp["maps"], out["maps"]))
    print(json.dumps({k: v for k, v in res.items() if k != "half_sweep_ms"}), flush=True)
    res["block_phantom_mwf_mae"] = {repr(k): v for k, v in mwf_mae(MU_GRID).items()}
    print(json.dumps(res))
    if out_path:
        with open(out_path, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
