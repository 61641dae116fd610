"""Timing of the per-voxel bootstrap (Met2Plan.bootstrap) on the config-2 phantom (96 x 96 x 60 x 32, 552 960 voxels,
spline FA + X2-I, seeded) for B = 20 and 100 replicates: CUDA-event times of replicate synthesis, refits and summary
on one GPU, the whole bootstrap on one GPU and, through pipeline.MultiGpuFit, on all GPUs; then the calibration of
tests/test_gpu_boot.py.  Prints one JSON line and, given a path as the first argument, writes the record there.
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

from multicomponent_t2_toolbox_b200 import _lib, batched, pipeline  # noqa: E402
from multicomponent_t2_toolbox_b200.batched import _ptr, _stream  # noqa: E402
from multicomponent_t2_toolbox_b200.phantom import make_phantom  # noqa: E402
from test_gpu_boot import calibration  # noqa: E402


def event():
    e = torch.cuda.Event(enable_timing=True)
    e.record()
    return e


def stage_times(plan, sig, fa, est, B, seed=0, max_replicates=1 << 21):
    """Met2Plan.bootstrap's chunk loop with an event between the stages; returns ms per stage summed over chunks."""
    V = sig.shape[0]
    chunk = min(V, max_replicates // B)
    rep_sig = torch.empty((chunk * B, plan.nTE), dtype=torch.float64, device=plan.dev)
    rep_fa = torch.empty(chunk * B, dtype=torch.int32, device=plan.dev)
    stats = torch.zeros((V, 6, 4), dtype=torch.float64, device=plan.dev)
    n_valid = torch.zeros(V, dtype=torch.int32, device=plan.dev)
    bufs, marks = None, []
    torch.cuda.synchronize()
    for lo in range(0, V, chunk):
        n = min(chunk, V - lo)
        R = n * B
        e0 = event()
        _lib.check(plan.lib.met2_boot_resample(_ptr(sig[lo:]), _ptr(est[lo:]), _ptr(fa[lo:]), n, plan.nTE, B, seed, lo,
                                               _ptr(rep_sig), _ptr(rep_fa), _stream()), "met2_boot_resample")
        e1 = event()
        fits = plan.t2_fit(rep_sig[:R], rep_fa[:R],
                           out=None if bufs is None else {k: v[:R] for k, v in bufs.items()})
        bufs = bufs if bufs is not None else fits
        e2 = event()
        _lib.check(plan.lib.met2_boot_summary(_ptr(fits["maps"]), _ptr(fits["status"]), n, B, _ptr(stats[lo:]),
                                              _ptr(n_valid[lo:]), _stream()), "met2_boot_summary")
        e3 = event()
        marks.append((e0, e1, e2, e3))
    torch.cuda.synchronize()
    t = np.array([[a.elapsed_time(b), b.elapsed_time(c), c.elapsed_time(d)] for a, b, c, d in marks]).sum(axis=0)
    times = dict(chunks=len(marks), resample_ms=float(t[0]), refits_ms=float(t[1]), summary_ms=float(t[2]))
    return times, stats, n_valid


def main():
    assert torch.cuda.is_available(), "gpu_boot_time.py needs a CUDA device"
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().split("\n")
    ngpu = torch.cuda.device_count()
    res = {"gpus": q, "n_gpus": ngpu, "volume": "config-2 phantom 96x96x60x32, seed 2, b1 FA, full mask",
           "method": "spline FA + X2-I"}
    ph = make_phantom((96, 96, 60), seed=2, fa_mode="b1", backend="gpu")
    sig_h = np.ascontiguousarray(ph["data"].reshape(-1, 32))
    V = sig_h.shape[0]
    res["voxels"] = V
    plan = batched.Met2Plan(32, 10.0, 1000.0, reg_method="X2", reg_matrix="I", FA_method="spline")
    sig = torch.as_tensor(sig_h).cuda()
    plan.fit(sig[:4096])                                            # warm-up
    torch.cuda.synchronize()
    e0 = event()
    fa_out, t2_out = plan.fit(sig)
    e1 = event()
    torch.cuda.synchronize()
    res["point_fit_ms"] = e0.elapsed_time(e1)
    fa, est = fa_out["fa_index"], t2_out["est_signal"]
    pin = torch.as_tensor(sig_h).pin_memory()
    multi = pipeline.MultiGpuFit.create(ngpu, 32, 10.0, 1000.0, reg_method="X2", reg_matrix="I", FA_method="spline")
    multi.fit(pin)
    t0 = time.perf_counter()
    multi.fit(pin)
    res["all_gpus_point_fit_s"] = time.perf_counter() - t0
    for B in (20, 100):
        r = {}
        plan.bootstrap(sig[:8192], fa[:8192], est[:8192], B=B)       # warm-up of this B's shapes
        r["stages_one_gpu"], stats, n_valid = stage_times(plan, sig, fa, est, B)
        s = r["stages_one_gpu"]
        tot = s["resample_ms"] + s["refits_ms"] + s["summary_ms"]
        s["summary_share"] = s["summary_ms"] / tot
        s["resample_share"] = s["resample_ms"] / tot
        torch.cuda.synchronize()
        e0 = event()
        st2, nv2 = plan.bootstrap(sig, fa, est, B=B)
        e1 = event()
        torch.cuda.synchronize()
        r["bootstrap_one_gpu_ms"] = e0.elapsed_time(e1)
        r["same_as_stage_loop"] = bool(torch.equal(st2, stats) and torch.equal(nv2, n_valid))
        r["replicate_fits_per_s_one_gpu"] = V * B / (r["bootstrap_one_gpu_ms"] * 1e-3)
        r["n_valid_fraction"] = float(n_valid.double().mean().item() / B)
        r["median_mwf_sd"] = float(stats[:, 0, 1].median().item())
        multi.fit(pin, n_bootstrap=B)
        t0 = time.perf_counter()
        out = multi.fit(pin, n_bootstrap=B)
        r["all_gpus_fit_plus_bootstrap_s"] = time.perf_counter() - t0
        r["all_gpus_same_as_one_gpu"] = bool(np.array_equal(out["boot_stats"], st2.cpu().numpy()) and
                                             np.array_equal(out["boot_n_valid"], nv2.cpu().numpy()))
        res["B%d" % B] = r
        print(json.dumps({"B": B, **r}), flush=True)
    res["calibration"] = calibration()
    print(json.dumps(res))
    if out_path:
        with open(out_path, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
