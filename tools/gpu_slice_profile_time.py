"""Cost and accuracy of the slice-profile dictionary (met2_epg_dictionary_profile, DESIGN §10g) on one GPU:
  - the build time of the fine (273 angles) and coarse (15 knots) dictionaries with their Gram tables, 60 bins, 32
    echoes, for K = 16, 64 and 256 positions and for the plain dictionary (CUDA events, median of 7 after a warm-up);
  - the echo-basis residual `tail` at ranks 16 and 24 and the rank the echo-space kernels then use, for the default
    profiles (TBW 2.7 and 6, refocusing slab 1x and 2x the excitation);
  - the point-fit time (spline FA + X2-I, Met2Plan.fit) on the config-2 phantom (96 x 96 x 60 x 32, seed 2, b1 FA) with
    the profile plan and with the plain plan (median of 5 after a warm-up);
  - the accuracy table of tests/test_gpu_slice_profile.py (FA, MWF, T2_IE errors, plain against profile dictionary,
    SNR 50-150 and noise-free) for the four profiles.
Prints one JSON line and, given a path as the first argument, writes the record there.  Needs a CUDA device."""
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

from multicomponent_t2_toolbox_b200 import batched, grids, pipeline  # noqa: E402
from multicomponent_t2_toolbox_b200.phantom import make_phantom  # noqa: E402
from test_gpu_slice_profile import accuracy_table  # noqa: E402


def event():
    e = torch.cuda.Event(enable_timing=True)
    e.record()
    return e


def timed(fn, n):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(n):
        e0 = event()
        fn()
        e1 = event()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return ts


def main():
    assert torch.cuda.is_available(), "gpu_slice_profile_time.py needs a CUDA device"
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().split("\n")
    dev = torch.device("cuda", 0)
    res = {"gpus": q, "build": {}, "echo_basis": {}, "point_fit": {}}
    T2s = grids.t2_grid(60)
    T1s = np.full(60, 1000.0)
    fine, knots = grids.fa_grids("spline")

    def build(prof):
        batched.Dictionary(fine, T2s, T1s, 32, 10.0, 1000.0, dev, profile=prof)
        batched.Dictionary(knots, T2s, T1s, 32, 10.0, 1000.0, dev, profile=prof)
    for K in (None, 16, 64, 256):
        prof = None if K is None else grids.slice_profile(K=K)
        ts = timed(lambda: build(prof), 7)
        res["build"]["plain" if K is None else "K%d" % K] = {"ms": ts, "ms_median": float(np.median(ts)),
                                                             "echo_trains": 288 * 60 * (1 if K is None else K)}
    print(json.dumps(res["build"]), flush=True)
    profiles = {"tbw2.7_ratio1": grids.slice_profile(), "tbw2.7_ratio2": grids.slice_profile(ratio=2.0),
                "tbw6_ratio1": grids.slice_profile(tbw=6.0), "tbw6_ratio2": grids.slice_profile(tbw=6.0, ratio=2.0)}
    for name, prof in list(profiles.items()) + [("plain", None)]:
        d = batched.Dictionary(fine, T2s, T1s, 32, 10.0, 1000.0, dev, profile=prof)
        red = d.echo_basis()
        res["echo_basis"][name] = {"tail_r16": d.echo_tables(16)[2], "tail_r24": d.echo_tables(24)[2],
                                   "rank_used": None if red is None else red[2]}
    print(json.dumps(res["echo_basis"]), flush=True)
    ph = make_phantom((96, 96, 60), seed=2, fa_mode="b1", backend="gpu", slice_profile=profiles["tbw2.7_ratio1"])
    _, sig_h = pipeline.masked_voxel_list(ph["data"], ph["mask"])
    sig = torch.as_tensor(sig_h).cuda()
    res["point_fit"]["voxels"] = int(sig.shape[0])
    res["point_fit"]["data"] = "config-2 phantom with the TBW 2.7 / ratio 1 / K 64 profile"
    for name, prof in (("plain", None), ("profile", profiles["tbw2.7_ratio1"])):
        plan = batched.Met2Plan(32, 10.0, 1000.0, reg_method="X2", reg_matrix="I", FA_method="spline",
                                slice_profile=prof)
        ts = timed(lambda: plan.fit(sig), 5)
        red = plan.dict_hr.echo_basis()
        res["point_fit"][name] = {"ms": ts, "ms_median": float(np.median(ts)),
                                  "echo_rank": None if red is None else red[2]}
    print(json.dumps(res["point_fit"]), flush=True)
    res["accuracy"] = {"phantom": "make_phantom((16, 16, 4), seed=5, fa_mode='b1'), spline + X2-I via recon_arrays",
                       "rows": {name: accuracy_table(profile=prof) for name, prof in profiles.items()}}
    print(json.dumps(res))
    if out_path:
        with open(out_path, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
