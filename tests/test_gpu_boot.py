"""Per-voxel bootstrap uncertainty on the GPU (Met2Plan.bootstrap, pipeline, motor_recon_met2): bitwise equal to the
NumPy restatement (tests/boot_oracle.py) with the plan's own t2_fit in between, independent of chunking, slabs and the
number of GPUs, and calibrated against repeated noise draws."""
import os

import numpy as np
import pytest
import torch

import boot_oracle as O
from multicomponent_t2_toolbox_b200 import batched, nifti_io, pipeline
from multicomponent_t2_toolbox_b200.phantom import epg_signal_batch, make_phantom

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def config2_voxels(golden_config2):
    return np.ascontiguousarray(golden_config2["sig"][::10][:2048])


def _point_fit(plan, sig):
    fa = plan.fa_fit(sig)
    t2 = plan.t2_fit(sig, fa["fa_index"])
    return fa["fa_index"].cpu().numpy(), t2["est_signal"].cpu().numpy(), t2["status"].cpu().numpy()


def _host(stats_nv):
    return stats_nv[0].cpu().numpy(), stats_nv[1].cpu().numpy()


@pytest.mark.parametrize("method, rm", [("X2", "I"), ("L_curve", "I"), ("BayesReg", "InvT2")])
def test_bootstrap_equals_restatement_through_t2_fit(config2_voxels, method, rm):
    sig = config2_voxels
    B, seed = 16, 20261020
    plan = batched.Met2Plan(32, 10.0, 1000.0, reg_method=method, reg_matrix=rm, FA_method="spline")
    fa, est, status = _point_fit(plan, sig)
    assert not (status & batched.ST_SKIPPED).any()
    rep, rep_fa = O.resample(sig, est, fa, B, seed)
    fits = plan.t2_fit(rep, rep_fa)
    ref, ref_n = O.summary(fits["maps"].cpu().numpy(), fits["status"].cpu().numpy(), B)
    stats, n_valid = _host(plan.bootstrap(sig, fa, est, B=B, seed=seed))
    assert np.array_equal(n_valid, ref_n) and (n_valid == B).mean() > 0.99
    assert np.array_equal(stats, ref, equal_nan=True)
    assert (stats[:, 0, 1] > 0).mean() > 0.9            # MWF varies between replicates


def test_chunks_slabs_and_seeds(config2_voxels):
    sig = config2_voxels
    B = 16
    plan = batched.Met2Plan(32, 10.0, 1000.0, reg_method="X2", reg_matrix="I", FA_method="spline")
    fa, est, _ = _point_fit(plan, sig)
    whole = _host(plan.bootstrap(sig, fa, est, B=B, seed=7))
    chunked = _host(plan.bootstrap(sig, fa, est, B=B, seed=7, max_replicates=16 * B))
    h = len(sig) // 2 + 3
    a = _host(plan.bootstrap(sig[:h], fa[:h], est[:h], B=B, seed=7))
    b = _host(plan.bootstrap(sig[h:], fa[h:], est[h:], B=B, seed=7, voxel_offset=h))
    again = _host(plan.bootstrap(sig, fa, est, B=B, seed=7))
    other = _host(plan.bootstrap(sig, fa, est, B=B, seed=8))
    for k in range(2):
        assert np.array_equal(chunked[k], whole[k])
        assert np.array_equal(np.concatenate([a[k], b[k]]), whole[k])
        assert np.array_equal(again[k], whole[k])
    assert not np.array_equal(other[0], whole[0])
    with pytest.raises(ValueError):
        plan.bootstrap(sig, fa, est, B=1025)
    with pytest.raises(ValueError):
        plan.bootstrap(sig, fa, est, B=4, seed=-1)


BOOT_VOLUMES = tuple(n + "_bootstrap" for n in pipeline.MAP_NAMES) + ("bootstrap_n_valid",)


def test_recon_arrays_slabs_equal_one_run():
    """One-process-per-GPU slabs (world_size 2, each rank's voxel_offset = its slab start) put together equal the
    unsharded run byte for byte; skipped and masked-out voxels are zero."""
    ph = make_phantom((12, 10, 6), seed=5, fa_mode="b1", mask_mode="ellipsoid")
    data = ph["data"].copy()
    data[6, 5, 3] = 0.0                                   # inside the mask but not fitted
    args = (data, ph["mask"], 10.0 * np.arange(1, 33), 1000.0, "X2", "I", "spline")
    one = pipeline.recon_arrays(*args, n_gpus=1, n_bootstrap=8, bootstrap_seed=3)
    parts = [pipeline.recon_arrays(*args, n_gpus=1, rank=r, world_size=2, n_bootstrap=8, bootstrap_seed=3)
             for r in range(2)]
    for k in BOOT_VOLUMES:
        assert np.array_equal(parts[0][k] + parts[1][k], one[k]), k
    fitted = (one["status"] & batched.ST_SKIPPED) == 0
    fitted &= ph["mask"] > 0
    assert one["MWF_bootstrap"].shape == (12, 10, 6, 4) and one["bootstrap_n_valid"].shape == (12, 10, 6)
    assert (one["bootstrap_n_valid"][fitted] == 8).all() and not one["bootstrap_n_valid"][~fitted].any()
    assert not one["MWF_bootstrap"][~fitted].any() and one["MWF_bootstrap"][fitted][:, 1].max() > 0


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_recon_arrays_two_gpus_equals_one_gpu():
    ph = make_phantom((16, 12, 8), seed=6, fa_mode="b1", mask_mode="ellipsoid")
    args = (ph["data"], ph["mask"], 10.0 * np.arange(1, 33), 1000.0, "X2", "I", "spline")
    one = pipeline.recon_arrays(*args, n_gpus=1, n_bootstrap=8)
    two = pipeline.recon_arrays(*args, n_gpus=2, n_bootstrap=8)
    for k in BOOT_VOLUMES + ("MWF", "status"):
        assert np.array_equal(one[k], two[k]), k


def test_motor_recon_met2_writes_bootstrap_volumes(tmp_path):
    from multicomponent_t2_toolbox_b200.motor.motor_recon_met2_real_data import (BOOTSTRAP_OUTPUTS, OUTPUTS,
                                                                                motor_recon_met2)
    ph = make_phantom((10, 8, 4), seed=9, fa_mode="b1", mask_mode="ellipsoid")
    nifti_io.save(ph["data"], str(tmp_path / "Data.nii.gz"))
    nifti_io.save(ph["mask"].astype(np.int16), str(tmp_path / "Mask.nii.gz"))
    TE = 10.0 * np.arange(1, 33)
    args = (str(tmp_path / "Data.nii.gz"), str(tmp_path / "Mask.nii.gz"))
    dirs = {}
    for tag, kw in (("plain", {}), ("zero", dict(n_bootstrap=0)), ("boot", dict(n_bootstrap=8, bootstrap_seed=1))):
        out = str(tmp_path / tag) + "/"
        os.mkdir(out)
        motor_recon_met2(TE, *args, out, 1000.0, "X2", "I", "None", "spline", "no", 40.0, -1, **kw)
        dirs[tag] = out
    listing = {t: sorted(os.listdir(d)) for t, d in dirs.items()}
    assert listing["zero"] == listing["plain"]
    assert sorted(set(listing["boot"]) - set(listing["plain"])) == sorted(n + ".nii.gz" for n in BOOTSTRAP_OUTPUTS)
    for name in listing["plain"]:
        with open(dirs["plain"] + name, "rb") as f0, open(dirs["zero"] + name, "rb") as f1:
            assert f0.read() == f1.read(), name
    for name in OUTPUTS:                                  # the bootstrap leaves the ten outputs as they were
        with open(dirs["plain"] + name + ".nii.gz", "rb") as f0, open(dirs["boot"] + name + ".nii.gz", "rb") as f1:
            assert f0.read() == f1.read(), name
    nv = nifti_io.load(dirs["boot"] + "bootstrap_n_valid.nii.gz").get_fdata()
    fitted = nifti_io.load(dirs["boot"] + "TWC.nii.gz").get_fdata() > 0
    assert (nv[fitted] == 8).all() and not nv[~fitted].any() and fitted.sum() > 50
    mwf = nifti_io.load(dirs["boot"] + "MWF_bootstrap.nii.gz").get_fdata()
    assert mwf.shape == (10, 8, 4, 4)
    assert (mwf[fitted][:, 2] <= mwf[fitted][:, 3]).all()


def calibration(n_vox=256, n_draws=64, B=100, seed=11):
    """Does the bootstrap SD mean anything?  n_vox voxels with fixed parameters (drawn like the phantom's, SNR in
    100-150, flip angles 120-180), n_draws independent Rician noise draws each, spline FA + X2-I.  Returns the median
    over voxels of (bootstrap SD of MWF from draw 0, B replicates) / (SD of the fitted MWF across the draws), with the
    fraction of voxels whose noise-free fit's MWF lies inside the bootstrap's 95 % interval from draw 0."""
    rng = np.random.default_rng(seed)
    mwf = rng.uniform(0.05, 0.25, n_vox)
    fwf = rng.uniform(0.0, 0.05, n_vox)
    t2m, t2ie = rng.uniform(15.0, 35.0, n_vox), rng.uniform(60.0, 90.0, n_vox)
    fa = rng.uniform(120.0, 180.0, n_vox)
    snr = rng.uniform(100.0, 150.0, n_vox)
    T1 = np.full(n_vox, 1000.0)
    clean = (mwf[:, None] * epg_signal_batch(32, 10.0, T1, t2m, fa)
             + (1.0 - mwf - fwf)[:, None] * epg_signal_batch(32, 10.0, T1, t2ie, fa)
             + fwf[:, None] * epg_signal_batch(32, 10.0, T1, np.full(n_vox, 2000.0), fa))
    clean *= 1000.0 * (1.0 - np.exp(-1.0))
    sigma = (clean[:, 0] / snr)[None, :, None]
    n1 = rng.standard_normal((n_draws,) + clean.shape) * sigma
    n2 = rng.standard_normal((n_draws,) + clean.shape) * sigma
    noisy = np.sqrt((clean[None] + n1) ** 2 + n2 ** 2)
    plan = batched.Met2Plan(32, 10.0, 1000.0, reg_method="X2", reg_matrix="I", FA_method="spline")
    sig = noisy.reshape(-1, 32)
    fa_i, est, status = _point_fit(plan, sig)
    assert not (status & batched.ST_SKIPPED).any()
    mwf_draws = plan.t2_fit(sig, fa_i)["maps"][:, 0].cpu().numpy().reshape(n_draws, n_vox)
    emp_sd = mwf_draws.std(axis=0, ddof=1)
    stats, n_valid = _host(plan.bootstrap(sig[:n_vox], fa_i[:n_vox], est[:n_vox], B=B, seed=seed))
    ratio = stats[:, 0, 1] / emp_sd
    truth_fit = plan.fit(clean)[1]["maps"][:, 0].cpu().numpy()
    inside = (stats[:, 0, 2] <= truth_fit) & (truth_fit <= stats[:, 0, 3])
    return dict(n_voxels=n_vox, n_draws=n_draws, B=B, median_sd_ratio=float(np.median(ratio)),
                sd_ratio_quartiles=[float(q) for q in np.percentile(ratio, [25, 75])],
                coverage_95=float(inside.mean()), n_valid_min=int(n_valid.min()),
                median_empirical_sd=float(np.median(emp_sd)), median_bootstrap_sd=float(np.median(stats[:, 0, 1])))


def test_bootstrap_sd_calibration():
    """Wild bootstrap of NNLS residuals comes out low: the fit absorbs part of the noise into the spectrum, so the
    residuals are smaller than the noise.  This seeded set-up measured a median ratio of 0.843 (quartiles 0.72 and
    0.99) on one B200 at a 1000 W power limit, and the 95 % intervals held the noise-free fit's MWF in 84 % of the
    voxels (profiles/r04_bootstrap_time.json).  The inputs are seeded, so the ratio moves only when the fit or the
    bootstrap changes; the band is +/- 0.1 around the measurement and lies inside [0.5, 2]."""
    c = calibration()
    print("calibration:", c)
    assert c["n_valid_min"] == c["B"]
    assert 0.74 <= c["median_sd_ratio"] <= 0.95, c
