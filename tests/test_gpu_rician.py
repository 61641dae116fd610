"""Met2Plan.rician_fit (met2_rician_fit + met2_spatial_finish) on the device: within 1e-9 of the NumPy restatement of
tests/rician_oracle.py with equal supports at a fixed number of MM iterations, on a crop and on 2 000 voxels of the
96 x 96 x 60 x 32 phantom; repeatable; equal across devices; the files of motor_recon_met2(rician_sigma=...); and the
bias table of DESIGN.md §10f through the whole pipeline, printed as measured."""
import os

import numpy as np
import pytest
import torch

import rician_oracle as R
from multicomponent_t2_toolbox_b200 import batched, nifti_io, pipeline
from multicomponent_t2_toolbox_b200.phantom import make_phantom

pytestmark = pytest.mark.gpu

TE = 10.0 * np.arange(1, 33)


@pytest.fixture(scope="module")
def phantom():
    ph = make_phantom((96, 96, 60), seed=2, fa_mode="b1", mask_mode="ellipsoid", backend="gpu", snr_range=(20.0, 40.0))
    flat, sig = pipeline.masked_voxel_list(ph["data"], ph["mask"])
    return flat, sig, ph["truth"]["sigma"].reshape(-1)[flat]


@pytest.fixture(scope="module")
def plan():
    return batched.Met2Plan(32, 10.0, 1000.0, reg_method="X2", reg_matrix="I", FA_method="spline")


def _point_fit(plan, sig):
    res = pipeline.fit_voxels(plan, sig)
    lam = plan.t2_fit(sig, res["fa_index"], flags=batched.REG_IS_LAMBDA)["reg"].cpu().numpy()
    return res, lam


def _check_against_restatement(plan, sig, sigma, res, lam, rf, pick, fast):
    dic = plan.dict_hr.dic.cpu().numpy()
    x = rf["x"].cpu().numpy()
    it = rf["iters"].cpu().numpy()
    worst = 0.0
    for v in pick:
        y = sig[v] / sig[v, 0]
        x0 = res["fsol"][v] / sig[v, 0]
        ref, iters, capped, _ = R.mm_fit(dic[res["fa_index"][v]], y, plan.Laplac, lam[v], sigma[v] / sig[v, 0], x0,
                                         max_iter=5, tol=0.0, fast=fast)
        assert capped or it[v] < 5
        assert np.array_equal(x[v] > 0, ref > 0), v
        worst = max(worst, np.abs(x[v] - ref).max() / np.abs(ref).max())
    print("largest relative difference to the restatement over %d voxels: %.3g" % (len(pick), worst))
    assert worst <= 1e-9


def test_fixed_iterations_on_a_crop(plan):
    ph = make_phantom((12, 12, 6), seed=4, fa_mode="b1", mask_mode="ellipsoid", snr_range=(20.0, 40.0))
    flat, sig = pipeline.masked_voxel_list(ph["data"], ph["mask"])
    sigma = ph["truth"]["sigma"].reshape(-1)[flat]
    res, lam = _point_fit(plan, sig)
    rf = plan.rician_fit(sig, res["fa_index"], lam, sigma, res["fsol"], res["status"], max_iter=5, tol=0.0)
    fitted = np.nonzero((res["status"] & batched.ST_SKIPPED) == 0)[0]
    _check_against_restatement(plan, sig, sigma, res, lam, rf, fitted, fast=False)
    # the outputs of met2_spatial_finish for this x
    x = rf["x"].cpu().numpy()
    assert np.allclose(rf["fsol"].cpu().numpy(), x * sig[:, :1], rtol=1e-15, atol=0.0)


def test_fixed_iterations_on_2000_voxels_and_repeatable(plan, phantom):
    flat, sig, sigma = phantom
    res, lam = _point_fit(plan, sig)
    d = [torch.as_tensor(a).cuda() for a in (sig, res["fa_index"], lam, sigma, res["fsol"], res["status"])]
    rf = plan.rician_fit(*d, max_iter=5, tol=0.0)
    pick = np.sort(np.random.default_rng(11).choice(len(flat), 2000, replace=False))
    pick = pick[(res["status"][pick] & batched.ST_SKIPPED) == 0]
    _check_against_restatement(plan, sig, sigma, res, lam, rf, pick, fast=True)
    a = plan.rician_fit(*d)
    b = plan.rician_fit(*d)
    for k in a:
        assert torch.equal(a[k], b[k]), k
    it = a["iters"].cpu().numpy()
    st = a["status"].cpu().numpy()
    fitted = (st & batched.ST_SKIPPED) == 0
    print("MM iterations on %d voxels: median %d, p90 %d, max %d; at the cap %d; ITMAX %d" % (
        fitted.sum(), np.median(it[fitted]), np.percentile(it[fitted], 90), it[fitted].max(),
        ((st & batched.ST_MM_CAP) != 0).sum(), ((st & batched.ST_ITMAX) != 0).sum()))
    zero = plan.rician_fit(*d[:3], torch.zeros_like(d[3]), *d[4:])
    assert not zero["iters"].any()
    assert torch.equal(zero["x"], torch.where(((d[5] & 1) == 0)[:, None], d[4] / d[0][:, :1], 0.0))


def test_multi_gpu_fit_equals_fit_voxels(plan):
    """MultiGpuFit copies each chunk's sigma beside its signals: two plans on one device (the chunk dealing) and, when
    there are two devices, one plan per device give the bytes of fit_voxels."""
    ph = make_phantom((20, 20, 8), seed=6, fa_mode="b1", snr_range=(20.0, 40.0))
    _, sig = pipeline.masked_voxel_list(ph["data"], ph["mask"])
    sigma = ph["truth"]["sigma"].reshape(-1)
    one = pipeline.fit_voxels(plan, sig, sigma=sigma)
    plans = [plan, batched.Met2Plan(32, 10.0, 1000.0, reg_method="X2", reg_matrix="I", FA_method="spline",
                                    device=torch.device("cuda", 1 if torch.cuda.device_count() > 1 else 0))]
    many = pipeline.MultiGpuFit(plans).fit(torch.as_tensor(sig).pin_memory(), sigma=sigma)
    for k in one:
        if k != "fsol_sum":          # summed per device
            assert np.array_equal(one[k], many[k]), k
    assert "rician_maps" in many and (one["rician_iters"] > 0).mean() > 0.9


def test_recon_arrays_on_two_gpus_equals_one():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    ph = make_phantom((16, 16, 6), seed=8, fa_mode="b1", mask_mode="ellipsoid", snr_range=(20.0, 40.0))
    args = (ph["data"], ph["mask"], TE, 1000.0, "X2", "I", "spline")
    a = pipeline.recon_arrays(*args, n_gpus=1, rician_sigma=ph["truth"]["sigma"])
    b = pipeline.recon_arrays(*args, n_gpus=2, rician_sigma=ph["truth"]["sigma"])
    for k in pipeline.RICIAN_VOLUMES:
        assert a[k].tobytes() == b[k].tobytes(), k


def test_motor_recon_met2_writes_the_rician_volumes(tmp_path):
    from multicomponent_t2_toolbox_b200.motor.motor_recon_met2_real_data import OUTPUTS, motor_recon_met2
    ph = make_phantom((10, 8, 6), seed=9, fa_mode="b1", mask_mode="ellipsoid", snr_range=(20.0, 40.0))
    nifti_io.save(ph["data"], str(tmp_path / "Data.nii.gz"))
    nifti_io.save(ph["mask"].astype(np.int16), str(tmp_path / "Mask.nii.gz"))
    files = (str(tmp_path / "Data.nii.gz"), str(tmp_path / "Mask.nii.gz"))
    outs = {}
    for tag, sigma in (("plain", None), ("number", 3.5), ("MPPCA", "MPPCA")):
        out = str(tmp_path / tag) + "/"
        os.mkdir(out)
        motor_recon_met2(TE, *files, out, 1000.0, "X2", "I", "None", "spline", "no", 40.0, -1, rician_sigma=sigma)
        outs[tag] = out
    load = lambda d, name: nifti_io.load(d + name + ".nii.gz").get_fdata()
    for tag in ("number", "MPPCA"):
        names = set(os.listdir(outs[tag]))
        assert {n + ".nii.gz" for n in tuple(OUTPUTS) + tuple(pipeline.RICIAN_VOLUMES)} <= names
        assert ("MPPCA_sigma.nii.gz" in names) == (tag == "MPPCA")
        for name in OUTPUTS:
            assert load(outs[tag], name).tobytes() == load(outs["plain"], name).tobytes(), (tag, name)
    data = nifti_io.load(files[0]).get_fdata()
    mask = nifti_io.load(files[1]).get_fdata().astype(np.int64)
    data = data * mask[..., None]
    data[data < 0.0] = 0.0
    sigma = batched.mppca_denoise(data, mask)[1].cpu().numpy()
    assert np.array_equal(load(outs["MPPCA"], "MPPCA_sigma"), sigma)
    for tag, s in (("number", 3.5), ("MPPCA", sigma)):
        vol = pipeline.recon_arrays(data, mask, TE, 1000.0, "X2", "I", "spline", premasked=True, rician_sigma=s)
        for name in pipeline.RICIAN_VOLUMES:
            assert np.array_equal(load(outs[tag], name), vol[name]), (tag, name)
        assert (vol["rician_iters"][mask == 1] > 0).mean() > 0.9
    with pytest.raises(ValueError):
        motor_recon_met2(TE, *files, outs["plain"], 1000.0, "X2", "I", "NESMA", "spline", "no", 40.0, -1,
                         rician_sigma=3.5)
    with pytest.raises(ValueError):
        motor_recon_met2(TE, *files, outs["plain"], 1000.0, "X2", "I", "None", "spline", "no", 40.0, -1,
                         degibbs=True, rician_sigma="MPPCA")
    with pytest.raises(ValueError):
        pipeline.recon_arrays(data, mask, TE, 1000.0, "X2", "I", "spline", spatial_mu=0.1, rician_sigma=3.5)


def bias_table(n_side=14, seed=3):
    """Mean errors (fit - truth) of MWF, FWF and T2_IE of the point fit and of the Rician fit through recon_arrays
    (spline FA), for NNLS and X2-I at SNR 20-40 and 50-150, with sigma = 0.8, 1 and 1.25 x the true noise SD, on
    make_phantom((n_side, n_side, 4), seed, "b1").  Returns a list of rows."""
    rows = []
    for snr in ((20.0, 40.0), (50.0, 150.0)):
        ph = make_phantom((n_side, n_side, 4), seed=seed, fa_mode="b1", snr_range=snr)
        tr = ph["truth"]
        for method in ("NNLS", "X2"):
            for scale in (1.0, 0.8, 1.25):
                vol = pipeline.recon_arrays(ph["data"], ph["mask"], TE, 1000.0, method, "I", "spline",
                                            rician_sigma=scale * tr["sigma"])
                row = dict(snr=snr, method=method, sigma_scale=scale,
                           iters=[int(np.median(vol["rician_iters"])), int(np.percentile(vol["rician_iters"], 90)),
                                  int(vol["rician_iters"].max())])
                for tag, suffix in (("gauss", ""), ("rician", "_rician")):
                    for key, name in (("mwf", "MWF"), ("fwf", "FWF"), ("t2ie", "T2_IE")):
                        err = vol[name + suffix] - tr[key]
                        row["%s_%s_bias" % (key, tag)] = float(err.mean())
                        row["%s_%s_mae" % (key, tag)] = float(np.abs(err).mean())
                rows.append(row)
    return rows


def test_bias_table():
    """Printed as measured; asserted only in the direction of the prototype (DESIGN.md §10f), with margin: at SNR 20-40
    with the true sigma, the Rician fit at least halves the FWF bias of NNLS and reduces the T2_IE bias of X2-I."""
    rows = bias_table()
    for r in rows:
        print("SNR %g-%g %-4s sigma x%.2f: MWF %+.4f -> %+.4f | FWF %+.4f -> %+.4f | T2_IE %+.2f -> %+.2f ms | "
              "MM iterations %s" % (*r["snr"], r["method"], r["sigma_scale"], r["mwf_gauss_bias"], r["mwf_rician_bias"],
                                    r["fwf_gauss_bias"], r["fwf_rician_bias"], r["t2ie_gauss_bias"],
                                    r["t2ie_rician_bias"], r["iters"]))
    get = {(r["snr"][0], r["method"], r["sigma_scale"]): r for r in rows}
    nn = get[(20.0, "NNLS", 1.0)]
    assert abs(nn["fwf_rician_bias"]) <= 0.5 * abs(nn["fwf_gauss_bias"])
    x2 = get[(20.0, "X2", 1.0)]
    assert abs(x2["t2ie_rician_bias"]) <= 0.8 * abs(x2["t2ie_gauss_bias"])
