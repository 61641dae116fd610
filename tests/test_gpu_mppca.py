"""batched.mppca_denoise (met2_mppca) on the device: bitwise equal to the NumPy restatement of tests/mppca_oracle.py on
a crop and on fixed voxels of the 96 x 96 x 60 x 32 ellipsoid phantom, repeatable, the files of
motor_recon_met2(denoise='MPPCA'), and the MWF error on the block phantom of test_gpu_spatial.py."""
import os

import numpy as np
import pytest

import mppca_oracle as O
from multicomponent_t2_toolbox_b200 import batched, nifti_io, pipeline
from multicomponent_t2_toolbox_b200.phantom import make_phantom

pytestmark = pytest.mark.gpu

TE = 10.0 * np.arange(1, 33)


@pytest.fixture(scope="module")
def phantom():
    ph = make_phantom((96, 96, 60), seed=2, fa_mode="b1", mask_mode="ellipsoid", backend="gpu")
    data = ph["data"] * ph["mask"][..., None]          # motor_recon_met2: data * mask, negatives clipped
    data[data < 0.0] = 0.0
    return np.ascontiguousarray(data), ph["mask"]


def test_bitwise_on_a_crop(phantom):
    """A 16 x 16 x 10 crop across the mask's edge (the restatement takes tens of ms per voxel on the host)."""
    data, mask = phantom
    crop = np.ascontiguousarray(data[0:16, 40:56, 25:35])
    cm = np.ascontiguousarray(mask[0:16, 40:56, 25:35])
    assert 0 < cm.sum() < cm.size
    ref = O.mppca(crop, cm, 2)
    got = [t.cpu().numpy() for t in batched.mppca_denoise(crop, cm)]
    for a, b, name in zip(got, ref, ("out", "sigma", "n_signal")):
        assert np.array_equal(a, b), name


def test_bitwise_on_fixed_voxels_of_the_full_volume_and_repeatable(phantom):
    import torch
    data, mask = phantom
    d = torch.as_tensor(data).cuda()
    m = torch.as_tensor(mask).cuda()
    a = batched.mppca_denoise(d, m)
    b = batched.mppca_denoise(d, m)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    out, sigma, nsig = (t.cpu().numpy() for t in a)
    assert not out[mask != 1].any() and not sigma[mask != 1].any() and not nsig[mask != 1].any()
    rng = np.random.default_rng(7)
    centres = np.argwhere(mask == 1)
    pick = centres[np.sort(rng.choice(len(centres), 2000, replace=False))]
    ref = O.mppca_batch(data, pick, 2)
    i, j, k = pick.T
    assert np.array_equal(out[i, j, k], ref["out"])
    assert np.array_equal(sigma[i, j, k], ref["sigma"])
    assert np.array_equal(nsig[i, j, k], ref["n_signal"])
    assert not ref["capped"].any()


def test_motor_recon_met2_writes_the_sigma_map(tmp_path):
    from multicomponent_t2_toolbox_b200.motor.motor_recon_met2_real_data import OUTPUTS, motor_recon_met2
    ph = make_phantom((10, 8, 6), seed=9, fa_mode="b1", mask_mode="ellipsoid")
    nifti_io.save(ph["data"], str(tmp_path / "Data.nii.gz"))
    nifti_io.save(ph["mask"].astype(np.int16), str(tmp_path / "Mask.nii.gz"))
    out = str(tmp_path / "out") + "/"
    os.mkdir(out)
    motor_recon_met2(TE, str(tmp_path / "Data.nii.gz"), str(tmp_path / "Mask.nii.gz"), out, 1000.0, "X2", "I", "MPPCA",
                     "spline", "no", 40.0, -1)
    names = set(os.listdir(out))
    assert {n + ".nii.gz" for n in OUTPUTS} | {"MPPCA_sigma.nii.gz"} <= names
    data = nifti_io.load(str(tmp_path / "Data.nii.gz")).get_fdata()
    mask = nifti_io.load(str(tmp_path / "Mask.nii.gz")).get_fdata().astype(np.int64)
    data = data * mask[..., None]
    data[data < 0.0] = 0.0
    den, sigma, _ = batched.mppca_denoise(data, mask)
    vol = pipeline.recon_arrays(den.cpu().numpy(), mask, TE, 1000.0, "X2", "I", "spline", myelin_T2=40.0,
                                diagnostics=True, premasked=True)
    for name in OUTPUTS:
        assert np.array_equal(nifti_io.load(out + name + ".nii.gz").get_fdata(), vol[name]), name
    assert np.array_equal(nifti_io.load(out + "MPPCA_sigma.nii.gz").get_fdata(), sigma.cpu().numpy())


def test_block_phantom_mwf_error_drops():
    """Inside the blocks of constant tissue the MWF error with MP-PCA is at most 0.85 x the error without denoising
    (measured values: DESIGN.md §10d)."""
    from test_gpu_spatial import block_phantom
    data, mask, truth, interior = block_phantom()
    mae = {}
    for name in ("None", "MPPCA"):
        d = data if name == "None" else batched.mppca_denoise(data, mask)[0].cpu().numpy()
        vol = pipeline.recon_arrays(d, mask, TE, 1000.0, "X2", "I", "spline", premasked=True)
        mae[name] = float(np.abs(vol["MWF"] - truth)[interior].mean())
    print("block phantom MWF MAE inside the blocks:", mae)
    assert mae["MPPCA"] <= 0.85 * mae["None"], mae
