"""batched.degibbs (met2_degibbs) on the device: bitwise equal to the NumPy restatement of tests/degibbs_oracle.py (fed
with libmet2.so's own tables) on a crop and on a sample of slices of the 96 x 96 x 60 x 32 phantom, repeatable, other
in-plane axes equal to a permuted call, the files of motor_recon_met2(degibbs=True, denoise='MPPCA'), and the MWF
error on a block phantom with ringing."""
import ctypes
import os

import numpy as np
import pytest
import torch

import degibbs_oracle as O
from multicomponent_t2_toolbox_b200 import _lib, batched, nifti_io, pipeline
from multicomponent_t2_toolbox_b200.phantom import epg_signal_batch, make_phantom

pytestmark = pytest.mark.gpu

TE = 10.0 * np.arange(1, 33)


def tables(n, nsh=O.NSH):
    """met2_degibbs_tables of libmet2.so."""
    lib = _lib.load()
    k = int(lib.met2_degibbs_tables(n, nsh, None))
    out = np.full(k, np.nan)
    assert lib.met2_degibbs_tables(n, nsh, out.ctypes.data_as(ctypes.c_void_p)) == k
    return out


@pytest.fixture(scope="module")
def phantom():
    ph = make_phantom((96, 96, 60), seed=2, fa_mode="b1", mask_mode="ellipsoid", backend="gpu")
    data = ph["data"] * ph["mask"][..., None]          # motor_recon_met2: data * mask, negatives clipped
    data[data < 0.0] = 0.0
    return np.ascontiguousarray(data), ph["mask"]


def test_bitwise_on_a_crop(phantom):
    data, _ = phantom
    crop = np.ascontiguousarray(data[10:42, 30:54, 28:30, :])
    ref = O.degibbs(crop, tables(32), tables(24))
    assert np.array_equal(batched.degibbs(crop).cpu().numpy(), ref)


def test_bitwise_on_sample_slices_of_the_full_volume_and_repeatable(phantom):
    data, _ = phantom
    d = torch.as_tensor(data).cuda()
    a = batched.degibbs(d)
    assert torch.equal(a, batched.degibbs(d))
    out = a.cpu().numpy()
    rng = np.random.default_rng(3)
    z, t = rng.integers(0, 60, 8), rng.integers(0, 32, 8)
    ref = O.degibbs(np.ascontiguousarray(data[:, :, z, t]), tables(96), tables(96))
    assert np.array_equal(out[:, :, z, t], ref)


@pytest.mark.parametrize("shape", [(1, 1, 2, 3), (1, 5, 2, 1), (6, 1, 1, 2)])
def test_smallest_in_plane_sizes(shape):
    """n = 1 with minW = maxW = 0: the padded positions of the last thread row wrap more than once."""
    vol = np.random.default_rng(4).standard_normal(shape) + 10.0
    ref = O.degibbs(vol, tables(shape[0]), tables(shape[1]), minW=0, maxW=0)
    assert np.array_equal(batched.degibbs(vol, minW=0, maxW=0).cpu().numpy(), ref)


def test_other_axes_equal_a_permuted_call(phantom):
    data, _ = phantom
    d = torch.as_tensor(np.ascontiguousarray(data[20:60, 30:62, 20:44, :4])).cuda()
    got = batched.degibbs(d, axes=(0, 2))
    ref = batched.degibbs(d.permute(0, 2, 1, 3)).permute(0, 2, 1, 3)
    assert got.shape == d.shape and torch.equal(got, ref)
    got = batched.degibbs(d, axes=(2, 1))
    ref = batched.degibbs(d.permute(2, 1, 0, 3)).permute(2, 1, 0, 3)
    assert torch.equal(got, ref)


def test_motor_recon_met2_with_degibbs_after_mppca(tmp_path):
    from multicomponent_t2_toolbox_b200.motor.motor_recon_met2_real_data import (OUTPUTS, degibbs_step1,
                                                                                 motor_recon_met2)
    ph = make_phantom((12, 10, 6), seed=9, fa_mode="b1", mask_mode="ellipsoid")
    nifti_io.save(ph["data"], str(tmp_path / "Data.nii.gz"))
    nifti_io.save(ph["mask"].astype(np.int16), str(tmp_path / "Mask.nii.gz"))
    out = str(tmp_path / "out") + "/"
    os.mkdir(out)
    motor_recon_met2(TE, str(tmp_path / "Data.nii.gz"), str(tmp_path / "Mask.nii.gz"), out, 1000.0, "X2", "I", "MPPCA",
                     "spline", "no", 40.0, -1, degibbs=True)
    assert {n + ".nii.gz" for n in OUTPUTS} | {"MPPCA_sigma.nii.gz"} <= set(os.listdir(out))
    data = nifti_io.load(str(tmp_path / "Data.nii.gz")).get_fdata()
    mask = nifti_io.load(str(tmp_path / "Mask.nii.gz")).get_fdata().astype(np.int64)
    data = data * mask[..., None]
    data[data < 0.0] = 0.0
    step1 = degibbs_step1(batched.mppca_denoise(data, mask)[0].cpu().numpy(), mask)
    assert (step1 >= 0.0).all() and not step1[mask != 1].any()
    vol = pipeline.recon_arrays(step1, mask, TE, 1000.0, "X2", "I", "spline", myelin_T2=40.0, diagnostics=True,
                                premasked=True)
    inside = mask == 1
    for name in OUTPUTS:
        written = nifti_io.load(out + name + ".nii.gz").get_fdata()
        assert np.array_equal(written, vol[name]), name
        assert np.isfinite(written[inside]).all(), name


def ringing_block_phantom(n=30, block=6, nz=4, snr=50.0, seed=21):
    """Blocks of constant tissue, a third of them CSF-like (free water only), on a 2n x 2n grid; every echo's k-space
    is truncated to the central n x n (the acquisition) and Rician noise at SNR 50 of the tissue's first echo is added.
    Returns (data [n, n, nz, 32], mask, truth MWF, tissue: voxels of non-CSF blocks, near: tissue voxels within two
    voxels of a CSF block)."""
    rng = np.random.default_rng(seed)
    nb = n // block
    csf = rng.random((nb, nb)) < 1.0 / 3.0
    mwf = np.where(csf, 0.0, rng.uniform(0.05, 0.3, (nb, nb)))
    fwf = np.where(csf, 1.0, rng.uniform(0.0, 0.05, (nb, nb)))
    t2m, t2ie = rng.uniform(15.0, 30.0, (nb, nb)), rng.uniform(60.0, 90.0, (nb, nb))
    B = nb * nb
    T1, fa = np.full(B, 1000.0), np.full(B, 170.0)
    sig = (mwf.ravel()[:, None] * epg_signal_batch(32, 10.0, T1, t2m.ravel(), fa)
           + (1.0 - mwf - fwf).ravel()[:, None] * epg_signal_batch(32, 10.0, T1, t2ie.ravel(), fa)
           + fwf.ravel()[:, None] * epg_signal_batch(32, 10.0, T1, np.full(B, 2000.0), fa))
    sig *= 1000.0 * (1.0 - np.exp(-1.0))
    f = 2 * block
    fine = np.repeat(np.repeat(sig.reshape(nb, nb, 32), f, axis=0), f, axis=1)          # [2n, 2n, 32]
    k = np.fft.fftfreq(n, 1.0 / n).astype(int) % (2 * n)
    coarse = np.real(np.fft.ifft2(np.fft.fft2(fine, axes=(0, 1))[np.ix_(k, k)], axes=(0, 1))) / 4.0
    clean = np.repeat(coarse[:, :, None, :], nz, axis=2)
    sigma = np.median(sig[~csf.ravel(), 0]) / snr
    data = np.sqrt((clean + sigma * rng.standard_normal(clean.shape)) ** 2
                   + (sigma * rng.standard_normal(clean.shape)) ** 2)
    lab = np.arange(n) // block
    csf_vox = csf[lab[:, None], lab[None, :]]
    near = ~csf_vox & np.array([[csf_vox[max(i - 2, 0):i + 3, max(j - 2, 0):j + 3].any() for j in range(n)]
                                for i in range(n)])
    rep = lambda a: np.repeat(a[:, :, None], nz, axis=2)
    truth = rep(mwf[lab[:, None], lab[None, :]])
    return data, np.ones((n, n, nz)), truth, rep(~csf_vox), rep(near)


def mwf_mae_with_and_without_degibbs():
    from multicomponent_t2_toolbox_b200.motor.motor_recon_met2_real_data import degibbs_step1
    data, mask, truth, tissue, near = ringing_block_phantom()
    res = {}
    for name in ("None", "degibbs"):
        d = data if name == "None" else degibbs_step1(data, mask)
        vol = pipeline.recon_arrays(d, mask, TE, 1000.0, "X2", "I", "spline", premasked=True)
        err = np.abs(vol["MWF"] - truth)
        res[name] = {"tissue": float(err[tissue].mean()), "near_csf": float(err[near].mean())}
    return res


def test_block_phantom_with_ringing_mwf_error():
    """MWF MAE (spline + X2-I) in the tissue of the ringing block phantom, with and without unringing.  Measured on a
    B200: tissue 0.0850 -> 0.0780 (ratio 0.917), tissue within two voxels of CSF 0.0999 -> 0.0855 (ratio 0.855);
    DESIGN.md §10e.  The bounds leave a few per cent of margin."""
    mae = mwf_mae_with_and_without_degibbs()
    print("ringing block phantom MWF MAE:", mae)
    assert mae["degibbs"]["tissue"] <= 0.95 * mae["None"]["tissue"], mae
    assert mae["degibbs"]["near_csf"] <= 0.9 * mae["None"]["near_csf"], mae
