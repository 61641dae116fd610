"""Module path of the reference's motor/motor_recon_met2_real_data.py.

`motor_recon_met2` keeps the reference's signature and NIfTI outputs (motor/motor_recon_met2_real_data.py:165-506) but
replaces the two joblib voxel loops (Steps 2 and 3, :349-373 and :428-441) and the Python metrics loop (Step 4,
:443-472) by one gather -> batched GPU fit -> scatter (pipeline.recon_arrays).  Host-side preprocessing that is not on
the accelerated path: the TV denoiser (:293-303) calls scikit-image on the host, exactly like the reference, when that
package is importable (it is not in this image; SURVEY.md §2, §8f).  The NESMA denoiser
(:305-333) and the Gaussian smoothing for the FA stage (:336-346) run on the GPU (met2_nesma_filter,
met2_gaussian_smooth); the data behind the mean-spectrum figure (:375-403) is computed on the GPU and written as a text
table (Mean_spectrum_from_all_voxels.txt) instead of a PNG (no matplotlib here).
"""
import os
import threading
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from .. import _lib, batched, nifti_io, pipeline
from ..reference_api import create_Laplacian_matrix, fitting_slice_T2  # noqa: F401

OUTPUTS = ("MWF", "IEWF", "FWF", "T2_M", "T2_IE", "TWC", "FA", "fsol_4D", "Est_Signal", "reg_param")
BOOTSTRAP_OUTPUTS = tuple(name + "_bootstrap" for name in pipeline.MAP_NAMES) + ("bootstrap_n_valid",)


def tv_denoise(data):
    """Step 1, denoise == 'TV' (motor...:293-303): per echo volume, scikit-image's Chambolle total-variation filter
    with weight 2 x the estimated noise sigma — host preprocessing, kept on scikit-image like the reference."""
    try:
        from skimage.restoration import denoise_tv_chambolle, estimate_sigma
    except ImportError as exc:
        raise NotImplementedError("denoise='TV' needs scikit-image (skimage.restoration), which is not installed here; "
                                  "use --denoise NESMA (GPU) or --denoise None") from exc
    for t in range(data.shape[3]):
        vol = np.squeeze(data[:, :, :, t])
        sigma_est = np.mean(estimate_sigma(vol, channel_axis=None))
        data[:, :, :, t] = denoise_tv_chambolle(vol, weight=2.0 * sigma_est, eps=0.0002, max_num_iter=200,
                                                channel_axis=None)
    return data


def n_gpus_from_num_cores(num_cores):
    """The reference's `num_cores` (joblib workers; -1 = all, motor...:280-286) becomes the number of GPUs the voxel
    list is spread over: -1 (or anything < 1) = all visible GPUs, k = min(k, visible GPUs)."""
    import torch
    avail = max(1, torch.cuda.device_count())
    if num_cores is None or int(num_cores) < 1:
        return avail
    return min(int(num_cores), avail)


def _warm_gpus(n_gpus):
    """Create the CUDA contexts of the GPUs the fit will use and load libmet2.so — run in a thread beside the NIfTI
    load (gunzip releases the GIL).  Errors are left for the fit itself to raise."""
    try:
        import torch
        _lib.load()
        for i in range(min(int(n_gpus), torch.cuda.device_count())):
            torch.zeros(1, device="cuda:%d" % i)
        torch.cuda.synchronize()
    except Exception:
        pass


def degibbs_step1(data, mask):
    """Gibbs-ringing removal of the Step-1 output data[nx, ny, nz, nt] (batched.degibbs, in-plane axes 0 and 1, MRtrix's
    defaults), masked again with negatives clipped to 0 like Step 1's input: the state recon_arrays(premasked=True)
    expects."""
    out = batched.degibbs(data).cpu().numpy()
    np.multiply(out, mask[..., None], out=out)
    out[out < 0.0] = 0.0
    return out


def motor_recon_met2(TE_array, path_to_data, path_to_mask, path_to_save_data, TR, reg_method, reg_matrix, denoise,
                     FA_method, FA_smooth, myelin_T2, num_cores, n_bootstrap=0, bootstrap_seed=0, spatial_mu=0.0,
                     spatial_sweeps=10, parametric=False, degibbs=False, rician_sigma=None):
    """Same arguments as the reference.  `num_cores` selects the number of GPUs (-1 = all visible; see
    n_gpus_from_num_cores): the masked voxels of the volume are spread over them by pipeline.MultiGpuFit.

    n_bootstrap > 0 (not in the reference): also the per-voxel bootstrap uncertainty of the six maps with that many
    wild-bootstrap replicates per voxel (pipeline.recon_arrays), written as <MAP>_bootstrap.nii.gz (4 frames: mean,
    sd, 2.5th and 97.5th percentile) and bootstrap_n_valid.nii.gz beside the ten outputs.

    spatial_mu > 0 (not in the reference): the six maps, fsol_4D and Est_Signal are those of the spatially regularised
    fit, spatial_sweeps red-black sweeps that couple each voxel's spectrum to its face neighbours' with weight
    spatial_mu (pipeline.recon_arrays); FA and reg_param stay the point fit's.  The same ten files are written.

    parametric=True (not in the reference): also the three-pool parametric fit started from each voxel's point fit
    (pipeline.recon_arrays), written as MWF_3pool, IEWF_3pool, FWF_3pool, T2_M_3pool, T2_IE_3pool, T2_FW_3pool,
    FA_3pool, TWC_3pool, SSE_3pool and Est_Signal_3pool (.nii.gz) beside the unchanged ten outputs.

    denoise='MPPCA' (not in the reference, reached from Python only): Step 1 is Marchenko-Pastur PCA denoising on the
    GPU (batched.mppca_denoise, patch radius 2), and its per-voxel noise sigma is written as MPPCA_sigma.nii.gz beside
    the ten outputs.

    degibbs=True (not in the reference, reached from Python only): after Step 1 (denoising first, as MRtrix advises:
    unringing correlates the noise), every axial slice of every echo is unrung on the GPU (degibbs_step1, the local
    subvoxel-shift method of MRtrix3's mrdegibbs), then masked again with negatives clipped to 0.  No file is added.

    rician_sigma (not in the reference, reached from Python only): also the Rician-likelihood fit started from each
    voxel's point fit (pipeline.recon_arrays), with the noise SD rician_sigma in the data's units: a number, an
    [nx, ny, nz] array, or 'MPPCA' for the sigma map of batched.mppca_denoise on the masked data (the denoised data are
    discarded; the map is written as MPPCA_sigma.nii.gz).  Written as MWF_rician, IEWF_rician, FWF_rician, T2_M_rician,
    T2_IE_rician, TWC_rician, fsol_4D_rician, Est_Signal_rician and rician_iters (.nii.gz) beside the unchanged ten
    outputs.  The likelihood describes raw magnitude data, so it needs denoise='None' and degibbs=False."""
    if rician_sigma is not None and (denoise != 'None' or degibbs):
        raise ValueError("rician_sigma describes the noise of the raw magnitude data: it needs denoise='None' and "
                         "degibbs=False")
    n_gpus = n_gpus_from_num_cores(num_cores)
    warm = threading.Thread(target=_warm_gpus, args=(n_gpus,), daemon=True)   # CUDA contexts + libmet2.so while the files load
    warm.start()
    img = nifti_io.load(path_to_data)
    data = img.get_fdata().astype(np.float64, copy=False)
    mask = nifti_io.load(path_to_mask).get_fdata().astype(np.int64, copy=False)
    print('--------- Data shape -----------------')
    print(data.shape)
    print('--------------------------------------')
    nx, ny, nz, nt = data.shape
    np.multiply(data, mask[..., None], out=data)   # motor...:178-180, all echoes in one pass (5x faster than per echo)
    data[data < 0.0] = 0.0
    if reg_matrix not in ('I', 'L1', 'L2', 'InvT2'):
        print('Error: Wrong reg_matrix option!')
        raise SystemExit(1)
    join = (lambda name: path_to_save_data + name) if path_to_save_data.endswith('/') else \
        (lambda name: os.path.join(path_to_save_data, name))
    warm.join()
    print('Using ', n_gpus, ' GPU(s)')
    if denoise == 'TV':
        print('Step #1: Denoising using Total Variation:')
        data = tv_denoise(data)
        nifti_io.save(data, join('Data_denoised.nii.gz'), affine=img.affine)      # motor...:302-303
    if denoise == 'NESMA':
        print('Step #1: Denoising using the NESMA filter:')
        data = batched.nesma_filter(data, mask).cpu().numpy()
    mppca_sigma = None
    if denoise == 'MPPCA':
        print('Step #1: Denoising using MP-PCA:')
        den, mppca_sigma, _ = batched.mppca_denoise(data, mask)
        data, mppca_sigma = den.cpu().numpy(), mppca_sigma.cpu().numpy()
    if isinstance(rician_sigma, str):
        if rician_sigma != 'MPPCA':
            raise ValueError("rician_sigma must be a number, an array or 'MPPCA'")
        print('Noise map for the Rician fit: MP-PCA')
        _, mppca_sigma, _ = batched.mppca_denoise(data, mask)
        rician_sigma = mppca_sigma = mppca_sigma.cpu().numpy()
    if degibbs:
        print('Step #1b: Gibbs-ringing removal:')
        data = degibbs_step1(data, mask)
    print('Step #2: Estimation of flip angles:')
    data_fa = None
    if FA_smooth == 'yes':
        # per-echo Gaussian smoothing, sigma = 2 (motor...:336-346) — on the GPU, bitwise equal to scipy.ndimage
        data_fa = batched.gaussian_smooth(data, sigma=2.0)
    print('Step #3: Estimation of T2 spectra:')
    vol = pipeline.recon_arrays(data, mask, np.asarray(TE_array, dtype=np.float64), TR, reg_method, reg_matrix,
                                FA_method, myelin_T2=myelin_T2, data_fa=data_fa, diagnostics=True, premasked=True,
                                n_gpus=n_gpus, n_bootstrap=n_bootstrap, bootstrap_seed=bootstrap_seed,
                                spatial_mu=spatial_mu, spatial_sweeps=spatial_sweeps, parametric=parametric,
                                rician_sigma=rician_sigma)
    print('Step #4: Estimation of quantitative metrics')
    # the ten volumes (motor...:474-503) are written concurrently, largest first: every writer deflates with all cores
    # (nifti_io), but the eight 3-D maps are too small to keep them busy one at a time (2.2 s -> 1.2 s on 8 cores)
    names = OUTPUTS + (BOOTSTRAP_OUTPUTS if n_bootstrap > 0 else ()) + \
        (tuple(pipeline.PARAM_VOLUMES) if parametric else ()) + \
        (tuple(pipeline.RICIAN_VOLUMES) if rician_sigma is not None else ())
    order = sorted(names, key=lambda name: -vol[name].size)
    with ThreadPoolExecutor(max_workers=4) as pool:
        list(pool.map(lambda name: nifti_io.save(vol[name], join(name + '.nii.gz'), affine=img.affine), order))
    if mppca_sigma is not None:
        nifti_io.save(mppca_sigma, join('MPPCA_sigma.nii.gz'), affine=img.affine)
    dg = vol.get("diagnostics")
    if dg is not None:
        np.savetxt(join('Mean_spectrum_from_all_voxels.txt'),
                   np.column_stack([dg["T2s"], dg["mean_T2_dist"], dg["dist_T2_mean1"], dg["dist_T2_mean2"]]),
                   header="T2(ms)  mean_T2_dist(all voxels, NNLS)  dist_T2_mean1(mean signal, NNLS)  "
                          "dist_T2_mean2(mean signal, NNLS-X2-I)")
    print('Done!')
    return vol
