"""Module path of the reference's motor/motor_recon_met2_real_data_ROI.py.

`motor_recon_met2_ROIs` keeps the reference's signature (:152) and tabular outputs (table_MWF.csv, table_Spectra.csv,
ROI_labels.csv, ROI_<label>/table_values.{txt,csv}; :474-503).  The FA stage is the batched GPU call of the voxel-wise
pipeline; the per-ROI mean signal / mean kernel (:405-423, a Python triple loop over the volume per ROI) is one
segmented reduction on the GPU (met2_segment_means) and the per-ROI X2 fits (factor 1.01, :427) are one batched
met2_t2_fit over the ROIs.  Figures are not produced (no matplotlib here).
"""
import os

import numpy as np
from tabulate import tabulate

from .. import batched, nifti_io, pipeline
from .motor_recon_met2_real_data import degibbs_step1, tv_denoise


def motor_recon_met2_ROIs(TE_array, path_to_data, path_to_mask, path_to_ROIs, path_to_save_data, TR, reg_matrix, denoise,
                          FA_method, FA_smooth, myelin_T2, num_cores, degibbs=False, slice_profile=None):
    """Same arguments as the reference.  slice_profile = (x, r, w) (not in the reference; grids.slice_profile): the
    flip-angle search and the ROI fits run on the slice-profile-integrated EPG dictionary of 2-D multi-slice data
    (pipeline.recon_arrays)."""
    img = nifti_io.load(path_to_data)
    data = img.get_fdata().astype(np.float64, copy=False)
    mask = nifti_io.load(path_to_mask).get_fdata().astype(np.int64, copy=False)
    ROIs = nifti_io.load(path_to_ROIs).get_fdata().astype(np.int64, copy=False)
    nx, ny, nz, nt = data.shape
    np.multiply(data, mask[..., None], out=data)   # :181-182, all echoes in one pass
    data[data < 0.0] = 0.0
    if reg_matrix not in ('I', 'L1', 'L2', 'InvT2'):
        print('Error: Wrong reg_matrix option!')
        raise SystemExit(1)
    if denoise == 'TV':
        data = tv_denoise(data)
    if denoise == 'NESMA':
        data = batched.nesma_filter(data, mask).cpu().numpy()
    if denoise == 'MPPCA':      # not in the reference: MP-PCA on the GPU (batched.mppca_denoise), reached from Python
        data = batched.mppca_denoise(data, mask)[0].cpu().numpy()
    if degibbs:                 # not in the reference: Gibbs-ringing removal after Step 1, as motor_recon_met2(degibbs=True)
        data = degibbs_step1(data, mask)
    data_fa = batched.gaussian_smooth(data, sigma=2.0) if FA_smooth == 'yes' else None
    vol = pipeline.recon_arrays(data, mask, np.asarray(TE_array, dtype=np.float64), TR, "X2", reg_matrix, FA_method,
                                myelin_T2=myelin_T2, data_fa=data_fa, diagnostics=True, rois=ROIs, premasked=True,
                                fa_only=True,   # the ROI estimator never fits voxel spectra (reference :349-445)
                                slice_profile=slice_profile)
    roi = vol["roi"]
    join = (lambda name: path_to_save_data + name) if path_to_save_data.endswith('/') else \
        (lambda name: os.path.join(path_to_save_data, name))
    for i, label in enumerate(roi["roi_values"]):
        d = join('ROI_' + repr(int(label)) + '/')
        os.makedirs(d, exist_ok=True)
        table = [['1. MWF       ', roi["MWF_ROIs"][i]], ['2. IEWF      ', roi["IEWF_ROIs"][i]],
                 ['3. FWF       ', roi["FWF_ROIs"][i]], ['4. T2M       ', roi["T2M_ROIs"][i]],
                 ['5. T2IE      ', roi["T2IE_ROIs"][i]], ['6. TWC       ', roi["TWC_ROIs"][i]]]
        with open(d + 'table_values.txt', 'w') as fh:
            fh.write(tabulate(table, headers=['Parameter    ', 'Mean value']))
        np.savetxt(d + 'table_values.csv', table, delimiter=",", fmt='%s')
    np.savetxt(join('table_MWF.csv'), roi["MWF_ROIs"], delimiter=",", fmt='%s')
    np.savetxt(join('table_Spectra.csv'), roi["fsol_ROIs"], delimiter=",", fmt='%s')
    np.savetxt(join('ROI_labels.csv'), roi["roi_values"], delimiter=",", fmt='%s')
    print('Done!')
    return vol
