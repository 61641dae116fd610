#!/usr/bin/env python
"""CLI of the voxel-wise MET2 reconstruction — same flags, types, defaults, `required` settings and output-folder naming
as the reference's run_real_data_script.py:18-62,82-93,119-122; the fit itself runs on the GPU(s)
(multicomponent_t2_toolbox_b200; --numcores = number of GPUs).
Plotting (--savefig) needs matplotlib + LaTeX, which this image lacks; the NIfTI outputs carry the same names the
reference's plot scripts read."""
from __future__ import division

import argparse
import os
import time

import numpy as np
from tabulate import tabulate

from multicomponent_t2_toolbox_b200.motor.motor_recon_met2_real_data import motor_recon_met2


# (flag, type, default, choices, required, help) — the reference's flags, types, defaults, choices and `required`
# settings (run_real_data_script.py:18-62): every flag is required there except --numcores (default -1 = all).
# tests/test_nifti_cli.py diffs this table against the reference's argparse block (tests/golden/reference_cli_flags.json).
_FLAGS = [
    ("--path_to_folder", str, None, None, True, "folder that holds the data, mask and the output directory (trailing '/')"),
    ("--input", str, None, None, True, "4-D multi-echo NIfTI file inside the folder"),
    ("--mask", str, None, None, True, "3-D brain-mask NIfTI file inside the folder"),
    ("--minTE", float, None, None, True, "first echo time = echo spacing, ms"),
    ("--nTE", int, 32, None, True, "number of echoes"),
    ("--TR", float, None, None, True, "repetition time, ms"),
    ("--FA_method", str, "spline", ["spline", "brute-force"], True,
     "flip-angle search: 15-knot spline + Brent, or exhaustive 1-degree grid"),
    ("--FA_smooth", str, "yes", ["yes", "no"], True, "Gaussian-smooth (sigma 2) the data used for the flip-angle search"),
    ("--denoise", str, "None", ["TV", "NESMA", "None"], True,
     "pre-processing denoiser (NESMA runs on the GPU; TV needs scikit-image on the host)"),
    ("--reg_method", str, "X2", ["NNLS", "T2SPARC", "X2", "L_curve", "GCV", "BayesReg"], True,
     "regularisation-weight selector"),
    ("--reg_matrix", str, "I", ["I", "L1", "L2", "InvT2"], True, "Tikhonov matrix"),
    ("--numcores", int, -1, None, False,
     "number of workers; here: number of GPUs the voxel slabs are spread over, -1 = all visible GPUs"),
    ("--myelin_T2_cutoff", float, 40, None, True, "upper T2 bound of the myelin-water compartment, ms"),
    ("--savefig", str, "yes", ["yes", "no"], True, "save PNG maps (needs matplotlib; skipped with a message if absent)"),
    ("--savefig_slice", int, 30, None, True, "axial slice for the PNG maps"),
]


def build_parser():
    parser = argparse.ArgumentParser(description='Myelin Water Imaging')
    for flag, typ, default, choices, required, text in _FLAGS:
        kw = dict(type=typ, default=default, help=text)
        if required:
            kw["required"] = True
        if choices:
            kw["choices"] = choices
        parser.add_argument(flag, **kw)
    return parser


def main(argv=None):
    args = build_parser().parse_args(argv)
    start_time = time.time()
    path_to_folder = args.path_to_folder
    path_to_data = path_to_folder + args.input
    path_to_mask = path_to_folder + args.mask
    reg_method, reg_matrix = args.reg_method, args.reg_matrix
    if reg_method in ('NNLS', 'T2SPARC'):
        path_to_save_data = path_to_folder + 'recon_all_' + reg_method + '/'
    else:
        path_to_save_data = path_to_folder + 'recon_all_' + reg_method + '-' + reg_matrix + '/'
    if reg_method == 'T2SPARC':
        reg_matrix = 'InvT2'
    headers = ['Selected options', '   ']
    table = [["Regularization method", reg_method], ["Regularization matrix", reg_matrix], ["Denoising method", args.denoise],
             ["TR (ms)", args.TR], ["Minimum TE (ms)", args.minTE], ["Number of TEs", args.nTE],
             ["Flip angle (FA) method", args.FA_method], ["Smooth image for FA estimation", args.FA_smooth],
             ["Myelin T2 cutoff (ms)", args.myelin_T2_cutoff], ["Number of GPUs (-1 = all)", args.numcores],
             ["Save figures", args.savefig]]
    print(tabulate(table, headers=headers, tablefmt="fancy_grid"))
    try:
        os.mkdir(path_to_save_data)
    except OSError:
        print("Creation of the directory %s failed" % path_to_save_data)
    else:
        print("Successfully created the directory %s " % path_to_save_data)
    TE_array = args.minTE * np.arange(1, args.nTE + 1)
    TE_array = np.array(TE_array)
    motor_recon_met2(TE_array, path_to_data, path_to_mask, path_to_save_data, args.TR, reg_method, reg_matrix,
                     args.denoise, args.FA_method, args.FA_smooth, args.myelin_T2_cutoff, args.numcores)
    if args.savefig == 'yes':
        print("--savefig: plotting needs matplotlib with LaTeX (not available here); the NIfTI maps were written to "
              + path_to_save_data)
    print("--- %s seconds ---" % (time.time() - start_time))


if __name__ == "__main__":
    main()
