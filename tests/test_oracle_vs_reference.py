"""Bitwise comparison of the oracle with the unmodified reference, through the reference's own outputs stored in
tests/golden/dictionary.npz and tests/golden/voxels.npz (written by oracle/make_golden.py from the reference's modules,
imported read-only through oracle/ref_shim.py).  The 48 stored voxels include an empty, a masked-out and an
M[0] == 0 voxel."""
import numpy as np
import pytest

import met2_oracle as O


@pytest.fixture(scope="module")
def setup(golden_voxels):
    T2s = golden_voxels["T2s"]
    T1s = 1000.0 * np.ones(60)
    a273, a91, a15 = np.linspace(90.0, 180.0, 273), np.linspace(90.0, 180.0, 91), np.linspace(90.0, 180.0, 15)
    mk = lambda a: O.create_Dic_3D(60, T2s, T1s, 32, 10.0, a, 1000.0)
    return dict(a273=a273, a91=a91, a15=a15, d273=mk(a273), d91=mk(a91), d15=mk(a15))


def test_dictionary_bitwise(golden_dictionary):
    g = golden_dictionary
    D = O.create_Dic_3D(60, g["T2s"], g["T1s"], int(g["nte"]), float(g["tau"]), g["alphas"], float(g["TR"]))
    assert np.array_equal(D, g["dic"])
    T2s100 = np.logspace(1, np.log10(2000.0), 100)
    D48 = O.create_Dic_3D(100, T2s100, 1000.0 * np.ones(100), 48, 8.0, np.array([90.0, 133.0, 180.0]), 2000.0)
    assert np.array_equal(D48, g["dic48"])


def test_fa_row_workers_bitwise(golden_voxels, setup):
    g, d = golden_voxels, setup
    nx = len(g["mask"])
    b = O.fitting_slice_FA_spline_method(d["d15"], d["d273"], g["sig"], g["mask"], d["a15"], nx, d["a273"])
    a = [g["fa_spline_" + k] for k in ("deg", "idx", "km", "fsum")]
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    b = O.fitting_slice_FA_brute_force(g["mask"], g["sig"], nx, d["d91"], d["a91"])
    a = [g["fa_brute_" + k] for k in ("deg", "idx", "km", "fsum")]
    assert all(np.array_equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("method,rm", [("X2", "I"), ("X2", "L2"), ("L_curve", "L1"), ("GCV", "I"), ("GCV", "L2"),
                                       ("BayesReg", "I"), ("BayesReg", "InvT2"), ("T2SPARC", "InvT2"), ("NNLS", "I")])
def test_t2_row_worker_bitwise(golden_voxels, setup, method, rm):
    g = golden_voxels
    nx = len(g["mask"])
    gr = O._grids(method, rm, "spline", 40.0, 32, 10.0, 1000.0, npc=60)
    assert np.array_equal(gr["lambda_reg"], g["lambda_reg"])
    a = [g["t2_%s_%s_%s" % (method, rm, k)] for k in ("f", "s", "reg")]
    b = O.fitting_slice_T2(g["mask"], g["sig"], g["fa_spline_idx"], nx, setup["d273"], gr["lambda_reg"], 60, 32, method,
                           gr["L"])
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
