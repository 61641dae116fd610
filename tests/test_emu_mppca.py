"""met2_mppca (csrc/met2_mppca.cu) under the SIMT emulator (tests/emu): the kernels' own source on the CPU, bitwise equal
to the NumPy restatement of tests/mppca_oracle.py for the denoised signals, sigma and n_signal, under the three lane
orders.  Outputs and workspaces are poisoned and canary-guarded (emu._Guarded)."""
import ctypes
import os

import numpy as np
import pytest

import mppca_oracle as O
from emu import emu

P = ctypes.c_void_p


@pytest.fixture(scope="module", autouse=True)
def _built():
    emu.build()
    L = emu.lib()
    L.met2_mppca_workspace_bytes.restype = ctypes.c_int64
    L.met2_mppca_workspace_bytes.argtypes = [ctypes.c_int] * 5
    L.met2_mppca.argtypes = [P, P] + [ctypes.c_int] * 5 + [P] * 5


def mppca(vol, mask, r):
    """met2_mppca on host arrays -> (out, sigma, n_signal)."""
    L = emu.lib()
    vol = np.ascontiguousarray(vol, dtype=np.float64)
    mask = np.ascontiguousarray(mask, dtype=np.int32)
    nx, ny, nz, nt = vol.shape
    gd = emu._Guarded()
    out = gd.array(vol.shape, np.float64, np.nan)
    sigma = gd.array(vol.shape[:3], np.float64, -7.0)
    nsig = gd.array(vol.shape[:3], np.int32, -7)
    nbytes = L.met2_mppca_workspace_bytes(nx, ny, nz, nt, r)
    assert nbytes > 0, L.met2_last_error()
    ws = gd.array(int(nbytes), np.uint8, 0xA5)
    emu._check(L.met2_mppca(emu._ptr(vol), emu._ptr(mask), nx, ny, nz, nt, r, emu._ptr(out), emu._ptr(sigma),
                            emu._ptr(nsig), emu._ptr(ws), None), "met2_mppca")
    gd.check("met2_mppca")
    return np.array(out), np.array(sigma), np.array(nsig)


def _volume(shape, nt, seed):
    """Decaying multi-echo signals with a smooth spatial variation and Gaussian noise, clipped at 0 like Step 1."""
    rng = np.random.default_rng(seed)
    nx, ny, nz = shape
    g = np.linspace(0.0, 1.0, nx)[:, None, None] + np.linspace(0.0, 0.5, ny)[None, :, None] + \
        np.linspace(0.0, 0.3, nz)[None, None, :]
    te = 10.0 * np.arange(1, nt + 1)
    clean = 400.0 * np.exp(-te / (60.0 + 20.0 * g[..., None])) + 80.0 * np.exp(-te / (20.0 + 5.0 * g[..., None]))
    vol = clean + 6.0 * rng.standard_normal(clean.shape)
    return np.maximum(vol, 0.0)


def _ellipsoid(shape):
    gx, gy, gz = (np.linspace(-1.0, 1.0, n)[s] for n, s in zip(shape, ((slice(None), None, None),
                                                                      (None, slice(None), None),
                                                                      (None, None, slice(None)))))
    return ((gx ** 2 + gy ** 2 + gz ** 2) <= 1.0).astype(np.int32)


def _check(vol, mask, r):
    ref = O.mppca(vol, mask, r)
    got = mppca(vol, mask, r)
    for a, b, name in zip(got, ref, ("out", "sigma", "n_signal")):
        assert np.array_equal(a, b, equal_nan=True), name
    return got


@pytest.mark.parametrize("nt, r, shape, masked", [
    (32, 2, (6, 5, 5), False),      # every window touches an edge
    (32, 1, (6, 6, 5), True),       # ellipsoid mask
    (48, 1, (5, 4, 4), True),
    (64, 1, (4, 4, 3), False),
    (33, 1, (4, 4, 3), False),      # odd N: the dummy index of the round-robin order
])
def test_bitwise_against_restatement(nt, r, shape, masked):
    vol = _volume(shape, nt, 40 + nt + r)
    mask = _ellipsoid(shape) if masked else np.ones(shape, dtype=np.int32)
    out, sigma, nsig = _check(vol, mask, r)
    assert (nsig[mask == 1] >= 1).any() and (out[mask != 1] == 0).all() and (sigma[mask != 1] == 0).all()


def test_single_slice_and_non_finite_window():
    """nz = 1 at r = 2: M = 25 < N = 32, so R = M - 1 and C has a null space; a NaN sample poisons exactly the voxels
    whose window holds it."""
    vol = _volume((7, 6, 1), 32, 50)
    _, _, nsig = _check(vol, np.ones((7, 6, 1)), 2)
    assert (nsig >= 0).all()
    vol[0, 0, 0, 5] = np.nan
    out, sigma, nsig = _check(vol, np.ones((7, 6, 1)), 2)
    bad = nsig == -1
    assert bad[:3, :3].all() and not bad[5:].any()
    assert np.isnan(sigma[bad]).all() and np.array_equal(out[bad], vol[bad], equal_nan=True)


@pytest.mark.parametrize("order", ["reverse", "shuffle"])
def test_lane_scheduling_orders(order):
    vol = _volume((5, 4, 4), 48, 60)
    vol[4, 3, 3, 0] = np.inf
    mask = _ellipsoid((5, 4, 4))
    base = mppca(vol, mask, 1)
    os.environ["SIMT_EMU_ORDER"] = order
    try:
        got = mppca(vol, mask, 1)
    finally:
        del os.environ["SIMT_EMU_ORDER"]
    for a, b in zip(got, base):
        assert np.array_equal(a, b, equal_nan=True)
    for a, b in zip(got, O.mppca(vol, mask, 1)):
        assert np.array_equal(a, b, equal_nan=True)


def test_argument_checks_launch_nothing():
    L = emu.lib()
    vol = np.ones((4, 3, 2, 2))
    mask = np.ones((4, 3, 2), dtype=np.int32)
    out, sigma, nsig = np.zeros_like(vol), np.zeros((4, 3, 2)), np.zeros((4, 3, 2), dtype=np.int32)
    ws = np.zeros(1 << 16, dtype=np.uint8)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    emu.counters(reset_only=True)
    launched = L.met2_launch_count()
    assert L.met2_mppca_workspace_bytes(4, 3, 2, 65, 2) == -1
    assert L.met2_mppca_workspace_bytes(4, 3, 2, 2, 0) == -1
    assert L.met2_mppca_workspace_bytes(1, 1, 1, 2, 1) == -1         # M = 1
    good = [p(vol), p(mask), 4, 3, 2, 2, 1, p(out), p(sigma), p(nsig), p(ws), None]
    for k, bad in ((0, None), (1, None), (7, None), (8, None), (9, None), (10, None), (5, 65), (5, 0), (6, 0),
                   (2, 0), (7, p(vol))):
        args = list(good)
        args[k] = bad
        assert L.met2_mppca(*args) == -1
        assert b"met2_mppca" in L.met2_last_error()
    args = list(good)
    args[2:5] = [1, 1, 1]
    assert L.met2_mppca(*args) == -1
    assert emu.counters()["launches"] == 0 and L.met2_launch_count() == launched
    mask[...] = 0                                                      # an empty mask: all-zero outputs
    out[...] = sigma[...] = 9.0
    nsig[...] = 9
    assert L.met2_mppca(*good) == 0 and emu.counters()["launches"] == 4
    assert not out.any() and not sigma.any() and not nsig.any()
