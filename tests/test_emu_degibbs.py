"""met2_degibbs (csrc/met2_degibbs.cu) under the SIMT emulator (tests/emu): the kernels' own source on the CPU, bitwise
equal to the NumPy restatement of tests/degibbs_oracle.py fed with the library's tables, under the three lane orders.
Outputs and workspaces are poisoned and canary-guarded (emu._Guarded)."""
import ctypes
import os

import numpy as np
import pytest

import degibbs_oracle as O
from emu import emu

P = ctypes.c_void_p


@pytest.fixture(scope="module", autouse=True)
def _built():
    _bind()


def _bind():
    emu.build()
    L = emu.lib()
    L.met2_degibbs_tables.restype = ctypes.c_int64
    L.met2_degibbs_tables.argtypes = [ctypes.c_int, ctypes.c_int, P]
    L.met2_degibbs_workspace_bytes.restype = ctypes.c_int64
    L.met2_degibbs_workspace_bytes.argtypes = [ctypes.c_int] * 7
    L.met2_degibbs.argtypes = [P] + [ctypes.c_int] * 7 + [P] * 3
    return L


def tables(n, nsh=O.NSH):
    """met2_degibbs_tables of the emulator build (the library's host function, compiled for the CPU)."""
    L = _bind()
    k = L.met2_degibbs_tables(n, nsh, None)
    assert k == n * (2 * nsh + 4), L.met2_last_error()
    out = np.full(k, np.nan)
    assert L.met2_degibbs_tables(n, nsh, emu._ptr(out)) == k
    return out


def degibbs(vol, nsh=O.NSH, minW=O.MINW, maxW=O.MAXW):
    """met2_degibbs on a host array [nx, ny, nz, nt]."""
    L = emu.lib()
    vol = np.ascontiguousarray(vol, dtype=np.float64)
    nx, ny, nz, nt = vol.shape
    gd = emu._Guarded()
    out = gd.array(vol.shape, np.float64, np.nan)
    nbytes = L.met2_degibbs_workspace_bytes(nx, ny, nz, nt, nsh, minW, maxW)
    assert nbytes > 0, L.met2_last_error()
    ws = gd.array(int(nbytes), np.uint8, 0xA5)
    emu._check(L.met2_degibbs(emu._ptr(vol), nx, ny, nz, nt, nsh, minW, maxW, emu._ptr(out), emu._ptr(ws), None),
               "met2_degibbs")
    gd.check("met2_degibbs")
    return np.array(out)


def _volume(shape, seed):
    """Blocks of constant intensity with a decay over the last axis, plus noise: edges that ring, and a TV argmin that
    is not always q = 0."""
    rng = np.random.default_rng(seed)
    nx, ny, nz, nt = shape
    x = np.arange(nx)[:, None, None, None]
    y = np.arange(ny)[None, :, None, None]
    img = 100.0 * ((np.abs(x - nx / 2) < nx / 4) & (np.abs(y - ny / 2) < ny / 3)) + 40.0 * (x > 0.7 * nx)
    img = img * np.exp(-np.arange(nt) / 10.0)[None, None, None, :] * np.ones((1, 1, nz, 1))
    return img + rng.standard_normal(shape)


def _check(vol, nsh=O.NSH, minW=O.MINW, maxW=O.MAXW):
    ref = O.degibbs(vol, tables(vol.shape[0], nsh), tables(vol.shape[1], nsh), nsh, minW, maxW)
    got = degibbs(vol, nsh, minW, maxW)
    assert np.array_equal(got, ref, equal_nan=True)
    return got


@pytest.mark.parametrize("shape, nsh, minW, maxW", [
    ((16, 16, 1, 1), 20, 1, 3),
    ((16, 16, 1, 32), 20, 1, 3),      # 32 slices: two CTAs of slices
    ((17, 24, 2, 3), 20, 1, 3),       # odd x even, non-square, a partial CTA of slices
    ((17, 24, 1, 1), 1, 2, 2),        # nsh = 1, minW = maxW
    ((64, 48, 1, 1), 20, 0, 0),
    ((9, 13, 1, 2), 20, 4, 4),        # maxW at its limit for n = 9
])
def test_bitwise_against_restatement(shape, nsh, minW, maxW):
    vol = _volume(shape, 3 + shape[0])
    out = _check(vol, nsh, minW, maxW)
    assert np.isfinite(out).all() and not np.array_equal(out, vol)


@pytest.mark.parametrize("shape", [(1, 1, 1, 3), (1, 5, 2, 1), (6, 1, 1, 2), (2, 2, 1, 1)])
def test_smallest_in_plane_sizes(shape):
    """n = 1 and 2 with minW = maxW = 0, the only window they allow: the padded positions of the last thread row wrap
    more than once (the emulator bounds-checks every shared-memory access)."""
    _check(_volume(shape, 11), minW=0, maxW=0)


def test_limit_size():
    """The largest in-plane size (256 x 256: 1024 threads per unringing CTA)."""
    _check(_volume((256, 256, 1, 1), 5), nsh=1)


def test_non_finite_slices():
    """A NaN in one slice and an Inf in another: the transforms spread them over their slice only."""
    vol = _volume((17, 24, 1, 3), 8)
    vol[3, 5, 0, 0] = np.nan
    vol[10, 2, 0, 2] = np.inf
    out = _check(vol)
    assert not np.isfinite(out[..., 0, 0]).any() and np.isfinite(out[..., 0, 1]).all()


@pytest.mark.parametrize("order", ["reverse", "shuffle"])
def test_lane_scheduling_orders(order):
    vol = _volume((17, 24, 1, 19), 9)
    vol[0, 0, 0, 4] = np.nan
    base = degibbs(vol)
    os.environ["SIMT_EMU_ORDER"] = order
    try:
        got = degibbs(vol)
    finally:
        del os.environ["SIMT_EMU_ORDER"]
    assert np.array_equal(got, base, equal_nan=True)
    assert np.array_equal(got, O.degibbs(vol, tables(17), tables(24)), equal_nan=True)


@pytest.mark.parametrize("n, nsh", [(16, 20), (17, 1), (96, 20), (256, 20)])
def test_tables(n, nsh):
    """Layout and values of met2_degibbs_tables against the closed forms the restatement expects."""
    cs, sn, c, h = O.split_tables(tables(n, nsh), n, nsh)
    r = np.arange(n)
    f = np.fft.fftfreq(n)
    s = O.shifts(nsh) / (2 * nsh)
    assert np.abs(cs - np.cos(2 * np.pi * r / n)).max() <= 1e-15
    assert np.abs(sn - np.sin(2 * np.pi * r / n)).max() <= 1e-15
    assert np.abs(c - (1.0 + np.cos(2 * np.pi * f))).max() <= 1e-15
    href = np.real(np.fft.ifft(np.exp(2j * np.pi * f[None, :] * s[:, None]), axis=1))
    assert np.abs(h - href).max() <= 1e-15
    assert h[0, 0] == 1.0 and np.abs(h[0, 1:]).max() <= 1e-15
    if n % 2 == 0:
        assert c[n // 2] == 0.0                       # exactly: G0's special case depends on it


def test_argument_checks_launch_nothing():
    L = emu.lib()
    vol = np.ones((8, 8, 2, 2))
    out = np.zeros_like(vol)
    ws = np.zeros(1 << 20, dtype=np.uint8)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    emu.counters(reset_only=True)
    launched = L.met2_launch_count()
    good = [p(vol), 8, 8, 2, 2, 20, 1, 3, p(out), p(ws), None]
    assert L.met2_degibbs_workspace_bytes(*good[1:8]) > 0
    bad_sizes = [(1, 0), (1, 257), (2, 0), (2, 257), (3, 0), (4, 0),
                 (5, 0), (6, -1), (6, 4), (7, 4), (7, 8)]              # nsh < 1, minW < 0, minW > maxW, maxW >= n/2
    for k, v in bad_sizes:
        args = list(good)
        args[k] = v
        assert L.met2_degibbs_workspace_bytes(*args[1:8]) == -1
        assert L.met2_degibbs(*args) == -1
        assert b"met2_degibbs" in L.met2_last_error()
    args = list(good)
    args[1:3] = [256, 256]
    args[5] = 41                                                        # (2 nsh + 33) 8 n > 227 KB
    assert L.met2_degibbs_workspace_bytes(*args[1:8]) == -1
    args[5] = 40
    assert L.met2_degibbs_workspace_bytes(*args[1:8]) > 0
    args = list(good)
    args[2], args[7] = 5, 3                                             # maxW >= n/2 on axis 1 only
    assert L.met2_degibbs(*args) == -1
    for k, v in ((0, None), (8, None), (9, None), (8, p(vol))):        # NULL pointers, out aliasing vol
        args = list(good)
        args[k] = v
        assert L.met2_degibbs(*args) == -1
        assert b"met2_degibbs" in L.met2_last_error()
    assert L.met2_degibbs_tables(0, 20, None) == -1 and L.met2_degibbs_tables(257, 20, None) == -1
    assert L.met2_degibbs_tables(16, 0, None) == -1
    assert emu.counters()["launches"] == 0 and L.met2_launch_count() == launched
    assert L.met2_degibbs(*good) == 0 and emu.counters()["launches"] == 7
