"""met2_noise_sigma and met2_tv_chambolle (csrc/met2_tv.cu) under the SIMT emulator (tests/emu): the kernels' own source
on the CPU, bitwise equal to the NumPy restatement of tests/tv_oracle.py for sigma, the denoised volume and the
iteration counts.  Outputs and workspaces are poisoned and canary-guarded (emu._Guarded)."""
import ctypes
import os

import numpy as np
import pytest

import tv_oracle as T
from emu import emu


P = ctypes.c_void_p


@pytest.fixture(scope="module", autouse=True)
def _built():
    emu.build()
    L = emu.lib()
    for name in ("met2_noise_sigma_workspace_bytes", "met2_tv_workspace_bytes"):
        getattr(L, name).restype = ctypes.c_int64
        getattr(L, name).argtypes = [ctypes.c_int] * 4
    L.met2_noise_sigma.argtypes = [P] + [ctypes.c_int] * 4 + [P, P, P]
    L.met2_tv_chambolle.argtypes = [P] + [ctypes.c_int] * 4 + [P, ctypes.c_double, ctypes.c_int, P, P, P, P]


def noise_sigma(vol):
    """met2_noise_sigma on host arrays: vol[nx, ny, nz, nt] -> sigma [nt] (poisoned, canary-guarded output and
    workspace)."""
    L = emu.lib()
    vol = np.ascontiguousarray(vol, dtype=np.float64)
    nx, ny, nz, nt = vol.shape
    gd = emu._Guarded()
    sigma = gd.array(nt, np.float64, -7.0)
    nbytes = L.met2_noise_sigma_workspace_bytes(nx, ny, nz, nt)
    assert nbytes >= 0, L.met2_last_error()
    ws = gd.array(int(nbytes), np.uint8, 0xA5)
    emu._check(L.met2_noise_sigma(emu._ptr(vol), nx, ny, nz, nt, emu._ptr(sigma), emu._ptr(ws), None),
               "met2_noise_sigma")
    gd.check("met2_noise_sigma")
    return np.array(sigma)


def tv_chambolle(vol, weight, eps=2e-4, max_iter=200):
    """met2_tv_chambolle on host arrays: vol[nx, ny, nz, nt], weight[nt] -> (out like vol, iterations [nt] int32)."""
    L = emu.lib()
    vol = np.ascontiguousarray(vol, dtype=np.float64)
    nx, ny, nz, nt = vol.shape
    weight = np.ascontiguousarray(np.broadcast_to(np.asarray(weight, dtype=np.float64), (nt,)))
    gd = emu._Guarded()
    out = gd.array(vol.shape, np.float64, np.nan)
    iters = gd.array(nt, np.int32, -7)
    nbytes = L.met2_tv_workspace_bytes(nx, ny, nz, nt)
    assert nbytes >= 0, L.met2_last_error()
    ws = gd.array(int(nbytes), np.uint8, 0xA5)
    emu._check(L.met2_tv_chambolle(emu._ptr(vol), nx, ny, nz, nt, emu._ptr(weight), float(eps), int(max_iter),
                                   emu._ptr(out), emu._ptr(iters), emu._ptr(ws), None), "met2_tv_chambolle")
    gd.check("met2_tv_chambolle")
    return np.array(out), np.array(iters)


def _check_against_restatement(vol, max_iter=200, weight=None):
    """sigma (always) and the TV filter with weight = 2 sigma, or with the given per-echo weights."""
    s = noise_sigma(vol)
    sigma = np.array([T.estimate_sigma(np.squeeze(vol[..., t])) for t in range(vol.shape[3])])
    assert np.array_equal(s, sigma, equal_nan=True)
    if weight is None:
        weight = 2.0 * sigma
    ref = np.empty_like(vol)
    iters = np.zeros(vol.shape[3], dtype=np.int32)
    for t in range(vol.shape[3]):
        den, iters[t] = T.denoise_tv_chambolle(np.squeeze(vol[..., t]), weight[t], 2e-4, max_iter)
        ref[..., t] = den.reshape(vol.shape[:3])
    out, it = tv_chambolle(vol, weight, 2e-4, max_iter)
    assert np.array_equal(it, iters), (it, iters)
    assert np.array_equal(out, ref, equal_nan=True)
    return out, it, s


def _noisy(shape, seed, level=100.0, noise=8.0):
    rng = np.random.default_rng(seed)
    return level + noise * rng.standard_normal(shape)


def test_volume_with_a_masked_out_region():
    vol = _noisy((11, 9, 7, 3), 21)
    vol[:4, :3] = 0.0
    out, it, s = _check_against_restatement(vol)
    assert (it > 1).all() and (it < 200).all() and np.isfinite(s).all()


def test_squeezed_axes():
    _check_against_restatement(_noisy((12, 10, 1, 2), 22))       # 2-D, tau = 1/4
    _check_against_restatement(_noisy((17, 1, 1, 1), 23))        # 1-D, tau = 1/2
    _check_against_restatement(_noisy((1, 6, 9, 2), 24))         # leading axis dropped


def test_iteration_cap():
    out, it, _ = _check_against_restatement(_noisy((9, 8, 6, 2), 25), max_iter=5)
    assert (it == 5).all()


def test_constant_and_all_zero_echoes():
    vol = _noisy((6, 5, 4, 3), 26)
    vol[..., 1] = 7.0            # constant: the db2 taps sum to ~1e-16, not 0, so sigma is tiny but not NaN
    vol[..., 2] = 0.0            # all zero: no nonzero coefficient -> sigma NaN, output NaN
    out, it, s = _check_against_restatement(vol, max_iter=30)
    assert np.isfinite(s[:2]).all() and s[1] < 1e-40 and np.isnan(s[2])
    assert np.isnan(out[..., 2]).all() and (it[1:] == 30).all()
    # a constant echo with a finite weight runs every iteration (E_init = 0) and comes back unchanged
    out, it, _ = _check_against_restatement(vol[..., 1:2].copy(), max_iter=30, weight=np.array([1.0]))
    assert it[0] == 30 and np.array_equal(out, vol[..., 1:2])


@pytest.mark.parametrize("n, parity", [(17, 0), (16, 1)])
def test_median_of_an_even_and_an_odd_count(n, parity):
    """1-D volumes of random data: every coefficient is nonzero, so the count is the band length (n + 3) // 2."""
    vol = _noisy((n, 1, 1, 2), 27 + n)
    assert np.count_nonzero(T.dwt_detail(vol[:, 0, 0, 0])) % 2 == parity
    _check_against_restatement(vol)
    # a 3-D band with a constant region, where many coefficients are exactly zero
    vol3 = _noisy((n, 5, 4, 1), 28 + n)
    vol3[: n // 2] = 3.0
    assert np.array_equal(noise_sigma(vol3), [T.estimate_sigma(vol3[..., 0])])


def test_larger_volume_with_several_partials_per_echo():
    """64 x 64 x 66 voxels: 2^11 depth-K nodes of NumPy's pairwise tree, 64 partial sums per echo field."""
    vol = _noisy((64, 64, 66, 1), 29)
    _check_against_restatement(vol, max_iter=3)


@pytest.mark.parametrize("order", ["reverse", "shuffle"])
def test_lane_scheduling_orders(order):
    vol = _noisy((10, 7, 5, 2), 30)
    vol[:3] = 0.0
    base_s = noise_sigma(vol)
    base = tv_chambolle(vol, 2.0 * base_s, 2e-4, 200)
    os.environ["SIMT_EMU_ORDER"] = order
    try:
        s = noise_sigma(vol)
        out = tv_chambolle(vol, 2.0 * s, 2e-4, 200)
    finally:
        del os.environ["SIMT_EMU_ORDER"]
    assert np.array_equal(s, base_s)
    assert np.array_equal(out[0], base[0]) and np.array_equal(out[1], base[1])


def test_argument_checks_launch_nothing():
    L = emu.lib()
    vol = np.ones((4, 3, 2, 2))
    out = np.zeros_like(vol)
    w = np.ones(2)
    it = np.zeros(2, dtype=np.int32)
    ws = np.zeros(1 << 20, dtype=np.uint8)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    emu.counters(reset_only=True)
    launched = L.met2_launch_count()
    assert L.met2_noise_sigma_workspace_bytes(1, 1, 1, 2) == -1
    assert L.met2_tv_workspace_bytes(4, 3, 0, 2) == -1
    assert L.met2_noise_sigma(p(vol), 1, 1, 1, 2, p(w), p(ws), None) == -1
    assert L.met2_noise_sigma(None, 4, 3, 2, 2, p(w), p(ws), None) == -1
    assert L.met2_noise_sigma(p(vol), 4, 3, 2, 0, p(w), p(ws), None) == -1
    good = [p(vol), 4, 3, 2, 2, p(w), 2e-4, 10, p(out), p(it), p(ws), None]
    for k, bad in ((0, None), (5, None), (8, None), (9, None), (10, None), (7, 0), (7, -1), (1, 0), (4, -3), (8, p(vol))):
        args = list(good)
        args[k] = bad
        assert L.met2_tv_chambolle(*args) == -1
        assert b"met2_tv_chambolle" in L.met2_last_error()
    args = list(good)
    args[1:4] = [1, 1, 1]
    assert L.met2_tv_chambolle(*args) == -1
    assert emu.counters()["launches"] == 0 and L.met2_launch_count() == launched
    assert L.met2_tv_chambolle(*good) == 0 and emu.counters()["launches"] == 3 + 4 * 10
