"""met2_rician_fit and met2_bessel_ratio (csrc/met2_rician.cu) under the SIMT emulator (tests/emu): the kernel's own
source on the CPU against the NumPy restatement of tests/rician_oracle.py, with a fixed number of MM iterations
(tol = 0), for 60 / 96 / 128 bins, 32 / 48 / 64 echoes, lambda = 0 and > 0, and L = I, L2 and InvT2."""
import ctypes
import os

import numpy as np
import pytest

import met2_oracle as O
import rician_oracle as R
from emu import emu
from multicomponent_t2_toolbox_b200.phantom import make_phantom

P = ctypes.c_void_p
FIT_ARGS = [P] * 6 + [ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int] + [P] * 3 + \
    [ctypes.c_int, ctypes.c_double] + [P] * 4
ALPHAS = np.array([115.0, 150.0, 178.0])
ST_SKIPPED, ST_ITMAX, ST_MM_CAP, ST_BAD_SIGMA = 1, 4, 128, 256


@pytest.fixture(scope="module", autouse=True)
def _built():
    emu.build()
    L = emu.lib()
    L.met2_rician_fit.argtypes = FIT_ARGS
    L.met2_bessel_ratio.argtypes = [P, ctypes.c_int64, P]
    L.met2_bessel_ratio.restype = ctypes.c_int64


def _p(a):
    return emu._ptr(a)


class Case:
    """V voxels of a low-SNR phantom with nTE echoes, three flip angles, nT2 bins and matrix rm; x0 = the oracle's
    solve at lambda (per voxel: alternately 0 and `lam`), sigma = the phantom's true noise SD."""

    def __init__(self, n, m, rm, lam, V=6, seed=7):
        g = O._grids("X2", rm, "brute-force", 40.0, m, 10.0, 1000.0, npc=n)
        self.T2s, self.L = g["T2s"], g["L"]
        self.Dic = O.create_Dic_3D(n, self.T2s, g["T1s"], m, 10.0, ALPHAS, 1000.0)
        self.dic, self.dicT, self.G, self.kband = emu.tables(self.Dic, self.L)
        ph = make_phantom((V, 1, 1), n_echoes=m, seed=seed, fa_mode="b1", snr_range=(20.0, 40.0))
        self.sig = np.ascontiguousarray(ph["data"].reshape(-1, m))
        self.sigma = np.ascontiguousarray(ph["truth"]["sigma"].ravel())
        rng = np.random.default_rng(seed)
        self.fa = rng.integers(0, len(ALPHAS), V).astype(np.int32)
        self.lam = np.where(np.arange(V) % 2 == 0, lam, 0.0)
        self.Y = self.sig / self.sig[:, :1]
        self.x0 = np.zeros((V, n))
        for v in range(V):
            self.x0[v], _ = R.solve(self.D(v), self.Y[v], self.L, self.lam[v])
        self.status = np.zeros(V, dtype=np.uint32)
        self.n, self.m, self.V = n, m, V

    def D(self, v):
        return self.Dic[:, :, self.fa[v]]

    def args(self, max_iter, tol, sigma=None, status=None, fa=None):
        gd = emu._Guarded()
        x = gd.array((self.V, self.n), np.float64, np.nan)
        iters = gd.array(self.V, np.int32, -7)
        status_out = gd.array(self.V, np.uint32, 0xDEAD)
        sigma = self.sigma if sigma is None else np.ascontiguousarray(sigma, dtype=np.float64)
        status = self.status if status is None else np.ascontiguousarray(status, dtype=np.uint32)
        fa = self.fa if fa is None else np.ascontiguousarray(fa, dtype=np.int32)
        keep = (sigma, status, fa)
        a = [_p(self.sig), _p(fa), _p(self.lam), _p(sigma), _p(self.x0), _p(status), self.V, self.m, self.n,
             len(ALPHAS), _p(self.G), _p(self.dicT), _p(self.kband), max_iter, tol, _p(x), _p(iters), _p(status_out),
             None]
        return a, (x, iters, status_out), gd, keep

    def fit(self, max_iter, tol=0.0, **kw):
        a, out, gd, _keep = self.args(max_iter, tol, **kw)
        emu._check(emu.lib().met2_rician_fit(*a), "met2_rician_fit")
        gd.check("met2_rician_fit")
        return tuple(np.array(o) for o in out)


_CASES = {}


def _case(n, m, rm, lam):
    key = (n, m, rm, lam)
    if key not in _CASES:
        _CASES[key] = Case(n, m, rm, lam, seed=len(_CASES) + 7)
    return _CASES[key]


CONFIGS = [(60, 32, "I", 0.05), (60, 32, "L2", 0.3), (96, 48, "InvT2", 0.02), (128, 64, "I", 0.1),
           (128, 32, "L2", 0.0)]


@pytest.mark.parametrize("n, m, rm, lam", CONFIGS)
@pytest.mark.parametrize("max_iter", [1, 5, 30])
def test_fixed_iterations_equal_restatement(n, m, rm, lam, max_iter):
    c = _case(n, m, rm, lam)
    x, iters, st = c.fit(max_iter)
    # tol = 0 stops only on an exact repeat of yt, i.e. at a fixed point of the iteration in floating point
    assert np.all((iters == max_iter) & (st == ST_MM_CAP) | (iters < max_iter) & (st == 0))
    assert (iters == max_iter).mean() >= 0.5
    for v in range(c.V):
        ref, it, capped, itmax = R.mm_fit(c.D(v), c.Y[v], c.L, c.lam[v], c.sigma[v] / c.sig[v, 0], c.x0[v],
                                          max_iter=max_iter, tol=0.0)
        assert not itmax and (capped or it >= 5)
        assert np.array_equal(x[v] > 0, ref > 0), v
        assert np.abs(x[v] - ref).max() <= 1e-9 * np.abs(ref).max(), v
        assert np.abs(x[v] - c.x0[v]).max() > 1e-6 * np.abs(ref).max()      # the iterations move the spectrum


def test_converged_fit_and_lane_orders_are_bitwise_identical():
    c = _case(60, 32, "I", 0.05)
    outs = []
    for order in (None, "reverse", "shuffle"):
        if order:
            os.environ["SIMT_EMU_ORDER"] = order
        try:
            outs.append(c.fit(200, 1e-9))
        finally:
            os.environ.pop("SIMT_EMU_ORDER", None)
    for o in outs[1:]:
        assert all(np.array_equal(a, b) for a, b in zip(outs[0], o))
    x, iters, st = outs[0]
    for v in range(c.V):
        ref, it, capped, _ = R.mm_fit(c.D(v), c.Y[v], c.L, c.lam[v], c.sigma[v] / c.sig[v, 0], c.x0[v])
        assert not capped and abs(int(iters[v]) - it) <= 1 and iters[v] >= 2
        assert np.abs(x[v] - ref).max() <= 1e-8 * np.abs(ref).max()
    assert np.all(st == 0)


def test_sigma_zero_reproduces_the_point_fit():
    c = _case(60, 32, "I", 0.05)
    x, iters, st = c.fit(200, 1e-9, sigma=np.zeros(c.V))
    assert np.all(iters == 0) and np.all(st == 0) and np.array_equal(x, c.x0)


def test_bad_sigma_and_skipped_voxels():
    c = _case(60, 32, "I", 0.05)
    sigma = c.sigma.copy()
    sigma[0], sigma[1], sigma[2] = np.nan, -np.inf, -1e-3
    status = c.status.copy()
    status[3] = ST_SKIPPED | 2
    fa = c.fa.copy()
    fa[4] = len(ALPHAS)
    x, iters, st = c.fit(200, 1e-9, sigma=sigma, status=status, fa=fa)
    assert np.all(st[:3] == ST_BAD_SIGMA | ST_SKIPPED) and st[3] == ST_SKIPPED | 2 and st[4] == 0
    assert not x[:5].any() and not iters[:5].any()
    ref, _, _ = c.fit(200, 1e-9)
    assert np.array_equal(x[5], ref[5]) and iters[5] > 0


def test_argument_checks_launch_nothing():
    L = emu.lib()
    c = _case(60, 32, "I", 0.05)
    good, out, gd, keep = c.args(5, 1e-9)
    emu.counters(reset_only=True)
    launched = L.met2_launch_count()
    bad = [(6, -1), (6, 1 << 31), (7, 0), (7, 65), (8, 0), (8, 129), (9, 0), (13, 0), (13, -1), (14, -1e-9),
           (14, float("nan")), (14, float("inf"))] + [(k, None) for k in (0, 1, 2, 3, 4, 5, 10, 11, 12, 15, 16, 17)]
    for k, b in bad:
        args = list(good)
        args[k] = b
        assert L.met2_rician_fit(*args) == -1, (k, b)
        assert b"met2_rician_fit" in L.met2_last_error()
    assert L.met2_rician_fit(*([None] * 6), 0, 32, 60, 3, None, None, None, 5, 1e-9, None, None, None, None) == 0
    assert emu.counters()["launches"] == 0 and L.met2_launch_count() == launched
    assert L.met2_rician_fit(*good) == 0
    assert emu.counters()["launches"] == 1 and L.met2_launch_count() == launched + 1
    z = np.zeros(3)
    assert L.met2_bessel_ratio(_p(z), -1, _p(z)) == -1 and L.met2_bessel_ratio(None, 3, _p(z)) == -1
    assert L.met2_bessel_ratio(_p(z), 3, None) == -1 and L.met2_bessel_ratio(None, 0, None) == 0


def test_bessel_ratio_hook_equals_restatement():
    z = np.concatenate(([0.0, -0.0, 8.0, np.nextafter(8.0, 9.0), np.inf, -np.inf, np.nan], np.linspace(-20.0, 20.0, 4001),
                        np.logspace(-300.0, 300.0, 3001)))
    out = np.full_like(z, -5.0)
    assert emu.lib().met2_bessel_ratio(_p(z), len(z), _p(out)) == len(z)
    ref = R.bessel_ratio(z)
    assert np.array_equal(out.view(np.uint64), ref.view(np.uint64))
    assert out[4] == 1.0 and out[5] == -1.0 and out[0] == 0.0
