"""met2_spatial_sweep and met2_spatial_finish (csrc/met2_spatial.cu) under the SIMT emulator (tests/emu): the kernels'
own source on the CPU against the NumPy restatement of tests/spatial_oracle.py, on a small masked volume with holes,
an in-mask voxel the point fit skips and voxels without fitted neighbours."""
import ctypes
import os

import numpy as np
import pytest

import met2_oracle as O
import spatial_oracle as S
from emu import emu
from multicomponent_t2_toolbox_b200 import pipeline
from multicomponent_t2_toolbox_b200.phantom import make_phantom

P = ctypes.c_void_p
SWEEP_ARGS = [P] * 5 + [ctypes.c_int64, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int, P, P, P,
                        ctypes.c_double, P, P, P]
FINISH_ARGS = [P] * 4 + [ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int] + [P] * 7
ALPHAS = np.array([115.0, 150.0, 178.0])


@pytest.fixture(scope="module", autouse=True)
def _built():
    emu.build()
    L = emu.lib()
    L.met2_spatial_sweep.argtypes = SWEEP_ARGS
    L.met2_spatial_finish.argtypes = FINISH_ARGS


def _p(a):
    return emu._ptr(a)


class Case:
    """A 7 x 6 x 3 volume (mask with holes, one in-mask voxel with zero signal), three flip angles, and the oracle's
    point fit of every fitted voxel: x0 (normalised spectrum) and the lambda it selected."""

    def __init__(self, method, rm, seed):
        g = O._grids(method, rm, "brute-force", 40.0, 32, 10.0, 1000.0)
        self.T2s, self.L, n = g["T2s"], g["L"], g["npc"]
        self.Dic = O.create_Dic_3D(n, self.T2s, g["T1s"], 32, 10.0, ALPHAS, 1000.0)      # [nTE, nT2, nA]
        self.dic, self.dicT, self.G, self.kband = emu.tables(self.Dic, self.L)
        shape = (7, 6, 3)
        ph = make_phantom(shape, seed=seed, fa_mode="b1")
        rng = np.random.default_rng(seed)
        mask = rng.random(shape) < 0.85
        mask[3, 3, 1] = True
        mask[0, 0, 0], mask[1, 0, 0], mask[0, 1, 0], mask[0, 0, 1] = True, False, False, False   # an isolated voxel
        data = ph["data"].copy()
        data[3, 3, 1] = 0.0                                                   # masked, not fitted
        self.flat = np.nonzero(mask.ravel())[0]
        self.shape = shape
        self.sig = np.ascontiguousarray(data.reshape(-1, 32)[self.flat])
        V = len(self.flat)
        self.fa = rng.integers(0, len(ALPHAS), V).astype(np.int32)
        self.fitted = self.sig.sum(axis=1) > 0
        self.status = np.where(self.fitted, 0, 1).astype(np.uint32)
        self.x0 = np.zeros((V, n))
        self.lam = np.zeros(V)
        self.Y = self.sig / np.where(self.fitted, self.sig[:, 0], 1.0)[:, None]
        for v in np.nonzero(self.fitted)[0]:
            D = self.Dic[:, :, self.fa[v]]
            if method == "X2":
                self.x0[v], self.lam[v], _ = O.nnls_x2(D, self.Y[v], self.L, 1.02)
            else:
                self.lam[v] = 1.8 if method == "T2SPARC" else O.nnls_lcurve_wrapper(D, self.Y[v], self.L, g["lambda_reg"])
                self.x0[v] = O.nnls_tik(D, self.Y[v], self.L, self.lam[v])
        self.nbr, self.colours = S.neighbours(self.flat, shape, self.fitted)
        self.Dv = lambda v: self.Dic[:, :, self.fa[v]]

    def sweep(self, x, status, vox, mu):
        x = np.ascontiguousarray(x)
        status = np.ascontiguousarray(status)
        vox = np.ascontiguousarray(vox, dtype=np.int32)
        emu._check(emu.lib().met2_spatial_sweep(
            _p(self.sig), _p(self.fa), _p(self.lam), _p(self.nbr), _p(vox), len(vox), len(self.flat), 32,
            self.dic.shape[2], len(ALPHAS), _p(self.G), _p(self.dicT), _p(self.kband), mu, _p(x), _p(status), None),
            "met2_spatial_sweep")
        return x, status

    def finish(self, x, status):
        V, n = x.shape
        comp = ((self.T2s <= 40.0) * 1 + ((self.T2s > 40.0) & (self.T2s <= 200.0)) * 2 + (self.T2s >= 200.0) * 4)
        comp = comp.astype(np.uint8)
        logT2 = np.log(self.T2s)
        gd = emu._Guarded()
        fsol = gd.array((V, n), np.float64, np.nan)
        est = gd.array((V, 32), np.float64, np.nan)
        maps = gd.array((V, 6), np.float64, np.nan)
        emu._check(emu.lib().met2_spatial_finish(_p(self.sig), _p(self.fa), _p(status), _p(x), V, 32, n, len(ALPHAS),
                                                 _p(self.dicT), _p(logT2), _p(comp), _p(fsol), _p(est), _p(maps), None),
                   "met2_spatial_finish")
        gd.check("met2_spatial_finish")
        return np.array(fsol), np.array(est), np.array(maps)


_CASES = {}


def _case(key):
    if key not in _CASES:
        method, rm = key.split("-")
        _CASES[key] = Case(method, rm, seed=len(_CASES) + 21)
    return _CASES[key]


def _close(x, ref, fitted):
    assert np.array_equal(x[fitted] > 0, ref[fitted] > 0)
    scale = np.abs(ref[fitted]).max(axis=1)
    return (np.abs(x[fitted] - ref[fitted]).max(axis=1) / scale).max()


def test_neighbour_table_equals_restatement():
    c = _case("X2-I")
    nbr, colours = pipeline.spatial_neighbours(c.flat, c.shape, c.fitted)
    assert np.array_equal(nbr, c.nbr) and all(np.array_equal(a, b) for a, b in zip(colours, c.colours))
    nv = (c.nbr >= 0).sum(axis=1)
    assert (nv[c.fitted] == 0).any() and (nv == 6).any() and not c.fitted.all()


@pytest.mark.parametrize("order", [None, "reverse", "shuffle"])
@pytest.mark.parametrize("key, mu", [("X2-I", 0.05), ("L_curve-L2", 0.3), ("T2SPARC-InvT2", 0.02)])
def test_sweeps_equal_restatement(key, mu, order):
    c = _case(key)
    if order:
        os.environ["SIMT_EMU_ORDER"] = order
    try:
        x, st = c.sweep(c.x0.copy(), c.status.copy(), c.colours[0], mu)
        ref, itmax = S.half_sweep(c.x0, c.colours[0], c.Y, c.Dv, c.lam, c.L, c.nbr, mu)
        assert not itmax and np.array_equal(st, c.status)
        assert _close(x, ref, c.fitted) <= 1e-9
        assert np.array_equal(x[c.colours[1]], c.x0[c.colours[1]])               # the other colour is untouched
        assert np.array_equal(x[~c.fitted], c.x0[~c.fitted])
        moved = np.abs(x - c.x0).max(axis=1)[c.colours[0]]
        assert (moved > 1e-6 * np.abs(c.x0).max()).mean() > 0.5                  # the prior moves most spectra
        x, st = c.sweep(x, st, c.colours[1], mu)
        for _ in range(2):
            for vox in c.colours:
                x, st = c.sweep(x, st, vox, mu)
        ref3, _ = S.sweeps(c.x0, c.colours, c.Y, c.Dv, c.lam, c.L, c.nbr, mu, 3)
        assert _close(x, ref3, c.fitted) <= 1e-9
        fsol, est, maps = c.finish(x, st)
    finally:
        os.environ.pop("SIMT_EMU_ORDER", None)
    km = c.sig[:, 0]
    f = c.fitted
    assert np.allclose(fsol[f], x[f] * km[f, None], rtol=1e-15, atol=0)
    D_est = np.einsum("vec,vc->ve", np.transpose(c.Dic, (2, 0, 1))[c.fa], x) * km[:, None]
    assert np.allclose(est[f], D_est[f], rtol=1e-12, atol=1e-12 * np.abs(D_est).max())
    ind = ((c.T2s <= 40.0), (c.T2s > 40.0) & (c.T2s <= 200.0), c.T2s >= 200.0)
    ref_maps = np.array([O.voxel_metrics(fsol[v], c.T2s, *ind) for v in range(len(x))])
    assert np.allclose(maps[f], ref_maps[f], rtol=1e-12, atol=1e-14)
    # a skipped voxel gets met2_t2_fit's outputs for a skipped voxel
    assert not fsol[~f].any() and not est[~f].any()
    assert np.array_equal(maps[~f], np.tile([0.0, 0.0, 0.0, 1.0, 1.0, 1e-16], ((~f).sum(), 1)))


def test_mu_zero_keeps_the_point_fit():
    c = _case("X2-I")
    x, st = c.x0.copy(), c.status.copy()
    for vox in c.colours:
        x, st = c.sweep(x, st, vox, 0.0)
    assert _close(x, c.x0, c.fitted) <= 1e-9


def test_argument_checks_launch_nothing():
    L = emu.lib()
    c = _case("X2-I")
    V, n = len(c.flat), c.dic.shape[2]
    x, st = c.x0.copy(), c.status.copy()
    vox = np.ascontiguousarray(c.colours[0])
    good = [_p(c.sig), _p(c.fa), _p(c.lam), _p(c.nbr), _p(vox), len(vox), V, 32, n, 3, _p(c.G), _p(c.dicT),
            _p(c.kband), 0.1, _p(x), _p(st), None]
    emu.counters(reset_only=True)
    launched = L.met2_launch_count()
    bad_sweep = [(5, -1), (5, V + 1), (6, 1 << 31), (6, -1), (7, 0), (7, 65), (8, 0), (8, 129), (9, 0), (13, -0.1),
                 (13, float("nan")), (13, float("inf"))] + [(k, None) for k in (0, 1, 2, 3, 4, 10, 11, 12, 14, 15)]
    for k, bad in bad_sweep:
        args = list(good)
        args[k] = bad
        assert L.met2_spatial_sweep(*args) == -1, (k, bad)
        assert b"met2_spatial_sweep" in L.met2_last_error()
    comp = np.zeros(n, dtype=np.uint8)
    out = np.zeros((V, n)), np.zeros((V, 32)), np.zeros((V, 6))
    good_f = [_p(c.sig), _p(c.fa), _p(st), _p(x), V, 32, n, 3, _p(c.dicT), _p(c.T2s), _p(comp), _p(out[0]),
              _p(out[1]), _p(out[2]), None]
    bad_finish = [(4, 1 << 31), (4, -1), (5, 0), (5, 65), (6, 0), (6, 129), (7, 0)] + \
        [(k, None) for k in (0, 1, 2, 3, 8, 9, 10, 11, 12, 13)]
    for k, bad in bad_finish:
        args = list(good_f)
        args[k] = bad
        assert L.met2_spatial_finish(*args) == -1, (k, bad)
        assert b"met2_spatial_finish" in L.met2_last_error()
    # nothing to do is a no-op, NULL pointers included
    assert L.met2_spatial_sweep(None, None, None, None, None, 0, V, 32, n, 3, None, None, None, 0.1, None, None,
                                None) == 0
    assert L.met2_spatial_finish(None, None, None, None, 0, 32, n, 3, *([None] * 7)) == 0
    assert emu.counters()["launches"] == 0 and L.met2_launch_count() == launched
    assert L.met2_spatial_sweep(*good) == 0 and L.met2_spatial_finish(*good_f) == 0
    assert emu.counters()["launches"] == 2 and L.met2_launch_count() == launched + 2
