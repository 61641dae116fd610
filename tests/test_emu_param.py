"""met2_param_fit (csrc/met2_param.cu) under the SIMT emulator (tests/emu): the kernel's own source on the CPU against
the NumPy restatement of tests/param_oracle.py, at 32 echoes / 60 bins from an X2-I start and at 48 echoes / 100 bins
from an NNLS start, with a skipped and a non-finite voxel.  The emulator runs about 0.05 s per model evaluation, so
the cases are a dozen voxels, some with a lowered max_iter (which also exercises MET2_ST_ITMAX)."""
import ctypes
import os

import numpy as np
import pytest

import met2_oracle as O
import param_oracle as PO
from emu import emu
from multicomponent_t2_toolbox_b200 import _lib, grids
from multicomponent_t2_toolbox_b200.phantom import make_phantom


@pytest.fixture(scope="module", autouse=True)
def _built():
    emu.build()
    emu.lib().met2_param_fit.argtypes = _lib.SIGNATURES["met2_param_fit"][1]


class Case:
    def __init__(self, nTE, nT2, V, seed, method):
        self.T2s = grids.t2_grid(nT2)
        ph = make_phantom((V, 1, 1), n_echoes=nTE, seed=seed, fa_mode="uniform")
        self.sig = np.ascontiguousarray(ph["data"].reshape(V, nTE))
        self.sig[1] = 0.0                                          # skipped by the point fit
        self.status = np.zeros(V, np.uint32)
        self.status[1] = 1
        self.status[2] = 2                                         # NaN in the signal
        alphas = np.linspace(90.0, 180.0, 91)
        ia = np.abs(alphas[None, :] - ph["truth"]["fa"].ravel()[:, None]).argmin(axis=1)
        self.fa = np.ascontiguousarray(alphas[ia] + 0.3)
        d, _, _ = PO.epg_curves(alphas[ia][:, None], self.T2s[None, :], 1000.0, 10.0, 1000.0, nTE)
        self.fsol = np.zeros((V, nT2))
        for v in range(V):
            if self.status[v]:
                continue
            y = self.sig[v] / self.sig[v, 0]
            f = O.nnls_x2(d[v].T, y, np.eye(nT2), 1.02)[0] if method == "X2" else O.nnls(d[v].T, y)[0]
            self.fsol[v] = f * self.sig[v, 0]
        self.sig[2, 3] = np.nan
        m, t, c = grids.compartment_masks(self.T2s, 40.0)
        self.comp = (m.astype(np.uint8) | (t.astype(np.uint8) << 1) | (c.astype(np.uint8) << 2))
        self.logT2 = np.log(self.T2s)

    def cfg(self, **kw):
        return PO.plan_cfg(self.T2s, **kw)

    def run(self, V=None, **kw):
        cfg = {**PO.DEFAULTS, **self.cfg(**kw)}
        V = len(self.sig) if V is None else V
        nTE = self.sig.shape[1]
        c = _lib.ParamCfg(nTE=nTE, nT2=len(self.T2s), max_iter=cfg["max_iter"], reserved=0, tau=10.0, TR=1000.0,
                          T1=1000.0, fa_lo=90.0, fa_hi=180.0, mu0=cfg["mu0"], mu_max=cfg["mu_max"], ftol=cfg["ftol"],
                          xtol=cfg["xtol"])
        for k in range(3):
            c.t2_lo[k], c.t2_hi[k] = cfg["t2_lo"][k], cfg["t2_hi"][k]
        gd = emu._Guarded()     # poisoned, canary-guarded outputs: every element must be written, nothing beyond
        out = dict(params=gd.array((V, 7), np.float64, np.nan), maps=gd.array((V, 6), np.float64, np.nan),
                   est_signal=gd.array((V, nTE), np.float64, np.nan), sse=gd.array(V, np.float64, np.nan),
                   iters=gd.array(V, np.int32, -7), status=gd.array(V, np.uint32, 0xFFFFFFFF))
        p = emu._ptr
        rc = emu.lib().met2_param_fit(p(self.sig), p(self.fa), p(self.fsol), p(self.status), V, ctypes.byref(c),
                                      p(self.logT2), p(self.comp), p(out["params"]), p(out["maps"]),
                                      p(out["est_signal"]), p(out["sse"]), p(out["iters"]), p(out["status"]), None)
        emu._check(rc, "met2_param_fit")
        gd.check("met2_param_fit")
        return {k: np.array(v) for k, v in out.items()}

    def oracle(self, V=None, **kw):
        V = len(self.sig) if V is None else V
        return PO.param_fit(self.sig[:V], self.fa[:V], self.fsol[:V], self.status[:V], self.logT2, self.comp,
                            self.cfg(**kw))


def compare(out, ref):
    np.testing.assert_array_equal(out["status"], ref["status"])
    np.testing.assert_allclose(out["params"], ref["params"], rtol=1e-8, atol=1e-8 * np.abs(ref["params"]).max())
    np.testing.assert_allclose(out["sse"], ref["sse"], rtol=1e-10, atol=0)
    np.testing.assert_allclose(out["est_signal"], ref["est_signal"], rtol=1e-8, atol=1e-8 * ref["est_signal"].max())
    np.testing.assert_allclose(out["maps"], ref["maps"], rtol=1e-8, atol=1e-8 * np.abs(ref["maps"]).max())
    same = float(np.mean(out["iters"] == ref["iters"]))
    assert same >= 0.95, same
    for v in (1, 2):                                               # skipped / non-finite: zeros
        for k in ("params", "maps", "est_signal", "sse", "iters"):
            assert np.all(out[k][v] == 0), (k, v)
    return same


@pytest.fixture(scope="module")
def case32():
    return Case(32, 60, 12, seed=21, method="X2")


def test_32_echoes_60_bins_against_restatement(case32):
    out = case32.run(max_iter=40)
    ref = case32.oracle(max_iter=40)
    same = compare(out, ref)
    print("32 echoes: iteration counts equal in %.0f %% of %d voxels" % (100 * same, len(out["sse"])))
    assert np.any(out["status"] & PO.ST_ITMAX) and np.any((out["status"] & PO.ST_ITMAX) == 0)


def test_48_echoes_100_bins_against_restatement():
    c = Case(48, 100, 6, seed=22, method="NNLS")
    out = c.run(max_iter=15)
    same = compare(out, c.oracle(max_iter=15))
    print("48 echoes: iteration counts equal in %.0f %% of %d voxels" % (100 * same, len(out["sse"])))


@pytest.mark.parametrize("order", ["reverse", "shuffle"])
def test_bitwise_equal_under_lane_orders(case32, order):
    base = case32.run(V=6, max_iter=6)
    os.environ["SIMT_EMU_ORDER"] = order
    try:
        other = case32.run(V=6, max_iter=6)
    finally:
        del os.environ["SIMT_EMU_ORDER"]
    for k in base:
        assert np.array_equal(base[k].view(np.uint8), other[k].view(np.uint8)), k


def test_argument_validation_and_empty_batch(case32):
    L = emu.lib()
    c = _lib.ParamCfg(nTE=32, nT2=60, max_iter=200, reserved=0, tau=10.0, TR=1000.0, T1=1000.0, fa_lo=90.0,
                      fa_hi=180.0, mu0=1e-3, mu_max=1e16, ftol=1e-12, xtol=1e-10)
    for k, (a, b) in enumerate(((10.0, 40.0), (40.0, 200.0), (200.0, 2000.0))):
        c.t2_lo[k], c.t2_hi[k] = a, b
    buf = np.zeros(64 * 128)
    P = buf.ctypes.data_as(ctypes.c_void_p)
    call = lambda V, cfg, ptr=P: L.met2_param_fit(ptr, P, P, P, V, ctypes.byref(cfg) if cfg else None, P, P, P, P, P,
                                                 P, P, P, None)
    n0 = emu.lib().met2_launch_count()
    assert call(0, c) == 0                                         # V = 0: no-op
    assert call(0, c, None) == 0
    assert call(1, c, None) == -1                                  # NULL pointer
    assert call(-1, c) == -1
    assert call(1, None) == -1
    for field, value in (("nTE", 65), ("nTE", 0), ("nT2", 129), ("max_iter", -1), ("fa_lo", 181.0), ("tau", 0.0),
                         ("mu0", 0.0), ("ftol", -1.0)):
        old = getattr(c, field)
        setattr(c, field, value)
        assert call(1, c) == -1, field
        assert b"met2_param_fit" in L.met2_last_error()
        setattr(c, field, old)
    c.t2_lo[1], c.t2_hi[1] = 200.0, 40.0                           # empty T2 box
    assert call(1, c) == -1
    assert emu.lib().met2_launch_count() == n0                     # nothing was launched


def test_struct_size_matches_header():
    # met2_param_cfg: 4 int32, tau / TR / T1, t2_lo[3], t2_hi[3], fa_lo / fa_hi, mu0 / mu_max, ftol / xtol
    assert ctypes.sizeof(_lib.ParamCfg) == 4 * 4 + 3 * 8 + 6 * 8 + 2 * 8 + 4 * 8
