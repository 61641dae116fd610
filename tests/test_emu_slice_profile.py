"""met2_epg_dictionary_profile and met2_epg_signals_profile (csrc/met2_epg.cu) under the SIMT emulator (tests/emu): the
kernels' own source on the CPU against the NumPy restatement of tests/slice_profile_oracle.py (the reference's dense
EPG summed over the slice positions in order), bitwise equal across three lane orders, K = 1 bitwise equal to
met2_epg_dictionary, and the argument checks."""
import ctypes
import os

import numpy as np
import pytest

import slice_profile_oracle as SP
from emu import emu
from multicomponent_t2_toolbox_b200 import grids

P = ctypes.c_void_p
DIC_ARGS = [P, ctypes.c_int, P, P, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_double, P, P, P, ctypes.c_int,
            P, P, P]
SIG_ARGS = [P, P, P, ctypes.c_int64, ctypes.c_int, ctypes.c_double, P, P, P, ctypes.c_int, P, P]


@pytest.fixture(scope="module", autouse=True)
def _built():
    emu.build()
    L = emu.lib()
    L.met2_epg_dictionary_profile.argtypes = DIC_ARGS
    L.met2_epg_signals_profile.argtypes = SIG_ARGS


def _p(a):
    return emu._ptr(a)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def dictionary(alphas, T2s, nTE, tau, TR, prof, T1=1000.0):
    alphas, T2s = _f64(alphas), _f64(T2s)
    T1s = np.full(len(T2s), T1)
    x, r, w = (_f64(a) for a in prof)
    g = emu._Guarded()
    dic = g.array((len(alphas), nTE, len(T2s)), np.float64, np.nan)
    dicT = g.array((len(alphas), len(T2s), nTE), np.float64, np.nan)
    rc = emu.lib().met2_epg_dictionary_profile(_p(alphas), len(alphas), _p(T2s), _p(T1s), len(T2s), nTE, tau, TR,
                                               _p(x), _p(r), _p(w), len(w), _p(dic), _p(dicT), None)
    emu._check(rc, "met2_epg_dictionary_profile")
    g.check("met2_epg_dictionary_profile")
    return np.array(dic), np.array(dicT)


def signals(alphas, T2s, T1s, nTE, tau, prof):
    alphas, T2s, T1s = _f64(alphas), _f64(T2s), _f64(T1s)
    x, r, w = (_f64(a) for a in prof)
    g = emu._Guarded()
    sig = g.array((len(alphas), nTE), np.float64, np.nan)
    emu._check(emu.lib().met2_epg_signals_profile(_p(alphas), _p(T2s), _p(T1s), len(alphas), nTE, tau, _p(x), _p(r),
                                                  _p(w), len(w), _p(sig), None), "met2_epg_signals_profile")
    g.check("met2_epg_signals_profile")
    return np.array(sig)


def _profile(K, seed=0):
    if K >= 7:
        return grids.as_slice_profile(grids.slice_profile(tbw=2.7, ratio=1.5, K=K))
    rng = np.random.default_rng(seed)     # a few arbitrary positions, unequal weights
    return grids.as_slice_profile((rng.uniform(0.2, 1.0, K), rng.uniform(0.2, 1.0, K), rng.uniform(0.5, 2.0, K)))


def _in_orders(fn):
    outs = []
    for order in (None, "reverse", "shuffle"):
        if order:
            os.environ["SIMT_EMU_ORDER"] = order
        try:
            outs.append(fn())
        finally:
            os.environ.pop("SIMT_EMU_ORDER", None)
    for o in outs[1:]:
        assert all(np.array_equal(a, b) for a, b in zip(outs[0], o))
    return outs[0]


@pytest.mark.parametrize("nTE, nT2, K, alphas", [
    (32, 60, 7, [95.0, 150.0]), (48, 96, 64, [120.0]), (64, 128, 1, [90.0, 133.0, 180.0]),
    (32, 8, 512, [140.0]), (64, 4, 64, [100.0, 170.0])])
def test_dictionary_against_restatement_in_three_lane_orders(nTE, nT2, K, alphas):
    prof = _profile(K)
    T2s = grids.t2_grid(nT2)
    cols = np.unique(np.linspace(0, nT2 - 1, min(nT2, 6)).astype(int))    # restated columns (the dense EPG is slow)
    dic, dicT = _in_orders(lambda: dictionary(alphas, T2s, nTE, 10.0, 1000.0, prof))
    assert np.array_equal(dicT, np.transpose(dic, (0, 2, 1)))
    ref = SP.dictionary(alphas, T2s[cols], np.full(len(cols), 1000.0), nTE, 10.0, 1000.0, *prof)
    assert np.all(np.isfinite(dic))
    assert np.max(np.abs(dic[:, :, cols] - ref)) <= 1e-14 * np.abs(ref).max()


def test_k1_is_the_plain_dictionary_bit_for_bit():
    T2s = grids.t2_grid(60)
    alphas = np.linspace(90.0, 180.0, 13)
    for nTE, tau, TR in ((32, 10.0, 1000.0), (48, 8.0, 2000.0), (64, 5.0, 1500.0)):
        plain, plainT = emu.epg_dictionary(alphas, T2s, np.full(60, 1000.0), nTE, tau, TR)
        dic, dicT = dictionary(alphas, T2s, nTE, tau, TR, (np.ones(1), np.ones(1), np.ones(1)))
        assert np.array_equal(dic, plain) and np.array_equal(dicT, plainT)


def test_signals_against_restatement_and_dictionary():
    prof = _profile(24)
    rng = np.random.default_rng(3)
    al, t2 = rng.uniform(95.0, 180.0, 5), rng.uniform(15.0, 300.0, 5)
    t1 = np.full(5, 1000.0)
    sig = _in_orders(lambda: (signals(al, t2, t1, 32, 10.0, prof),))[0]
    ref = SP.signals(al, t2, t1, 32, 10.0, *prof)
    assert np.max(np.abs(sig - ref)) <= 1e-14 * np.abs(ref).max()
    # the dictionary entry is the signal times (1 - exp(-TR/T1)), bit for bit
    dic, _ = dictionary(al[:1], t2[:1], 32, 10.0, 1000.0, prof)
    assert np.array_equal(dic[0, :, 0], (1.0 - np.exp(-1.0)) * sig[0])


def test_argument_errors_before_any_launch():
    L = emu.lib()
    a, t2, t1 = _f64([120.0]), _f64([50.0]), _f64([1000.0])
    out = np.zeros(64 * 200)
    good = (_f64([1.0, 0.5]), _f64([1.0, 0.5]), _f64([0.5, 0.5]))

    def dic(K=2, nT2=1, nTE=32, prof=good, alphas=a):
        x, r, w = prof
        return L.met2_epg_dictionary_profile(_p(alphas), 1, _p(t2), _p(t1), nT2, nTE, 10.0, 1000.0, _p(x), _p(r), _p(w),
                                             K, _p(out), None, None)

    def sig(K=2, N=1, prof=good):
        x, r, w = prof
        return L.met2_epg_signals_profile(_p(a), _p(t2), _p(t1), N, 32, 10.0, _p(x), _p(r), _p(w), K, _p(out), None)
    emu.counters(reset_only=True)
    assert dic() == 0 and sig() == 0
    assert emu.counters()["launches"] == 2
    bads = []
    for i in range(3):
        for v in (np.nan, -0.1, np.inf, -np.inf):
            p = [q.copy() for q in good]
            p[i][1] = v
            bads.append(tuple(p))
    for p in bads:
        assert dic(prof=p) == -1 and sig(prof=p) == -1
        assert b"slice profile" in L.met2_last_error()
    assert dic(K=0) == -1 and sig(K=0) == -1 and dic(K=513) == -1 and sig(K=513) == -1
    assert dic(nT2=129) == -1 and dic(nTE=65) == -1 and dic(nTE=0) == -1 and dic(alphas=None) == -1
    assert dic(prof=(None, good[1], good[2])) == -1 and sig(N=-1) == -1
    assert emu.counters()["launches"] == 0
    assert sig(N=0) == 0 and emu.counters()["launches"] == 0
