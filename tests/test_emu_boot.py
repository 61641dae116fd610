"""met2_boot_resample and met2_boot_summary (csrc/met2_boot.cu) under the SIMT emulator (tests/emu): the kernels' own
source on the CPU, bitwise equal to the NumPy restatement of tests/boot_oracle.py.  Outputs are poisoned and
canary-guarded (emu._Guarded)."""
import ctypes
import os

import numpy as np
import pytest

import boot_oracle as O
from emu import emu

P = ctypes.c_void_p


@pytest.fixture(scope="module", autouse=True)
def _built():
    emu.build()
    L = emu.lib()
    L.met2_boot_resample.argtypes = [P, P, P, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_uint64,
                                     ctypes.c_int64, P, P, P]
    L.met2_boot_summary.argtypes = [P, P, ctypes.c_int64, ctypes.c_int, P, P, P]


def resample(sig, est, fa, B, seed, voxel_offset):
    L = emu.lib()
    sig = np.ascontiguousarray(sig, dtype=np.float64)
    est = np.ascontiguousarray(est, dtype=np.float64)
    fa = np.ascontiguousarray(fa, dtype=np.int32)
    V, nTE = sig.shape
    gd = emu._Guarded()
    rep = gd.array((V * B, nTE), np.float64, np.nan)
    rep_fa = gd.array(V * B, np.int32, -7)
    emu._check(L.met2_boot_resample(emu._ptr(sig), emu._ptr(est), emu._ptr(fa), V, nTE, B, seed, voxel_offset,
                                    emu._ptr(rep), emu._ptr(rep_fa), None), "met2_boot_resample")
    gd.check("met2_boot_resample")
    return np.array(rep), np.array(rep_fa)


def summary(maps, status, B):
    L = emu.lib()
    maps = np.ascontiguousarray(maps, dtype=np.float64)
    status = np.ascontiguousarray(status, dtype=np.uint32)
    V = maps.shape[0] // B
    gd = emu._Guarded()
    stats = gd.array((V, 6, 4), np.float64, -7.0)
    n = gd.array(V, np.int32, -7)
    emu._check(L.met2_boot_summary(emu._ptr(maps), emu._ptr(status), V, B, emu._ptr(stats), emu._ptr(n), None),
               "met2_boot_summary")
    gd.check("met2_boot_summary")
    return np.array(stats), np.array(n)


def _signals(V, nTE, seed):
    rng = np.random.default_rng(seed)
    est = 1000.0 * np.exp(-np.arange(1, nTE + 1) * 10.0 / rng.uniform(30, 120, (V, 1)))
    return est + rng.normal(0, 8.0, (V, nTE)), est, rng.integers(0, 273, V).astype(np.int32)


@pytest.mark.parametrize("B, nTE", [(1, 32), (2, 48), (7, 64), (100, 32), (1024, 64)])
def test_resample_equals_restatement(B, nTE):
    V = 3 if B == 1024 else 9
    sig, est, fa = _signals(V, nTE, B + nTE)
    seed, off = 0xDEADBEEF12345678, 123457
    rep, rep_fa = resample(sig, est, fa, B, seed, off)
    ref, ref_fa = O.resample(sig, est, fa, B, seed, off)
    assert np.array_equal(rep, ref) and np.array_equal(rep_fa, ref_fa)
    if nTE == 64 and B > 1:        # bit 63 of the word is used, and takes both values
        neg = O.signs(V, B, nTE, seed, off)[..., 63]
        assert neg.any() and not neg.all()


def _replicate_maps(V, B, seed, skip_frac=0.3):
    rng = np.random.default_rng(seed)
    maps = rng.normal(0.15, 0.04, (V * B, 6))
    maps[:, 3:5] = rng.uniform(10, 90, (V * B, 2))
    maps[rng.random(V * B) < 0.2, 0] = 0.0                       # ties
    maps[:, 5] = np.round(maps[:, 5], 2)                          # many ties
    status = np.where(rng.random(V * B) < skip_frac, 1, 0).astype(np.uint32)
    status |= np.where(rng.random(V * B) < 0.1, 4, 0).astype(np.uint32)    # ITMAX alone does not invalidate
    return maps, status


@pytest.mark.parametrize("B", [1, 2, 7, 100, 1024])
def test_summary_equals_restatement(B):
    V = 5 if B == 1024 else 13
    maps, status = _replicate_maps(V, B, B)
    st = status.reshape(V, B)
    st[0] |= 1                                                   # no valid replicate
    if B > 1:
        st[1, 1:] |= 1                                           # exactly one
        st[2] &= ~np.uint32(1)                                   # all valid
    maps[B * 3 + (B - 1), 2] = np.nan                            # a NaN in one map of voxel 3
    maps[(B * 4):(B * 5), 1] = 0.25                              # a constant map
    stats, n = summary(maps, status, B)
    ref, ref_n = O.summary(maps, status, B)
    assert np.array_equal(n, ref_n)
    assert np.array_equal(stats, ref, equal_nan=True)
    assert np.array_equal(stats[0], np.zeros((6, 4)))
    if B > 1:
        assert n[1] == 1 and np.all(stats[1, :, 1] == 0.0) and n[2] == B


@pytest.mark.parametrize("order", ["reverse", "shuffle"])
def test_lane_scheduling_orders(order):
    B = 37
    maps, status = _replicate_maps(6, B, 99)
    base = summary(maps, status, B)
    os.environ["SIMT_EMU_ORDER"] = order
    try:
        got = summary(maps, status, B)
    finally:
        del os.environ["SIMT_EMU_ORDER"]
    ref = O.summary(maps, status, B)
    for a, b, r in zip(got, base, ref):
        assert np.array_equal(a, b) and np.array_equal(a, r)


def test_argument_checks_launch_nothing():
    L = emu.lib()
    sig = np.ones((4, 32))
    fa = np.zeros(4, dtype=np.int32)
    rep = np.zeros((4 * 8, 32))
    rep_fa = np.zeros(4 * 8, dtype=np.int32)
    maps = np.zeros((4 * 8, 6))
    status = np.zeros(4 * 8, dtype=np.uint32)
    stats = np.zeros((4, 6, 4))
    n = np.zeros(4, dtype=np.int32)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    emu.counters(reset_only=True)
    launched = L.met2_launch_count()
    good = [p(sig), p(sig), p(fa), 4, 32, 8, 0, 0, p(rep), p(rep_fa), None]
    for k, bad in ((5, 0), (5, -1), (5, 1025), (4, 0), (4, 65), (3, -1), (7, -1), (0, None), (1, None), (2, None),
                   (8, None), (9, None)):
        args = list(good)
        args[k] = bad
        assert L.met2_boot_resample(*args) == -1
        assert b"met2_boot_resample" in L.met2_last_error()
    good_s = [p(maps), p(status), 4, 8, p(stats), p(n), None]
    for k, bad in ((3, 0), (3, 1025), (2, -1), (0, None), (1, None), (4, None), (5, None)):
        args = list(good_s)
        args[k] = bad
        assert L.met2_boot_summary(*args) == -1
        assert b"met2_boot_summary" in L.met2_last_error()
    # V = 0 is a no-op, NULL pointers included
    assert L.met2_boot_resample(None, None, None, 0, 32, 8, 0, 0, None, None, None) == 0
    assert L.met2_boot_summary(None, None, 0, 8, None, None, None) == 0
    assert emu.counters()["launches"] == 0 and L.met2_launch_count() == launched
    assert L.met2_boot_resample(*good) == 0 and L.met2_boot_summary(*good_s) == 0
    assert emu.counters()["launches"] == 2 and L.met2_launch_count() == launched + 2
