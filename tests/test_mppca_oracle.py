"""The NumPy restatement of met2_mppca (tests/mppca_oracle.py) on its own: its Jacobi iteration against
numpy.linalg.eigh, and the statistics of the method — sigma and n_signal on pure Gaussian noise, and the signal error on
the B1 phantom against the noiseless EPG signal."""
import numpy as np
import pytest

import mppca_oracle as O
from multicomponent_t2_toolbox_b200.phantom import epg_signal_batch, make_phantom


def _eigh(C):
    return np.linalg.eigh(C)


def _both(vol, r=2):
    """The restatement with its own Jacobi and with eigh, on every voxel of vol."""
    centres = np.argwhere(np.ones(vol.shape[:3], dtype=bool))
    return O.mppca_batch(vol, centres, r), O.mppca_batch(vol, centres, r, eig=_eigh), centres


@pytest.fixture(scope="module")
def noise():
    rng = np.random.default_rng(0)
    return _both(100.0 + 5.0 * rng.standard_normal((12, 12, 12, 32)))


@pytest.fixture(scope="module")
def phantom():
    ph = make_phantom((16, 16, 8), seed=3, fa_mode="b1")
    data = ph["data"] * ph["mask"][..., None]
    data[data < 0.0] = 0.0
    return ph, _both(np.ascontiguousarray(data))


@pytest.fixture(scope="module")
def echoes48():
    ph = make_phantom((8, 8, 6), n_echoes=48, seed=4, fa_mode="b1")
    return _both(np.ascontiguousarray(ph["data"]))


def _against_eigh(jac, ref):
    scale = np.abs(ref["ev"]).max(axis=1, keepdims=True)
    assert (np.abs(jac["ev"] - ref["ev"]) <= 1e-12 * scale).all()
    assert np.array_equal(jac["n_signal"], ref["n_signal"])
    den = np.abs(ref["out"]).max(axis=1, keepdims=True)
    assert (np.abs(jac["out"] - ref["out"]) <= 1e-9 * den).all()
    assert not jac["capped"].any(), "a voxel reached the sweep cap"
    print("sweeps per voxel: mean %.2f, max %d" % (jac["sweeps"].mean(), jac["sweeps"].max()))


@pytest.mark.parametrize("case", ["noise", "phantom", "echoes48"])
def test_jacobi_against_eigh(case, request):
    res = request.getfixturevalue(case)
    jac, ref, _ = res[1] if case == "phantom" else res
    _against_eigh(jac, ref)


def test_pure_noise_sigma_and_rank(noise):
    jac, _, _ = noise
    med = np.median(jac["sigma"])
    zero = (jac["n_signal"] == 0).mean()
    print("pure noise: median sigma %.4f, n_signal = 0 in %.1f %%, histogram %s"
          % (med, 100 * zero, np.bincount(jac["n_signal"]).tolist()))
    assert abs(med - 5.0) <= 0.02 * 5.0
    assert zero >= 0.8


def test_phantom_signal_error_drops(phantom):
    ph, (jac, _, centres) = phantom
    tr = ph["truth"]
    V = tr["mwf"].size
    T1 = np.full(V, 1000.0)
    fa = tr["fa"].ravel()
    clean = (tr["mwf"].ravel()[:, None] * epg_signal_batch(32, 10.0, T1, tr["t2m"].ravel(), fa)
             + tr["iewf"].ravel()[:, None] * epg_signal_batch(32, 10.0, T1, tr["t2ie"].ravel(), fa)
             + tr["fwf"].ravel()[:, None] * epg_signal_batch(32, 10.0, T1, np.full(V, 2000.0), fa))
    clean *= 1000.0 * (1.0 - np.exp(-1.0))
    clean = clean.reshape(ph["data"].shape)[centres[:, 0], centres[:, 1], centres[:, 2]]
    noisy = ph["data"][centres[:, 0], centres[:, 1], centres[:, 2]]
    before = np.sqrt(np.mean((noisy - clean) ** 2))
    after = np.sqrt(np.mean((jac["out"] - clean) ** 2))
    print("phantom signal RMSE %.3f -> %.3f (ratio %.3f), n_signal %s"
          % (before, after, after / before, np.bincount(jac["n_signal"]).tolist()))
    assert after <= 0.7 * before


def test_window_shifts_at_edges():
    s, w = O.window_starts(10, np.array([0, 1, 2, 5, 8, 9]), 2)
    assert w == 5 and s.tolist() == [0, 0, 0, 3, 5, 5]
    s, w = O.window_starts(3, np.array([0, 1, 2]), 2)
    assert w == 3 and s.tolist() == [0, 0, 0]
