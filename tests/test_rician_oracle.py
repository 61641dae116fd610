"""The NumPy restatement of the Rician-likelihood fit (tests/rician_oracle.py) against closed forms and SciPy: the
Bessel ratio, monotone MM, the optimality conditions of Phi, the sigma = 0 case, and the bias it removes on a low-SNR
phantom (the dictionary at each voxel's true flip angle, so no flip-angle search)."""
import numpy as np
import scipy.special as sp

import met2_oracle as O
import rician_oracle as R
from multicomponent_t2_toolbox_b200.phantom import epg_signal_batch, make_phantom

T2S = np.logspace(1.0, np.log10(2000.0), 60)
IND = (T2S <= 40.0, (T2S > 40.0) & (T2S <= 200.0), T2S >= 200.0)


def test_bessel_ratio_against_scipy():
    z = np.concatenate(([0.0], np.linspace(0.0, 20.0, 2001), np.logspace(-8.0, 12.0, 2001)))
    ref = sp.i1e(z) / sp.i0e(z)
    got = R.bessel_ratio(z)
    pos = z > 0
    assert np.max(np.abs(got[pos] - ref[pos]) / ref[pos]) <= 4e-16
    assert R.bessel_ratio(np.inf) == 1.0 and R.bessel_ratio(0.0) == 0.0
    assert np.array_equal(R.bessel_ratio(-z), -got)


def _voxel(seed=5, snr=(20.0, 40.0)):
    ph = make_phantom((2, 2, 1), seed=seed, fa_mode="b1", snr_range=snr)
    tr = {k: v.ravel() for k, v in ph["truth"].items()}
    sig = ph["data"].reshape(-1, 32)
    D = epg_signal_batch(32, 10.0, np.full(60, 1000.0), T2S, np.full(60, tr["fa"][0])).T
    return D, sig[0] / sig[0, 0], tr["sigma"][0] / sig[0, 0]


def test_objective_never_increases_and_kkt_holds():
    D, y, sn = _voxel()
    L = np.eye(60)
    for lam in (0.0, 0.05):
        x0, _ = R.solve(D, y, L, lam)
        trace = []
        x, iters, capped, itmax = R.mm_fit(D, y, L, lam, sn, x0, trace=trace)
        assert not capped and not itmax and iters >= 3
        phi = [R.objective(t, D, y, L, lam, sn) for t in [x0] + trace]
        assert all(b <= a + 1e-13 * abs(a) for a, b in zip(phi, phi[1:]))
        assert phi[-1] < phi[0]
        g = R.gradient(x, D, y, L, lam, sn)
        on = x > 0
        assert np.abs(g[on]).max() <= 1e-7 and g[~on].min() >= -1e-7


def test_sigma_zero_returns_the_start():
    D, y, _ = _voxel()
    x0, _ = R.solve(D, y, np.eye(60), 0.0)
    x, iters, capped, _ = R.mm_fit(D, y, np.eye(60), 0.0, 0.0, x0)
    assert iters == 0 and not capped and np.array_equal(x, x0)


def _bias(lam_mode, n_side, snr, seed=3):
    """Gaussian (point) and Rician fits of every voxel of make_phantom((n_side, n_side, 4), seed, "b1", snr) with sigma
    from the truth; returns the mean errors (fit - truth) of MWF, FWF and T2_IE for both, and the MM iteration counts."""
    ph = make_phantom((n_side, n_side, 4), seed=seed, fa_mode="b1", snr_range=snr)
    tr = {k: v.ravel() for k, v in ph["truth"].items()}
    sig = ph["data"].reshape(-1, 32)
    L = np.eye(60)
    err = {"g": [], "r": []}
    its = []
    for v in range(sig.shape[0]):
        D = epg_signal_batch(32, 10.0, np.full(60, 1000.0), T2S, np.full(60, tr["fa"][v])).T
        y = sig[v] / sig[v, 0]
        lam = 0.0 if lam_mode == "NNLS" else O.nnls_x2(D, y, L, 1.02)[1]
        x0, _ = R.solve(D, y, L, lam, fast=True)
        x, iters, _, _ = R.mm_fit(D, y, L, lam, tr["sigma"][v] / sig[v, 0], x0, fast=True)
        its.append(iters)
        for tag, s in (("g", x0), ("r", x)):
            mwf, _, fwf, _, t2ie, _ = O.voxel_metrics(s, T2S, *IND)
            err[tag].append((mwf - tr["mwf"][v], fwf - tr["fwf"][v], t2ie - tr["t2ie"][v]))
    return {k: np.mean(v, axis=0) for k, v in err.items()}, np.array(its)


def test_rician_fit_reduces_the_low_snr_bias():
    e, its = _bias("NNLS", 10, (20.0, 40.0))
    print("\nNNLS, SNR 20-40, 400 voxels: MWF/FWF/T2_IE bias Gaussian %+.4f %+.4f %+.2f ms, Rician %+.4f %+.4f %+.2f ms; "
          "MM iterations median %d p90 %d max %d" % (*e["g"], *e["r"], np.median(its), np.percentile(its, 90), its.max()))
    assert abs(e["r"][1]) * 2.0 <= abs(e["g"][1])          # FWF
    e, its = _bias("X2", 10, (20.0, 40.0))
    print("X2, SNR 20-40, 400 voxels: MWF/FWF/T2_IE bias Gaussian %+.4f %+.4f %+.2f ms, Rician %+.4f %+.4f %+.2f ms; "
          "MM iterations median %d p90 %d max %d" % (*e["g"], *e["r"], np.median(its), np.percentile(its, 90), its.max()))
    assert abs(e["r"][2]) < abs(e["g"][2])                  # T2_IE
