"""The physics behind the slice-profile dictionary, on the CPU: the EPG recurrence with an excitation angle apart from
the refocusing angle against an isochromat Bloch simulation, and the slice-profile generator (grids.slice_profile)
against the small-tip Fourier limit, symmetry in z and the exact angle of a rectangular pulse on resonance."""
import numpy as np
import pytest

import met2_oracle as O
import slice_profile_oracle as SP
from multicomponent_t2_toolbox_b200 import grids


@pytest.mark.parametrize("refoc, exc, T2", [(150.0, 30.0, np.inf), (100.0, 80.0, np.inf), (20.0, 5.0, np.inf),
                                            (170.0, 89.0, np.inf), (150.0, 75.0, 30.0), (120.0, 45.0, 60.0)])
def test_decoupled_recurrence_matches_bloch(refoc, exc, T2):
    n, tau = 8, 10.0
    ref = O.epg_signal(n, tau, 1.0 / 1000.0 if np.isfinite(T2) else 1e-12, 1.0 / T2 if np.isfinite(T2) else 1e-12,
                       np.deg2rad(refoc), np.deg2rad(exc))
    bl = SP.bloch_cpmg(n, tau, refoc, exc, T2=T2 if np.isfinite(T2) else 1e12, T1=1000.0 if np.isfinite(T2) else 1e12)
    assert np.max(np.abs(ref - bl)) <= 1e-12


def test_small_tip_limit_is_the_fourier_transform_of_the_waveform():
    """At a tiny flip angle the rotation is 2|beta| = |sum_j b_j sinc(g / 2) e^{-i g j}| with g the gradient phase per
    step (the hard-pulse discretisation's sinc), up to O(flip^3)."""
    for wave in (grids.hann_sinc(2.7, 256), grids.hann_sinc(6.0, 256), np.hanning(200)):
        flip = 1e-3
        f = np.linspace(-4.0, 4.0, 41)
        got = grids.pulse_rotation(wave, flip, f)
        b = np.deg2rad(flip) * wave / wave.sum()
        g = 2.0 * np.pi * f / len(b)
        ft = np.abs(np.exp(-1j * np.outer(g, np.arange(len(b)))) @ b) * np.sinc(g / (2.0 * np.pi))
        assert np.max(np.abs(got - np.rad2deg(ft))) <= 1e-6 * flip


def test_profile_is_symmetric_in_z():
    for ratio in (1.0, 2.0):
        x, r, w = grids.slice_profile(tbw=2.7, ratio=ratio, K=65)
        assert np.max(np.abs(x - x[::-1])) <= 1e-12 and np.max(np.abs(r - r[::-1])) <= 1e-12
        assert abs(x[32] - 1.0) <= 1e-12 and abs(r[32] - 1.0) <= 1e-12
        assert np.all(x <= 1.0 + 1e-12) and np.all(r <= 1.0 + 1e-12) and np.all(w == 1.0 / 65)


def test_rectangular_pulse_on_resonance_gives_its_angle():
    for flip in (30.0, 90.0, 137.0, 180.0):
        assert abs(grids.pulse_rotation(np.ones(64), flip, [0.0])[0] - flip) <= 1e-12
    x, r, w = grids.slice_profile(K=1, waveform_exc=np.ones(32), waveform_ref=np.ones(32))
    assert abs(x[0] - 1.0) <= 1e-12 and abs(r[0] - 1.0) <= 1e-12 and w[0] == 1.0


def test_wider_refocusing_slab_flattens_the_refocusing_profile():
    _, r1, _ = grids.slice_profile(ratio=1.0)
    x2, r2, _ = grids.slice_profile(ratio=2.0)
    assert r2.mean() > r1.mean() + 0.1


def test_profile_arguments_are_checked():
    x, r, w = grids.slice_profile(K=8)
    xs, rs, ws = grids.as_slice_profile((x, r, 3.0 * w))
    assert np.array_equal(xs, x) and abs(ws.sum() - 1.0) <= 1e-15
    for bad in ((x, r), (x, r[:4], w), (x, r, -w), (x * np.nan, r, w), (x, r, 0 * w), (np.ones(513),) * 3):
        with pytest.raises(ValueError):
            grids.as_slice_profile(bad)
    with pytest.raises(ValueError):
        grids.slice_profile(K=0)
