"""The NumPy restatement of met2_degibbs (tests/degibbs_oracle.py) against independent arithmetic: numpy.fft for the
split and the shifted lines, exact identities of the split, images the method must leave (nearly) alone, and the
ringing it must remove.  The tables are the library's (met2_degibbs_tables of the emulator build)."""
import numpy as np
import pytest

import degibbs_oracle as O
from test_emu_degibbs import tables

SIZES = [(16, 16), (17, 24), (63, 80), (96, 96)]


def _rel(a, b):
    return np.abs(a - b).max() / np.abs(b).max()


@pytest.mark.parametrize("n0, n1", SIZES)
def test_split_against_numpy_fft(n0, n1):
    rng = np.random.default_rng(n0 * n1)
    u = rng.standard_normal((n0, n1, 3)) + 5.0
    v0, v1, mid = O.split(u, tables(n0), tables(n1))
    a = mid["A"][0] + 1j * mid["A"][1]
    assert _rel(a, np.fft.fft(u, axis=1)) <= 1e-12
    U = np.fft.fft2(u, axes=(0, 1))
    assert _rel(mid["U"][0] + 1j * mid["U"][1], U) <= 1e-12
    f0, f1 = np.fft.fftfreq(n0), np.fft.fftfreq(n1)
    c0, c1 = 1.0 + np.cos(2 * np.pi * f0), 1.0 + np.cos(2 * np.pi * f1)
    den = c0[:, None] + c1[None, :]
    G0 = np.where(den == 0.0, 0.5, c1[None, :] / np.where(den == 0.0, 1.0, den))
    assert _rel(mid["B"][0] + 1j * mid["B"][1], np.fft.ifft(U * G0[:, :, None], axis=1) * n1) <= 1e-12
    ref_v0 = np.real(np.fft.ifft2(U * G0[:, :, None], axes=(0, 1)))
    assert _rel(v0, ref_v0) <= 1e-12
    # v1 is u - v0 bit for bit, so v0 + v1 is u up to the rounding of the two subtractions / additions
    assert np.array_equal(v1, u - v0)
    scale = np.maximum(np.maximum(np.abs(u), np.abs(v0)), np.abs(v1))
    assert (np.abs((v0 + v1) - u) <= 2.0 ** -52 * scale).all()


@pytest.mark.parametrize("n", [16, 17, 96])
def test_shifted_lines_against_numpy_fft(n):
    rng = np.random.default_rng(n)
    x = rng.standard_normal((5, n))
    h = O.split_tables(tables(n), n, O.NSH)[3]
    Y = O.shifted_lines(x, h)
    f = np.fft.fftfreq(n)
    for q, m in enumerate(O.shifts(O.NSH)):
        ref = np.real(np.fft.ifft(np.fft.fft(x, axis=-1) * np.exp(2j * np.pi * f * m / (2 * O.NSH)), axis=-1))
        assert _rel(Y[q], ref) <= 1e-12
    assert np.array_equal(Y[0], x * 1.0)                 # h_0 is an exact delta in the library's table


@pytest.mark.parametrize("n0, n1", SIZES)
def test_constant_image_unchanged(n0, n1):
    u = np.full((n0, n1, 2), 123.25)
    out = O.degibbs(u, tables(n0), tables(n1))
    assert np.abs(out - u).max() <= 1e-12 * 123.25


@pytest.mark.parametrize("n0, n1", SIZES)
def test_band_limited_image_within_the_interpolation_bound(n0, n1):
    """A smooth image (periods >= 16 pixels) is not ringing, but the method still moves it: each part is shifted by
    some s_q, |s_q| <= 1/2, and linearly interpolated back.  Linear interpolation of the band-limited line at fraction
    s errs by at most s (1 - s) / 2 max |x''| <= max |x''| / 8, so |out - u| <= (max |v0''_0| + max |v1''_1|) / 8, the
    second derivatives along each part's unringing axis (exact, by spectral differentiation)."""
    x = np.arange(n0)[:, None, None]
    y = np.arange(n1)[None, :, None]
    u = 50.0 + 20.0 * np.cos(2 * np.pi * x / 16.0 + 0.3) * np.cos(2 * np.pi * y / 24.0 + 1.1) + \
        10.0 * np.sin(2 * np.pi * (x / 32.0 + y / 20.0))
    u = u * np.ones((1, 1, 2))
    out = O.degibbs(u, tables(n0), tables(n1))
    v0, v1, _ = O.split(u, tables(n0), tables(n1))

    def d2(v, axis):
        f = np.fft.fftfreq(v.shape[axis]).reshape([-1 if a == axis else 1 for a in range(3)])
        return np.real(np.fft.ifft(np.fft.fft(v, axis=axis) * -(2 * np.pi * f) ** 2, axis=axis))

    bound = (np.abs(d2(v0, 0)).max() + np.abs(d2(v1, 1)).max()) / 8.0
    change = np.abs(out - u).max()
    print("band-limited %d x %d: max change %.3g, bound %.3g" % (n0, n1, change, bound))
    assert 0.0 < change <= bound


def _phantom(N0, N1):
    """Piecewise-constant phantom on a fine grid: an ellipse, a darker rectangle and a bright disc."""
    x = np.arange(N0)[:, None] / N0
    y = np.arange(N1)[None, :] / N1
    img = np.zeros((N0, N1))
    img[(x - 0.5) ** 2 / 0.37 ** 2 + (y - 0.5) ** 2 / 0.41 ** 2 <= 1] = 100.0
    img[(np.abs(x - 0.41) < 0.11) & (np.abs(y - 0.56) < 0.143)] = 40.0
    img[(x - 0.63) ** 2 + (y - 0.39) ** 2 <= 0.083 ** 2] = 160.0
    return img


def truncated_phantom(n0, n1):
    """(ringing image, reference): the phantom on a 2 n0 x 2 n1 grid, its k-space truncated to the central half and
    reconstructed on the n0 x n1 grid (the acquisition's truncation), and the untruncated phantom at the same
    resolution (2 x 2 means of the fine grid)."""
    fine = _phantom(2 * n0, 2 * n1)
    F = np.fft.fft2(fine)
    k0 = np.fft.fftfreq(n0, 1.0 / n0).astype(int)
    k1 = np.fft.fftfreq(n1, 1.0 / n1).astype(int)
    ring = np.real(np.fft.ifft2(F[np.ix_(k0 % (2 * n0), k1 % (2 * n1))])) / 4.0
    return ring, fine.reshape(n0, 2, n1, 2).mean(axis=(1, 3))


@pytest.mark.parametrize("n0, n1", [(96, 96), (63, 80)])
def test_ringing_is_reduced(n0, n1):
    """RMSE against the untruncated phantom: over the whole image it falls by >= 1.1x (measured 1.120 at 96 x 96, 1.107
    at 63 x 80: the partial-volume blur of the edges dominates and is not ringing); more than two pixels from every edge,
    where only the ripples are left, by >= 5.5x (measured 7.48 and 5.89)."""
    from scipy import ndimage
    ring, ref = truncated_phantom(n0, n1)
    out = O.degibbs(ring[:, :, None], tables(n0), tables(n1))[:, :, 0]
    edge = ndimage.maximum_filter(ref, 3) != ndimage.minimum_filter(ref, 3)
    far = ~ndimage.binary_dilation(edge, iterations=1)
    rmse = lambda a, m: float(np.sqrt(np.mean((a - ref)[m] ** 2)))
    whole = np.ones(ref.shape, bool)
    f_whole = rmse(ring, whole) / rmse(out, whole)
    f_far = rmse(ring, far) / rmse(out, far)
    print("ringing %d x %d: RMSE factor whole %.3f, away from edges %.3f" % (n0, n1, f_whole, f_far))
    assert f_whole >= 1.1 and f_far >= 5.5
