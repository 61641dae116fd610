"""The NumPy restatement of Step 1 with --denoise TV (tests/tv_oracle.py) checked without scikit-image or PyWavelets:
the db2 detail band against a dense analysis matrix, the noise estimate on white noise of known sigma, and properties of
the Chambolle iteration that follow from its definition."""
import numpy as np
import pytest

import tv_oracle as T


def _analysis_matrix(n):
    """W [m][n] with band = W @ x: row o holds dec_hi[j] at the sample ext(2o + 1 - j) of the half-sample symmetric
    extension x0 .. x_{n-1}, x_{n-1} .. x0 repeated with period 2n."""
    period = np.concatenate([np.arange(n), np.arange(n)[::-1]])
    m = (n + 3) // 2
    W = np.zeros((m, n))
    for o in range(m):
        for j, h in enumerate(T.DB2_DEC_HI):
            W[o, period[(2 * o + 1 - j) % (2 * n)]] += h
    return W


@pytest.mark.parametrize("n", range(2, 10))
def test_dwt_detail_equals_the_dense_analysis_matrix(n):
    rng = np.random.default_rng(n)
    W = _analysis_matrix(n)
    x = rng.standard_normal(n)
    assert np.allclose(T.dwt_detail(x), W @ x, rtol=0, atol=1e-14)
    a = rng.standard_normal((n, n + 1))
    ref2 = _analysis_matrix(n) @ a @ _analysis_matrix(n + 1).T
    assert np.allclose(T.dwt_detail(a), ref2, rtol=0, atol=1e-13)
    b = rng.standard_normal((3, n, 2))
    ref3 = np.einsum("ai,bj,ck,ijk->abc", _analysis_matrix(3), _analysis_matrix(n), _analysis_matrix(2), b)
    assert np.allclose(T.dwt_detail(b), ref3, rtol=0, atol=1e-13)


def test_estimate_sigma_on_white_noise():
    """Gaussian white noise of known sigma on 64^3.  Away from the volume's faces the db2 high-pass has unit energy, so the
    MAD estimate over the interior coefficients is within 2 %.  The first and last coefficient along each axis mix
    repeated samples of the symmetric extension (variance 3/4 of the others), which lowers the estimate over the whole
    band by 2-3 % at this size."""
    rng = np.random.default_rng(11)
    for sigma in (0.5, 3.0, 40.0):
        img = 100.0 + sigma * rng.standard_normal((64, 64, 64))
        inner = T.dwt_detail(img)[1:-1, 1:-1, 1:-1]
        assert abs(np.median(np.abs(inner)) / T.NORM_PPF_075 / sigma - 1.0) < 0.02
        assert 0.95 < T.estimate_sigma(img) / sigma < 1.0


def test_estimate_sigma_edge_cases():
    assert np.isnan(T.estimate_sigma(np.zeros((6, 5, 4))))            # no nonzero coefficient
    assert 0.0 < T.estimate_sigma(np.full((6, 5), 3.0)) < 1e-15         # constant: the db2 taps sum to -5.6e-17
    x = np.random.default_rng(3).standard_normal((7, 6))
    x[2, 3] = np.nan
    assert np.isnan(T.estimate_sigma(x))


def test_tv_preserves_the_sum():
    """The last slice of every p[ax] stays 0, so d has zero sum and out the sum of the image (to rounding)."""
    rng = np.random.default_rng(12)
    img = 50.0 + 5.0 * rng.standard_normal((13, 9, 5))
    out, it = T.denoise_tv_chambolle(img, 2.0 * T.estimate_sigma(img))
    assert 1 < it < 200 and not np.array_equal(out, img)
    assert abs(out.sum() - img.sum()) < 1e-11 * np.abs(img).sum()


def test_constant_image_runs_every_iteration_and_is_unchanged():
    """E_init = 0 for a constant image, so |E_prev - E| < eps * E_init never holds."""
    img = np.full((7, 6, 5), 5.0)
    out, it = T.denoise_tv_chambolle(img, 1.0, max_num_iter=37)
    assert it == 37 and np.array_equal(out, img)


def test_single_slice_volume_is_the_2d_filter():
    """A 40 x 33 x 1 volume is squeezed to 2-D (tau = 1/4) by tv_denoise, like the reference's np.squeeze."""
    rng = np.random.default_rng(13)
    data = 20.0 + rng.standard_normal((40, 33, 1, 2))
    out, sigma, iters = T.tv_denoise(data)
    for t in range(2):
        ref, it = T.denoise_tv_chambolle(data[:, :, 0, t], 2.0 * T.estimate_sigma(data[:, :, 0, t]))
        assert sigma[t] == T.estimate_sigma(data[:, :, 0, t]) and iters[t] == it
        assert np.array_equal(out[:, :, 0, t], ref)
    out3, it3 = T.denoise_tv_chambolle(data[..., 0], 2.0 * sigma[0])        # unsqueezed: tau = 1/6, another result
    assert not np.array_equal(out3[:, :, 0], out[:, :, 0, 0])
