"""TEST INFRASTRUCTURE ONLY — NumPy restatement of Step 1 with `--denoise TV` (motor/motor_recon_met2_real_data.py:293-303
of the reference): scikit-image's `estimate_sigma` (a wavelet MAD noise estimate on PyWavelets' single-level db2
transform) and `denoise_tv_chambolle` (`_denoise_tv_chambolle_nd`), stated line for line.  The GPU kernels of
csrc/met2_tv.cu are compared with these functions bit for bit (tests/test_emu_tv.py, tests/test_gpu_tv.py).

Written without scikit-image or PyWavelets available: neither library could be run beside it, so the restatement follows
their published source, and the db2 filter values below are PyWavelets' stored table as quoted, not checked against a
run of that library.  Only tests/ and tools/ import this module; the product package never does.
"""
import numpy as np

# PyWavelets' db2 decomposition high-pass filter (the stored values; the closed form differs by ~3e-13)
DB2_DEC_HI = (-0.48296291314469025, 0.836516303737469, -0.22414386804185735, -0.12940952255092145)
NORM_PPF_075 = 0.6744897501960817        # scipy.stats.norm.ppf(0.75)


def _sym_index(k, n):
    """PyWavelets' 'symmetric' mode: half-sample symmetric extension of x[0..n) with period 2n."""
    k = np.mod(k, 2 * n)
    return np.where(k < n, k, 2 * n - 1 - k)


def dwt_detail_axis(x, axis):
    """Single-level db2 high-pass band of `x` along `axis`: out[o] = sum_j dec_hi[j] * ext(2o + 1 - j), o < (n + 3) // 2,
    summed from 0.0 with j ascending."""
    x = np.moveaxis(np.asarray(x, dtype=np.float64), axis, -1)
    n = x.shape[-1]
    o = np.arange((n + 3) // 2)
    out = np.zeros(x.shape[:-1] + (len(o),))
    for j, h in enumerate(DB2_DEC_HI):
        out = out + h * x[..., _sym_index(2 * o + 1 - j, n)]
    return np.moveaxis(out, -1, axis)


def dwt_detail(image):
    """pywt.dwtn(image, 'db2')['d' * ndim]: the high-pass pass along axis 0, then 1, then 2, each on the previous output."""
    c = np.asarray(image, dtype=np.float64)
    for ax in range(c.ndim):
        c = dwt_detail_axis(c, ax)
    return c


def estimate_sigma(image):
    """skimage.restoration.estimate_sigma(image, channel_axis=None) -> _sigma_est_dwt: median(|c|) / norm.ppf(0.75) over
    the nonzero detail coefficients.  NaN if any coefficient is NaN or none is nonzero."""
    c = dwt_detail(image).ravel()
    c = c[np.nonzero(c)]
    if c.size == 0:
        return np.nan                     # np.median of an empty array (with a RuntimeWarning)
    return np.median(np.abs(c)) / NORM_PPF_075


def denoise_tv_chambolle(image, weight, eps=2.0e-4, max_num_iter=200):
    """skimage.restoration._denoise._denoise_tv_chambolle_nd for a float64 image.  Returns (out, iterations), the number of
    times `out` was formed."""
    image = np.asarray(image, dtype=np.float64)
    ndim = image.ndim
    p = np.zeros((image.ndim,) + image.shape, dtype=image.dtype)
    g = np.zeros_like(p)
    d = np.zeros_like(image)
    i = 0
    with np.errstate(all="ignore"):
        while i < max_num_iter:
            if i > 0:
                # d will be the (negative) divergence of p
                d = -p.sum(0)
                slices_d = [slice(None)] * ndim
                slices_p = [slice(None)] * (ndim + 1)
                for ax in range(ndim):
                    slices_d[ax] = slice(1, None)
                    slices_p[ax + 1] = slice(0, -1)
                    slices_p[0] = ax
                    d[tuple(slices_d)] += p[tuple(slices_p)]
                    slices_d[ax] = slice(None)
                    slices_p[ax + 1] = slice(None)
                out = image + d
            else:
                out = image
            E = (d ** 2).sum()
            # g stores the gradients of out along each axis; the last element of each axis stays 0
            slices_g = [slice(None)] * (ndim + 1)
            for ax in range(ndim):
                slices_g[ax + 1] = slice(0, -1)
                slices_g[0] = ax
                g[tuple(slices_g)] = np.diff(out, axis=ax)
                slices_g[ax + 1] = slice(None)
            norm = np.sqrt((g ** 2).sum(axis=0))[np.newaxis, ...]
            E += weight * norm.sum()
            tau = 1.0 / (2.0 * ndim)
            norm *= tau / weight
            norm += 1.0
            p -= tau * g
            p /= norm
            E /= float(image.size)
            if i == 0:
                E_init = E
                E_previous = E
            else:
                if np.abs(E_previous - E) < eps * E_init:
                    break
                else:
                    E_previous = E
            i += 1
    return out, (i + 1 if i < max_num_iter else max_num_iter)


def tv_denoise(data, eps=2.0e-4, max_num_iter=200):
    """Step 1 as the reference writes it: per echo t, vol = np.squeeze(data[..., t]) and
    denoise_tv_chambolle(vol, 2 * estimate_sigma(vol), eps, max_num_iter).  Returns (denoised data, sigma[nt],
    iterations[nt])."""
    data = np.asarray(data, dtype=np.float64)
    out = np.empty_like(data)
    nt = data.shape[3]
    sigma = np.zeros(nt)
    iters = np.zeros(nt, dtype=np.int32)
    for t in range(nt):
        vol = np.squeeze(data[:, :, :, t])
        sigma[t] = estimate_sigma(vol)
        den, iters[t] = denoise_tv_chambolle(vol, 2.0 * sigma[t], eps, max_num_iter)
        out[:, :, :, t] = den.reshape(data.shape[:3])
    return out, sigma, iters
