"""NumPy restatement of met2_degibbs (csrc/met2_degibbs.cu, whose header holds the definition), operation for operation:
the same IEEE +, -, *, / and |.| in the same order, vectorised across lines and slices (elementwise IEEE operations do
not depend on the batch).  It takes the library's tables (met2_degibbs_tables) as input, so that a last-bit difference
between two cos / sin implementations cannot move a TV argmin.

Volumes are handled as [n0, n1, S] (S = nz * nt, the slice index fastest, as in the C-order volume)."""
import numpy as np

NSH, MINW, MAXW = 20, 1, 3


def split_tables(tab, n, nsh):
    """The table of one in-plane size -> (cos[n], sin[n], c[n], h[2 nsh + 1][n])."""
    tab = np.asarray(tab, dtype=np.float64)
    assert tab.shape == (n * (2 * nsh + 4),)
    return tab[:n], tab[n:2 * n], tab[2 * n:3 * n], tab[3 * n:].reshape(2 * nsh + 1, n)


def shifts(nsh):
    """m_q for q = 0..2 nsh: 0, +1, .., +nsh, -1, .., -nsh."""
    return np.array([q if q <= nsh else nsh - q for q in range(2 * nsh + 1)])


def _dft(re, im, cs, sn, axis, fwd, real_part_only=False):
    """Direct DFT of every line along `axis` (0 or 1) of [n0, n1, S] arrays: out[k] = sum_x in[x] w[(k x) mod n],
    x ascending from 0.0, w = (cos, -sin) forward and (cos, sin) inverse.  im None: real input."""
    n = re.shape[axis]
    k = np.arange(n)
    shape = [1, 1, 1]
    shape[axis] = n
    acc_re = np.zeros(re.shape)
    acc_im = np.zeros(re.shape)
    for x in range(n):
        idx = (k * x) % n
        c = cs[idx].reshape(shape)
        w = (-sn[idx] if fwd else sn[idx]).reshape(shape)
        ar = np.take(re, [x], axis=axis)
        if im is None:
            acc_re = acc_re + ar * c
            acc_im = acc_im + ar * w
        else:
            ai = np.take(im, [x], axis=axis)
            acc_re = acc_re + (ar * c - ai * w)
            if not real_part_only:
                acc_im = acc_im + (ar * w + ai * c)
    return acc_re, acc_im


def g0(c0, c1):
    den = c0[:, None] + c1[None, :]
    with np.errstate(divide="ignore", invalid="ignore"):
        g = c1[None, :] / den
    return np.where(den == 0.0, 0.5, g)


def split(u, tab0, tab1, nsh=NSH):
    """Step 1: u [n0, n1, S] -> (v0, v1) and the intermediate spectra (A rows, P = U G0, B)."""
    n0, n1, _ = u.shape
    cs0, sn0, c0, _ = split_tables(tab0, n0, nsh)
    cs1, sn1, c1, _ = split_tables(tab1, n1, nsh)
    a_re, a_im = _dft(u, None, cs1, sn1, 1, True)
    u_re, u_im = _dft(a_re, a_im, cs0, sn0, 0, True)
    g = g0(c0, c1)[:, :, None]
    p_re, p_im = u_re * g, u_im * g
    b_re, b_im = _dft(p_re, p_im, cs1, sn1, 1, False)
    s_re, _ = _dft(b_re, b_im, cs0, sn0, 0, False, real_part_only=True)
    v0 = s_re / float(n0 * n1)
    return v0, u - v0, dict(A=(a_re, a_im), U=(u_re, u_im), P=(p_re, p_im), B=(b_re, b_im))


def shifted_lines(x, h):
    """y_q[..., j] = sum_d h[q][d] x[..., (j - d) mod n] for every q -> [2 nsh + 1, ..., n]."""
    ys = []
    for hq in h:
        y = np.zeros(x.shape)
        for d in range(x.shape[-1]):
            y = y + hq[d] * np.roll(x, d, axis=-1)
        ys.append(y)
    return np.stack(ys)


def unring_lines(x, h, nsh=NSH, minW=MINW, maxW=MAXW):
    """Step 2 on lines x[..., n] (the last axis) with the kernel table h [2 nsh + 1][n]."""
    Y = shifted_lines(x, h)
    best = np.full(x.shape, np.inf)
    sel = np.zeros(x.shape, dtype=np.int64)
    for q in range(len(h)):
        y = Y[q]
        tvl = np.zeros(x.shape)
        for w in range(minW, maxW + 1):
            tvl = tvl + np.abs(np.roll(y, w, axis=-1) - np.roll(y, w + 1, axis=-1))
        tvr = np.zeros(x.shape)
        for w in range(minW, maxW + 1):
            tvr = tvr + np.abs(np.roll(y, -w, axis=-1) - np.roll(y, -w - 1, axis=-1))
        for tv in (tvl, tvr):
            upd = tv < best
            best = np.where(upd, tv, best)
            sel = np.where(upd, q, sel)
    y0 = np.take_along_axis(Y, sel[None], 0)[0]
    yp = np.take_along_axis(np.roll(Y, 1, axis=-1), sel[None], 0)[0]      # y[j - 1]
    yn = np.take_along_axis(np.roll(Y, -1, axis=-1), sel[None], 0)[0]     # y[j + 1]
    s = shifts(nsh)[sel] / float(2 * nsh)
    a = np.abs(s)
    with np.errstate(invalid="ignore"):
        return np.where(s > 0.0, (1.0 - s) * y0 + s * yp, (1.0 - a) * y0 + a * yn)


def degibbs(vol, tab0, tab1, nsh=NSH, minW=MINW, maxW=MAXW):
    """met2_degibbs on a volume [nx, ny, ...] (trailing axes are slices) with the library's tables of sizes nx, ny."""
    vol = np.asarray(vol, dtype=np.float64)
    n0, n1 = vol.shape[:2]
    u = vol.reshape(n0, n1, -1)
    with np.errstate(invalid="ignore", over="ignore"):
        v0, v1, _ = split(u, tab0, tab1, nsh)
        h0 = split_tables(tab0, n0, nsh)[3]
        h1 = split_tables(tab1, n1, nsh)[3]
        r0 = np.moveaxis(unring_lines(np.moveaxis(v0, 0, -1), h0, nsh, minW, maxW), -1, 0)
        r1 = np.moveaxis(unring_lines(np.moveaxis(v1, 1, -1), h1, nsh, minW, maxW), -1, 1)
        out = r0 + r1
    return out.reshape(vol.shape)
