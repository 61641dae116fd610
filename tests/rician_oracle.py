"""NumPy restatement of the Rician-likelihood spectrum fit (definition in csrc/met2_rician.cu, DESIGN.md §10f).

A(z) = I1(z) / I0(z) in the kernel's operation order, from the Chebyshev tables the kernel source carries (the test
against scipy.special.i1e / i0e checks them); the MM iteration with one Lawson-Hanson solve of the stacked system
[D; sqrt(lam) L] per iteration (oracle/met2_oracle.py: lh_nnls); the objective Phi and its gradient.  Spectra are in the
reference's normalised units (fsol / sig[0])."""
import os
import re

import numpy as np

import met2_oracle as O

_SRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "multicomponent_t2_toolbox_b200",
                    "csrc", "met2_rician.cu")


def _tables():
    src = open(_SRC).read()
    out = {}
    for name, n in (("A0", 30), ("A1", 29), ("B0", 25), ("B1", 25)):
        body = re.search(r"const double %s\[%d\] = \{(.*?)\};" % (name, n), src, re.S).group(1)
        vals = [float(v) for v in re.findall(r"[-+]?\d\.\d+E[-+]\d+", body)]
        assert len(vals) == n, name
        out[name] = vals
    return out


T = _tables()


def chbevl(x, c):
    """Cephes' chbevl, elementwise: b0 = c[0]; b0 <- x b1 - b2 + c[k]; 0.5 (b0 - b2)."""
    x = np.asarray(x, dtype=np.float64)
    b0, b1, b2 = np.full_like(x, c[0]), np.zeros_like(x), np.zeros_like(x)
    for ck in c[1:]:
        b2 = b1
        b1 = b0
        b0 = x * b1 - b2 + ck
    return 0.5 * (b0 - b2)


def bessel_ratio(z):
    """A(z) = I1(z) / I0(z), the kernel's rc_bessel_ratio operation for operation; A(-z) = -A(z)."""
    z = np.asarray(z, dtype=np.float64)
    a = np.where(z < 0.0, -z, z)
    with np.errstate(all="ignore"):    # both branches are evaluated everywhere
        t1 = a / 2.0 - 2.0
        small = (a * chbevl(t1, T["A1"])) / chbevl(t1, T["A0"])
        t2 = 32.0 / a - 2.0
        large = chbevl(t2, T["B1"]) / chbevl(t2, T["B0"])
    r = np.where(a <= 8.0, small, large)
    return np.where(z < 0.0, -r, r)


def modified_data(y, f, s2):
    """yt = y * A((y * f) / s2); y itself when s2 = 0."""
    if not s2 > 0.0:
        return np.array(y, dtype=np.float64, copy=True)
    return y * bessel_ratio((y * f) / s2)


def objective(x, D, y, L, lam, sn):
    """Phi(x) = sum_e [f_e^2 - 2 s2 log I0(y_e f_e / s2)] + lam ||L x||^2 with log I0(z) = log i0e(z) + z, i.e.
    sum_e [f_e^2 - 2 y_e f_e - 2 s2 log i0e(z_e)] + lam ||L x||^2 (the sn -> 0 limit is ||D x - y||^2 - ||y||^2 + ...)."""
    import scipy.special as sp
    f = D @ x
    s2 = sn * sn
    lik = np.sum(f * f - 2.0 * y * f - 2.0 * s2 * np.log(sp.i0e((y * f) / s2)))
    return lik + lam * np.sum((L @ x) ** 2)


def gradient(x, D, y, L, lam, sn):
    """Half the gradient of Phi: D^T (f - y A(y f / s2)) + lam K x."""
    f = D @ x
    return D.T @ (f - modified_data(y, f, sn * sn)) + lam * (L.T @ (L @ x))


def solve(D, yt, L, lam, fast=False):
    """argmin_{x >= 0} ||D x - yt||^2 + lam ||L x||^2 by Lawson-Hanson (fast: SciPy's compiled routine instead of the
    restatement); returns (x, hit itmax)."""
    if lam > 0.0:
        A = np.concatenate((D, np.sqrt(lam) * L))
        b = np.concatenate((yt, np.zeros(L.shape[0])))
    else:
        A, b = D, yt
    if fast:
        return O.nnls(A, b)[0], False
    x, _, mode = O.lh_nnls(A, b)
    return x, mode == 3


def mm_fit(D, y, L, lam, sn, x0, max_iter=200, tol=1e-9, trace=None, fast=False):
    """The MM loop of the definition from x0.  Returns (x, iters, capped, itmax); `trace` (a list) gets every iterate;
    fast: see `solve`."""
    x = np.array(x0, dtype=np.float64, copy=True)
    yt_prev = np.array(y, dtype=np.float64, copy=True)
    s2 = sn * sn
    itmax = False
    for k in range(1, max_iter + 1):
        yt = modified_data(y, D @ x, s2)
        if np.max(np.abs(yt - yt_prev)) <= tol:
            return x, k - 1, False, itmax
        x, hit = solve(D, yt, L, lam, fast)
        itmax |= hit
        yt_prev = yt
        if trace is not None:
            trace.append(x)
    return x, max_iter, True, itmax
