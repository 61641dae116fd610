"""NumPy restatement of the slice-profile-integrated EPG curves of csrc/met2_epg.cu (met2_epg_dictionary_profile,
met2_epg_signals_profile): the reference's dense EPG (oracle/met2_oracle.py:epg_signal) at the per-position angles,
weighted and summed over the positions k = 0, 1, ..., K-1 in that order.  Also an isochromat Bloch simulation of the
same CPMG train, the independent check of the recurrence with an excitation angle apart from the refocusing angle."""
import numpy as np

import met2_oracle as O

RAD = np.pi / 180.0


def profile_curve(n, tau, T2, T1, alpha_deg, x, r, w):
    """sum_k w[k] EPG(T2, T1, refocusing alpha r[k], excitation (alpha / 2) x[k]) [n], without (1 - exp(-TR/T1))."""
    acc = np.zeros(n)
    for k in range(len(w)):
        acc = acc + w[k] * O.epg_signal(n, tau, 1.0 / T1, 1.0 / T2, alpha_deg * r[k] * RAD,
                                        alpha_deg / 2.0 * x[k] * RAD)
    return acc


def dictionary(alphas, T2s, T1s, n, tau, TR, x, r, w):
    """dic [nA][n][nT2] of met2_epg_dictionary_profile."""
    dic = np.zeros((len(alphas), n, len(T2s)))
    for a, al in enumerate(alphas):
        for j, (t2, t1) in enumerate(zip(T2s, T1s)):
            dic[a, :, j] = (1.0 - np.exp(-TR / t1)) * profile_curve(n, tau, t2, t1, al, x, r, w)
    return dic


def signals(alphas, T2s, T1s, n, tau, x, r, w):
    """sig [N][n] of met2_epg_signals_profile."""
    return np.stack([profile_curve(n, tau, t2, t1, al, x, r, w) for al, t2, t1 in zip(alphas, T2s, T1s)])


def bloch_cpmg(n, tau, refoc_deg, exc_deg, T2=np.inf, T1=np.inf, spins=720):
    """Echo magnitudes [n] of a CPMG train by isochromats: excitation about x, then per echo precession over tau/2,
    refocusing about y, precession over tau/2, with `spins` isochromats spread evenly over one cycle of dephasing
    (ideal crushers) and T2 / T1 decay without T1 recovery, the convention of the EPG recurrence."""
    ph = 2.0 * np.pi * np.arange(spins) / spins
    e2, e1 = np.exp(-(tau / 2.0) / T2), np.exp(-(tau / 2.0) / T1)
    c, s = np.cos(ph), np.sin(ph)
    th = np.deg2rad(exc_deg)
    mx, my, mz = np.zeros(spins), np.full(spins, np.sin(th)), np.full(spins, np.cos(th))   # (0, 0, 1) rotated about x
    q = np.deg2rad(refoc_deg)
    cq, sq = np.cos(q), np.sin(q)

    def precess(mx, my, mz):
        return (c * mx - s * my) * e2, (s * mx + c * my) * e2, mz * e1
    out = np.empty(n)
    for i in range(n):
        mx, my, mz = precess(mx, my, mz)
        mx, mz = cq * mx - sq * mz, sq * mx + cq * mz
        mx, my, mz = precess(mx, my, mz)
        out[i] = np.hypot(mx.mean(), my.mean())
    return out
