"""Host-side grids of the MET2 inverse problem (T2 grid, flip-angle grids, lambda grid, regularisation matrices).

Mirrors the hard-coded set-up of the reference orchestrator
(motor/motor_recon_met2_real_data.py:204-273 and :86-111).  Pure numpy, tiny, runs once per reconstruction.
"""
import math

import numpy as np

REG_MATRICES = ("I", "L1", "L2", "InvT2")
REG_METHODS = ("NNLS", "T2SPARC", "X2", "L_curve", "GCV", "BayesReg")
FA_METHODS = ("spline", "brute-force")


def t2_grid(npc, t2_min=10.0, t2_max=2000.0):
    """`T2s = logspace(log10(10), log10(2000), Npc)` (motor...:215-220)."""
    return np.logspace(math.log10(t2_min), math.log10(t2_max), num=npc, endpoint=True, base=10.0)


def default_npc(reg_method):
    """Npc = 96 for T2SPARC else 60 (motor...:207-213)."""
    return 96 if reg_method == "T2SPARC" else 60


def compartment_masks(T2s, myelin_T2, t2_tissue=200.0):
    """ind_m / ind_t / ind_csf (motor...:222-224).  Note ind_t and ind_csf overlap at T2 == 200 exactly."""
    ind_m = T2s <= myelin_T2
    ind_t = (T2s > myelin_T2) & (T2s <= t2_tissue)
    ind_csf = T2s >= t2_tissue
    return ind_m, ind_t, ind_csf


def fa_grids(FA_method, n_alphas=None):
    """Flip-angle grids (motor...:231-245): spline -> 273-grid + 15 knots; brute-force -> 91-grid."""
    if FA_method == "spline":
        alpha_values = np.linspace(90.0, 180.0, 91 * 3 if n_alphas is None else n_alphas)
        alpha_values_spline = np.linspace(90.0, 180.0, 15)
        return alpha_values, alpha_values_spline
    if FA_method == "brute-force":
        alpha_values = np.linspace(90.0, 180.0, 91 if n_alphas is None else n_alphas)
        return alpha_values, None
    raise ValueError("Error: Wrong FA_method option!")


def lambda_grid(num=50, lam_min=1e-8, lam_max=10.0):
    """L-curve grid: lambda_reg[0] = 0, lambda_reg[1:] = logspace(1e-8, 10, 49) (motor...:248-251)."""
    lam = np.zeros((num,))
    lam[1:] = np.logspace(math.log10(lam_min), math.log10(lam_max), num=num - 1, endpoint=True, base=10.0)
    return lam


def create_Laplacian_matrix(Npc, order):
    """Dense regularisation matrix of order 0 (I), 1 (lower bidiagonal) or 2 (tridiagonal, Neumann corners).

    Same matrices as motor/motor_recon_met2_real_data.py:86-111, built directly instead of through scipy.sparse.
    """
    if order == 0:
        return np.eye(Npc)
    if order == 1:
        L = np.eye(Npc)
        L[np.arange(1, Npc), np.arange(0, Npc - 1)] = -1.0
        return L
    if order == 2:
        L = 2.0 * np.eye(Npc)
        L[np.arange(1, Npc), np.arange(0, Npc - 1)] = -1.0
        L[np.arange(0, Npc - 1), np.arange(1, Npc)] = -1.0
        L[0, 0] = 1.0
        L[-1, -1] = 1.0
        return L
    raise ValueError("order must be 0, 1 or 2")


def reg_matrix(name, T2s):
    """`Laplac` for reg_matrix in {I, L1, L2, InvT2} (motor...:254-273)."""
    npc = len(T2s)
    if name == "I":
        return create_Laplacian_matrix(npc, 0)
    if name == "L1":
        return create_Laplacian_matrix(npc, 1)
    if name == "L2":
        return create_Laplacian_matrix(npc, 2)
    if name == "InvT2":
        T2s_mod = np.concatenate((np.array([T2s[0] - 1.0]), T2s[:-1]))
        deltaT2 = T2s - T2s_mod
        deltaT2[0] = deltaT2[1]
        return np.diag(1.0 / deltaT2)
    raise ValueError("Error: Wrong reg_matrix option!")


def hann_sinc(tbw, n=512):
    """Hann-windowed sinc of time-bandwidth product `tbw`, sampled at the midpoints of n steps over the pulse."""
    t = (np.arange(n) + 0.5) / n - 0.5
    return np.sinc(tbw * t) * (0.5 + 0.5 * np.cos(2.0 * np.pi * t))


def pulse_rotation(waveform, flip_deg, freq):
    """Rotation angle (deg) of an RF pulse at the off-resonance frequencies `freq` (cycles per pulse duration), by a
    hard-pulse Cayley-Klein Bloch simulation: the waveform (any real samples, scaled so that their sum is flip_deg) is
    applied as len(waveform) instantaneous rotations about (b_j, 0, 2 pi freq / n).  Returns 2 arcsin|beta| (evaluated
    as 2 atan2(|beta|, |alpha|)); the phase of the result is dropped."""
    b = np.asarray(waveform, dtype=np.float64)
    b = b * (np.deg2rad(float(flip_deg)) / b.sum())
    g = 2.0 * np.pi * np.asarray(freq, dtype=np.float64) / len(b)
    a, bb = np.ones(g.shape, complex), np.zeros(g.shape, complex)
    for bj in b:
        phi = np.hypot(bj, g)
        s = np.sin(phi / 2.0)
        with np.errstate(invalid="ignore", divide="ignore"):
            nx = np.where(phi > 0.0, bj / phi, 0.0)
            nz = np.where(phi > 0.0, g / phi, 0.0)
        al = np.cos(phi / 2.0) - 1j * nz * s
        be = -1j * nx * s
        a, bb = al * a - np.conj(be) * bb, be * a + np.conj(al) * bb
    return np.rad2deg(2.0 * np.arctan2(np.abs(bb), np.abs(a)))   # 2 arcsin|beta|, well conditioned near 180


def slice_profile(tbw=2.7, ratio=1.0, K=64, extent=1.5, waveform_exc=None, waveform_ref=None):
    """Slice profile (x, r, w) of a 2-D multi-slice CPMG acquisition for the profile-integrated EPG dictionary
    (`batched.Dictionary(profile=...)`, csrc/met2_epg.cu): K positions z evenly spaced over [-extent, extent] in units of
    the excitation slice thickness, equal weights w = 1 / K, and the effective angles of the excitation (nominal 90)
    and refocusing (nominal 180) pulses there as fractions of the nominal angle: x[k] = theta_exc(z_k) / 90,
    r[k] = theta_ref(z_k) / 180.

    Each pulse is simulated by `pulse_rotation` (hard-pulse Cayley-Klein Bloch).  The default pulse is a Hann-windowed
    sinc of time-bandwidth product `tbw` (`hann_sinc`); waveform_exc / waveform_ref replace either by the caller's
    samples (scaled to the nominal angle).  Position z lies at tbw * z cycles per pulse off resonance for the excitation
    and at tbw * z / ratio for the refocusing pulse, whose slab is `ratio` times the excitation thickness.  The
    excitation phase across the slice is ignored: only the rotation angle 2 arcsin|beta| enters the model, as in the
    single-angle dictionary.  A caller with its own pulse simulation passes its own (x, r, w) instead."""
    K = int(K)
    if not 1 <= K <= 512:
        raise ValueError("K must be in 1..512")
    if not (tbw > 0 and ratio > 0 and extent >= 0):
        raise ValueError("tbw and ratio must be > 0 and extent >= 0")
    z = np.linspace(-extent, extent, K) if K > 1 else np.zeros(1)
    exc = hann_sinc(tbw) if waveform_exc is None else waveform_exc
    ref = hann_sinc(tbw) if waveform_ref is None else waveform_ref
    x = pulse_rotation(exc, 90.0, tbw * z) / 90.0
    r = pulse_rotation(ref, 180.0, tbw * z / ratio) / 180.0
    return x, r, np.full(K, 1.0 / K)


def as_slice_profile(profile):
    """(x, r, w) as three float64 arrays of one length K in 1..512, all finite and >= 0, with w normalised to sum 1."""
    try:
        x, r, w = (np.ascontiguousarray(np.asarray(a, dtype=np.float64).reshape(-1)) for a in profile)
    except (TypeError, ValueError):
        raise ValueError("a slice profile is a tuple (x, r, w) of three arrays")
    if not (len(x) == len(r) == len(w) and 1 <= len(x) <= 512):
        raise ValueError("a slice profile needs x, r, w of one length K in 1..512")
    if not all(np.all(np.isfinite(a)) and np.all(a >= 0.0) for a in (x, r, w)) or not w.sum() > 0.0:
        raise ValueError("slice profile entries must be finite and >= 0, with a positive sum of weights")
    return x, r, np.ascontiguousarray(w / w.sum())
