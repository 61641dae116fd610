"""Seeded synthetic 3-compartment MET2 phantom (SURVEY.md §8d).

Input generator only (not on the fitted path): builds `[nx, ny, nz, nTE]` float64 multi-echo volumes whose voxels are a
myelin / intra-extra-cellular / free-water mixture pushed through the stimulated-echo EPG forward model at a
per-voxel (continuous) flip angle, with Rician noise.  The recipe follows the reference's Monte-Carlo scripts
(scripts_synthetic_data_evaluation/Paper_Comparison/evaluate_all_methods_two_lobes_SNR50_150.py:40-57,156-176,386-394)
with discrete compartments.  The EPG forward model here is a vectorised numpy recurrence over voxels that applies the
same operator sequence as epg/epg.py:64-153 (shift, relax tau/2, RF, shift, relax tau/2 per echo).
"""
import numpy as np


def epg_signal_batch(n_echoes, tau, T1, T2, alpha_deg, chunk=65536, exc_deg=None):
    """EPG multi-echo decay for arrays of (T1, T2, alpha) — one decay curve per element.

    State layout follows epg/epg.py:97-147: index 0 is F0, block k=1..n holds (F+k, F-k, Zk).  The excitation is
    alpha/2 (or exc_deg, an array like alpha_deg) and the start state is x[0]=sin(a_exc), F-1 slot = cos(a_exc)
    (epg/epg.py:57,143-147).  Returns [N, n_echoes] (no (1-exp(-TR/T1)) factor).
    """
    T1 = np.asarray(T1, dtype=np.float64).ravel()
    T2 = np.asarray(T2, dtype=np.float64).ravel()
    alpha_deg = np.asarray(alpha_deg, dtype=np.float64).ravel()
    if exc_deg is not None:
        exc_deg = np.broadcast_to(np.asarray(exc_deg, dtype=np.float64).ravel(), alpha_deg.shape)
    N = T2.shape[0]
    out = np.empty((N, n_echoes))
    n = n_echoes
    for s in range(0, N, chunk):
        e = min(N, s + chunk)
        a = alpha_deg[s:e] * (np.pi / 180.0)
        a_exc = (alpha_deg[s:e] / 2.0 if exc_deg is None else exc_deg[s:e]) * (np.pi / 180.0)
        e2 = np.exp(-(tau / 2.0) / T2[s:e])
        e1 = np.exp(-(tau / 2.0) / T1[s:e])
        c2 = np.cos(a / 2.0) ** 2
        s2 = np.sin(a / 2.0) ** 2
        sa = np.sin(a)
        ca = np.cos(a)
        m = e - s
        # Fp[k], Fm[k], Z[k] for k = 0..n+1 (k=0 and k=n+1 are padding that stays zero); F0 separately.
        F0 = np.sin(a_exc)
        Fp = np.zeros((n + 2, m))
        Fm = np.zeros((n + 2, m))
        Z = np.zeros((n + 2, m))
        Fm[1] = np.cos(a_exc)
        for iecho in range(n):
            for half in range(2):
                # shift: F0 <- F-1 ; F+1 <- F0 ; F+k <- F+(k-1) ; F-k <- F-(k+1) ; Z unchanged
                newF0 = Fm[1].copy()
                Fp[2:n + 1] = Fp[1:n].copy()
                Fp[1] = F0
                Fm[1:n] = Fm[2:n + 1].copy()
                Fm[n] = 0.0
                F0 = newF0
                # relax over tau/2
                F0 = F0 * e2
                Fp[1:n + 1] *= e2
                Fm[1:n + 1] *= e2
                Z[1:n + 1] *= e1
                if half == 0:
                    # RF mixing on every block k >= 1; F0 is left untouched (T[0,0] = 1, epg/epg.py:125)
                    fp = Fp[1:n + 1]
                    fm = Fm[1:n + 1]
                    z = Z[1:n + 1]
                    nfp = c2 * fp + s2 * fm + sa * z
                    nfm = s2 * fp + c2 * fm - sa * z
                    nz = -0.5 * sa * fp + 0.5 * sa * fm + ca * z
                    Fp[1:n + 1] = nfp
                    Fm[1:n + 1] = nfm
                    Z[1:n + 1] = nz
            out[s:e, iecho] = F0
    return out


def b1_field(shape, rng, jitter=3.0):
    """Smooth flip-angle field FA = 180 (1 - 0.3 r^2) + U(-jitter, jitter), clipped to [95, 180] (SURVEY.md §8d)."""
    nx, ny, nz = shape
    gx = np.linspace(-1.0, 1.0, nx)[:, None, None] if nx > 1 else np.zeros((1, 1, 1))
    gy = np.linspace(-1.0, 1.0, ny)[None, :, None] if ny > 1 else np.zeros((1, 1, 1))
    gz = np.linspace(-1.0, 1.0, nz)[None, None, :] if nz > 1 else np.zeros((1, 1, 1))
    r2 = (gx ** 2 + gy ** 2 + gz ** 2) / 3.0
    fa = 180.0 * (1.0 - 0.3 * r2) + rng.uniform(-jitter, jitter, size=shape)
    return np.clip(fa, 95.0, 180.0)


def epg_profile_signal_batch(n_echoes, tau, T1, T2, alpha_deg, profile):
    """Slice-profile-integrated curves of met2_epg_signals_profile on the host: sum over the positions k, in order, of
    w[k] * epg_signal_batch at refocusing alpha r[k] and excitation (alpha / 2) x[k]."""
    x, r, w = profile
    alpha_deg = np.asarray(alpha_deg, dtype=np.float64).ravel()
    acc = np.zeros((alpha_deg.shape[0], n_echoes))
    for k in range(len(w)):
        acc = acc + w[k] * epg_signal_batch(n_echoes, tau, T1, T2, alpha_deg * r[k], exc_deg=alpha_deg / 2.0 * x[k])
    return acc


def _epg_signal_batch_gpu(n_echoes, tau, T1, T2, alpha_deg, profile=None):
    """Same curves as epg_signal_batch (epg_profile_signal_batch with a profile), computed by libmet2's EPG kernels
    (met2_epg_signals, met2_epg_signals_profile)."""
    import ctypes

    import torch

    from . import _lib
    lib = _lib.load()
    dev = torch.device("cuda", torch.cuda.current_device())
    a = torch.as_tensor(np.ascontiguousarray(alpha_deg, dtype=np.float64)).to(dev)
    t2 = torch.as_tensor(np.ascontiguousarray(T2, dtype=np.float64)).to(dev)
    t1 = torch.as_tensor(np.ascontiguousarray(T1, dtype=np.float64)).to(dev)
    out = torch.empty((a.numel(), n_echoes), dtype=torch.float64, device=dev)
    if profile is not None:
        x, r, w = (ctypes.c_void_p(q.ctypes.data) for q in profile)    # host arrays
        _lib.check(lib.met2_epg_signals_profile(ctypes.c_void_p(a.data_ptr()), ctypes.c_void_p(t2.data_ptr()),
                                                ctypes.c_void_p(t1.data_ptr()), a.numel(), n_echoes, float(tau), x, r,
                                                w, len(profile[2]), ctypes.c_void_p(out.data_ptr()),
                                                ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)),
                   "met2_epg_signals_profile")
        return out.cpu().numpy()
    _lib.check(lib.met2_epg_signals(ctypes.c_void_p(a.data_ptr()), ctypes.c_void_p(t2.data_ptr()),
                                    ctypes.c_void_p(t1.data_ptr()), a.numel(), n_echoes, float(tau),
                                    ctypes.c_void_p(out.data_ptr()),
                                    ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), "met2_epg_signals")
    return out.cpu().numpy()


def make_phantom(shape=(16, 16, 4), n_echoes=32, tau=10.0, TR=1000.0, T1=1000.0, seed=1, fa_mode="uniform",
                 snr_range=(50.0, 150.0), Km=1000.0, mask_mode="full", backend="numpy", slice_profile=None):
    """Return dict(data[nx,ny,nz,nTE], mask[nx,ny,nz], truth={...}); truth["sigma"] is the SD of the Rician noise in
    the data's units.

    fa_mode: "uniform" -> FA ~ U(100, 180) per voxel (config 1); "b1" -> smooth B1 field (configs 2, 3, 5).
    mask_mode: "full" -> all ones; "ellipsoid" -> ~52 % fill, exercises the gather/scatter of masked voxels.
    backend: "numpy" (host recurrence) or "gpu" (libmet2's EPG kernel; for the half-million-voxel bench volumes).
    The two backends agree to ~1e-15 relative; the random draws are identical.
    slice_profile = (x, r, w) (`grids.slice_profile`): the curves are integrated over that slice profile, as 2-D
    multi-slice data are (met2_epg_signals_profile; truth["fa"] is the nominal angle at the slice centre).  The random
    draws are those of the same call without a profile.
    """
    rng = np.random.default_rng(seed)
    nx, ny, nz = shape
    V = nx * ny * nz
    mwf = rng.uniform(0.05, 0.25, V)
    fwf = rng.uniform(0.0, 0.05, V)
    iewf = 1.0 - mwf - fwf
    t2m = rng.uniform(15.0, 35.0, V)
    t2ie = rng.uniform(60.0, 90.0, V)
    t2fw = np.full(V, 2000.0)
    if fa_mode == "uniform":
        fa = rng.uniform(100.0, 180.0, V)
    elif fa_mode == "b1":
        fa = b1_field(shape, rng).ravel()
    else:
        raise ValueError(fa_mode)
    snr = rng.uniform(snr_range[0], snr_range[1], V)
    T1v = np.full(V, float(T1))
    epg = _epg_signal_batch_gpu if backend == "gpu" else epg_signal_batch
    if slice_profile is not None:
        from .grids import as_slice_profile
        prof = as_slice_profile(slice_profile)
        epg = (lambda *a: _epg_signal_batch_gpu(*a, profile=prof)) if backend == "gpu" else \
            (lambda *a: epg_profile_signal_batch(*a, prof))
    sig = mwf[:, None] * epg(n_echoes, tau, T1v, t2m, fa)
    sig += iewf[:, None] * epg(n_echoes, tau, T1v, t2ie, fa)
    sig += fwf[:, None] * epg(n_echoes, tau, T1v, t2fw, fa)
    sig *= Km * (1.0 - np.exp(-TR / T1))
    sigma = sig[:, 0] / snr
    n1 = rng.standard_normal(sig.shape) * sigma[:, None]
    n2 = rng.standard_normal(sig.shape) * sigma[:, None]
    noisy = np.sqrt((sig + n1) ** 2 + n2 ** 2)
    if mask_mode == "full":
        mask = np.ones(shape, dtype=np.int64)
    elif mask_mode == "ellipsoid":
        gx = np.linspace(-1.0, 1.0, nx)[:, None, None]
        gy = np.linspace(-1.0, 1.0, ny)[None, :, None]
        gz = np.linspace(-1.0, 1.0, nz)[None, None, :]
        mask = ((gx ** 2 + gy ** 2 + gz ** 2) <= 1.0).astype(np.int64)
    else:
        raise ValueError(mask_mode)
    data = noisy.reshape(nx, ny, nz, n_echoes) * mask[..., None]
    truth = dict(mwf=mwf.reshape(shape), fwf=fwf.reshape(shape), iewf=iewf.reshape(shape), t2m=t2m.reshape(shape),
                 t2ie=t2ie.reshape(shape), fa=fa.reshape(shape), snr=snr.reshape(shape), sigma=sigma.reshape(shape))
    return dict(data=data, mask=mask, truth=truth, TE_array=tau * np.arange(1, n_echoes + 1), TR=TR)


def tile_volume(data, mask, reps=(2, 2, 2)):
    """Config 5: tile the config-2 volume (SURVEY.md §8d)."""
    return np.tile(data, reps + (1,)), np.tile(mask, reps)
