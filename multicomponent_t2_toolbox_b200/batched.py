"""Batched host API over libmet2.so: one call per stage for all voxels instead of the reference's joblib row loops.

`Met2Plan` owns the device-resident tables of one reconstruction set-up (EPG dictionaries, Gram tables, band forms of
the regularisation matrix, grids) — what motor/motor_recon_met2_real_data.py:204-277 builds on the host — and exposes

    fa_fit(signals[V, nTE])                -> FA index / angle / km / sum of spectra      (Step 2, motor...:349-373)
    t2_fit(signals[V, nTE], fa_index[V])   -> spectra, fitted signals, reg, six maps      (Steps 3+4, motor...:428-472)

PyTorch is used only for device buffers and streams.  There is no CPU path: constructing a plan without CUDA raises.
"""
import ctypes
import math

import numpy as np
import torch

from . import _lib, grids

FA_METHOD_CODE = {"brute-force": 0, "spline": 1}
REG_METHOD_CODE = {"NNLS": 0, "T2SPARC": 1, "X2": 2, "L_curve": 3, "GCV": 4, "BayesReg": 5}

ST_SKIPPED, ST_NONFINITE, ST_ITMAX, ST_SSE_ZERO, ST_NOT_PD = 1, 2, 4, 8, 16
ST_AT_BOUND = 64
ST_MM_CAP, ST_BAD_SIGMA = 128, 256    # met2_rician_fit
# Levenberg-Marquardt settings of the three-pool parametric fit (csrc/met2_param.cu)
PARAM_DEFAULTS = dict(mu0=1e-3, mu_max=1e16, ftol=1e-12, xtol=1e-10, max_iter=2000)
# majorize-minimize settings of the Rician-likelihood fit (csrc/met2_rician.cu)
RICIAN_DEFAULTS = dict(max_iter=200, tol=1e-9)
REG_IS_LAMBDA, NO_NORMALISE, COLD_START, GCV_EVAL, FULL_START, GCV_GRID, ECHO_SPACE = 1, 2, 4, 8, 16, 32, 64   # MET2_T2_FLAG_*
# Largest residual of the reduction (max_j |d_j - U C_j| / max_j |d_j| over the flip angles, measured by
# met2_echo_basis) for which a rank of the reduced echo space is used.  24 (MET2_ECHO_RANK): the rounding of the
# dictionary's own entries (8e-16 .. 1e-15 measured).  16 (MET2_ECHO_RANK_SMALL): 4e-12 — the reference's 32-echo
# protocol measures 1.6e-12 (60 bins) / 1.9e-12 (96 bins) and reproduces the unmodified reference on 20 480 voxels with 0
# active-set disagreements and spectra within 7.8e-9, the accuracy class of the Gram-domain kernels (1.7e-9), 19 % less
# time per volume (profiles/r02_ab_echo_rank.json); the 48-echo protocol of config 4 measures 2.2e-11 and stays at rank
# 24; a dictionary that misses that bound too runs the Gram-domain kernels.
ECHO_TAIL_MAX = {24: 1e-15, 16: 4e-12}


def _require_cuda(device):
    if not torch.cuda.is_available():
        raise _lib.Met2Error("met2: no CUDA device available — this package has no CPU fallback")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.type != "cuda":
        raise _lib.Met2Error("met2: device must be a CUDA device, got %s" % dev)
    return dev


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dev_f64(a, dev):
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).to(dev)


def gaussian_smooth(data, sigma=2.0, truncate=4.0, device=None):
    """Per-echo 3-D Gaussian smoothing of data[nx, ny, nz, nt] on the GPU, bitwise equal to
    `scipy.ndimage.gaussian_filter(data[..., c], sigma, 0)` for every c (motor...:336-346).  Returns a CUDA tensor."""
    dev = _require_cuda(device)
    lib = _lib.load()
    if isinstance(data, np.ndarray):
        data = torch.as_tensor(np.ascontiguousarray(data, dtype=np.float64))
    vol = data.to(device=dev, dtype=torch.float64).contiguous()
    if vol.dim() != 4:
        raise ValueError("data must be [nx, ny, nz, nt]")
    radius = int(truncate * float(sigma) + 0.5)
    k = np.arange(-radius, radius + 1)
    w = np.exp(-0.5 / (sigma * sigma) * k ** 2)     # scipy.ndimage._filters._gaussian_kernel1d, order 0
    w = w / w.sum()
    wd = _dev_f64(w, dev)
    out = torch.empty_like(vol)
    tmp = torch.empty_like(vol)
    nx, ny, nz, nt = vol.shape
    with torch.cuda.device(dev):
        _lib.check(lib.met2_gaussian_smooth(_ptr(vol), nx, ny, nz, nt, _ptr(wd), radius, _ptr(out), _ptr(tmp), _stream()),
                   "met2_gaussian_smooth")
    return out


def nesma_filter(data, mask, half_window=6, threshold=2.5, device=None):
    """NESMA denoiser of motor/motor_recon_met2_real_data.py:305-333 on the GPU (met2_nesma_filter): every voxel with
    mask == 1 becomes the mean of the signals in its [-6, +6) window whose relative L1 distance to it is < 2.5 %.
    data[nx, ny, nz, nt], mask[nx, ny, nz]; returns a CUDA tensor like data."""
    dev = _require_cuda(device)
    lib = _lib.load()
    if isinstance(data, np.ndarray):
        data = torch.as_tensor(np.ascontiguousarray(data, dtype=np.float64))
    if isinstance(mask, np.ndarray):
        mask = torch.as_tensor(np.ascontiguousarray(mask))
    vol = data.to(device=dev, dtype=torch.float64).contiguous()
    msk = mask.to(device=dev, dtype=torch.int32).contiguous()
    if vol.dim() != 4 or tuple(msk.shape) != tuple(vol.shape[:3]):
        raise ValueError("data must be [nx, ny, nz, nt] and mask [nx, ny, nz]")
    out = torch.empty_like(vol)
    tmp = torch.empty_like(vol)
    nx, ny, nz, nt = vol.shape
    with torch.cuda.device(dev):
        _lib.check(lib.met2_nesma_filter(_ptr(vol), _ptr(msk), nx, ny, nz, nt, int(half_window), float(threshold),
                                         _ptr(out), _ptr(tmp), _stream()), "met2_nesma_filter")
    return out


def _volume(data, dev):
    if isinstance(data, np.ndarray):
        data = torch.as_tensor(np.ascontiguousarray(data, dtype=np.float64))
    vol = data.to(device=dev, dtype=torch.float64).contiguous()
    if vol.dim() != 4:
        raise ValueError("data must be [nx, ny, nz, nt]")
    return vol


def noise_sigma(data, device=None):
    """Per-echo noise estimate of Step 1 with --denoise TV (motor...:296) on the GPU (met2_noise_sigma): for every echo
    t, skimage.restoration.estimate_sigma(np.squeeze(data[..., t]), channel_axis=None), the median absolute db2 detail
    coefficient over 0.6745.  data[nx, ny, nz, nt]; returns a CUDA float64 tensor [nt]."""
    dev = _require_cuda(device)
    lib = _lib.load()
    vol = _volume(data, dev)
    nx, ny, nz, nt = vol.shape
    sigma = torch.empty(nt, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        nbytes = lib.met2_noise_sigma_workspace_bytes(nx, ny, nz, nt)
        if nbytes < 0:
            _lib.check(int(nbytes), "met2_noise_sigma_workspace_bytes")
        ws = torch.empty(int(nbytes), dtype=torch.uint8, device=dev)
        _lib.check(lib.met2_noise_sigma(_ptr(vol), nx, ny, nz, nt, _ptr(sigma), _ptr(ws), _stream()), "met2_noise_sigma")
    return sigma


def tv_denoise(data, weight=None, eps=2e-4, max_num_iter=200, device=None):
    """Chambolle total-variation denoising of every echo volume on the GPU (met2_tv_chambolle):
    skimage.restoration.denoise_tv_chambolle(np.squeeze(data[..., t]), weight[t], eps, max_num_iter) for every t.
    weight=None uses 2 * noise_sigma(data), Step 1 of the reference with --denoise TV (motor...:293-303); otherwise a
    scalar or one weight per echo.  Returns (denoised CUDA tensor like data, iterations run per echo, int32 [nt])."""
    dev = _require_cuda(device)
    lib = _lib.load()
    vol = _volume(data, dev)
    nx, ny, nz, nt = vol.shape
    if weight is None:
        w = 2.0 * noise_sigma(vol, dev)
    else:
        w = torch.as_tensor(weight, dtype=torch.float64).to(dev).reshape(-1)
        if w.numel() == 1:
            w = w.expand(nt)
        if w.numel() != nt:
            raise ValueError("weight must be a scalar or have one value per echo (%d)" % nt)
        w = w.contiguous()
    out = torch.empty_like(vol)
    iterations = torch.empty(nt, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        nbytes = lib.met2_tv_workspace_bytes(nx, ny, nz, nt)
        if nbytes < 0:
            _lib.check(int(nbytes), "met2_tv_workspace_bytes")
        ws = torch.empty(int(nbytes), dtype=torch.uint8, device=dev)
        _lib.check(lib.met2_tv_chambolle(_ptr(vol), nx, ny, nz, nt, _ptr(w), float(eps), int(max_num_iter), _ptr(out),
                                         _ptr(iterations), _ptr(ws), _stream()), "met2_tv_chambolle")
    return out, iterations


def mppca_denoise(data, mask, patch_radius=2, device=None):
    """Marchenko-Pastur PCA denoising on the GPU (met2_mppca; definition in csrc/met2_mppca.cu): every voxel with
    mask == 1 is rebuilt from the signal components of the PCA of its (2 patch_radius + 1)^3 window.  data[nx, ny, nz,
    nt], mask[nx, ny, nz].  Returns CUDA tensors (denoised like data, noise sigma [nx, ny, nz], number of signal
    components [nx, ny, nz] int32; 0 outside the mask, -1 where the window holds a non-finite sample)."""
    dev = _require_cuda(device)
    lib = _lib.load()
    vol = _volume(data, dev)
    if isinstance(mask, np.ndarray):
        mask = torch.as_tensor(np.ascontiguousarray(mask))
    msk = mask.to(device=dev, dtype=torch.int32).contiguous()
    if tuple(msk.shape) != tuple(vol.shape[:3]):
        raise ValueError("mask must be [nx, ny, nz] like data[..., 0]")
    nx, ny, nz, nt = vol.shape
    out = torch.empty_like(vol)
    sigma = torch.empty((nx, ny, nz), dtype=torch.float64, device=dev)
    n_signal = torch.empty((nx, ny, nz), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        nbytes = lib.met2_mppca_workspace_bytes(nx, ny, nz, nt, int(patch_radius))
        if nbytes < 0:
            _lib.check(int(nbytes), "met2_mppca_workspace_bytes")
        ws = torch.empty(int(nbytes), dtype=torch.uint8, device=dev)
        _lib.check(lib.met2_mppca(_ptr(vol), _ptr(msk), nx, ny, nz, nt, int(patch_radius), _ptr(out), _ptr(sigma),
                                  _ptr(n_signal), _ptr(ws), _stream()), "met2_mppca")
    return out, sigma, n_signal


def degibbs(data, nsh=20, minW=1, maxW=3, axes=(0, 1), device=None):
    """Gibbs-ringing removal by local subvoxel shifts on the GPU (met2_degibbs; definition in csrc/met2_degibbs.cu), the
    method of MRtrix3's mrdegibbs (Kellner et al. 2016), applied to every 2-D slice spanned by `axes` of data[nx, ny, nz,
    nt] (axes=(0, 2) or (1, 2) for sagittal or coronal slices).  Partial-Fourier data are out of scope.  Returns a CUDA
    tensor like data."""
    dev = _require_cuda(device)
    lib = _lib.load()
    vol = _volume(data, dev)
    a0, a1 = (int(a) % 4 for a in axes)
    if a0 == a1 or 3 in (a0, a1):
        raise ValueError("axes must be two distinct spatial axes of [nx, ny, nz, nt]")
    perm = [a0, a1] + [a for a in range(4) if a not in (a0, a1)]
    vol = vol.permute(perm).contiguous()
    n0, n1, n2, n3 = vol.shape
    out = torch.empty_like(vol)
    with torch.cuda.device(dev):
        nbytes = lib.met2_degibbs_workspace_bytes(n0, n1, n2, n3, int(nsh), int(minW), int(maxW))
        if nbytes < 0:
            _lib.check(int(nbytes), "met2_degibbs_workspace_bytes")
        ws = torch.empty(int(nbytes), dtype=torch.uint8, device=dev)
        _lib.check(lib.met2_degibbs(_ptr(vol), n0, n1, n2, n3, int(nsh), int(minW), int(maxW), _ptr(out), _ptr(ws),
                                    _stream()), "met2_degibbs")
    inv = [perm.index(a) for a in range(4)]
    return out.permute(inv).contiguous()


def segment_means(sig, fa_index, labels, n_seg, dictionary):
    """Per-segment mean signal and mean kernel (met2_segment_means; motor...:377-392 and
    motor_recon_met2_real_data_ROI.py:408-423).  sig[V, nTE], fa_index[V], labels[V] in [0, n_seg) (else: no segment).
    Returns (mean_signal[n_seg, nTE], mean_kernel[n_seg, nTE, nT2], counts[n_seg]) as CUDA tensors."""
    lib = _lib.load()
    dev = dictionary.dic.device
    if isinstance(sig, np.ndarray):
        sig = torch.as_tensor(np.ascontiguousarray(sig, dtype=np.float64))
    sig = sig.to(device=dev, dtype=torch.float64).contiguous()
    as_i32 = lambda a: (torch.as_tensor(np.ascontiguousarray(a)) if isinstance(a, np.ndarray) else a).to(
        device=dev, dtype=torch.int32).contiguous()
    fa_index, labels = as_i32(fa_index), as_i32(labels)
    V = sig.shape[0]
    if sig.dim() != 2 or sig.shape[1] != dictionary.nTE or fa_index.shape != (V,) or labels.shape != (V,):
        raise ValueError("segment_means: sig[V, nTE], fa_index[V], labels[V] expected")
    n_seg = int(n_seg)
    mean_signal = torch.empty((n_seg, dictionary.nTE), dtype=torch.float64, device=dev)
    mean_kernel = torch.empty((n_seg, dictionary.nTE, dictionary.nT2), dtype=torch.float64, device=dev)
    counts = torch.empty(n_seg, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        ws = torch.empty(int(lib.met2_segment_workspace_bytes(n_seg, dictionary.nA)), dtype=torch.uint8, device=dev)
        _lib.check(lib.met2_segment_means(_ptr(sig), _ptr(fa_index), _ptr(labels), V, dictionary.nTE, dictionary.nT2,
                                          dictionary.nA, n_seg, _ptr(dictionary.dic), _ptr(mean_signal),
                                          _ptr(mean_kernel), _ptr(counts), _ptr(ws), _stream()), "met2_segment_means")
    return mean_signal, mean_kernel, counts


class Dictionary:
    """Device EPG dictionary of one angle grid: dic [nA][nTE][nT2], dicT [nA][nT2][nTE], G [nA][nT2][nT2]."""

    def __init__(self, alphas, T2s, T1s, n_echoes, tau, TR, dev):
        lib = _lib.load()
        self.alphas_host = np.ascontiguousarray(alphas, dtype=np.float64)
        self.nA, self.nT2, self.nTE = len(self.alphas_host), len(T2s), int(n_echoes)
        self.alphas = _dev_f64(self.alphas_host, dev)
        t2 = _dev_f64(T2s, dev)
        t1 = _dev_f64(T1s, dev)
        self.dic = torch.empty((self.nA, self.nTE, self.nT2), dtype=torch.float64, device=dev)
        self.dicT = torch.empty((self.nA, self.nT2, self.nTE), dtype=torch.float64, device=dev)
        self.G = torch.empty((self.nA, self.nT2, self.nT2), dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            _lib.check(lib.met2_epg_dictionary(_ptr(self.alphas), self.nA, _ptr(t2), _ptr(t1), self.nT2, self.nTE,
                                               float(tau), float(TR), _ptr(self.dic), _ptr(self.dicT), _stream()),
                       "met2_epg_dictionary")
            _lib.check(lib.met2_gram_tables(_ptr(self.dic), self.nA, self.nTE, self.nT2, None, _ptr(self.G), None, None,
                                            _stream()), "met2_gram_tables")

    @classmethod
    def from_reference_layout(cls, Dic_3D, alphas, dev):
        """Device tables for a dictionary given on the host as Dic_3D[nTE, nT2, nA] (any forward model)."""
        lib = _lib.load()
        self = cls.__new__(cls)
        Dic_3D = np.asarray(Dic_3D, dtype=np.float64)
        if Dic_3D.ndim == 2:
            Dic_3D = Dic_3D[:, :, None]
        self.nTE, self.nT2, self.nA = Dic_3D.shape
        self.alphas_host = np.ascontiguousarray(alphas if alphas is not None else np.zeros(self.nA), dtype=np.float64)
        self.alphas = _dev_f64(self.alphas_host, dev)
        self.dic = _dev_f64(np.transpose(Dic_3D, (2, 0, 1)), dev)
        self.dicT = _dev_f64(np.transpose(Dic_3D, (2, 1, 0)), dev)
        self.G = torch.empty((self.nA, self.nT2, self.nT2), dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            _lib.check(lib.met2_gram_tables(_ptr(self.dic), self.nA, self.nTE, self.nT2, None, _ptr(self.G), None, None,
                                            _stream()), "met2_gram_tables")
        return self

    @classmethod
    def from_device(cls, dic, alphas=None):
        """Tables for a dictionary already on the GPU as dic[nA, nTE, nT2] (e.g. the per-segment mean kernels of
        `segment_means`)."""
        lib = _lib.load()
        self = cls.__new__(cls)
        dev = dic.device
        self.dic = dic.to(torch.float64).contiguous()
        self.nA, self.nTE, self.nT2 = self.dic.shape
        self.alphas_host = np.ascontiguousarray(alphas if alphas is not None else np.zeros(self.nA), dtype=np.float64)
        self.alphas = _dev_f64(self.alphas_host, dev)
        self.dicT = self.dic.transpose(1, 2).contiguous()
        self.G = torch.empty((self.nA, self.nT2, self.nT2), dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            _lib.check(lib.met2_gram_tables(_ptr(self.dic), self.nA, self.nTE, self.nT2, None, _ptr(self.G), None, None,
                                            _stream()), "met2_gram_tables")
        return self

    def echo_tables(self, R):
        """met2_echo_basis at rank R (built on first use, kept): (basis [nA, nTE, R], coef [nA, nT2, R], tail) with
        tail = the largest residual of the reduction over the flip angles, max_j |d_j - U C_j| / max_j |d_j|."""
        cache = self.__dict__.setdefault("_echo_tables", {})
        if R not in cache:
            lib = _lib.load()
            dev = self.dic.device
            basis = torch.empty((self.nA, self.nTE, R), dtype=torch.float64, device=dev)
            coef = torch.empty((self.nA, self.nT2, R), dtype=torch.float64, device=dev)
            tail = torch.empty(self.nA, dtype=torch.float64, device=dev)
            with torch.cuda.device(dev):
                _lib.check(lib.met2_echo_basis(_ptr(self.dic), self.nA, self.nTE, self.nT2, R, _ptr(basis),
                                               _ptr(coef), _ptr(tail), _stream()), "met2_echo_basis")
            cache[R] = (basis, coef, float(tail.max()))
        return cache[R]

    def echo_basis(self, ranks=None):
        """Reduced echo basis the echo-space kernels run on: (basis, coef, R) for the smallest rank R among `ranks`
        (default: both ranks the library is built for, 16 and 24) whose measured residual is within ECHO_TAIL_MAX[R], or
        None when none is (then the Gram-domain kernels run)."""
        if ranks is None:
            lib = _lib.load()
            ranks = (int(lib.met2_echo_rank(1)), int(lib.met2_echo_rank(0)))
        for R in sorted(ranks):
            basis, coef, tail = self.echo_tables(R)
            if tail <= ECHO_TAIL_MAX[R]:
                return basis, coef, R
        return None

    def to_reference_layout(self):
        """Host copy in the reference's layout Dic_3D[nTE, nT2, nA] (epg/epg.py:155-162)."""
        return np.ascontiguousarray(self.dic.permute(1, 2, 0).cpu().numpy())


class Met2Plan:
    def __init__(self, n_echoes, tau, TR, reg_method="X2", reg_matrix="I", FA_method="spline", myelin_T2=40.0,
                 npc=None, n_alphas=None, T1=1000.0, device=None, lambda_reg=None, Laplac=None, Dic_3D=None,
                 Dic_3D_LR=None, alpha_values=None, alpha_values_spline=None, T2s=None, t2_flags=0, echo_space=True,
                 echo_ranks=None):
        """Tables for one reconstruction set-up.  By default everything is built like motor...:204-277 (EPG dictionary
        on the GPU); `Dic_3D` (+ `Dic_3D_LR`, `alpha_values`, `alpha_values_spline`, `T2s`, `Laplac`) lets a caller bring
        its own dictionary in the reference layout [nTE, nT2, nA] — used by the drop-in row workers and per-voxel API."""
        if reg_method not in REG_METHOD_CODE:
            raise ValueError("unknown reg_method %r" % (reg_method,))
        if FA_method not in FA_METHOD_CODE:
            raise ValueError("Error: Wrong FA_method option!")
        self.dev = _require_cuda(device)
        self.lib = _lib.load()
        self.reg_method, self.reg_matrix, self.FA_method = reg_method, reg_matrix, FA_method
        self.t2_flags = int(t2_flags)    # MET2_T2_FLAG_* applied to every t2_fit of this plan (e.g. GCV_GRID)
        # reduced-echo-space kernels wherever they apply (X2 and T2SPARC with a diagonal matrix: I, InvT2), where they
        # measured 1.4-3x faster than the Gram-domain ones (profiles/r02_ab_*); echo_space=False keeps the latter
        self.echo_space = bool(echo_space)
        # ranks of the reduced space this plan may use (None: the smallest of 16 / 24 the dictionary is exact at, see
        # ECHO_TAIL_MAX; (24,) pins the rank that is exact to the rounding of the dictionary's entries)
        self.echo_ranks = None if echo_ranks is None else tuple(int(r) for r in echo_ranks)
        self.nTE, self.tau, self.TR = int(n_echoes), float(tau), float(TR)
        if Dic_3D is not None:
            Dic_3D = np.asarray(Dic_3D, dtype=np.float64)
            if Dic_3D.ndim == 2:
                Dic_3D = Dic_3D[:, :, None]
            npc = Dic_3D.shape[1]
            if Dic_3D.shape[0] != self.nTE:
                raise ValueError("Dic_3D has %d echoes, expected %d" % (Dic_3D.shape[0], self.nTE))
        self.npc = grids.default_npc(reg_method) if npc is None else int(npc)
        self.T2s = grids.t2_grid(self.npc) if T2s is None else np.asarray(T2s, dtype=np.float64)
        self.T1s = float(T1) * np.ones_like(self.T2s)
        self.myelin_T2 = float(myelin_T2)
        self.ind_m, self.ind_t, self.ind_csf = grids.compartment_masks(self.T2s, myelin_T2)
        self.alpha_values, self.alpha_spline = grids.fa_grids(FA_method, n_alphas)
        if Dic_3D is not None:
            self.alpha_values = (np.asarray(alpha_values, dtype=np.float64) if alpha_values is not None
                                 else np.zeros(Dic_3D.shape[2]))
            if len(self.alpha_values) != Dic_3D.shape[2]:
                raise ValueError("alpha_values does not match Dic_3D")
            if FA_method == "spline":
                if Dic_3D_LR is None or alpha_values_spline is None:
                    if alpha_values is not None:
                        raise ValueError("spline FA with a caller dictionary needs Dic_3D_LR and alpha_values_spline")
                    self.alpha_spline = None
                else:
                    self.alpha_spline = np.asarray(alpha_values_spline, dtype=np.float64)
        self.lambda_reg = grids.lambda_grid() if lambda_reg is None else np.asarray(lambda_reg, dtype=np.float64)
        self.Laplac = grids.reg_matrix(reg_matrix, self.T2s) if Laplac is None else np.asarray(Laplac, np.float64)
        K = self.Laplac.T @ self.Laplac
        off = np.abs(np.subtract.outer(np.arange(self.npc), np.arange(self.npc))) > 2
        if np.any(K[off] != 0.0) or np.any(self.Laplac[off] != 0.0):
            raise ValueError("regularisation matrix must be banded (|i-j| <= 2), like I, L1, L2, InvT2")
        with torch.cuda.device(self.dev):
            self.dict_lr = None
            if Dic_3D is not None:
                self.dict_hr = Dictionary.from_reference_layout(Dic_3D, self.alpha_values, self.dev)
                if FA_method == "spline" and self.alpha_spline is not None:
                    self.dict_lr = Dictionary.from_reference_layout(Dic_3D_LR, self.alpha_spline, self.dev)
                    self.knots = _dev_f64(self.alpha_spline, self.dev)
            else:
                self.dict_hr = Dictionary(self.alpha_values, self.T2s, self.T1s, self.nTE, tau, TR, self.dev)
                if FA_method == "spline":
                    self.dict_lr = Dictionary(self.alpha_spline, self.T2s, self.T1s, self.nTE, tau, TR, self.dev)
                    self.knots = _dev_f64(self.alpha_spline, self.dev)
            self.L_dev = _dev_f64(self.Laplac, self.dev)
            self.kband = torch.zeros((10, self.npc), dtype=torch.float64, device=self.dev)
            self.band_err = torch.zeros(1, dtype=torch.int32, device=self.dev)
            _lib.check(self.lib.met2_gram_tables(None, 0, self.nTE, self.npc, _ptr(self.L_dev), None, _ptr(self.kband),
                                                 _ptr(self.band_err), _stream()), "met2_gram_tables(L)")
            self.lambdas = _dev_f64(self.lambda_reg, self.dev)
            self.logT2 = _dev_f64(np.log(self.T2s), self.dev)
            comp = (self.ind_m.astype(np.uint8) | (self.ind_t.astype(np.uint8) << 1) | (self.ind_csf.astype(np.uint8) << 2))
            self.comp = torch.as_tensor(comp).to(self.dev)
        self._ws = {}

    # ------------------------------------------------------------------ configs
    def fa_cfg(self, final_solve=True):
        return _lib.FaCfg(method=FA_METHOD_CODE[self.FA_method], nTE=self.nTE, nT2=self.npc, nA=len(self.alpha_values),
                          nKnots=(len(self.alpha_spline) if self.alpha_spline is not None else 0),
                          final_solve=int(final_solve), brent_lo=90.0, brent_hi=180.0, brent_xatol=1e-5,
                          brent_maxfun=500, reserved=0)

    def t2_cfg(self, reg_method=None, flags=0, **overrides):
        method = self.reg_method if reg_method is None else reg_method
        cfg = _lib.T2Cfg(method=REG_METHOD_CODE[method], nTE=self.nTE, nT2=self.npc, nA=len(self.alpha_values),
                         nLambda=len(self.lambda_reg), maxfun=300, factor=1.02, lambda_fixed=1.8, brent_lo=0.0,
                         brent_hi=10.0, brent_xatol=1e-5, log_det_L=0.0, flags=int(flags) | self.t2_flags, echo_rank=0)
        if method == "GCV":
            cfg.brent_lo = 1e-8
        if method == "BayesReg":
            cfg.brent_lo, cfg.brent_hi, cfg.maxfun = 1e-8, 2.0, 200
            with np.errstate(divide="ignore"):
                cfg.log_det_L = float(np.log(np.linalg.det(self.Laplac)))
        if method == "X2" and np.array_equal(self.Laplac, np.eye(self.npc)):
            cfg.flags |= FULL_START
        if self.echo_space and self._diagonal_L() and not (cfg.flags & COLD_START):
            # measured on the config-2 volume (profiles/r02_ab_*): X2-I 365 -> 211 ms, X2-InvT2 262 -> 190 ms,
            # T2SPARC (96 bins) 282 -> 91 ms
            # L-curve and BayesReg (met2_t2_echo_reg_impl.cuh): see profiles/r02_ab_echo_reg.json
            if (method == "X2" and self.npc <= 64) or (method in ("T2SPARC", "L_curve", "BayesReg") and self.npc <= 128):
                cfg.flags |= ECHO_SPACE
        for k, v in overrides.items():   # e.g. factor=..., lambda_fixed=..., maxfun=...
            setattr(cfg, k, v)
        return cfg

    def _diagonal_L(self):
        L = self.Laplac
        return bool(np.all(L[~np.eye(self.npc, dtype=bool)] == 0.0) and np.all(np.diag(L) > 0.0))

    def _workspace(self, key, nbytes):
        ws = self._ws.get(key)
        if ws is None or ws.numel() < nbytes:
            ws = torch.empty(int(nbytes), dtype=torch.uint8, device=self.dev)
            self._ws[key] = ws
        return ws

    def _signals(self, sig):
        if isinstance(sig, np.ndarray):
            sig = torch.as_tensor(np.ascontiguousarray(sig, dtype=np.float64))
        sig = sig.to(device=self.dev, dtype=torch.float64).contiguous()
        if sig.dim() != 2 or sig.shape[1] != self.nTE:
            raise ValueError("signals must be [V, %d], got %s" % (self.nTE, tuple(sig.shape)))
        return sig

    # ------------------------------------------------------------------ Step 2
    def fa_fit(self, sig, final_solve=True, out=None):
        """Flip-angle estimation for all voxels.  Returns dict(fa_index int32[V], fa_deg[V], km[V], fsol_sum[nT2], status)."""
        sig = self._signals(sig)
        V = sig.shape[0]
        dev = self.dev
        if out is None:
            out = dict(fa_index=torch.empty(V, dtype=torch.int32, device=dev),
                       fa_deg=torch.empty(V, dtype=torch.float64, device=dev),
                       km=torch.empty(V, dtype=torch.float64, device=dev),
                       fsol_sum=torch.zeros(self.npc, dtype=torch.float64, device=dev),
                       status=torch.empty(V, dtype=torch.int32, device=dev))
        if V == 0:
            return out
        if self.FA_method == "spline" and self.dict_lr is None:
            raise ValueError("this plan was built without a coarse (spline) dictionary")
        cfg = self.fa_cfg(final_solve)
        with torch.cuda.device(dev):
            nbytes = self.lib.met2_fa_workspace_bytes(V, ctypes.byref(cfg))
            if nbytes < 0:
                _lib.check(-1, "met2_fa_workspace_bytes")
            ws = self._workspace("fa", nbytes)
            hr, lr = self.dict_hr, self.dict_lr
            _lib.check(self.lib.met2_fa_fit(
                _ptr(sig), V, ctypes.byref(cfg), _ptr(hr.dic), _ptr(hr.dicT), _ptr(hr.G), _ptr(hr.alphas),
                _ptr(lr.dic) if lr else None, _ptr(lr.dicT) if lr else None, _ptr(lr.G) if lr else None,
                _ptr(self.knots) if lr else None, _ptr(out["fa_index"]), _ptr(out["fa_deg"]), _ptr(out["km"]),
                _ptr(out["fsol_sum"]) if final_solve else None, _ptr(out["status"]), _ptr(ws), _stream()), "met2_fa_fit")
        return out

    # ------------------------------------------------------------------ Steps 3 + 4
    def t2_fit(self, sig, fa_index, reg_method=None, out=None, flags=0, dictionary=None, **cfg_overrides):
        """Spectrum fit + metrics.  Returns dict(fsol[V,nT2], est_signal[V,nTE], reg[V], maps[V,6], status[V]).
        `dictionary` (a `Dictionary` with this plan's nTE / nT2) replaces the plan's own kernel set for this call."""
        sig = self._signals(sig)
        V = sig.shape[0]
        dev = self.dev
        if isinstance(fa_index, np.ndarray):
            fa_index = torch.as_tensor(fa_index)
        fa_index = fa_index.to(device=dev, dtype=torch.int32).contiguous()
        if fa_index.shape != (V,):
            raise ValueError("fa_index must be [V]")
        if out is None:
            out = dict(fsol=torch.empty((V, self.npc), dtype=torch.float64, device=dev),
                       est_signal=torch.empty((V, self.nTE), dtype=torch.float64, device=dev),
                       reg=torch.empty(V, dtype=torch.float64, device=dev),
                       maps=torch.empty((V, 6), dtype=torch.float64, device=dev),
                       status=torch.empty(V, dtype=torch.int32, device=dev))
        if V == 0:
            return out
        cfg = self.t2_cfg(reg_method, flags, **cfg_overrides)
        hr = self.dict_hr if dictionary is None else dictionary
        if (hr.nTE, hr.nT2) != (self.nTE, self.npc):
            raise ValueError("dictionary shape does not match the plan")
        cfg.nA = hr.nA
        lambdas = self.lambdas
        if cfg.flags & GCV_GRID:    # GCV over the positive part of the L-curve grid (lambda_reg[1:]; lambda_reg[0] = 0)
            lambdas = self.lambdas[1:].contiguous()
            cfg.nLambda = lambdas.numel()
        red = None
        if cfg.flags & ECHO_SPACE:
            if not self._diagonal_L():
                raise ValueError("MET2_T2_FLAG_ECHO_SPACE needs a diagonal regularisation matrix (I, InvT2)")
            red = hr.echo_basis(self.echo_ranks)
            if red is None:      # dictionary not of numerical rank <= 24: Gram-domain kernels
                cfg.flags &= ~ECHO_SPACE
            else:
                cfg.echo_rank = red[2]
        with torch.cuda.device(dev):
            nbytes = self.lib.met2_t2_workspace_bytes(V, ctypes.byref(cfg))
            if nbytes < 0:
                _lib.check(-1, "met2_t2_workspace_bytes")
            ws = self._workspace("t2", nbytes)
            _lib.check(self.lib.met2_t2_fit_echo(
                _ptr(sig), _ptr(fa_index), V, ctypes.byref(cfg), _ptr(hr.dic), _ptr(hr.dicT), _ptr(hr.G),
                _ptr(self.kband), _ptr(lambdas), _ptr(self.logT2), _ptr(self.comp),
                _ptr(red[0]) if red else None, _ptr(red[1]) if red else None, _ptr(out["fsol"]),
                _ptr(out["est_signal"]), _ptr(out["reg"]), _ptr(out["maps"]), _ptr(out["status"]), _ptr(ws), _stream()),
                "met2_t2_fit_echo")
        return out

    def fit(self, sig, sig_fa=None):
        """Steps 2-4 for a batch of voxels: FA search on `sig_fa` (defaults to `sig`), spectrum fit on `sig`."""
        sig = self._signals(sig)
        fa = self.fa_fit(sig if sig_fa is None else sig_fa)
        t2 = self.t2_fit(sig, fa["fa_index"])
        return fa, t2

    # ------------------------------------------------------------------ spatially regularised fit
    def spatial_half_sweep(self, sig, fa_index, lam, x, nbr, vox, mu, status):
        """One half-sweep of met2_spatial_sweep: block updates of the voxels `vox` (all of one colour) of the
        normalised spectra x[V, nT2] (CUDA float64, updated in place); status[V] (CUDA int32) gets MET2_ST_ITMAX where a
        solve hit itmax.  sig[V, nTE], fa_index[V], lam[V] and nbr[V, 6] as for `spatial_fit`, already on this device."""
        V = sig.shape[0]
        hr = self.dict_hr
        with torch.cuda.device(self.dev):
            _lib.check(self.lib.met2_spatial_sweep(
                _ptr(sig), _ptr(fa_index), _ptr(lam), _ptr(nbr), _ptr(vox), vox.numel(), V, self.nTE, self.npc, hr.nA,
                _ptr(hr.G), _ptr(hr.dicT), _ptr(self.kband), float(mu), _ptr(x), _ptr(status), _stream()),
                "met2_spatial_sweep")

    def spatial_fit(self, sig, fa_index, lam, fsol, nbr, colours, mu, n_sweeps=10, status=None):
        """Spatially regularised spectra (definition in csrc/met2_spatial.cu): n_sweeps red-black sweeps of
        neighbour-coupled block updates with coupling weight mu >= 0, started from a point fit of this plan.

        sig[V, nTE] is the signal the point fit used, fa_index[V] its flip-angle indices, lam[V] the lambda it selected
        (`t2_fit(..., flags=REG_IS_LAMBDA)["reg"]`), fsol[V, nT2] its spectra and status[V] its status (None: the
        voxels in neither colour list count as skipped).  nbr[V, 6] and colours come from
        `pipeline.spatial_neighbours`.  The sweeps solve in the Gram domain, whichever kernels the point fit ran.
        Returns CUDA tensors fsol[V, nT2], est_signal[V, nTE], maps[V, 6], status[V] (the point fit's, with
        MET2_ST_ITMAX added where a sweep solve hit itmax) and x[V, nT2] = fsol / sig[0].  All work is enqueued on the
        current stream."""
        mu, n_sweeps = float(mu), int(n_sweeps)
        if not (math.isfinite(mu) and mu >= 0.0):
            raise ValueError("mu must be finite and >= 0, got %r" % mu)
        if n_sweeps < 0:
            raise ValueError("n_sweeps must be >= 0")
        sig = self._signals(sig)
        V = sig.shape[0]
        dev = self.dev
        i32 = lambda a: torch.as_tensor(a).to(device=dev, dtype=torch.int32).contiguous()
        fa_index, nbr = i32(fa_index), i32(nbr)
        colours = [i32(c).reshape(-1) for c in colours]
        lam = torch.as_tensor(lam).to(device=dev, dtype=torch.float64).contiguous()
        fsol = torch.as_tensor(fsol).to(device=dev, dtype=torch.float64)
        if (fa_index.shape != (V,) or lam.shape != (V,) or tuple(fsol.shape) != (V, self.npc)
                or tuple(nbr.shape) != (V, 6) or len(colours) != 2):
            raise ValueError("spatial_fit: sig[V, nTE], fa_index[V], lam[V], fsol[V, nT2], nbr[V, 6] and two colour "
                             "lists expected")
        for c in colours:
            if c.numel() and (int(c.min()) < 0 or int(c.max()) >= V):
                raise ValueError("spatial_fit: colour lists hold positions in [0, V)")
        if nbr.numel() and (int(nbr.min()) < -1 or int(nbr.max()) >= V):
            raise ValueError("spatial_fit: nbr holds positions in [0, V) or -1")
        if status is None:
            status = torch.full((V,), ST_SKIPPED, dtype=torch.int32, device=dev)
            for c in colours:
                status[c.long()] = 0
        else:
            status = i32(status).clone()
            if status.shape != (V,):
                raise ValueError("status must be [V]")
        out = dict(fsol=torch.empty((V, self.npc), dtype=torch.float64, device=dev),
                   est_signal=torch.empty((V, self.nTE), dtype=torch.float64, device=dev),
                   maps=torch.empty((V, 6), dtype=torch.float64, device=dev), status=status)
        if V == 0:
            out["x"] = torch.empty((0, self.npc), dtype=torch.float64, device=dev)
            return out
        with torch.cuda.device(dev):
            fitted = (status & ST_SKIPPED) == 0
            x = torch.where(fitted[:, None], fsol / sig[:, :1], 0.0).contiguous()
            for _ in range(n_sweeps):
                for vox in colours:
                    self.spatial_half_sweep(sig, fa_index, lam, x, nbr, vox, mu, status)
            hr = self.dict_hr
            _lib.check(self.lib.met2_spatial_finish(
                _ptr(sig), _ptr(fa_index), _ptr(status), _ptr(x), V, self.nTE, self.npc, hr.nA, _ptr(hr.dicT),
                _ptr(self.logT2), _ptr(self.comp), _ptr(out["fsol"]), _ptr(out["est_signal"]), _ptr(out["maps"]),
                _stream()), "met2_spatial_finish")
        out["x"] = x
        return out

    # ------------------------------------------------------------------ Rician-likelihood fit
    def rician_fit(self, sig, fa_index, lam, sigma, fsol, status, **cfg):
        """Rician-likelihood spectra (definition in csrc/met2_rician.cu): majorize-minimize iterations of warm-started
        Tikhonov NNLS solves with modified data, started from a point fit of this plan.  sig[V, nTE] is the signal the
        point fit used, fa_index[V] its flip-angle indices, lam[V] its lambda (`t2_fit(..., flags=REG_IS_LAMBDA)["reg"]`),
        fsol[V, nT2] its spectra and status[V] its status; sigma is the noise SD in the signal's units, a number or
        one value per voxel.  cfg overrides RICIAN_DEFAULTS.  The solves run in the Gram domain, whichever kernels the
        point fit ran.  Returns CUDA tensors fsol[V, nT2], est_signal[V, nTE] (the noiseless model D x sig[0]),
        maps[V, 6], iters[V] (int32, MM solves run), status[V] (the point fit's plus MET2_ST_MM_CAP, MET2_ST_ITMAX and
        MET2_ST_BAD_SIGMA | MET2_ST_SKIPPED) and x[V, nT2] (normalised spectra).  All work is enqueued on the current
        stream."""
        unknown = set(cfg) - set(RICIAN_DEFAULTS)
        if unknown:
            raise ValueError("unknown rician_fit settings %s" % sorted(unknown))
        o = {**RICIAN_DEFAULTS, **cfg}
        sig = self._signals(sig)
        V = sig.shape[0]
        dev = self.dev
        fa_index = torch.as_tensor(fa_index).to(device=dev, dtype=torch.int32).contiguous()
        lam = torch.as_tensor(lam).to(device=dev, dtype=torch.float64).contiguous()
        sigma = torch.as_tensor(sigma, dtype=torch.float64).to(dev).reshape(-1)
        if sigma.numel() == 1:
            sigma = sigma.expand(V)
        sigma = sigma.contiguous()
        fsol = torch.as_tensor(fsol).to(device=dev, dtype=torch.float64)
        status = torch.as_tensor(status).to(device=dev, dtype=torch.int32).contiguous()
        if (fa_index.shape != (V,) or lam.shape != (V,) or sigma.shape != (V,) or tuple(fsol.shape) != (V, self.npc)
                or status.shape != (V,)):
            raise ValueError("rician_fit: sig[V, nTE], fa_index[V], lam[V], sigma (a number or [V]), fsol[V, nT2] and "
                             "status[V] expected")
        out = dict(fsol=torch.empty((V, self.npc), dtype=torch.float64, device=dev),
                   est_signal=torch.empty((V, self.nTE), dtype=torch.float64, device=dev),
                   maps=torch.empty((V, 6), dtype=torch.float64, device=dev),
                   iters=torch.empty(V, dtype=torch.int32, device=dev),
                   status=torch.empty(V, dtype=torch.int32, device=dev),
                   x=torch.empty((V, self.npc), dtype=torch.float64, device=dev))
        if V == 0:
            return out
        hr = self.dict_hr
        with torch.cuda.device(dev):
            fitted = (status & ST_SKIPPED) == 0
            x0 = torch.where(fitted[:, None], fsol / sig[:, :1], 0.0).contiguous()
            _lib.check(self.lib.met2_rician_fit(
                _ptr(sig), _ptr(fa_index), _ptr(lam), _ptr(sigma), _ptr(x0), _ptr(status), V, self.nTE, self.npc,
                hr.nA, _ptr(hr.G), _ptr(hr.dicT), _ptr(self.kband), int(o["max_iter"]), float(o["tol"]), _ptr(out["x"]),
                _ptr(out["iters"]), _ptr(out["status"]), _stream()), "met2_rician_fit")
            _lib.check(self.lib.met2_spatial_finish(
                _ptr(sig), _ptr(fa_index), _ptr(out["status"]), _ptr(out["x"]), V, self.nTE, self.npc, hr.nA,
                _ptr(hr.dicT), _ptr(self.logT2), _ptr(self.comp), _ptr(out["fsol"]), _ptr(out["est_signal"]),
                _ptr(out["maps"]), _stream()), "met2_spatial_finish")
        return out

    # ------------------------------------------------------------------ three-pool parametric fit
    def param_cfg(self, **overrides):
        """met2_param_cfg of this plan: T2 boxes T2s[0]..myelin_T2, myelin_T2..200, 200..T2s[-1] (motor...:215-220),
        flip angle 90..180, the plan's tau / TR / T1, and PARAM_DEFAULTS unless overridden."""
        unknown = set(overrides) - set(PARAM_DEFAULTS)
        if unknown:
            raise ValueError("unknown param_fit settings %s" % sorted(unknown))
        o = {**PARAM_DEFAULTS, **overrides}
        T2s = self.T2s
        return _lib.ParamCfg(nTE=self.nTE, nT2=self.npc, max_iter=int(o["max_iter"]), reserved=0, tau=self.tau,
                             TR=self.TR, T1=float(self.T1s[0]),
                             t2_lo=(ctypes.c_double * 3)(T2s[0], self.myelin_T2, 200.0),
                             t2_hi=(ctypes.c_double * 3)(self.myelin_T2, 200.0, T2s[-1]), fa_lo=90.0, fa_hi=180.0,
                             mu0=float(o["mu0"]), mu_max=float(o["mu_max"]), ftol=float(o["ftol"]),
                             xtol=float(o["xtol"]))

    def param_fit(self, sig, fa_deg, fsol, status, **cfg):
        """Three-pool parametric fit (definition in csrc/met2_param.cu): bounded Levenberg-Marquardt over the
        amplitudes and continuous T2s of a myelin, an intra/extra-cellular and a free-water EPG pool with one shared
        continuous flip angle, started from a point fit of this plan.  sig[V, nTE] is the signal the point fit used,
        fa_deg[V] the FA stage's angles, fsol[V, nT2] and status[V] the `t2_fit` results; cfg overrides
        PARAM_DEFAULTS.  Returns CUDA tensors params[V, 7] (amplitudes in signal units, T2_m, T2_ie, T2_fw in ms,
        flip angle in deg), maps[V, 6] (met2_t2_fit's columns), est_signal[V, nTE], sse[V], iters[V] (int32) and
        status[V] (int32).  Voxels the point fit skipped get zeros.  All work is enqueued on the current stream."""
        c = self.param_cfg(**cfg)
        sig = self._signals(sig)
        V = sig.shape[0]
        dev = self.dev
        fa_deg = torch.as_tensor(fa_deg).to(device=dev, dtype=torch.float64).contiguous()
        fsol = torch.as_tensor(fsol).to(device=dev, dtype=torch.float64).contiguous()
        status = torch.as_tensor(status).to(device=dev, dtype=torch.int32).contiguous()
        if fa_deg.shape != (V,) or tuple(fsol.shape) != (V, self.npc) or status.shape != (V,):
            raise ValueError("param_fit: sig[V, nTE], fa_deg[V], fsol[V, nT2] and status[V] expected")
        out = dict(params=torch.empty((V, 7), dtype=torch.float64, device=dev),
                   maps=torch.empty((V, 6), dtype=torch.float64, device=dev),
                   est_signal=torch.empty((V, self.nTE), dtype=torch.float64, device=dev),
                   sse=torch.empty(V, dtype=torch.float64, device=dev),
                   iters=torch.empty(V, dtype=torch.int32, device=dev),
                   status=torch.empty(V, dtype=torch.int32, device=dev))
        with torch.cuda.device(dev):
            _lib.check(self.lib.met2_param_fit(
                _ptr(sig), _ptr(fa_deg), _ptr(fsol), _ptr(status), V, ctypes.byref(c), _ptr(self.logT2),
                _ptr(self.comp), _ptr(out["params"]), _ptr(out["maps"]), _ptr(out["est_signal"]), _ptr(out["sse"]),
                _ptr(out["iters"]), _ptr(out["status"]), _stream()), "met2_param_fit")
        return out

    # ------------------------------------------------------------------ bootstrap uncertainty of the maps
    def bootstrap(self, sig, fa_index, est_signal, B=100, seed=0, voxel_offset=0, max_replicates=1 << 21):
        """Per-voxel wild-bootstrap uncertainty of the six maps (definition in csrc/met2_boot.cu).

        sig[V, nTE] is the signal the point fit used, fa_index[V] and est_signal[V, nTE] are that fit's results.  Each
        voxel gets B replicates (1 <= B <= 1024), refitted by this plan's `t2_fit` at the point fit's flip angle, with
        lambda re-selected.  voxel_offset is the position of voxel 0 in the whole voxel list: a voxel's replicates
        depend only on that position and `seed`, so any split of the list gives the same result.  Voxels are processed
        in chunks of max_replicates // B (replicate buffers of about 1 KB per replicate at 32 echoes and 60 bins).
        Returns CUDA tensors stats[V, 6, 4] (mean, sd, p2.5, p97.5 of MWF, IEWF, FWF, T2_M, T2_IE, TWC) and n_valid[V]
        (int32, the replicates whose fit was not skipped).  All work is enqueued on the current stream."""
        B = int(B)
        if not 1 <= B <= 1024:
            raise ValueError("B must be in [1, 1024], got %d" % B)
        seed, voxel_offset = int(seed), int(voxel_offset)
        if not 0 <= seed < 1 << 64:
            raise ValueError("seed must be an unsigned 64-bit integer")
        if voxel_offset < 0:
            raise ValueError("voxel_offset must be >= 0")
        if int(max_replicates) < B:
            raise ValueError("max_replicates must be at least B")
        sig = self._signals(sig)
        est = self._signals(est_signal)
        V = sig.shape[0]
        dev = self.dev
        fa_index = torch.as_tensor(fa_index).to(device=dev, dtype=torch.int32).contiguous()
        if fa_index.shape != (V,) or est.shape[0] != V:
            raise ValueError("sig, fa_index and est_signal must describe the same V voxels")
        stats = torch.zeros((V, 6, 4), dtype=torch.float64, device=dev)
        n_valid = torch.zeros(V, dtype=torch.int32, device=dev)
        if V == 0:
            return stats, n_valid
        chunk = min(V, int(max_replicates) // B)
        with torch.cuda.device(dev):
            rep_sig = torch.empty((chunk * B, self.nTE), dtype=torch.float64, device=dev)
            rep_fa = torch.empty(chunk * B, dtype=torch.int32, device=dev)
            bufs = None       # the refits' outputs, allocated by the first chunk and reused by the others
            for lo in range(0, V, chunk):
                n = min(chunk, V - lo)
                R = n * B
                _lib.check(self.lib.met2_boot_resample(_ptr(sig[lo:]), _ptr(est[lo:]), _ptr(fa_index[lo:]), n, self.nTE,
                                                       B, seed, voxel_offset + lo, _ptr(rep_sig), _ptr(rep_fa),
                                                       _stream()), "met2_boot_resample")
                fits = self.t2_fit(rep_sig[:R], rep_fa[:R],
                                   out=None if bufs is None else {k: v[:R] for k, v in bufs.items()})
                bufs = bufs if bufs is not None else fits
                _lib.check(self.lib.met2_boot_summary(_ptr(fits["maps"]), _ptr(fits["status"]), n, B, _ptr(stats[lo:]),
                                                      _ptr(n_valid[lo:]), _stream()), "met2_boot_summary")
        return stats, n_valid
