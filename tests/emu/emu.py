"""TEST INFRASTRUCTURE ONLY — the CUDA sources of multicomponent_t2_toolbox_b200/csrc compiled by g++ against the
single-threaded SIMT emulator (simt_emu.h) into tests/emu/_build/libmet2_emu.so.  The library exports the SAME C ABI as
libmet2.so (include/met2.h): the host code of every entry point (argument checks, workspace carving, geometry, launch
sequence) runs unchanged and its MET2_LAUNCH sites drive the emulator, so the `-m "not gpu"` tests exercise the kernels'
real source — control flow, shared-memory indexing (bounds-checked), warp collectives, the blocked FP64-MMA
factorisation — with HOST (numpy) pointers.  Not a fallback: nothing in the product package imports this, and
multicomponent_t2_toolbox_b200/_lib.py only ever loads libmet2.so."""
import ctypes
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(ROOT, "multicomponent_t2_toolbox_b200", "csrc")
BUILD = os.path.join(HERE, "_build")
LIB = os.path.join(BUILD, "libmet2_emu.so")

METHODS = {"NNLS": 0, "T2SPARC": 1, "X2": 2, "L_curve": 3, "GCV": 4, "BayesReg": 5}
P = ctypes.c_void_p


class T2Cfg(ctypes.Structure):   # met2_t2_cfg of include/met2.h
    _fields_ = [("method", ctypes.c_int32), ("nTE", ctypes.c_int32), ("nT2", ctypes.c_int32), ("nA", ctypes.c_int32),
                ("nLambda", ctypes.c_int32), ("maxfun", ctypes.c_int32),
                ("factor", ctypes.c_double), ("lambda_fixed", ctypes.c_double),
                ("brent_lo", ctypes.c_double), ("brent_hi", ctypes.c_double), ("brent_xatol", ctypes.c_double),
                ("log_det_L", ctypes.c_double), ("flags", ctypes.c_int32), ("echo_rank", ctypes.c_int32)]


class FaCfg(ctypes.Structure):   # met2_fa_cfg of include/met2.h
    _fields_ = [("method", ctypes.c_int32), ("nTE", ctypes.c_int32), ("nT2", ctypes.c_int32), ("nA", ctypes.c_int32),
                ("nKnots", ctypes.c_int32), ("final_solve", ctypes.c_int32),
                ("brent_lo", ctypes.c_double), ("brent_hi", ctypes.c_double), ("brent_xatol", ctypes.c_double),
                ("brent_maxfun", ctypes.c_int32), ("reserved", ctypes.c_int32)]


def _sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu")) + \
        [os.path.join(HERE, "emu_runtime.cpp")]


def build(force=False):
    """g++ every csrc/*.cu (as C++, -DMET2_HOST_EMU) + emu_runtime.cpp -> libmet2_emu.so.  Rebuilds when a source is
    newer than the library."""
    deps = _sources() + [os.path.join(HERE, "simt_emu.h"), os.path.join(ROOT, "include", "met2.h")]
    deps += [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    if not force and os.path.exists(LIB) and all(os.path.getmtime(d) <= os.path.getmtime(LIB) for d in deps):
        return LIB
    os.makedirs(BUILD, exist_ok=True)
    flags = ["-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-DMET2_HOST_EMU=1", "-x", "c++", "-I", HERE, "-I", CSRC,
             "-I", os.path.join(ROOT, "include")]

    def compile_one(src):
        obj = os.path.join(BUILD, os.path.basename(src) + ".o")
        r = subprocess.run(["g++"] + flags + ["-c", src, "-o", obj], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("g++ failed on %s (SIMT emulation build):\n%s" % (src, r.stderr[-6000:]))
        return obj

    with ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:
        objs = list(ex.map(compile_one, _sources()))
    r = subprocess.run(["g++", "-shared", "-o", LIB] + objs, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link of libmet2_emu.so failed:\n" + r.stderr[-4000:])
    return LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
        _lib.met2_last_error.restype = ctypes.c_char_p
        _lib.met2_t2_workspace_bytes.restype = ctypes.c_int64
        _lib.met2_t2_workspace_bytes.argtypes = [ctypes.c_int64, ctypes.POINTER(T2Cfg)]
        _lib.met2_fa_workspace_bytes.restype = ctypes.c_int64
        _lib.met2_fa_workspace_bytes.argtypes = [ctypes.c_int64, ctypes.POINTER(FaCfg)]
        _lib.met2_segment_workspace_bytes.restype = ctypes.c_int64
        _lib.met2_segment_workspace_bytes.argtypes = [ctypes.c_int, ctypes.c_int]
        _lib.met2_launch_count.restype = ctypes.c_int64
    return _lib


def _ptr(a):
    return a.ctypes.data_as(P) if a is not None else None


def _check(rc, what):
    if rc != 0:
        raise RuntimeError("%s failed (%d): %s" % (what, rc, lib().met2_last_error().decode()))


_GUARD = 512      # bytes of canary either side of every output / workspace array


class _Guarded:
    """Output arrays carved out of byte buffers with canaries either side: a kernel writing just outside one of its
    output or workspace arrays is caught by `check()` after the call."""

    def __init__(self):
        self.bufs = []

    def array(self, shape, dtype, fill):
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * dtype.itemsize
        raw = np.full(n + 2 * _GUARD, 0xC3, dtype=np.uint8)
        view = raw[_GUARD:_GUARD + n].view(dtype).reshape(shape)
        view[...] = fill
        self.bufs.append((raw, n))
        return view

    def check(self, what):
        for raw, n in self.bufs:
            if not (np.all(raw[:_GUARD] == 0xC3) and np.all(raw[_GUARD + n:] == 0xC3)):
                raise AssertionError("%s wrote outside one of its output / workspace arrays" % what)


def counters(reset_only=False):
    """Work since the last call: per-THREAD counts of fma(), shared-memory accesses, __syncwarp, warp collectives
    (divide by 32 for warp level) and the number of kernel launches."""
    cnt = (ctypes.c_longlong * 5)()
    lib().emu_counters(cnt)
    return None if reset_only else dict(fma=int(cnt[0]), smem=int(cnt[1]), syncwarp=int(cnt[2]),
                                        collectives=int(cnt[3]), launches=int(cnt[4]))


def tables(Dic_3D, L):
    """numpy versions of what met2_epg_dictionary / met2_gram_tables hand to the fit kernels:
    dic [nA][nTE][nT2], dicT [nA][nT2][nTE], G [nA][nT2][nT2], kband [10][nT2]."""
    dic = np.ascontiguousarray(np.transpose(Dic_3D, (2, 0, 1)))
    dicT = np.ascontiguousarray(np.transpose(Dic_3D, (2, 1, 0)))
    G = np.ascontiguousarray(np.einsum("aec,aed->acd", dic, dic))
    n = dic.shape[2]
    K = L.T @ L
    kband = np.zeros((10, n))
    for d in range(5):
        for c in range(n):
            r = c + d - 2
            if 0 <= r < n:
                kband[d, c] = K[r, c]          # kband[d][c] = K[c + d - 2][c]
        for r in range(n):
            c = r + d - 2
            if 0 <= c < n:
                kband[5 + d, r] = L[r, c]      # kband[5 + d][r] = L[r][r + d - 2]
    return dic, dicT, G, kband


def epg_dictionary(alphas, T2s, T1s, nTE, tau, TR):
    """met2_epg_dictionary -> (dic [nA][nTE][nT2], dicT [nA][nT2][nTE])."""
    alphas = np.ascontiguousarray(alphas, dtype=np.float64)
    T2s = np.ascontiguousarray(T2s, dtype=np.float64)
    T1s = np.ascontiguousarray(T1s, dtype=np.float64)
    dic = np.zeros((len(alphas), nTE, len(T2s)))
    dicT = np.zeros((len(alphas), len(T2s), nTE))
    fn = lib().met2_epg_dictionary
    fn.argtypes = [P, ctypes.c_int, P, P, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_double, P, P, P]
    _check(fn(_ptr(alphas), len(alphas), _ptr(T2s), _ptr(T1s), len(T2s), nTE, tau, TR, _ptr(dic), _ptr(dicT), None),
           "met2_epg_dictionary")
    return dic, dicT


def gram_tables(dic, L):
    """met2_gram_tables -> (G [nA][nT2][nT2], kband [10][nT2], band_err)."""
    dic = np.ascontiguousarray(dic, dtype=np.float64)
    nA, nTE, n = dic.shape
    L = np.ascontiguousarray(L, dtype=np.float64)
    G = np.zeros((nA, n, n))
    kband = np.full((10, n), np.nan)
    err = np.full(1, -1, dtype=np.int32)
    fn = lib().met2_gram_tables
    fn.argtypes = [P, ctypes.c_int, ctypes.c_int, ctypes.c_int, P, P, P, P, P]
    _check(fn(_ptr(dic), nA, nTE, n, _ptr(L), _ptr(G), _ptr(kband), _ptr(err), None), "met2_gram_tables")
    return G, kband, int(err[0])


def echo_basis(dic, R=None):
    """met2_echo_basis -> (basis [nA][nTE][R], coef [nA][nT2][R], tail [nA]); R defaults to the library's MET2_ECHO_RANK."""
    if R is None:
        R = int(lib().met2_echo_rank(0))
    dic = np.ascontiguousarray(dic, dtype=np.float64)
    nA, m, n = dic.shape
    basis = np.full((nA, m, R), np.nan)
    coef = np.full((nA, n, R), np.nan)
    tail = np.full(nA, np.nan)
    fn = lib().met2_echo_basis
    fn.argtypes = [P, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, P, P, P, P]
    _check(fn(_ptr(dic), nA, m, n, R, _ptr(basis), _ptr(coef), _ptr(tail), None), "met2_echo_basis")
    return basis, coef, tail


def t2_fit(sig, fa_index, Dic_3D, L, T2s, method="X2", flags=0, echo=False, lambdas=None, myelin_T2=40.0, warps=2,
           factor=1.02, lambda_fixed=1.8, echo_rank=0):
    """met2_t2_fit on host arrays (counting sort, tile list, shared full-set factor tables and the fit kernel, all
    emulated).  `warps` caps the warps per block (MET2_T2_WARPS).  Returns dict(fsol, est_signal, reg, maps, status,
    counters)."""
    counters(reset_only=True)
    sig = np.ascontiguousarray(sig, dtype=np.float64)
    fa_index = np.ascontiguousarray(fa_index, dtype=np.int32)
    V, m = sig.shape
    dic, dicT, G, kband = tables(np.asarray(Dic_3D, dtype=np.float64), np.asarray(L, dtype=np.float64))
    nA, _, n = dic.shape
    T2s = np.asarray(T2s, dtype=np.float64)
    comp = ((T2s <= myelin_T2) * 1 + ((T2s > myelin_T2) & (T2s <= 200.0)) * 2 + (T2s >= 200.0) * 4).astype(np.uint8)
    logT2 = np.ascontiguousarray(np.log(T2s))
    lam = np.ascontiguousarray(lambdas if lambdas is not None else np.zeros(1), dtype=np.float64)
    cfg = T2Cfg(method=METHODS[method], nTE=m, nT2=n, nA=nA, nLambda=len(lam), maxfun=300, factor=factor,
                lambda_fixed=lambda_fixed, brent_lo=0.0, brent_hi=10.0, brent_xatol=1e-5, log_det_L=0.0,
                flags=int(flags) | (64 if echo else 0), echo_rank=int(echo_rank))
    if method == "GCV":                      # algorithms.py:280
        cfg.brent_lo = 1e-8
    if method == "BayesReg":                 # bayesian_interpolation.py:100-101
        cfg.brent_lo, cfg.brent_hi, cfg.maxfun = 1e-8, 2.0, 200
        with np.errstate(divide="ignore"):
            cfg.log_det_L = float(np.log(np.linalg.det(np.asarray(L, dtype=np.float64))))
    gd = _Guarded()      # poisoned, canary-guarded outputs: every element must be written, nothing beyond
    out = dict(fsol=gd.array((V, n), np.float64, np.nan), est_signal=gd.array((V, m), np.float64, np.nan),
               reg=gd.array(V, np.float64, np.nan), maps=gd.array((V, 6), np.float64, np.nan),
               status=gd.array(V, np.uint32, 0xFFFFFFFF))
    old = os.environ.get("MET2_T2_WARPS")
    os.environ["MET2_T2_WARPS"] = str(warps)
    try:
        nbytes = lib().met2_t2_workspace_bytes(V, ctypes.byref(cfg))
        if nbytes < 0:
            raise RuntimeError("met2_t2_workspace_bytes: " + lib().met2_last_error().decode())
        ws = gd.array(int(nbytes), np.uint8, 0xA5)               # poisoned like a fresh torch.empty
        basis = coef = None
        if echo:                                                 # reduced echo basis from the library's own kernel
            basis, coef, tail = echo_basis(dic, echo_rank if echo_rank else None)
            assert tail.max() <= (4e-12 if echo_rank == 16 else 1e-15), tail.max()      # batched.ECHO_TAIL_MAX
        fn = lib().met2_t2_fit_echo
        fn.argtypes = [P, P, ctypes.c_int64, ctypes.POINTER(T2Cfg)] + [P] * 16
        _check(fn(_ptr(sig), _ptr(fa_index), V, ctypes.byref(cfg), _ptr(dic), _ptr(dicT), _ptr(G), _ptr(kband),
                  _ptr(lam), _ptr(logT2), _ptr(comp), _ptr(basis), _ptr(coef), _ptr(out["fsol"]),
                  _ptr(out["est_signal"]), _ptr(out["reg"]), _ptr(out["maps"]), _ptr(out["status"]), _ptr(ws), None),
               "met2_t2_fit_echo")
        gd.check("met2_t2_fit")
    finally:
        if old is None:
            del os.environ["MET2_T2_WARPS"]
        else:
            os.environ["MET2_T2_WARPS"] = old
    out["counters"] = counters()
    return out


def fa_fit(sig, Dic_3D, alpha_values, Dic_3D_LR=None, alpha_values_spline=None):
    """met2_fa_fit on host arrays: brute force over `alpha_values`, or the spline method when the coarse dictionary is
    given.  Returns dict(fa_index, fa_deg, km, fsol_sum, status)."""
    counters(reset_only=True)
    sig = np.ascontiguousarray(sig, dtype=np.float64)
    V, m = sig.shape
    eye = np.eye(Dic_3D.shape[1])
    dic, dicT, G, _ = tables(np.asarray(Dic_3D, dtype=np.float64), eye)
    nA, _, n = dic.shape
    alphas = np.ascontiguousarray(alpha_values, dtype=np.float64)
    spline = Dic_3D_LR is not None
    dic_s = dicT_s = G_s = knots = None
    if spline:
        dic_s, dicT_s, G_s, _ = tables(np.asarray(Dic_3D_LR, dtype=np.float64), eye)
        knots = np.ascontiguousarray(alpha_values_spline, dtype=np.float64)
    cfg = FaCfg(method=1 if spline else 0, nTE=m, nT2=n, nA=nA, nKnots=(len(knots) if spline else 0), final_solve=1,
                brent_lo=90.0, brent_hi=180.0, brent_xatol=1e-5, brent_maxfun=500, reserved=0)
    gd = _Guarded()
    out = dict(fa_index=gd.array(V, np.int32, -7), fa_deg=gd.array(V, np.float64, np.nan), km=gd.array(V, np.float64, np.nan),
               fsol_sum=gd.array(n, np.float64, np.nan), status=gd.array(V, np.uint32, 0xFFFFFFFF))
    nbytes = lib().met2_fa_workspace_bytes(V, ctypes.byref(cfg))
    if nbytes < 0:
        raise RuntimeError("met2_fa_workspace_bytes: " + lib().met2_last_error().decode())
    ws = gd.array(int(nbytes), np.uint8, 0xA5)
    fn = lib().met2_fa_fit
    fn.argtypes = [P, ctypes.c_int64, ctypes.POINTER(FaCfg)] + [P] * 15
    _check(fn(_ptr(sig), V, ctypes.byref(cfg), _ptr(dic), _ptr(dicT), _ptr(G), _ptr(alphas), _ptr(dic_s), _ptr(dicT_s),
              _ptr(G_s), _ptr(knots), _ptr(out["fa_index"]), _ptr(out["fa_deg"]), _ptr(out["km"]), _ptr(out["fsol_sum"]),
              _ptr(out["status"]), _ptr(ws), None), "met2_fa_fit")
    gd.check("met2_fa_fit")
    out["counters"] = counters()
    return out


def gaussian_smooth(vol, sigma=2.0, truncate=4.0):
    """met2_gaussian_smooth with scipy.ndimage's kernel (radius = int(truncate * sigma + 0.5))."""
    vol = np.ascontiguousarray(vol, dtype=np.float64)
    nx, ny, nz, nt = vol.shape
    radius = int(truncate * sigma + 0.5)
    x = np.arange(-radius, radius + 1)
    w = np.exp(-0.5 / (sigma * sigma) * x ** 2)
    w = np.ascontiguousarray(w / w.sum())
    out, tmp = np.zeros_like(vol), np.zeros_like(vol)
    fn = lib().met2_gaussian_smooth
    fn.argtypes = [P] + [ctypes.c_int] * 4 + [P, ctypes.c_int, P, P, P]
    _check(fn(_ptr(vol), nx, ny, nz, nt, _ptr(w), radius, _ptr(out), _ptr(tmp), None), "met2_gaussian_smooth")
    return out


def nesma_filter(vol, mask, half_window=6, threshold=2.5):
    vol = np.ascontiguousarray(vol, dtype=np.float64)
    mask = np.ascontiguousarray(mask, dtype=np.int32)
    nx, ny, nz, nt = vol.shape
    out, tmp = np.zeros_like(vol), np.zeros_like(vol)
    fn = lib().met2_nesma_filter
    fn.argtypes = [P, P] + [ctypes.c_int] * 5 + [ctypes.c_double, P, P, P]
    _check(fn(_ptr(vol), _ptr(mask), nx, ny, nz, nt, half_window, threshold, _ptr(out), _ptr(tmp), None),
           "met2_nesma_filter")
    return out


def segment_means(sig, fa_index, label, nSeg, dic):
    """met2_segment_means -> (mean_signal [nSeg][nTE], mean_kernel [nSeg][nTE][nT2], counts [nSeg])."""
    sig = np.ascontiguousarray(sig, dtype=np.float64)
    fa_index = np.ascontiguousarray(fa_index, dtype=np.int32)
    label = np.ascontiguousarray(label, dtype=np.int32)
    dic = np.ascontiguousarray(dic, dtype=np.float64)
    V, m = sig.shape
    nA, _, n = dic.shape
    ms, mk, cnt = np.zeros((nSeg, m)), np.zeros((nSeg, m, n)), np.zeros(nSeg, dtype=np.int32)
    ws = np.full(int(lib().met2_segment_workspace_bytes(nSeg, nA)) + 512, 0xA5, dtype=np.uint8)
    fn = lib().met2_segment_means
    fn.argtypes = [P, P, P, ctypes.c_int64] + [ctypes.c_int] * 4 + [P] * 6
    _check(fn(_ptr(sig), _ptr(fa_index), _ptr(label), V, m, n, nA, nSeg, _ptr(dic), _ptr(ms), _ptr(mk), _ptr(cnt),
              _ptr(ws), None), "met2_segment_means")
    return ms, mk, cnt
