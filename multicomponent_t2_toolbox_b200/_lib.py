"""ctypes binding of libmet2.so (C ABI in include/met2.h).  No fallback: a missing library or GPU is an error."""
import ctypes
import os

from . import build as _build

_LIB = None

c_double_p = ctypes.c_void_p   # device pointers are passed as integers
c_void_p = ctypes.c_void_p


class FaCfg(ctypes.Structure):
    _fields_ = [("method", ctypes.c_int32), ("nTE", ctypes.c_int32), ("nT2", ctypes.c_int32), ("nA", ctypes.c_int32),
                ("nKnots", ctypes.c_int32), ("final_solve", ctypes.c_int32),
                ("brent_lo", ctypes.c_double), ("brent_hi", ctypes.c_double), ("brent_xatol", ctypes.c_double),
                ("brent_maxfun", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class T2Cfg(ctypes.Structure):
    _fields_ = [("method", ctypes.c_int32), ("nTE", ctypes.c_int32), ("nT2", ctypes.c_int32), ("nA", ctypes.c_int32),
                ("nLambda", ctypes.c_int32), ("maxfun", ctypes.c_int32),
                ("factor", ctypes.c_double), ("lambda_fixed", ctypes.c_double),
                ("brent_lo", ctypes.c_double), ("brent_hi", ctypes.c_double), ("brent_xatol", ctypes.c_double),
                ("log_det_L", ctypes.c_double), ("flags", ctypes.c_int32), ("echo_rank", ctypes.c_int32)]


class ParamCfg(ctypes.Structure):
    _fields_ = [("nTE", ctypes.c_int32), ("nT2", ctypes.c_int32), ("max_iter", ctypes.c_int32),
                ("reserved", ctypes.c_int32), ("tau", ctypes.c_double), ("TR", ctypes.c_double), ("T1", ctypes.c_double),
                ("t2_lo", ctypes.c_double * 3), ("t2_hi", ctypes.c_double * 3), ("fa_lo", ctypes.c_double),
                ("fa_hi", ctypes.c_double), ("mu0", ctypes.c_double), ("mu_max", ctypes.c_double),
                ("ftol", ctypes.c_double), ("xtol", ctypes.c_double)]


# every symbol include/met2.h declares, with its ctypes signature
SIGNATURES = {
    "met2_epg_dictionary": (ctypes.c_int, [c_void_p, ctypes.c_int, c_void_p, c_void_p, ctypes.c_int, ctypes.c_int,
                                           ctypes.c_double, ctypes.c_double, c_void_p, c_void_p, c_void_p]),
    "met2_epg_signals": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_double,
                                        c_void_p, c_void_p]),
    "met2_epg_dictionary_profile": (ctypes.c_int, [c_void_p, ctypes.c_int, c_void_p, c_void_p, ctypes.c_int,
                                                   ctypes.c_int, ctypes.c_double, ctypes.c_double, c_void_p, c_void_p,
                                                   c_void_p, ctypes.c_int, c_void_p, c_void_p, c_void_p]),
    "met2_epg_signals_profile": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, ctypes.c_int64, ctypes.c_int,
                                                ctypes.c_double, c_void_p, c_void_p, c_void_p, ctypes.c_int, c_void_p,
                                                c_void_p]),
    "met2_gram_tables": (ctypes.c_int, [c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_void_p]),
    "met2_fa_workspace_bytes": (ctypes.c_int64, [ctypes.c_int64, ctypes.POINTER(FaCfg)]),
    "met2_fa_fit": (ctypes.c_int, [c_void_p, ctypes.c_int64, ctypes.POINTER(FaCfg)] + [c_void_p] * 15),
    "met2_t2_workspace_bytes": (ctypes.c_int64, [ctypes.c_int64, ctypes.POINTER(T2Cfg)]),
    "met2_t2_fit": (ctypes.c_int, [c_void_p, c_void_p, ctypes.c_int64, ctypes.POINTER(T2Cfg)] + [c_void_p] * 14),
    "met2_t2_fit_echo": (ctypes.c_int, [c_void_p, c_void_p, ctypes.c_int64, ctypes.POINTER(T2Cfg)] + [c_void_p] * 16),
    "met2_echo_basis": (ctypes.c_int, [c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_void_p,
                                       c_void_p, c_void_p, c_void_p]),
    "met2_gaussian_smooth": (ctypes.c_int, [c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_void_p,
                                            ctypes.c_int, c_void_p, c_void_p, c_void_p]),
    "met2_segment_workspace_bytes": (ctypes.c_int64, [ctypes.c_int, ctypes.c_int]),
    "met2_segment_means": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_int,
                                          ctypes.c_int, ctypes.c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                          c_void_p]),
    "met2_nesma_filter": (ctypes.c_int, [c_void_p, c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                         ctypes.c_int, ctypes.c_double, c_void_p, c_void_p, c_void_p]),
    "met2_noise_sigma_workspace_bytes": (ctypes.c_int64, [ctypes.c_int] * 4),
    "met2_noise_sigma": (ctypes.c_int, [c_void_p] + [ctypes.c_int] * 4 + [c_void_p, c_void_p, c_void_p]),
    "met2_tv_workspace_bytes": (ctypes.c_int64, [ctypes.c_int] * 4),
    "met2_tv_chambolle": (ctypes.c_int, [c_void_p] + [ctypes.c_int] * 4 + [c_void_p, ctypes.c_double, ctypes.c_int,
                                                                          c_void_p, c_void_p, c_void_p, c_void_p]),
    "met2_mppca_workspace_bytes": (ctypes.c_int64, [ctypes.c_int] * 5),
    "met2_mppca": (ctypes.c_int, [c_void_p, c_void_p] + [ctypes.c_int] * 5 + [c_void_p] * 5),
    "met2_degibbs_tables": (ctypes.c_int64, [ctypes.c_int, ctypes.c_int, c_void_p]),
    "met2_degibbs_workspace_bytes": (ctypes.c_int64, [ctypes.c_int] * 7),
    "met2_degibbs": (ctypes.c_int, [c_void_p] + [ctypes.c_int] * 7 + [c_void_p] * 3),
    "met2_boot_resample": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_int,
                                          ctypes.c_uint64, ctypes.c_int64, c_void_p, c_void_p, c_void_p]),
    "met2_boot_summary": (ctypes.c_int, [c_void_p, c_void_p, ctypes.c_int64, ctypes.c_int, c_void_p, c_void_p,
                                         c_void_p]),
    "met2_spatial_sweep": (ctypes.c_int, [c_void_p] * 5 + [ctypes.c_int64, ctypes.c_int64, ctypes.c_int, ctypes.c_int,
                                                          ctypes.c_int, c_void_p, c_void_p, c_void_p, ctypes.c_double,
                                                          c_void_p, c_void_p, c_void_p]),
    "met2_spatial_finish": (ctypes.c_int, [c_void_p] * 4 + [ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int]
                            + [c_void_p] * 7),
    "met2_param_fit": (ctypes.c_int, [c_void_p] * 4 + [ctypes.c_int64, ctypes.POINTER(ParamCfg)] + [c_void_p] * 9),
    "met2_rician_fit": (ctypes.c_int, [c_void_p] * 6 + [ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int]
                        + [c_void_p] * 3 + [ctypes.c_int, ctypes.c_double] + [c_void_p] * 4),
    "met2_bessel_ratio": (ctypes.c_int64, [c_void_p, ctypes.c_int64, c_void_p]),
    "met2_last_error": (ctypes.c_char_p, []),
    "met2_version": (ctypes.c_int, []),
    "met2_echo_rank": (ctypes.c_int, [ctypes.c_int]),
    "met2_launch_count": (ctypes.c_int64, []),
}


class Met2Error(RuntimeError):
    pass


def library_path():
    return _build.LIB_PATH


def load(build_if_missing=True):
    """Load libmet2.so (building it in-tree with nvcc first if it is missing or stale and nvcc exists)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = _build.LIB_PATH
    if build_if_missing and _build.needs_build():
        try:
            _build.build_library()
        except Exception as exc:  # stale-but-present library is still usable; a missing one is fatal
            if not os.path.exists(path):
                raise Met2Error("libmet2.so is missing and could not be built: %s" % exc)
    if not os.path.exists(path):
        raise Met2Error("libmet2.so not found at %s (run __graft_entry__.build())" % path)
    lib = ctypes.CDLL(path)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the library does not export a declared symbol
        fn.restype = restype
        fn.argtypes = argtypes
    _LIB = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().met2_last_error()
        raise Met2Error("%s failed (%d): %s" % (what, rc, msg.decode() if msg else "?"))
