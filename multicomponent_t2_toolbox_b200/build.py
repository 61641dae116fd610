"""Build libmet2.so (hand-written sm_100a CUDA + the C ABI of include/met2.h) in-tree with nvcc."""
import os
import shutil
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libmet2.so")
SOURCES = ["met2_api.cu", "met2_epg.cu", "met2_basis.cu", "met2_smooth.cu", "met2_aux.cu", "met2_fa.cu", "met2_t2.cu", "met2_t2_m_nnls.cu", "met2_t2_m_t2sparc.cu",
           "met2_t2_m_x2.cu", "met2_t2_m_lcurve.cu", "met2_t2_m_bayesreg.cu", "met2_t2_m_gcv.cu", "met2_t2_echo_r16.cu", "met2_t2_echo_r24.cu",
           "met2_t2_echo_reg_r16.cu", "met2_t2_echo_reg_r24.cu", "met2_tv.cu", "met2_mppca.cu", "met2_degibbs.cu", "met2_boot.cu",
           "met2_spatial.cu", "met2_param.cu", "met2_rician.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    # no implicit FMA contraction: Brent / corner-selection comparisons must round like the reference's separate
    # multiply and add; the hot loops use explicit fma()
    "-fmad=false",
    "-Xcompiler", "-fPIC", "-Xptxas", "-v",
]


def _nvcc():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: libmet2.so cannot be built")
    return nvcc


def _deps():
    """Source files the library depends on (NOT the objects / ptxas.log the build itself writes into csrc/)."""
    return [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh", ".h"))] + \
        [os.path.join(PKG_DIR, "..", "include", "met2.h")]


def needs_build():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(d) > t for d in _deps())


def build_library(force=False, verbose=False):
    """Compile every .cu under csrc/ for sm_100a into libmet2.so.  Returns the library path.

    Safe against concurrent callers (torchrun ranks): the build runs under an exclusive file lock, objects go to a
    private temporary directory and the finished library is moved into place atomically, so a process that is loading
    libmet2.so never sees a half-written file."""
    import fcntl
    import tempfile
    if not force and not needs_build():
        return LIB_PATH
    nvcc = _nvcc()
    from concurrent.futures import ThreadPoolExecutor
    with open(os.path.join(PKG_DIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        if not force and not needs_build():      # another process built it while we waited
            return LIB_PATH
        with tempfile.TemporaryDirectory(prefix="met2_build_") as tmp:
            def compile_one(src):
                obj = os.path.join(tmp, src.replace(".cu", ".o"))
                cmd = [nvcc] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
                r = subprocess.run(cmd, capture_output=True, text=True)
                if r.returncode != 0:
                    raise RuntimeError("nvcc failed on %s:\n%s" % (src, r.stderr[-8000:]))
                return obj, r.stderr

            with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 4)) as ex:
                results = list(ex.map(compile_one, SOURCES))
            objs = [o for o, _ in results]
            logs = [l for _, l in results]
            # registers / spills / stack per kernel (compile times dropped: they change every build); written BEFORE the
            # library so that it is never newer than libmet2.so
            with open(os.path.join(CSRC, "ptxas.log"), "w") as fh:
                fh.write("\n".join(l for log in logs for l in log.split("\n") if "Compile time" not in l))
            tmp_lib = LIB_PATH + ".tmp.%d" % os.getpid()
            cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", tmp_lib] + objs
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError("nvcc link failed:\n%s" % r.stderr[-4000:])
            os.replace(tmp_lib, LIB_PATH)
        if verbose:
            print("\n".join(logs))
    return LIB_PATH


EXAMPLE_SRC = os.path.join(PKG_DIR, "..", "examples", "c_host", "met2_host_demo.cpp")
EXAMPLE_BIN = os.path.join(PKG_DIR, "..", "examples", "c_host", "met2_host_demo")


def build_c_host_example():
    """Compile the C-ABI-only host program (examples/c_host) against libmet2.so.  Returns the binary path."""
    nvcc = _nvcc()
    cmd = [nvcc, "-std=c++17", "-O2", "-I", os.path.join(PKG_DIR, "..", "include"), EXAMPLE_SRC, "-L", PKG_DIR, "-lmet2",
           "-Xlinker", "-rpath", "-Xlinker", "$ORIGIN/../../multicomponent_t2_toolbox_b200", "-o", EXAMPLE_BIN]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed on the C host example:\n%s" % r.stderr[-4000:])
    return EXAMPLE_BIN


if __name__ == "__main__":
    print(build_library(force=True, verbose=True))
