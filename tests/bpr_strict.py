"""ctypes binding of tests/bpr_strict_reference.cpp, the StrictMath BPR epoch that defines the reference-order BPR mode.

TEST INFRASTRUCTURE ONLY (tests/ and bench_configs.py --only bprref).  The library is compiled on first use into a per-user
directory under the system's temporary directory, named by the source's hash, so that a read-only checkout works and a changed
source is never served by a stale build."""
import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "bpr_strict_reference.cpp")
_lib = None

_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_i64p = np.ctypeslib.ndpointer(np.int64, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")


def _build():
    with open(_SRC, "rb") as f:
        tag = hashlib.sha256(f.read()).hexdigest()[:16]
    out_dir = os.path.join(tempfile.gettempdir(), "lrk_bpr_strict-%d" % os.getuid())
    so = os.path.join(out_dir, "libbpr_strict-%s.so" % tag)
    if not os.path.exists(so):
        os.makedirs(out_dir, exist_ok=True)
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else (shutil.which("g++") or "g++")
        tmp = "%s.%d.tmp" % (so, os.getpid())
        subprocess.check_call([cxx, "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math",
                               "-fvisibility=hidden", "-o", tmp, _SRC])
        os.replace(tmp, so)
    return so


def lib():
    """lro_fdlibm_exp, lro_jrandom_state / lro_set_jrandom_state, lro_bpr_epoch_strict (arguments as the oracle's lro_bpr_epoch)"""
    global _lib
    if _lib is not None:
        return _lib
    L = C.CDLL(_build())
    L.lro_fdlibm_exp.restype = C.c_double
    L.lro_fdlibm_exp.argtypes = [C.c_double]
    L.lro_jrandom_state.restype = C.c_uint64
    L.lro_jrandom_state.argtypes = []
    L.lro_set_jrandom_state.argtypes = [C.c_uint64]
    L.lro_bpr_epoch_strict.restype = C.c_double
    L.lro_bpr_epoch_strict.argtypes = [C.c_int32, C.c_int32, _i64p, _i32p, C.c_int32, _f64p, _f64p,
                                       C.c_float, C.c_float, C.c_float, C.c_int64, C.c_void_p, C.c_void_p]
    _lib = L
    return L
