"""Loader of tests/minpath_oracle.c -- TEST INFRASTRUCTURE ONLY: the CPU reference of the smallest path weight m_s of every
string, and with the oracle's forward-backward (oracle/oracle.py) the smallest path posterior rmin = min_s exp(m_s - log q_s).

The C source is compiled on first use into the temporary directory (the tree may be read-only), once per version of it."""
import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle import oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "minpath_oracle.c")
ORACLE_INC = os.path.join(os.path.dirname(HERE), "oracle")
F64P = C.POINTER(C.c_double)
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(SRC, "rb").read() + open(os.path.join(ORACLE_INC, "wfsa_oracle.h"), "rb").read()
        d = os.path.join(tempfile.gettempdir(), "wfsa_minpath_oracle_%d" % os.getuid())
        os.makedirs(d, exist_ok=True)
        so = os.path.join(d, "libminpath_%s.so" % hashlib.sha256(src).hexdigest()[:16])
        if not os.path.exists(so):
            cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else (shutil.which("gcc") or "cc")     # (as oracle/Makefile: OpenMP)
            tmp = "%s.%d.tmp" % (so, os.getpid())
            subprocess.run([cc, "-std=c11", "-O2", "-fPIC", "-shared", "-fopenmp", "-I", ORACLE_INC, "-o", tmp, SRC, "-lm"],
                           check=True, capture_output=True)
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.minpath_dp.argtypes = [C.c_void_p, C.c_void_p, F64P, F64P, F64P, C.c_int]
        _lib = L
    return _lib


def dp_minpath(low, ltw, lew, nthreads=0):
    """m[s] = smallest summed log-weight of a path of string s (+inf: not recognised); ltw / lew as oracle.dp_eval."""
    fd, cd = low.fsa_desc(), low.corpus_desc()
    n = int(cd.n_strings)
    m = np.zeros(max(n, 1))
    ltw = np.ascontiguousarray(ltw, dtype=np.float64); lew = np.ascontiguousarray(lew, dtype=np.float64)
    lib().minpath_dp(C.byref(fd), C.byref(cd), ltw.ctypes.data_as(F64P), lew.ctypes.data_as(F64P), m.ctypes.data_as(F64P), nthreads)
    return m[:n]


def rmin(low, ltw, lew, nthreads=0):
    """Smallest path posterior over all strings, min_s exp(m_s - log q_s), capped at 1 (no string with a choice)."""
    _, lq, _ = O.dp_eval(low, ltw, lew, nthreads=nthreads, want_grad=False)
    m = dp_minpath(low, ltw, lew, nthreads=nthreads)
    ok = np.isfinite(lq) & np.isfinite(m)
    return float(np.exp(min(0.0, float(np.min(m[ok] - lq[ok])) if ok.any() else 0.0)))
