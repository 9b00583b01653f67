"""Loader of tests/hessian_oracle.c -- TEST INFRASTRUCTURE ONLY: the CPU reference of H_f @ V by a tangent
forward-backward in long double, without enumerating paths (so at any corpus size, any number of paths per string).

The C source is compiled on first use into the temporary directory (the tree may be read-only), once per version of it."""
import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "hessian_oracle.c")
ORACLE_INC = os.path.join(os.path.dirname(HERE), "oracle")
F64P = C.POINTER(C.c_double)
I32P = C.POINTER(C.c_int32)
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(SRC, "rb").read() + open(os.path.join(ORACLE_INC, "wfsa_oracle.h"), "rb").read()
        d = os.path.join(tempfile.gettempdir(), "wfsa_hessian_oracle_%d" % os.getuid())
        os.makedirs(d, exist_ok=True)
        so = os.path.join(d, "libhessian_%s.so" % hashlib.sha256(src).hexdigest()[:16])
        if not os.path.exists(so):
            cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else (shutil.which("gcc") or "cc")     # (as oracle/Makefile: OpenMP)
            tmp = "%s.%d.tmp" % (so, os.getpid())
            subprocess.run([cc, "-std=c11", "-O2", "-fPIC", "-shared", "-fopenmp", "-I", ORACLE_INC, "-o", tmp, SRC, "-lm"],
                           check=True, capture_output=True)
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.hessian_oracle_hv.argtypes = [C.c_void_p, C.c_void_p, F64P, F64P, I32P, C.c_int32, F64P, C.c_int32, F64P, C.c_int]
        _lib = L
    return _lib


def edge_param(low, trimmed):
    """Trimmed parameter of every edge (transitions then emissions), -1 where none."""
    params = np.concatenate([low.trans_param, low.emis_param])
    return np.array([trimmed[r] if r >= 0 and trimmed[r] >= 0 else -1 for r in params], dtype=np.int32)


def hv(low, trimmed, x, V, nthreads=0):
    """H_f @ V at x (trimmed parameters) over every string of `low`, V of shape (n, m) or (n,)."""
    ltw, lew = low.edge_logweights(x, trimmed)
    ltw = np.ascontiguousarray(ltw, dtype=np.float64); lew = np.ascontiguousarray(lew, dtype=np.float64)
    V = np.asarray(V, dtype=np.float64)
    vec = V.ndim == 1
    V = np.ascontiguousarray(V.reshape(len(x), -1))
    n, m = V.shape
    out = np.zeros((max(n, 1), max(m, 1)))[:n, :m].copy()
    ep = edge_param(low, trimmed)
    fd, cd = low.fsa_desc(), low.corpus_desc()
    lib().hessian_oracle_hv(C.byref(fd), C.byref(cd), ltw.ctypes.data_as(F64P), lew.ctypes.data_as(F64P), ep.ctypes.data_as(I32P),
                            n, V.ctypes.data_as(F64P), m, out.ctypes.data_as(F64P), nthreads)
    return out[:, 0] if vec else out


def full(low, trimmed, x, nthreads=0):
    """The whole H_f (V = I)."""
    return hv(low, trimmed, x, np.eye(len(x)), nthreads)


def directions(n, seed, n_gauss=32, n_unit=16):
    """The test directions: n_gauss Gaussian columns and n_unit unit columns at random coordinates."""
    rng = np.random.RandomState(seed)
    U = np.zeros((n, min(n_unit, n)))
    for k, j in enumerate(rng.choice(n, U.shape[1], replace=False)):
        U[j, k] = 1.0
    return np.concatenate([rng.normal(size=(n, n_gauss)), U], axis=1)
