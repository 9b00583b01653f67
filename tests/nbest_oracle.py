"""Loader of tests/nbest_oracle.c -- TEST INFRASTRUCTURE ONLY: the CPU reference of the k most probable paths of every
string (their summed log weights and their steps), for the N-best tests.

The C source is compiled on first use into the temporary directory (the tree may be read-only), once per version of it."""
import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "nbest_oracle.c")
ORACLE_INC = os.path.join(os.path.dirname(HERE), "oracle")
F64P = C.POINTER(C.c_double)
I64P = C.POINTER(C.c_int64)
I32P = C.POINTER(C.c_int32)
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(SRC, "rb").read() + open(os.path.join(ORACLE_INC, "wfsa_oracle.h"), "rb").read()
        d = os.path.join(tempfile.gettempdir(), "wfsa_nbest_oracle_%d" % os.getuid())
        os.makedirs(d, exist_ok=True)
        so = os.path.join(d, "libnbest_%s.so" % hashlib.sha256(src).hexdigest()[:16])
        if not os.path.exists(so):
            cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else (shutil.which("gcc") or "cc")
            tmp = "%s.%d.tmp" % (so, os.getpid())
            subprocess.run([cc, "-std=c11", "-O2", "-fPIC", "-shared", "-fopenmp", "-I", ORACLE_INC, "-o", tmp, SRC, "-lm"],
                           check=True, capture_output=True)
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.nbest_kbest.argtypes = [C.c_void_p, C.c_void_p, F64P, F64P, C.c_int, F64P, I64P, I32P, C.c_int, C.c_int]
        _lib = L
    return _lib


def nbest(low, ltw, lew, k, nthreads=0):
    """(best [n, k], paths): best[s, r] = summed log-weight of the r-th most probable path of string s (-inf: s has at most r
    paths), paths[s][r] = its steps as (transition edge, emission edge) pairs, emission -1 on the final transition (empty:
    none)."""
    fd, cd = low.fsa_desc(), low.corpus_desc()
    n = int(cd.n_strings)
    lens = np.diff(np.asarray(low.offsets[:n + 1]))
    n_eps = sum(1 for s in range(low.n_states) if s not in (low.start, low.end)
                and any(low.emis_tok_off[e + 1] == low.emis_tok_off[e] for e in range(low.emis_row[s], low.emis_row[s + 1])))
    cap = (int(lens.max(initial=0)) + 2) * (n_eps + 1)
    m = max(n, 1) * k
    best = np.zeros(m)
    nst = np.zeros(m, dtype=np.int64)
    steps = np.zeros(m * cap * 2, dtype=np.int32)
    ltw = np.ascontiguousarray(ltw, dtype=np.float64); lew = np.ascontiguousarray(lew, dtype=np.float64)
    assert lib().nbest_kbest(C.byref(fd), C.byref(cd), ltw.ctypes.data_as(F64P), lew.ctypes.data_as(F64P), k,
                             best.ctypes.data_as(F64P), nst.ctypes.data_as(I64P), steps.ctypes.data_as(I32P), cap, nthreads) == 0
    assert (nst[:n * k] >= 0).all()
    st = steps.reshape(m, cap, 2)
    return best[:n * k].reshape(n, k), [[[(int(a), int(b)) for a, b in st[s * k + r, :nst[s * k + r]]] for r in range(k)]
                                        for s in range(n)]
