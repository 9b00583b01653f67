"""Loader of tests/maxpath_oracle.c -- TEST INFRASTRUCTURE ONLY: the CPU reference of the most probable path of every
string (its summed log weight and its steps), for the Viterbi tests.

The C source is compiled on first use into the temporary directory (the tree may be read-only), once per version of it."""
import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "maxpath_oracle.c")
ORACLE_INC = os.path.join(os.path.dirname(HERE), "oracle")
F64P = C.POINTER(C.c_double)
I64P = C.POINTER(C.c_int64)
I32P = C.POINTER(C.c_int32)
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(SRC, "rb").read() + open(os.path.join(ORACLE_INC, "wfsa_oracle.h"), "rb").read()
        d = os.path.join(tempfile.gettempdir(), "wfsa_maxpath_oracle_%d" % os.getuid())
        os.makedirs(d, exist_ok=True)
        so = os.path.join(d, "libmaxpath_%s.so" % hashlib.sha256(src).hexdigest()[:16])
        if not os.path.exists(so):
            cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else (shutil.which("gcc") or "cc")
            tmp = "%s.%d.tmp" % (so, os.getpid())
            subprocess.run([cc, "-std=c11", "-O2", "-fPIC", "-shared", "-fopenmp", "-I", ORACLE_INC, "-o", tmp, SRC, "-lm"],
                           check=True, capture_output=True)
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.maxpath_dp.argtypes = [C.c_void_p, C.c_void_p, F64P, F64P, F64P, I64P, I32P, C.c_int, C.c_int]
        _lib = L
    return _lib


def viterbi(low, ltw, lew, nthreads=0):
    """(best, paths): best[s] = largest summed log-weight of a path of string s (-inf: not recognised), paths[s] = its steps
    as (transition edge, emission edge) pairs, emission -1 on the final transition (empty: no path)."""
    fd, cd = low.fsa_desc(), low.corpus_desc()
    n = int(cd.n_strings)
    lens = np.diff(np.asarray(low.offsets[:n + 1]))
    n_eps = sum(1 for s in range(low.n_states) if s not in (low.start, low.end)
                and any(low.emis_tok_off[e + 1] == low.emis_tok_off[e] for e in range(low.emis_row[s], low.emis_row[s + 1])))
    cap = (int(lens.max(initial=0)) + 2) * (n_eps + 1)
    best = np.zeros(max(n, 1))
    nst = np.zeros(max(n, 1), dtype=np.int64)
    steps = np.zeros(max(n, 1) * cap * 2, dtype=np.int32)
    ltw = np.ascontiguousarray(ltw, dtype=np.float64); lew = np.ascontiguousarray(lew, dtype=np.float64)
    lib().maxpath_dp(C.byref(fd), C.byref(cd), ltw.ctypes.data_as(F64P), lew.ctypes.data_as(F64P), best.ctypes.data_as(F64P),
                     nst.ctypes.data_as(I64P), steps.ctypes.data_as(I32P), cap, nthreads)
    assert (nst[:n] >= 0).all()
    st = steps.reshape(max(n, 1), cap, 2)
    return best[:n], [[(int(a), int(b)) for a, b in st[s, :nst[s]]] for s in range(n)]


def path_logweight(steps, ltw, lew):
    """Left-to-right sum of the log weights of a path: (acc + log a) + log b per step, + log a(u, end) at the end."""
    acc = 0.0
    for t, e in steps:
        acc = acc + float(ltw[t])
        if e >= 0:
            acc = acc + float(lew[e])
    return acc
