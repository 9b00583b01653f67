"""Loader of tests/sample_oracle.c -- TEST INFRASTRUCTURE ONLY: the CPU reference of path sampling (log q, and the draws
with their summed log weights and their steps), for the sampling tests; and a Python copy of Philox4x32-10.

The C source is compiled on first use into the temporary directory (the tree may be read-only), once per version of it."""
import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "sample_oracle.c")
ORACLE_INC = os.path.join(os.path.dirname(HERE), "oracle")
F64P = C.POINTER(C.c_double)
I64P = C.POINTER(C.c_int64)
I32P = C.POINTER(C.c_int32)
U32P = C.POINTER(C.c_uint32)
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(SRC, "rb").read() + open(os.path.join(ORACLE_INC, "wfsa_oracle.h"), "rb").read()
        d = os.path.join(tempfile.gettempdir(), "wfsa_sample_oracle_%d" % os.getuid())
        os.makedirs(d, exist_ok=True)
        so = os.path.join(d, "libsample_%s.so" % hashlib.sha256(src).hexdigest()[:16])
        if not os.path.exists(so):
            cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else (shutil.which("gcc") or "cc")
            tmp = "%s.%d.tmp" % (so, os.getpid())
            subprocess.run([cc, "-std=c11", "-O2", "-fPIC", "-shared", "-fopenmp", "-I", ORACLE_INC, "-o", tmp, SRC, "-lm"],
                           check=True, capture_output=True)
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.sample_draws.argtypes = [C.c_void_p, C.c_void_p, F64P, F64P, C.c_int, C.c_uint64, F64P, F64P, I64P, I32P, C.c_int,
                                   C.c_int]
        L.sample_philox4x32_10.argtypes = [U32P, U32P, U32P]
        L.sample_philox4x32_10.restype = None
        _lib = L
    return _lib


def philox4x32_10(ctr, key):
    """Philox4x32-10 in Python integers: 4 words out of a 4-word counter and a 2-word key."""
    c, k = [int(v) & 0xffffffff for v in ctr], [int(v) & 0xffffffff for v in key]
    for i in range(10):
        if i:
            k = [(k[0] + 0x9E3779B9) & 0xffffffff, (k[1] + 0xBB67AE85) & 0xffffffff]
        p0, p1 = 0xD2511F53 * c[0], 0xCD9E8D57 * c[2]
        c = [(p1 >> 32) ^ c[1] ^ k[0], p1 & 0xffffffff, (p0 >> 32) ^ c[3] ^ k[1], p0 & 0xffffffff]
    return c


def philox4x32_10_c(ctr, key):
    """The C reference's copy of Philox4x32-10."""
    c = np.ascontiguousarray(ctr, dtype=np.uint32); k = np.ascontiguousarray(key, dtype=np.uint32)
    out = np.zeros(4, dtype=np.uint32)
    lib().sample_philox4x32_10(c.ctypes.data_as(U32P), k.ctypes.data_as(U32P), out.ctypes.data_as(U32P))
    return [int(v) for v in out]


def sample(low, ltw, lew, n, seed, nthreads=0):
    """(logq [n_strings], logw [n_strings, n], paths): draw r of string s has summed log weight logw[s, r] (-inf: s has no
    path) and steps paths[s][r], (transition edge, emission edge) pairs with emission -1 on the final transition."""
    fd, cd = low.fsa_desc(), low.corpus_desc()
    ns = int(cd.n_strings)
    lens = np.diff(np.asarray(low.offsets[:ns + 1]))
    n_eps = sum(1 for s in range(low.n_states) if s not in (low.start, low.end)
                and any(low.emis_tok_off[e + 1] == low.emis_tok_off[e] for e in range(low.emis_row[s], low.emis_row[s + 1])))
    cap = (int(lens.max(initial=0)) + 2) * (n_eps + 1)
    m = max(ns, 1) * n
    logq = np.zeros(max(ns, 1))
    logw = np.zeros(m)
    nst = np.zeros(m, dtype=np.int64)
    steps = np.zeros(m * cap * 2, dtype=np.int32)
    ltw = np.ascontiguousarray(ltw, dtype=np.float64); lew = np.ascontiguousarray(lew, dtype=np.float64)
    assert lib().sample_draws(C.byref(fd), C.byref(cd), ltw.ctypes.data_as(F64P), lew.ctypes.data_as(F64P), n, seed,
                              logq.ctypes.data_as(F64P), logw.ctypes.data_as(F64P), nst.ctypes.data_as(I64P),
                              steps.ctypes.data_as(I32P), cap, nthreads) == 0
    assert (nst[:ns * n] >= 0).all()
    st = steps.reshape(m, cap, 2)
    return logq[:ns], logw[:ns * n].reshape(ns, n), [[[(int(a), int(b)) for a, b in st[s * n + r, :nst[s * n + r]]]
                                                      for r in range(n)] for s in range(ns)]
