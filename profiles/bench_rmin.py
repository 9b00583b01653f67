#!/usr/bin/env python3
"""profiles/bench_rmin.py -- times the rmin column of the QuasiNewton optimiser: wfsa_dev_hessian(h, x, NULL, &rmin),
next to the evaluation it follows in every epoch.

    python profiles/bench_rmin.py [--config c5|c4] [--strings 1000000] [--reps 5] [--lib PATH/libwfsa_b200.so]

config 5 (default): K7, the (min, +) sweep k7_minfwd2 beside the forward sweep of the evaluation.  config 4: the segmented
kernel, rmin from its compiled region types.  Every call ends in a device synchronise (the result is copied to the host),
so host wall-clock time around a call is the call.  --lib times another build of the library (A/B runs alternate
processes).  Prints one JSON line with the card name and power limit read in the same run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "w-fsa_b200", "python"))
sys.path.insert(0, ROOT)
import wfsa_b200 as W  # noqa: E402
from wfsa_b200 import synth  # noqa: E402

CFG = {"c4": dict(n_states=256, n_sym=64, n_succ=8, n_emis=4, seed=1234),
       "c5": dict(n_states=4096, n_sym=256, n_succ=64, n_emis=16, seed=4321)}


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c5", choices=["c4", "c5"])
    ap.add_argument("--strings", type=int, default=1000000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--lib", default=None, help="another build of libwfsa_b200.so")
    a = ap.parse_args()
    if a.lib:
        W.LIB_PATH = os.path.abspath(a.lib)
    model = synth.make_model(**CFG[a.config])
    low = model.lowered()
    offs, toks, w = model.corpus(a.strings, 32, 128, seed=1235)
    low.set_tokens(offs, toks, w / w.sum())
    t0 = time.perf_counter()
    dev = W.Device(low)
    rec, pc, used = dev.structure()
    trimmed = np.where(used > 0, 0, -2).astype(np.int32)
    n = 0
    for i in range(low.n_raw):
        if trimmed[i] == 0:
            trimmed[i] = n
            n += 1
    dev.set_param_map(trimmed, n, rec)
    setup_s = time.perf_counter() - t0
    info = dev.info()
    x = np.random.RandomState(7).normal(-1.0, 0.3, size=n)
    rm = C.c_double()
    xp = W._p(x, W.F64P)

    def rmin_call():
        dev._ck(dev.L.wfsa_dev_hessian(dev.h, xp, None, C.byref(rm)))
        return rm.value

    def timed(fn):
        fn()                                                # warm-up (first calls allocate and build what they keep)
        ts = []
        for _ in range(a.reps):
            t = time.perf_counter(); fn(); ts.append((time.perf_counter() - t) * 1e3)
        return float(np.median(ts)), [round(v, 3) for v in ts]

    eval_ms, eval_all = timed(lambda: dev.eval(x, want_logq=False))
    rmin_ms, rmin_all = timed(rmin_call)
    epoch_ms, epoch_all = timed(lambda: (dev.eval(x, want_logq=False), rmin_call()))
    print(json.dumps({"config": a.config, "strings": a.strings, "symbols": int(offs[-1]), "kernel": info["kernel"],
                      "lib": a.lib or "this tree", "card": card(), "setup_s": round(setup_s, 2),
                      "eval_ms": eval_ms, "rmin_ms": rmin_ms, "epoch_ms": epoch_ms,
                      "eval_ms_all": eval_all, "rmin_ms_all": rmin_all, "epoch_ms_all": epoch_all, "rmin": rmin_call(),
                      "timing": "host wall clock around calls that end in a device synchronise; median of --reps"}))
    dev.close()


if __name__ == "__main__":
    main()
