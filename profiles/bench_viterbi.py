#!/usr/bin/env python3
"""profiles/bench_viterbi.py -- times Viterbi decoding: wfsa_dev_viterbi (the device part; the call ends in a device
synchronise, its logw copy-out included) and wfsa_dev_viterbi_paths (the copy-out of the steps) separately.

    python profiles/bench_viterbi.py [--config c4|c5] [--strings N] [--reps 5]

config 4 (default 1 M strings): the segmented kernel's handle, decoded by k3_viterbi with a warp per string (at most 32
candidates per symbol).  config 5 (default 300 k strings): a K7 handle, decoded by k3_viterbi with a CTA per string (up
to 320 candidates).  The two configurations sit on the two sides of the warp / CTA selection.  Prints one JSON line with
the card name and power limit read in the same run."""
import argparse
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
STRINGS = {"c4": 1000000, "c5": 300000}


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c4", choices=["c4", "c5"])
    ap.add_argument("--strings", type=int, default=None)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    ns = a.strings or STRINGS[a.config]
    model = synth.make_model(**CFG[a.config])
    low = model.lowered()
    offs, toks, w = model.corpus(ns, 32, 128, seed=1235)
    low.set_tokens(offs, toks, w / w.sum())
    dev = W.Device(low)
    rec, pc, used = dev.structure()
    trimmed = np.where(used > 0, 0, -2).astype(np.int32)
    n = 0
    for i in range(low.n_raw):
        if trimmed[i] == 0:
            trimmed[i] = n
            n += 1
    dev.set_param_map(trimmed, n, rec)
    info = dev.info()
    x = np.random.RandomState(7).normal(-1.0, 0.3, size=n)
    xp = W._p(x, W.F64P)
    logw = np.zeros(max(ns, 1))
    off = np.zeros(ns + 1, dtype=np.int64)

    def vit():
        dev._ck(dev.L.wfsa_dev_viterbi(dev.h, xp, W._p(logw, W.F64P), W._p(off, W.I64P)))

    vit()
    tr = np.zeros(max(int(off[-1]), 1), dtype=np.int32)
    em = np.zeros_like(tr)

    def paths():
        dev._ck(dev.L.wfsa_dev_viterbi_paths(dev.h, W._p(tr, W.I32P), W._p(em, W.I32P)))

    def timed(fn):
        fn()                                                # warm-up
        ts = []
        for _ in range(a.reps):
            t = time.perf_counter(); fn(); ts.append((time.perf_counter() - t) * 1e3)
        return float(np.median(ts)), [round(v, 3) for v in ts]

    vit_ms, vit_all = timed(vit)
    paths_ms, paths_all = timed(paths)
    eval_ms, _ = timed(lambda: dev.eval(x, want_logq=False))
    symbols = int(offs[-1])
    print(json.dumps({"config": a.config, "strings": ns, "symbols": symbols, "kernel": info["kernel"],
                      "max_candidates": info["max_candidates"], "group": "warp" if info["max_candidates"] <= 32 else "CTA",
                      "card": card(), "viterbi_ms": vit_ms, "viterbi_paths_ms": paths_ms, "eval_ms": eval_ms,
                      "viterbi_symbols_per_s": symbols / (vit_ms * 1e-3), "steps": int(off[-1]),
                      "decoded": int(np.isfinite(logw[:ns]).sum()), "viterbi_ms_all": vit_all, "viterbi_paths_ms_all": paths_all,
                      "timing": "host wall clock around calls that end in a device synchronise; median of --reps"}))
    dev.close()


if __name__ == "__main__":
    main()
