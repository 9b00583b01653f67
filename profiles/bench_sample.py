#!/usr/bin/env python3
"""profiles/bench_sample.py -- times path sampling: wfsa_dev_sample (the draw: the device part; the call ends in a device
synchronise, its logw and log q copy-out included) and wfsa_dev_viterbi_paths (the copy-out of the steps) separately, for
several n, beside wfsa_dev_viterbi on the same handle.

    python profiles/bench_sample.py [--config c4|c5] [--strings N] [--n 1,4,16] [--reps 5]

config 4 (default 1 M strings, n = 1, 4, 16): the segmented kernel's handle, sampled by k3_sample with a warp per string.
config 5 (default 300 k strings, n = 1, 4): a K7 handle, sampled by k3_sample with a CTA per string.  Prints one JSON line
for Viterbi and one per n, with the card name and power limit read in the same run.  The copy-out of n draws of every
string needs about 2 x 8 n (tokens + strings) bytes of host memory besides the caller's arrays; when MemAvailable cannot
hold that, the line says so and times the draw only."""
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
NS = {"c4": "1,4,16", "c5": "1,4"}


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def mem_available():
    with open("/proc/meminfo") as f:
        for line in f:
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) * 1024
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c4", choices=["c4", "c5"])
    ap.add_argument("--strings", type=int, default=None)
    ap.add_argument("--n", default=None, help="comma-separated list of n (1..256)")
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    ns = a.strings or STRINGS[a.config]
    ns_draws = [int(v) for v in (a.n or NS[a.config]).split(",")]
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
    symbols = int(offs[-1])
    name = card()

    def timed(fn):
        fn()                                                # warm-up
        ts = []
        for _ in range(a.reps):
            t = time.perf_counter(); fn(); ts.append((time.perf_counter() - t) * 1e3)
        return float(np.median(ts)), [round(v, 3) for v in ts]

    eval_ms, _ = timed(lambda: dev.eval(x, want_logq=False))
    for k in [None] + ns_draws:                             # None: wfsa_dev_viterbi
        m = k or 1
        logw = np.zeros(max(ns * m, 1))
        logq = np.zeros(max(ns, 1))
        off = np.zeros(ns * m + 1, dtype=np.int64)
        lw, lq, op = W._p(logw, W.F64P), W._p(logq, W.F64P), W._p(off, W.I64P)

        def draw():
            if k is None:
                dev._ck(dev.L.wfsa_dev_viterbi(dev.h, xp, lw, op))
            else:
                dev._ck(dev.L.wfsa_dev_sample(dev.h, xp, k, 1, lw, lq, op))

        dec_ms, dec_all = timed(draw)
        steps = int(off[-1])
        need = 2 * 4 * (steps + m * (symbols + ns))          # the caller's arrays and the padded host copy
        line = {"config": a.config, "strings": ns, "symbols": symbols, "call": "viterbi" if k is None else "sample", "n": m,
                "kernel": info["kernel"], "max_candidates": info["max_candidates"],
                "group": "warp" if info["max_candidates"] <= 32 else "CTA", "card": name, "draw_ms": dec_ms,
                "draw_ms_all": dec_all, "eval_ms": eval_ms, "draw_symbols_per_s": symbols / (dec_ms * 1e-3), "steps": steps,
                "paths_found": int(np.isfinite(logw[:ns * m]).sum()), "host_mem_available": mem_available()}
        if need < 0.8 * line["host_mem_available"]:
            tr = np.zeros(max(steps, 1), dtype=np.int32)
            em = np.zeros_like(tr)
            paths_ms, paths_all = timed(lambda: dev._ck(dev.L.wfsa_dev_viterbi_paths(dev.h, W._p(tr, W.I32P), W._p(em, W.I32P))))
            line.update(paths_ms=paths_ms, paths_ms_all=paths_all)
            del tr, em
        else:
            line.update(paths_ms=None, paths_skipped="the copy-out needs %d bytes of host memory" % need)
        line["timing"] = "host wall clock around calls that end in a device synchronise; median of --reps"
        print(json.dumps(line), flush=True)
        del logw, logq, off
    dev.close()


if __name__ == "__main__":
    main()
