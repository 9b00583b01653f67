#!/usr/bin/env python3
"""bench.py -- forward-backward + gradient throughput (symbols/s) of the w-fsa evaluation path.

One "step" = one objective + gradient evaluation (what one optimiser epoch needs,
/root/reference/src/QuasiNewtonLearner.cpp:162-168) over a synthetic corpus of BASELINE.json's
config 4: WFSA 256 states / 64 symbols / 8 480 combined arcs, 1M strings of length 32-128.
N = 1: the whole corpus on one GPU.  N > 1: STRONG scaling, the same 1M-string corpus cut into N
ranges of equal symbol count (north_star's multi-GPU target); [loglik, per-edge sums] are exchanged as
exact 64-bit integers through NVLink peer memory inside the evaluation kernel.  The weak-scaling
number (1M strings per GPU) is measured in the same run and reported under the key "weak".

  python bench.py [--gpus N] [--steps K] [--warmup W]          our arm (one JSON line on stdout)
  python bench.py --impl reference ...                           the reference's CPU implementation
  torchrun ... bench.py --gpus N ...                             one rank per GPU
  python bench.py ... --dump-outputs DIR                         also write what the last timed step returned, DIR/<name>.npy

`--dump-outputs DIR` writes, in float64, the log-likelihood (loglik.npy), the gradient (grad.npy) and log q of every string
in corpus order (logq.npy, the ranks' strings one after another) that the timed evaluations returned in their last step.
The inputs are seeded, so two builds run with the same arguments can be compared output for output.  Above DUMP_BYTES in
all, logq.npy holds a fixed, seeded sample of the strings, in corpus order.

`value`  : kernel-resident throughput -- x already on the device, K evaluations timed with CUDA
           events on the library's own stream, max over ranks.
`e2e`    : the same metric through the C-ABI call a w-fsa maintainer would make
           (wfsa_dev_eval with HOST buffers): H2D of x from pinned memory, all kernels,
           D2H of [loglik, grad], every step.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "w-fsa_b200", "python"))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "fwd-bwd+grad symbols/sec"
UNIT = "symbols/s"
C4 = dict(n_states=256, n_sym=64, n_succ=8, n_emis=4, seed=1234)
C5 = dict(n_states=4096, n_sym=256, n_succ=64, n_emis=16, seed=4321)    # config 5 (dense, CTA-per-string kernel)
DUMP_BYTES = 64 * 10**6                   # --dump-outputs: at most this much in all, .npy headers included


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu):
        self.gpu, self.proc, self.lines = gpu, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))
    return rank, world, local


# ------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """The reference's own CPU implementation (oracle/_ref/wfsa_ref = unmodified reference sources +
    MKL stand-in, single-threaded like the reference's mkl_sequential build) on a bounded sample of
    the same workload: a step = one QuasiNewtonLearner::OptimizationStep.  Falls back to the CPU
    port (oracle/wfsa_oracle.c) when the reference binary is not present."""
    if rank != 0:
        return
    from wfsa_b200 import synth
    model = synth.make_model(**C4)
    ref_bin = os.path.join(ROOT, "oracle", "_ref", "wfsa_ref")
    steps, warm = args.steps, args.warmup
    if os.path.exists(ref_bin) and not args.cpu_port:
        n = args.ref_strings
        offs, toks, w = model.corpus(n, 32, 128, seed=1235)
        with tempfile.TemporaryDirectory() as tmp:
            fa, fc = os.path.join(tmp, "c4.wfsa"), os.path.join(tmp, "c4.corpus")
            open(fa, "w").write(model.text())
            open(fc, "w").write(model.corpus_text(offs, toks, w))

            def run(epochs):
                t = time.perf_counter()
                subprocess.run([ref_bin, "-a", fa, "-c", fc, "-opt", "QuasiNewton", "-i", "7", "-e", str(epochs), "-tol", "0", "-s"],
                               check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
                return time.perf_counter() - t
            # a step is timed as the difference of two whole runs, so the run with the steps must be long against the
            # jitter of the 8 s one-time part: at least 20 epochs, the one-time part as the smaller of two runs, and four
            # times the epochs if the difference still drowns
            epochs = max(warm + steps, 20)
            t0 = min(run(0), run(0))          # load + path enumeration (Learner::BuildFrom), one-time
            t1 = run(epochs)
            if t1 - t0 < 0.05 * t0:
                epochs *= 4
                t1 = run(epochs)
        per_step = max(t1 - t0, 1e-6) / epochs
        tokens = int(offs[-1])
        kind, cores = "reference", 1
        sample = "%d strings (%d symbols) of config 4; one-time path enumeration %.1f s excluded" % (n, tokens, t0)
    else:
        from oracle import oracle as O
        low = model.lowered()
        n = args.cpu_strings
        offs, toks, w = model.corpus(n, 32, 128, seed=1235)
        low.set_tokens(offs, toks, w / w.sum())
        zt, ze = np.zeros(low.n_trans), np.zeros(low.n_emis)
        cores = O.max_threads()
        for _ in range(warm):
            O.dp_eval(low, zt, ze, nthreads=cores)
        t = time.perf_counter()
        for _ in range(steps):
            O.dp_eval(low, zt, ze, nthreads=cores)
        per_step = (time.perf_counter() - t) / steps
        tokens = int(offs[-1])
        kind = "port"
        sample = "%d strings (%d symbols) of config 4, CPU forward-backward port" % (n, tokens)
    value = tokens / per_step
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps,
            "warmup": warm, "ms_per_step": per_step * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "config 4: WFSA 256 states / 64 symbols / ~8k arcs, strings of length 32-128 (bounded sample)",
                       "strings": n, "symbols": tokens},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def cpu_baseline(model, budget_s=12.0):
    """CPU forward-backward port (oracle) on a bounded sample, all host cores."""
    from oracle import oracle as O
    low = model.lowered()
    cores = O.max_threads()
    n = 20000
    offs, toks, w = model.corpus(n, 32, 128, seed=99)
    low.set_tokens(offs, toks, w / w.sum())
    zt, ze = np.zeros(low.n_trans), np.zeros(low.n_emis)
    t = time.perf_counter()
    O.dp_eval(low, zt, ze, nthreads=cores)
    dt = time.perf_counter() - t
    reps = int(max(1, min(50, budget_s / max(dt, 1e-3))))
    t = time.perf_counter()
    for _ in range(reps):
        O.dp_eval(low, zt, ze, nthreads=cores)
    dt = (time.perf_counter() - t) / reps
    return {"value": float(offs[-1]) / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "%d strings (%d symbols) of config 4 x %d repetitions, oracle/wfsa_oracle.c forward-backward, OpenMP" % (n, int(offs[-1]), reps)}


def _trim_all_used(used):
    trimmed = np.where(used > 0, 0, -2).astype(np.int32)
    n = 0
    for i in range(len(trimmed)):            # the synthetic configs have no lone survivors; plain compaction
        if trimmed[i] == 0:
            trimmed[i] = n
            n += 1
    return trimmed, n


def dump_outputs(out_dir, loglik, grad, logq):
    grad, logq = np.asarray(grad, dtype=np.float64), np.asarray(logq, dtype=np.float64)
    room = (DUMP_BYTES - 3 * 256 - 8 - grad.nbytes) // 8
    if len(logq) > room:
        logq = logq[np.sort(np.random.RandomState(0).choice(len(logq), room, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("loglik", np.array([loglik], dtype=np.float64)), ("grad", grad), ("logq", logq)):
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measure(dev, x, args, barrier, want_e2e=True):
    """Device-timed steps (one event pair per evaluation, L2 flushed between evaluations), then the host-buffer call."""
    dev.upload_x(x)
    for _ in range(args.warmup):
        dev.eval_launch()
    dev.sync()
    launches0 = dev.info()["kernels_launched"]
    barrier()

    def timed_loop(detail):
        (dev.timer_begin if detail else dev.timer_begin_steps)()
        for _ in range(args.steps):
            if not args.no_flush:
                dev.l2_flush()
            dev.rank_barrier()      # N > 1: the flushes of the ranks differ by several us; line the ranks up again (on the device)
            dev.eval_launch()
        return dev.timer_end()

    # pass 1, the headline: one event pair per evaluation and nothing else in the stream
    bracket_ms = timed_loop(False)
    barrier()
    ms, nsteps = dev.timer_step_ms()
    assert nsteps == args.steps
    launches = dev.info()["kernels_launched"] - launches0
    # pass 2, for the roofline: the same evaluations with a second event pair around the dominant kernel (the extra
    # events cost a few us per step) and the in-kernel phase stamps of k_eval6
    dev.eval6_phases(True)
    timed_loop(True)
    barrier()
    kms, klaunches = dev.timer_kernel_ms()
    phases = dev.timer_phase_ms()
    inker = [float(v) / args.steps / 1e3 for v in dev.eval6_phases(True)]
    ll, grad = dev.eval_fetch()
    out = {"ms": ms, "bracket_ms": bracket_ms, "kms": kms, "klaunches": klaunches, "phases": phases, "in_kernel_us": inker,
           "launches": launches, "ll": ll, "grad": grad, "e2e_s": None}
    if want_e2e:
        for _ in range(max(1, args.warmup // 2)):
            dev.eval(x, want_logq=False)
        barrier()
        e2e_s = 0.0
        for i in range(args.steps):
            dev.l2_flush()
            dev.rank_barrier()
            dev.sync()
            t0 = time.perf_counter()
            ll_e, _, g_e = dev.eval(x, want_logq=False)
            e2e_s += time.perf_counter() - t0
        barrier()
        assert ll_e == ll and np.array_equal(g_e, grad), "resident and host-buffer evaluations must agree bitwise"
        out["e2e_s"] = e2e_s
    return out


def run_ours(args, rank, world, local):
    import torch
    import torch.distributed as dist
    import wfsa_b200 as W
    from wfsa_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the w-fsa B200 backend has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cfg = C5 if args.config == "c5" else C4
    model = synth.make_model(**cfg)
    low = model.lowered()
    n_strings = args.strings
    # N > 1: the headline is STRONG scaling on the 1M-string corpus of the metric (north_star); the weak-scaling number
    # (1M strings per GPU) is measured in the same run and reported under "weak"
    scaling = args.scaling or ("strong" if world > 1 else "weak")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def all_max(vals):
        if world == 1:
            return [float(v) for v in vals]
        v = torch.tensor(vals, dtype=torch.float64, device="cuda")
        dist.all_reduce(v, op=dist.ReduceOp.MAX)
        return [float(a) for a in v.tolist()]

    def all_sum(vals):
        if world == 1:
            return [float(v) for v in vals]
        v = torch.tensor(vals, dtype=torch.float64, device="cuda")
        dist.all_reduce(v)
        return [float(a) for a in v.tolist()]

    def make_shard(mode):
        if mode == "strong":
            offs, toks, w = model.corpus(n_strings, 32, 128, seed=1235)
            total_w = float(w.sum())
            cuts = synth.balanced_ranges(offs, world)
            a, b = cuts[rank], cuts[rank + 1]
            toks = toks[offs[a]:offs[b]]
            offs = offs[a:b + 1] - offs[a]
            w = w[a:b]
        else:
            offs, toks, w = model.corpus(n_strings, 32, 128, seed=1235 + 7919 * rank)
            total_w = all_sum([float(w.sum())])[0]
        return offs, toks, w, total_w

    def make_device(offs, toks, w, total_w):
        low.set_tokens(offs, toks, w / total_w)
        variant = args.variant | (args.replicas << 8) | (2 if args.noacc else 0) | (args.K << 16) | ((args.threads // 32) << 24)
        dev = W.Device(low, device=local, force_kernel=args.kernel, accum_mode=args.accum, accum_variant=variant)
        if world > 1:
            uid = np.zeros(W.UNIQUE_ID_BYTES, dtype=np.uint8)
            if rank == 0:
                W.lib().wfsa_dev_comm_unique_id(uid.ctypes.data_as(W.C.c_void_p))
            t = torch.from_numpy(uid).cuda()
            dist.broadcast(t, 0)
            dev.comm_init(t.cpu().numpy().tobytes(), rank, world)
        t0 = time.perf_counter()
        rec, pc, used = dev.structure()
        assert rec.all(), "synthetic strings are random walks of the automaton: all must be recognised"
        trimmed, n = _trim_all_used(used)
        dev.set_param_map(trimmed, n, rec)
        setup_s = time.perf_counter() - t0
        return dev, n, setup_s

    offs, toks, w, total_w = make_shard(scaling)
    my_tokens = int(offs[-1])
    dev, n, setup_s = make_device(offs, toks, w, total_w)
    info = dev.info()
    x = np.random.RandomState(0).normal(-1.0, 0.3, size=n)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    M = measure(dev, x, args, barrier)
    # the same call when the caller also wants log q of every string (ks_strings runs on demand, 8 B per string go back)
    lq_s = 0.0
    for i in range(min(args.steps, 5)):
        dev.l2_flush()
        dev.rank_barrier()
        dev.sync()
        t0 = time.perf_counter()
        ll_q, lq, g_q = dev.eval(x, want_logq=True)
        lq_s += time.perf_counter() - t0
    lq_ms = lq_s * 1e3 / min(args.steps, 5)
    barrier()
    assert ll_q == M["ll"] and np.array_equal(g_q, M["grad"])
    logq_all = lq
    if args.dump_outputs and world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, lq)
        logq_all = np.concatenate(parts)
    # self check on every run, any number of ranks: the log-likelihood never went through the per-string values, and with
    # N > 1 it went through the exchange over peer memory -- compare it with sum_s p_s log q_s over all ranks
    ll_strings = all_sum([float(np.dot(w / total_w, lq))])[0]
    ll_check = abs(ll_strings - M["ll"]) <= 1e-11 * abs(M["ll"])
    assert ll_check, (ll_strings, M["ll"])
    tok_total = all_sum([float(my_tokens)])[0]
    ms_max, e2e_max, kms_max = all_max([M["ms"], M["e2e_s"], M["kms"]])
    phases_all, inker_all = [M["phases"]], [M["in_kernel_us"]]
    if world > 1:
        ph = torch.tensor(M["phases"] + M["in_kernel_us"], dtype=torch.float64, device="cuda")
        allph = [torch.zeros_like(ph) for _ in range(world)]
        dist.all_gather(allph, ph)
        phases_all = [p.tolist()[:3] for p in allph]
        inker_all = [p.tolist()[3:] for p in allph]
    if ms_max < 600.0:
        # the timed regions are shorter than nvidia-smi's sampling period: keep the same load running (untimed)
        # for ~0.6 s so that `clocks` describes the GPU under this workload.  Every rank runs the same number of
        # evaluations (they contain a collective), derived from the all-reduced step time.
        extra = int(min(20000, max(50, 600.0 / max(ms_max / args.steps, 1e-3))))
        for i in range(extra):
            dev.eval_launch()
            if i % 200 == 199:
                dev.sync()
        dev.sync()
        barrier()
    clocks = sampler.stop() if rank == 0 else None
    n_local_strings = len(w)
    dev.close()

    # ---- extra measurements (untimed by the driver's contract, reported as additional keys)
    extra_keys = {}
    if world > 1 and not args.no_extra:
        # weak scaling: 1M strings per GPU
        other = "weak" if scaling == "strong" else "strong"
        o2, t2, w2, tw2 = make_shard(other)
        dev2, n2, _ = make_device(o2, t2, w2, tw2)
        x2 = np.random.RandomState(0).normal(-1.0, 0.3, size=n2)
        barrier()
        M2 = measure(dev2, x2, args, barrier, want_e2e=False)
        tok2 = all_sum([float(int(o2[-1]))])[0]
        ms2 = all_max([M2["ms"]])[0]
        extra_keys[other] = {"value": tok2 * args.steps / (ms2 * 1e-3), "unit": UNIT, "ms_per_step": ms2 / args.steps,
                             "strings_per_gpu": len(w2), "symbols_total": tok2, "scaling": other}
        dev2.close()
    if world == 1 and not args.no_extra and args.config == "c4":
        # the GPU arm on the SAME bounded sample the reference arm runs (--impl reference: 8 000 strings), so that one
        # ratio compares like with like
        o3, t3, w3 = model.corpus(args.ref_strings, 32, 128, seed=1235)
        dev3, n3, _ = make_device(o3, t3, w3, float(w3.sum()))
        x3 = np.zeros(n3)
        M3 = measure(dev3, x3, args, barrier)
        extra_keys["same_config_as_reference"] = {
            "strings": args.ref_strings, "symbols": int(o3[-1]), "value": int(o3[-1]) * args.steps / (M3["ms"] * 1e-3), "unit": UNIT,
            "ms_per_step": M3["ms"] / args.steps, "e2e_value": int(o3[-1]) * args.steps / M3["e2e_s"], "e2e_ms_per_step": M3["e2e_s"] * 1e3 / args.steps}
        dev3.close()

    if rank == 0:
        steps = args.steps
        value = tok_total * steps / (ms_max * 1e-3)
        e2e = tok_total * steps / e2e_max
        peak, peak_src = peaks()
        # SURVEY 8(d): tokens + per string (int32 offset, FP64 p_s in, FP64 log q_s out) + gradient + automaton;
        # the segmented path does not write log q_s unless asked (not asked here), so those 8 B are not counted
        alg_bytes = 4.0 * my_tokens + (12.0 if info["kernel"] == 6 else 20.0) * n_local_strings + 8.0 * n + float(info["table_bytes"])
        a_lat = None
        if info["kernel"] in (2, 7):
            # CTA-per-string kernel: the alpha lattice of a string does not fit on chip; SURVEY 8(d) charges 16 B per
            # live alpha entry (8 B written by the forward sweep, 8 B read back).  The kernel keeps one entry per
            # candidate state of the position's symbol (exactly max_candidates for the synthetic config 5).
            a_lat = float(info["max_candidates"]) * my_tokens
            alg_bytes += 16.0 * a_lat
        k_ms = kms_max / max(M["klaunches"], 1)
        achieved = alg_bytes / (k_ms * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp) and info["kernel"] == 6 and args.config == "c4" and args.strings == 1000000 and world == 1:
            try:                      # ncu capture of exactly this workload (the evaluation kernel, one launch)
                traffic = json.load(open(tp)).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        single = bool(info["eval_path"] & 1)
        kname = {1: "k2_fwdbwd", 2: "k3_fwdbwd", 3: "kg_fwdbwd", 4: "kt_fwdbwd", 5: "kl_fwdbwd", 6: "k_eval6" if single else "kr_regions",
                 7: "k7_fwd + k7_bwd (one launch each per position)"}[info["kernel"]]
        collective = "none"
        if world > 1:
            collective = ("exchange of [loglik, per-edge sums] (exact 64-bit integers) through NVLink peer memory inside the evaluation kernel"
                          if info["eval_path"] & 2 else "ncclAllReduce(uint64 sum) of [loglik, per-edge sums] per step")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": args.warmup,
            "ms_per_step": ms_max / steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "config %s: synthetic WFSA %d states / %d symbols / %d combined arcs, %d strings of length 32-128 %s"
                                   % (args.config[1:], cfg["n_states"], cfg["n_sym"], info["n_arcs"], n_strings,
                                      "per GPU" if scaling == "weak" else "in total, cut into %d ranges of equal symbol count" % world),
                       "strings_per_gpu": n_local_strings, "symbols_per_gpu": my_tokens, "symbols_total": tok_total, "parameters": n,
                       "kernel": {1: "K2 warp-per-string", 2: "K3 CTA-per-string", 3: "generic", 4: "KT thread-per-string (+ warp-per-string for overflow strings)",
                                  5: "KL thread-per-string over compiled lattices (+ warp-per-string for overflow strings)",
                                  7: "K7 position-synchronous, pair-batched: all strings of a batch advance one position per launch, grouped by symbol pair; "
                                     "alpha lattice of the batch resident in HBM (%d batch(es))" % info["pool_slots"],
                                  6: "segmented compiled lattices: forward-backward over the distinct region types (thread per type), "
                                     + ("weights, region types, grid barrier, fold and rank exchange in ONE persistent launch (k_eval6); " if single else "kr_regions + fold kernels; ")
                                     + "bridge edges are folded into constants when the corpus is compiled; log q per string (ks_strings) only on request"}[info["kernel"]],
                       "accumulators": {1: "shared memory (64-bit fixed point)", 2: "global REDs (64-bit fixed point)"}[info["accum_mode"]],
                       "grid": info["grid"], "block": info["block"], "smem_bytes": info["smem_bytes"],
                       **({"lattice": {"edges": info["lattice_edges"], "bridge_edges": info["lattice_bridge_edges"],
                                       "stream_words": info["lattice_words"], "overflow_strings": info["n_overflow_strings"],
                                       "pool_slots": info["pool_slots"]}} if info["kernel"] >= 5 else {}),
                       **({"segments": {"region_types": info["seg_types"], "region_instances": info["seg_region_instances"],
                                        "region_edges": info["seg_region_edges"], "type_edges": info["seg_type_edges"]}} if info["kernel"] == 6 else {}),
                       "l2_policy": "L2 flushed between timed evaluations (memset of 2x the L2 size on the evaluation stream, outside the "
                                    "per-evaluation event pairs; with N > 1 followed by a device-side barrier over the ranks, also outside); ms_per_step = sum of the event pairs / steps",
                       "bracket_ms_incl_flush": M["bracket_ms"],
                       "collective": collective,
                       "seeds": {"automaton": cfg["seed"], "strings": 1235}},
            # one-time cost per parameter map, outside the metric: structural pass on the device + corpus compile on the host cores
            "setup": {"structure_plus_set_param_map_s": setup_s, "corpus_compile_host_ms": info["seg_host_ms"] if info["kernel"] in (6, 7) else None},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "dram_frac": (traffic / (k_ms * 1e-3) / 1e9 / peak) if traffic else None,
                         "peak_source": peak_src, "kernel": kname,
                         "kernel_ms": k_ms, **({"alpha_lattice_entries": a_lat} if a_lat else {}),
                         "algorithmic_bytes_per_launch": alg_bytes,
                         "kernel_share_of_step": kms_max / max(ms_max, 1e-9),
                         # per rank, us per step: CUDA events [start of the evaluation -> kernel, kernel, kernel -> end]
                         "phases_us_per_rank": [[round(1e3 * v / steps, 2) for v in p] for p in phases_all],
                         # per rank, us per step, globaltimer stamps of CTA 0 inside k_eval6: [arc weights, region types, wait at
                         # the grid barrier, fold + rank exchange + conversion]
                         **({"in_kernel_us_per_rank": [[round(v, 2) for v in p] for p in inker_all]} if single else {})},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": 8 * (n + 1), "d2h_bytes_per_step": 8 * (n + 3),
                    "ms_per_step": e2e_max * 1e3 / steps, "with_logq_ms_per_step": lq_ms,
                    "with_logq_d2h_bytes_per_step": 8 * (n + 3) + 8 * n_local_strings,
                    "call": "wfsa_dev_eval(x, &loglik, NULL, grad) with host buffers" + (": one CUDA graph launch of ONE kernel node -- CTA 0 of k_eval6 fetches x from the mapped pinned staging buffer and publishes it to the grid, the kernel writes [loglik, grad] and a completion word straight into mapped pinned host memory, the host polls that word" if single else "")},
            "gpu_launches": int(M["launches"]),
            "self_check": {"loglik_vs_sum_p_logq_all_ranks": bool(ll_check), "resident_vs_host_buffer_bitwise": True},
            **extra_keys,
            **({"INVALID": "--noacc timing experiment: gradient accumulation skipped"} if args.noacc else {}),
            **({"INVALID": "--no-flush timing experiment: L2 warm from the previous step"} if args.no_flush else {}),
            "clocks": clocks,
            "loglik": M["ll"],
        }
        if world == 1 and not args.no_cpu and args.config == "c4":
            line["cpu_baseline"] = cpu_baseline(model)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, M["ll"], M["grad"], logq_all)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--strings", type=int, default=1000000, help="strings per GPU (weak) or in total (strong)")
    ap.add_argument("--scaling", default=None, choices=["weak", "strong"], help="default: weak at N = 1, strong (the 1M-string corpus cut into N ranges) at N > 1")
    ap.add_argument("--no-extra", action="store_true", help="skip the additional measurements (the other scaling mode at N > 1; the reference-sized sample at N = 1)")
    ap.add_argument("--kernel", type=int, default=0)
    ap.add_argument("--accum", type=int, default=0)
    ap.add_argument("--variant", type=int, default=0)
    ap.add_argument("--config", default="c4", choices=["c4", "c5"], help="BASELINE.json config 4 (default, the metric's workload) or 5")
    ap.add_argument("--K", type=int, default=0, help="thread-per-string kernel: active-set capacity per string (0 = default 12)")
    ap.add_argument("--threads", type=int, default=0, help="compiled-lattice kernel: threads per CTA (0 = as many as fit, <= 1024)")
    ap.add_argument("--replicas", type=int, default=0, help="copies of the global accumulators (0 = library default)")
    ap.add_argument("--noacc", action="store_true", help="timing experiment: skip gradient accumulation (INVALID as a result)")
    ap.add_argument("--no-flush", action="store_true", help="experiment: do not evict the L2 between steps (INVALID as a result)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--ref-strings", type=int, default=8000, help="--impl reference: strings in the bounded sample")
    ap.add_argument("--cpu-strings", type=int, default=20000)
    ap.add_argument("--cpu-port", action="store_true", help="--impl reference: time the CPU port instead of oracle/_ref")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write loglik, grad and log q per string of the last timed step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs: only the GPU arm (--impl ours) has outputs to write")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank, world, local = dist_env()
    if world == 1 and args.gpus > 1 and args.impl == "ours":
        # launched without torchrun: re-launch one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local)


if __name__ == "__main__":
    main()
