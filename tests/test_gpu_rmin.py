"""The smallest path posterior (the rmin column of the optimisers) on every kernel, without path blocks and without
enumerating paths: wfsa_dev_hessian(h, x, NULL, &rmin) runs a forward sweep in the (min, +) semiring over the lattice of
the evaluation; the CPU computes the same from tests/minpath_oracle.c and the oracle's forward-backward."""
import ctypes as C
import gc
import math
import os
import subprocess

import numpy as np
import pytest

import wfsa_b200 as W
from helpers import fnum, golden_to_mine, good_cases, key
import minpath_oracle as MP
from oracle import oracle as O
from wfsa_b200 import synth

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
EXE = os.path.join(os.path.dirname(HERE), "w-fsa_b200", "_build", "wfsa")


def rmin_call(dev, x, with_hf=False):
    """(return code, rmin) of wfsa_dev_hessian(h, x, Hf or NULL, &rmin)."""
    xx = np.ascontiguousarray(x, dtype=np.float64)
    rm = C.c_double(-1.0)
    H = np.zeros((dev.n, dev.n)) if with_hf else None
    rc = dev.L.wfsa_dev_hessian(dev.h, W._p(xx, W.F64P), W._p(H, W.F64P), C.byref(rm))
    return rc, rm.value


def mapped_device(low, **kw):
    dev = W.Device(low, **kw)
    rec, pc, used = dev.structure()
    params = np.concatenate([low.trans_param, low.emis_param])
    trimmed, n, _ = O.trim(low, np.array([r < 0 or used[r] for r in params]))
    dev.set_param_map(trimmed, n, rec)
    return dev, trimmed, n


def oracle_rmin(low, trimmed, x):
    ltw, lew = low.edge_logweights(x, trimmed)
    return MP.rmin(low, ltw, lew)


def synth_low(n_states, n_sym, n_succ, n_emis, seed, n_strings, lmin, lmax):
    low = synth.make_model(n_states, n_sym, n_succ, n_emis, seed=seed).lowered()
    offs, toks, w = synth.make_model(n_states, n_sym, n_succ, n_emis, seed=seed).corpus(n_strings, lmin, lmax, seed=seed + 1)
    low.set_tokens(offs, toks, w / w.sum())
    return low


@pytest.fixture(scope="module")
def c4():
    return synth_low(256, 64, 8, 4, 31, 600, 64, 128)


@pytest.mark.parametrize("kernel", [1, 2, 3, 4, 6, 7])
@pytest.mark.parametrize("mu,sigma", [(-1.0, 0.3), (-3.0, 1.0)])
def test_every_kernel_without_blocks(c4, kernel, mu, sigma):
    """At x ~ N(-3, 1) and strings of up to 128 symbols single path weights fall below 1e-308: only a log-domain minimum
    is right there."""
    dev, trimmed, n = mapped_device(c4, force_kernel=kernel, count=300 if kernel == 3 else None)
    assert dev.info()["kernel"] == kernel
    x = np.random.RandomState(kernel).normal(mu, sigma, size=n)
    rc, rm = rmin_call(dev, x)
    assert rc == 0, dev.L.wfsa_dev_last_error(dev.h).decode()
    low = c4
    if kernel == 3:
        low = W.Lowered.__new__(W.Lowered); low.__dict__.update(c4.__dict__)
        low.set_tokens(c4.offsets[:301], c4.tokens[:c4.offsets[300]], c4.p[:300])
    ref = oracle_rmin(low, trimmed, x)
    assert 0.0 < ref < 1e-3 and abs(rm - ref) <= 1e-12 * ref, (rm, ref)
    ll, _, _ = dev.eval(x, want_logq=False)                   # the evaluation after an rmin call is the usual one
    assert math.isfinite(ll)
    dev.close()


def golden_eval_cases():
    out = []
    for case in good_cases(("random",)):
        for i, ev in enumerate(case.get("evals", [])):
            out.append(pytest.param(case, ev, id="%s-x%d" % (case["name"], i)))
    return out


@pytest.mark.parametrize("kernel", [2, 3])
@pytest.mark.parametrize("case,ev", golden_eval_cases())
def test_golden_posteriors(case, ev, kernel):
    """The reference's own path posteriors (multi-token and empty emissions: the generic kernel's MODE_MINPATH)."""
    low = W.Lowered(W.parse(case["fsa_text"], case["corpus_text"]))
    try:
        dev, trimmed, n = mapped_device(low, force_kernel=kernel)
    except W.WfsaError as e:
        assert kernel == 2 and "fast kernel" in e.message
        pytest.skip("emissions of other than one token: no fast tables")
    params = np.concatenate([low.trans_param, low.emis_param])
    mine = {key(e): (trimmed[r] if r >= 0 else -1) for e, r in zip(low.edges, params)}
    perm = np.full(case["n"], -1, dtype=np.int64)
    for e in case["edges"]:
        if e["trimmed"] >= 0:
            perm[e["trimmed"]] = mine[key(e)]
    x = np.zeros(n)
    x[perm] = [fnum(v) for v in ev["x"]]
    rc, rm = rmin_call(dev, x)
    assert rc == 0, dev.L.wfsa_dev_last_error(dev.h).decode()
    ref = min((fnum(v) for v in ev["r"]), default=1.0)
    assert abs(rm - ref) <= 1e-12 * ref, (rm, ref)
    dev.close()


def test_config5_true_shape():
    """BASELINE config 5 at its named shape, several K7 batches: K7's sweep equals the oracle and the CTA-per-string
    kernel (the same sums and minima in the same order)."""
    low = synth_low(4096, 256, 64, 16, 4321, 300, 32, 128)
    os.environ["WFSA_K7_ROWS"] = "9000"
    try:
        dev7, trimmed, n = mapped_device(low, force_kernel=7)
    finally:
        os.environ.pop("WFSA_K7_ROWS", None)
    assert dev7.info()["kernel"] == 7 and dev7.info()["pool_slots"] >= 2
    dev3, trimmed3, n3 = mapped_device(low, force_kernel=2)
    assert n3 == n and np.array_equal(trimmed3, trimmed)
    for seed, (mu, sigma) in enumerate([(-1.0, 0.3), (-3.0, 1.0)]):
        x = np.random.RandomState(seed).normal(mu, sigma, size=n)
        rc7, r7 = rmin_call(dev7, x)
        rc3, r3 = rmin_call(dev3, x)
        assert rc7 == 0 and rc3 == 0
        ref = oracle_rmin(low, trimmed, x)
        assert abs(r7 - ref) <= 1e-12 * ref and abs(r7 - r3) <= 1e-13 * r3, (r7, r3, ref)
    dev7.close(); dev3.close()


def test_segmented_overflow_strings():
    """Kernel 6 with four pool slots: the strings that overflow them run on the secondary kernel and are not in the
    per-string layout; the sweep takes them into rmin.  The corpus is chosen so that one of them holds the minimum."""
    model = synth.make_model(256, 64, 8, 4, seed=21)
    low = model.lowered()
    offs, toks, w = model.corpus(3000, 32, 128, seed=22)
    low.set_tokens(offs, toks, w / w.sum())
    _, _, ee0 = O.dp_eval(low, np.zeros(low.n_trans), np.zeros(low.n_emis))
    trimmed, n, _ = O.trim(low, ee0 > 0)
    seg = W.segmented_compile(low, trimmed, n_slots=4)
    over = sorted(set(seg["overflow"].tolist()) | set(seg["rejected"].tolist()))
    keep = over + [s for s in range(3000) if s not in set(over)][:60]            # the overflow strings and 60 others
    o2, t2 = [0], []
    for s in keep:
        t2.extend(toks[offs[s]:offs[s + 1]]); o2.append(len(t2))
    low.set_tokens(np.array(o2), np.array(t2, dtype=np.int32), w[keep] / w[keep].sum())
    dev, trimmed, n = mapped_device(low, force_kernel=6, accum_variant=4 << 16)
    assert dev.info()["n_overflow_strings"] == len(over) > 0
    x = np.random.RandomState(0).normal(-1.0, 0.3, size=n)
    ltw, lew = low.edge_logweights(x, trimmed)
    _, lq, _ = O.dp_eval(low, ltw, lew, want_grad=False)
    m = MP.dp_minpath(low, ltw, lew)
    assert int(np.argmin(m - lq)) < len(over)                                   # precondition: an overflow string
    rc, rm = rmin_call(dev, x)
    ref = oracle_rmin(low, trimmed, x)
    assert rc == 0 and abs(rm - ref) <= 1e-12 * ref, (rm, ref)
    dev.close()


def test_segmented_region_types_beyond_the_block_limit():
    """Eight emissions per state: region types with more than 2^20 paths, no H_f blocks.  rmin alone is a sweep over every
    string; H_f still needs the blocks."""
    low = synth_low(256, 64, 8, 8, 1, 1500, 32, 128)
    dev, trimmed, n = mapped_device(low, force_kernel=6)
    x = np.random.RandomState(3).normal(-1.0, 0.3, size=n)
    rc, rm = rmin_call(dev, x)
    assert rc == 0, dev.L.wfsa_dev_last_error(dev.h).decode()
    ref = oracle_rmin(low, trimmed, x)
    assert abs(rm - ref) <= 1e-12 * ref, (rm, ref)
    rc, _ = rmin_call(dev, x, with_hf=True)
    assert rc == 6                                                              # WFSA_ERR_LIMIT
    rc, rm2 = rmin_call(dev, x)
    assert rc == 0 and rm2 == rm
    dev.close()


def qn_runs():
    out = []
    for case in good_cases():
        for run in case.get("runs", []):
            if "reference_error" in run or run["optimizer"] != "QuasiNewton":
                continue
            for k in (2, 3):
                out.append(pytest.param(case, run, k, id="%s-i%d-e%d-k%d" % (case["name"], run["flags"], run["epochs"], k)))
    return out


@pytest.mark.parametrize("case,run,kernel", qn_runs())
def test_quasinewton_trajectory_forced_kernel(case, run, kernel):
    """The golden QuasiNewton runs on the CTA-per-string and the generic kernel: their rmin column comes from the sweep."""
    try:
        s = W.Session(case["fsa_text"], case["corpus_text"], "QuasiNewton", force_kernel=kernel)
    except W.WfsaError as e:
        assert kernel == 2 and "fast kernel" in e.message
        pytest.skip("emissions of other than one token: no fast tables")
    perm = golden_to_mine(case, s.describe()["edges"])
    s.init(run["flags"])
    ref_rows = run["trajectory"]
    n_cmp = len(ref_rows) - (1 if run["error"] else 0)
    for row in ref_rows[:n_cmp]:
        info = s.step(run["eta"])
        ref = [fnum(v) for v in row["info"]]
        for c in [0, 1, 2, 3, 4]:
            assert math.isclose(info[c], ref[c], rel_tol=2e-6, abs_tol=2e-8), (row["epoch"], c, info[c], ref[c])
        if not case["unique_paths"]:
            assert math.isclose(info[5], ref[5], rel_tol=2e-6, abs_tol=1e-12), ("rmin", row["epoch"], info[5], ref[5])
        if "x" in row:
            assert np.allclose(s.x()[perm], np.array([fnum(v) for v in row["x"]][:case["n"]]), rtol=1e-6, atol=1e-6), row["epoch"]
        if s.halt(run["tol"]) and run["tol"] > 0:
            break
    s.close()


@pytest.fixture(scope="module")
def dense_files(tmp_path_factory):
    """1024 states / 64 symbols / 16 successors / 8 emissions: ~131 k combined arcs (beyond the segmented kernel), two
    paths per position on average, 2 000 strings of 32..64 symbols: far more paths than any enumeration could list."""
    model = synth.make_model(1024, 64, 16, 8, seed=5)
    offs, toks, w = model.corpus(2000, 32, 64, seed=6)
    d = tmp_path_factory.mktemp("dense")
    fsa, corpus = d / "dense.wfsa", d / "dense.corpus"
    fsa.write_text(model.text())
    corpus.write_text(model.corpus_text(offs, toks, w))
    return str(fsa), str(corpus)


def test_quasinewton_on_dense_automaton(dense_files):
    fsa, corpus = dense_files
    fsa_text, corpus_text = open(fsa).read(), open(corpus).read()
    low = W.Lowered(W.parse(fsa_text, corpus_text))
    dev = W.Device(low)
    assert dev.info()["kernel"] == 2                   # the shape the CLI gets (it cannot force a kernel)
    rec, pc, _ = dev.structure()
    assert rec.all() and pc[pc > 1].sum() > 1e9
    dev.close()
    # full precision through the Session (the same Learner): rmin of epoch 1 at the initial x
    s = W.Session(fsa_text, corpus_text, "QuasiNewton")
    mine = {key(e): e["trimmed"] for e in s.describe()["edges"]}
    trimmed = np.full(low.n_raw, -2, dtype=np.int32)
    for e in low.edges:
        if e["raw"] >= 0:
            trimmed[e["raw"]] = mine[key(e)]
    s.init(7)
    x0 = s.x()
    info = s.step(1.0)
    ref = oracle_rmin(low, trimmed, x0)
    assert 0.0 < ref < 1.0 and abs(info[5] - ref) <= 1e-9 * ref, (info[5], ref)
    s.close()
    r = subprocess.run([EXE, "-a", fsa, "-c", corpus, "-opt", "QuasiNewton", "-i", "7", "-e", "3"], capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stderr[-3000:]
    rows = [ln.split() for ln in r.stderr.splitlines() if ln[:1].isdigit() and "\t" in ln]
    assert len(rows) == 3, r.stderr[-3000:]
    assert math.isclose(float(rows[0][6]), ref, rel_tol=1e-2)        # (printed with three significant digits)


def test_quasinewton_on_dense_automaton_two_gpus(dense_files):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    fsa, corpus = dense_files
    tables = []
    for gpus in (1, 2):
        r = subprocess.run([EXE, "-a", fsa, "-c", corpus, "-opt", "QuasiNewton", "-i", "7", "-e", "3", "--gpus", str(gpus)],
                           capture_output=True, text=True, timeout=1800)
        assert r.returncode == 0, r.stderr[-3000:]
        tables.append([ln.split() for ln in r.stderr.splitlines() if ln[:1].isdigit() and "\t" in ln])
    assert len(tables[0]) == 3 and tables[0] == tables[1]


def held_bytes():
    gc.collect()
    return W.lib().wfsa_dev_held_bytes()


@pytest.mark.parametrize("kernel", [2, 7])
def test_rmin_buffers_are_given_back(c4, kernel):
    held = held_bytes()
    dev, trimmed, n = mapped_device(c4, force_kernel=kernel)
    x = np.random.RandomState(1).normal(-1.5, 0.8, size=n)
    dev.eval(x)
    rc, rm = rmin_call(dev, x)
    assert rc == 0 and 0.0 < rm <= 1.0
    dev.close()
    assert held_bytes() == held
