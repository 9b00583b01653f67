"""Path sampling on the device (wfsa_dev_sample / wfsa_dev_viterbi_paths): draws from the path posterior of every string on
every kernel.  Every draw is a valid path whose value is the left-to-right sum of its steps, bit for bit; log q is the
evaluation's; the draws are a function of (x, seed, string, draw) only (prefixes, determinism, the same bits on every
handle with fast tables, the CPU reference's draws without them); their distribution is the posterior (chi-square against
N-best posteriors where every path is known, Monte-Carlo expected counts against the gradient on long strings, the
reference's posteriors on the golden cases); no effect on the evaluation, memory, error codes and the CLI's --sample."""
import gc
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

import maxpath_oracle as MX
import sample_oracle as SO
import wfsa_b200 as W
from helpers import load_cases
from oracle import oracle as O
from test_cpu_sample import check_case_sample, chi2_terms
from test_cpu_viterbi import CASES
from test_gpu_nbest import same_bits, sub_corpus
from test_gpu_rmin import mapped_device, synth_low
from test_gpu_viterbi import as_paths, check_valid_path

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
EXE = os.path.join(os.path.dirname(HERE), "w-fsa_b200", "_build", "wfsa")


@pytest.fixture(scope="module")
def c4():
    return synth_low(256, 64, 8, 4, 31, 600, 64, 128)


def steps_of(res):
    logw, logq, off, tr, em = res
    return as_paths(off, tr, em)


def check_draws(low, trimmed, x, res):
    """Every draw of a string with a path is a valid path and the left-to-right sum of its steps; the others have none."""
    logw, logq, off, tr, em = res
    ns, n = logw.shape
    ltw, lew = low.edge_logweights(x, trimmed)
    paths = steps_of(res)
    assert len(paths) == ns * n
    for s in range(ns):
        assert (logw[s] == -np.inf).all() == (logq[s] == -np.inf), s
        for r in range(n):
            p = paths[s * n + r]
            if logw[s, r] == -np.inf:
                assert p == [], (s, r)
                continue
            check_valid_path(low, s, p)
            assert MX.path_logweight(p, ltw, lew) == logw[s, r], (s, r)       # the summation-order identity, bit for bit


@pytest.fixture(scope="module")
def c4_runs(c4):
    """Per kernel and scale of x: the handle's evaluation log q, the kernel-2 evaluation's log q, and draws at n = 4 / 32
    under seed 7 (twice at 32) and n = 32 under seed 8."""
    out = {}
    for mu, sigma in [(-1.0, 0.3), (-3.0, 1.0)]:
        for kernel in [2, 1, 3, 4, 6, 7]:
            dev, trimmed, n = mapped_device(c4, force_kernel=kernel, count=300 if kernel == 3 else None)
            assert dev.info()["kernel"] == kernel
            x = np.random.RandomState(17).normal(mu, sigma, size=n)
            _, lq, _ = dev.eval(x)
            out[kernel, mu] = dict(x=x, trimmed=trimmed, lq=lq, s4=dev.sample(x, 4, 7), s32=dev.sample(x, 32, 7),
                                   again=dev.sample(x, 32, 7), other=dev.sample(x, 32, 8))
            dev.close()
            if kernel == 3:                         # the same 300 strings on a K3 handle
                dev, trimmed2, n2 = mapped_device(c4, force_kernel=2, count=300)
                assert np.array_equal(trimmed2, trimmed)
                out[kernel, mu]["k3"] = dev.sample(x, 32, 7)
                dev.close()
    return out


@pytest.mark.parametrize("kernel", [1, 2, 3, 4, 6, 7])
@pytest.mark.parametrize("mu", [-1.0, -3.0])
def test_every_kernel(c4, c4_runs, kernel, mu):
    """At x ~ N(-3, 1) path weights of strings of up to 128 symbols fall below 1e-308: the sweep rescales, the values are
    log-domain sums.  The automaton has fast tables, so every handle (the generic kernel 3 too) samples with k3_sample and
    returns the same bits."""
    run = c4_runs[kernel, mu]
    low = sub_corpus(c4, 300) if kernel == 3 else c4
    x, trimmed, s32 = run["x"], run["trimmed"], run["s32"]
    logw, logq = s32[0], s32[1]
    assert np.isfinite(logw[:, 0]).sum() > len(logw) // 2
    check_draws(low, trimmed, x, s32)
    ok = np.isfinite(run["lq"])
    assert np.array_equal(np.isfinite(logq), ok)
    assert np.all(np.abs(logq[ok] - run["lq"][ok]) <= 1e-12 * np.abs(run["lq"][ok]))
    if kernel != 3:
        assert same_bits(logq, c4_runs[2, mu]["lq"])                          # K3's log q, to the last bit
    s4 = run["s4"]
    assert same_bits(s4[0], s32[0][:, :4]) and same_bits(s4[1], s32[1])
    p4, p32 = steps_of(s4), steps_of(s32)
    assert all(p4[s * 4 + r] == p32[s * 32 + r] for s in range(len(logw)) for r in range(4))
    assert all(same_bits(a, b) for a, b in zip(s32, run["again"]))            # the same seed: the same bits
    assert steps_of(run["other"]) != p32                                       # another seed: other draws
    same = c4_runs[2, mu]["s32"] if kernel != 3 else run["k3"]                 # every handle with fast tables: the same bits
    assert all(same_bits(a, b) for a, b in zip(s32, same))


def test_short_strings_against_nbest():
    """Strings of 4..12 symbols, most with 2..16 paths: nbest(x, 16) lists every path of those; every draw is one of them
    with its N-best value bit for bit, and the draw counts pass chi-square against exp(logw_nbest - log q), on every kernel."""
    low = synth_low(256, 64, 8, 4, 91, 400, 4, 12)
    for kernel in [1, 2, 3, 4, 6, 7]:
        dev = W.Device(low, force_kernel=kernel)
        rec, pc, used = dev.structure()
        params = np.concatenate([low.trans_param, low.emis_param])
        trimmed, n, _ = O.trim(low, np.array([r < 0 or used[r] for r in params]))
        dev.set_param_map(trimmed, n, rec)
        x = np.random.RandomState(4).normal(-1.0, 0.5, size=n)
        nb_w, nb_off, nb_tr, nb_em = dev.nbest(x, 16)
        nb_p = as_paths(nb_off, nb_tr, nb_em)
        sel = [s for s in range(len(pc)) if 2 <= pc[s] <= 16]
        assert len(sel) > 100, len(sel)
        stat, dof = 0.0, 0
        obs = {s: {} for s in sel}
        for seed in range(4):
            res = dev.sample(x, 256, seed)
            logw, logq = res[0], res[1]
            paths = steps_of(res)
            for s in sel:
                known = {tuple(nb_p[s * 16 + r]): nb_w[s, r] for r in range(16) if nb_w[s, r] > -np.inf}
                for r in range(256):
                    p = tuple(paths[s * 256 + r])
                    assert p in known, (kernel, s, r)
                    assert logw[s, r] == known[p], (kernel, s, r)
                    obs[s][p] = obs[s].get(p, 0) + 1
        for s in sel:
            want = {tuple(nb_p[s * 16 + r]): np.exp(nb_w[s, r] - logq[s]) for r in range(16) if nb_w[s, r] > -np.inf}
            t, f = chi2_terms(obs[s], want, 4 * 256)
            stat += t; dof += f
        assert dof > 100 and stats.chi2.sf(stat, dof) >= 1e-6, (kernel, stat, dof)
        dev.close()


def mc_gradient(low, trimmed, n_par, res):
    """-sum_s p_s (1/n) sum_r c_i(pi_sr) over the trimmed parameters, from the draws."""
    logw, logq, off, tr, em = res
    ns, n = logw.shape
    sid = np.repeat(np.repeat(np.arange(ns), n), np.diff(off))
    wt = np.asarray(low.p[:ns])[sid] / n
    tp = np.asarray(low.trans_param)[tr]
    ep = np.where(em >= 0, np.asarray(low.emis_param)[np.maximum(em, 0)], -1)
    out = np.zeros(n_par)
    for p in (tp, ep):
        tt = np.where(p >= 0, np.asarray(trimmed)[np.maximum(p, 0)], -1)
        m = tt >= 0
        out -= np.bincount(tt[m], weights=wt[m], minlength=n_par)
    return out


def check_mc_gradient(low, trimmed, n_par, x, g, res):
    logw = res[0]
    n = logw.shape[1]
    ok = np.isfinite(logw[:, 0])
    lens = np.diff(np.asarray(low.offsets[:len(logw) + 1]))
    pmax = float(np.asarray(low.p[:len(logw)])[ok].max())
    lmax = int(lens.max()) + 1
    gh = mc_gradient(low, trimmed, n_par, res)
    bound = 6.0 * np.sqrt(pmax * lmax * np.abs(g) / n)
    assert np.all(np.abs(gh - g) <= bound + 1e-15), np.argsort(-(np.abs(gh - g) - bound))[:5]


@pytest.mark.parametrize("kernel", [1, 2, 3, 4, 6, 7])
def test_expected_counts_match_gradient(c4, kernel):
    """Long strings, no enumeration: the Monte-Carlo expected counts of 64 draws per string agree with the evaluation's
    gradient within 6 standard deviations (the variance bounded through c_i <= L_max)."""
    dev, trimmed, n = mapped_device(c4, force_kernel=kernel, count=300 if kernel == 3 else None)
    low = sub_corpus(c4, 300) if kernel == 3 else c4
    x = np.random.RandomState(23).normal(-1.0, 0.3, size=n)
    _, _, g = dev.eval(x)
    check_mc_gradient(low, trimmed, n, x, g, dev.sample(x, 64, 3))
    dev.close()


def test_config5_true_shape():
    """BASELINE config 5 at its named shape (4096 states / 256 symbols: a CTA per string), several K7 batches: the K7
    handle against a forced CTA-per-string handle (same bits), valid draws, and the expected counts against the gradient."""
    low = synth_low(4096, 256, 64, 16, 4321, 300, 32, 128)
    os.environ["WFSA_K7_ROWS"] = "9000"
    try:
        dev7, trimmed, n = mapped_device(low, force_kernel=7)
    finally:
        os.environ.pop("WFSA_K7_ROWS", None)
    assert dev7.info()["kernel"] == 7 and dev7.info()["max_candidates"] > 32
    dev2, trimmed2, n2 = mapped_device(low, force_kernel=2)
    assert n2 == n and np.array_equal(trimmed2, trimmed)
    x = np.random.RandomState(0).normal(-1.0, 0.3, size=n)
    r7, r2 = dev7.sample(x, 64, 5), dev2.sample(x, 64, 5)
    assert all(same_bits(a, b) for a, b in zip(r7, r2))
    _, lq, g = dev7.eval(x)
    ok = np.isfinite(lq)
    assert np.array_equal(np.isfinite(r7[1]), ok) and np.all(np.abs(r7[1][ok] - lq[ok]) <= 1e-12 * np.abs(lq[ok]))
    check_draws(low, trimmed, x, r7)
    check_mc_gradient(low, trimmed, n, x, g, r7)
    dev7.close(); dev2.close()


@pytest.mark.parametrize("kernel", [2, 3])
@pytest.mark.parametrize("case", CASES, ids=lambda c: c["name"])
def test_golden_posteriors(case, kernel):
    """The reference's own path posteriors and counts through the device; without fast tables (multi-token or empty
    emissions) the draws are the CPU reference's."""
    low = W.Lowered(W.parse(case["fsa_text"], case["corpus_text"]))
    inner = [s for s in range(low.n_states) if s not in (low.start, low.end)]
    no_fast = any(low.emis_tok_off[e + 1] - low.emis_tok_off[e] != 1 for s in inner for e in range(low.emis_row[s], low.emis_row[s + 1]))
    if kernel == 2 and no_fast:
        pytest.skip("emissions of other than one token: no fast tables")

    held = {}

    def draw(low, trimmed, x, ltw, lew, n, seed):
        if held.get("x") is None or not np.array_equal(held["x"], x):        # one handle per stored x
            if "dev" in held:
                held["dev"].close()
            held["dev"] = W.Device(low, force_kernel=kernel)
            rec, _, _ = held["dev"].structure()
            held["dev"].set_param_map(trimmed, len(x), rec)
            held["x"] = x.copy()
        res = held["dev"].sample(x, n, seed)
        p = steps_of(res)
        steps = [[tuple(p[s * n + r]) for r in range(n)] for s in range(len(res[0]))]
        if no_fast:
            rq, rw, rp = SO.sample(low, ltw, lew, n, seed)
            assert same_bits(res[0], rw) and steps == [[tuple(q) for q in ps] for ps in rp]
        return res[1], res[0], steps
    try:
        check_case_sample(case, draw)
    finally:
        if "dev" in held:
            held["dev"].close()


@pytest.mark.parametrize("kernel", [2, 3, 6, 7])
def test_evaluation_and_decodes_are_unchanged(c4, kernel):
    """A sample between two evaluations, and between eval_launch and eval_fetch, changes no bit of what the evaluation
    returns; viterbi_paths after a sample gives the sample's steps; a later viterbi / nbest is unchanged."""
    dev, trimmed, n = mapped_device(c4, force_kernel=kernel, count=300 if kernel == 3 else None)
    x = np.random.RandomState(11).normal(-1.0, 0.3, size=n)
    y = np.random.RandomState(12).normal(-2.0, 0.5, size=n)
    ll0, lq0, g0 = dev.eval(x)
    v0, nb0 = dev.viterbi(y), dev.nbest(y, 4)
    res = dev.sample(y, 8, 1)
    ll1, lq1, g1 = dev.eval(x)
    assert ll1 == ll0 and np.array_equal(lq1, lq0) and np.array_equal(g1, g0)
    dev.upload_x(x)
    dev.eval_launch()
    again = dev.sample(y, 8, 1)
    ll2, lq2, g2 = dev.eval_fetch(want_logq=True)
    assert ll2 == ll0 and np.array_equal(lq2, lq0) and np.array_equal(g2, g0)
    assert all(same_bits(a, b) for a, b in zip(res, again))
    tr = np.zeros(max(int(res[2][-1]), 1), dtype=np.int32); em = np.zeros_like(tr)
    assert dev.L.wfsa_dev_viterbi_paths(dev.h, W._p(tr, W.I32P), W._p(em, W.I32P)) == 0
    assert np.array_equal(tr[:res[2][-1]], res[3]) and np.array_equal(em[:res[2][-1]], res[4])
    v1, nb1 = dev.viterbi(y), dev.nbest(y, 4)
    assert all(same_bits(a, b) for a, b in zip(v0, v1)) and all(same_bits(a, b) for a, b in zip(nb0, nb1))
    dev.close()


def held_bytes():
    gc.collect()
    return W.lib().wfsa_dev_held_bytes()


@pytest.mark.parametrize("kernel", [2, 3, 7])
def test_memory_and_errors(c4, kernel):
    held = held_bytes()
    dev = W.Device(c4, force_kernel=kernel, count=300 if kernel == 3 else None)
    L, h = dev.L, dev.h
    logw = np.zeros(dev.n_strings * 256)
    logq = np.zeros(dev.n_strings)
    off = np.zeros(dev.n_strings * 256 + 1, dtype=np.int64)
    x = np.zeros(1)
    F, I = W.F64P, W.I64P
    assert L.wfsa_dev_sample(h, W._p(x, F), 4, 0, W._p(logw, F), W._p(logq, F), W._p(off, I)) == 5   # before set_param_map
    dev.close()
    dev, trimmed, n = mapped_device(c4, force_kernel=kernel, count=300 if kernel == 3 else None)
    L, h = dev.L, dev.h
    x = np.random.RandomState(1).normal(-1.5, 0.8, size=n)
    for k in (0, 257, -1):
        assert L.wfsa_dev_sample(h, W._p(x, F), k, 0, W._p(logw, F), W._p(logq, F), W._p(off, I)) == 1
    assert L.wfsa_dev_sample(h, None, 4, 0, W._p(logw, F), W._p(logq, F), W._p(off, I)) == 1
    assert L.wfsa_dev_sample(h, W._p(x, F), 4, 0, None, W._p(logq, F), W._p(off, I)) == 1
    assert L.wfsa_dev_sample(h, W._p(x, F), 4, 0, W._p(logw, F), W._p(logq, F), None) == 1
    assert L.wfsa_dev_sample(h, W._p(x, F), 4, 0, W._p(logw, F), None, W._p(off, I)) == 0              # logq may be NULL
    dev.eval(x)
    for k in (256, 3):
        lw, lq, off2, tr2, em2 = dev.sample(x, k, 2)
        assert off2[-1] > 0 and np.isfinite(lw[:, 0]).any()
    dev.close()
    assert held_bytes() == held


FIXTURES = [("test3.wfsa", "test.corpus"), ("talk.wfsa", "talk.corpus"), ("test5.wfsa", "test5.corpus"),
            ("test.list.wfsa", "test.corpus"), ("test.loop.wfsa", "test.corpus")]


@pytest.mark.parametrize("fsa,corpus", FIXTURES)
def test_cli_sample_paths_are_reference_paths(fsa, corpus, tmp_path):
    """`wfsa -e 0 -s --sample N S --seed 5 --nbest 4 B`: N lines per corpus string in corpus order, draws numbered from 1,
    every path a -pr line of the reference binary for that word, ratio w/q in (0, 1]; a second run gives the same file; the
    N-best file is written too."""
    name = fsa + "+" + corpus
    case = [c for c in load_cases("fixtures") if c["name"] == name][0]
    (tmp_path / fsa).write_bytes(case["fsa_text"].encode())
    (tmp_path / corpus).write_bytes(case["corpus_text"].encode())
    N = 12
    outs = []
    for i in range(2):
        out, nb = tmp_path / ("sample%d.tsv" % i), tmp_path / ("nbest%d.tsv" % i)
        r = subprocess.run([EXE, "-a", str(tmp_path / fsa), "-c", str(tmp_path / corpus), "-e", "0", "-s", "--sample", str(N),
                            str(out), "--seed", "5", "--nbest", "4", str(nb)], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-3000:]
        assert nb.read_text().count("\n") >= len(case["corpus"])
        outs.append(out.read_text())
    assert outs[0] == outs[1]
    want = set(load_cases("path_listing")[name])
    lines = outs[0].split("\n")
    assert lines[-1] == ""
    i = 0
    for w in case["corpus"]:
        if w["paths"] == 0:
            assert lines[i].split("\t") == [w["word"], "0", "-inf", "0", ""]
            i += 1
            continue
        block = [ln.split("\t") for ln in lines[i:i + N]]
        i += N
        assert [b[0] for b in block] == [w["word"]] * N and [b[1] for b in block] == [str(r + 1) for r in range(N)]
        for b in block:
            assert len(b) == 5 and w["word"] + ": " + b[4] in want, b
            assert 0.0 < float(b[3]) <= 1.0 + 1e-12 and np.isfinite(float(b[2]))
    assert i == len(lines) - 1
