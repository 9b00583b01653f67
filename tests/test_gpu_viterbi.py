"""Viterbi decoding on the device (wfsa_dev_viterbi / wfsa_dev_viterbi_paths): the most probable path of every string on
every kernel, against the CPU reference (tests/maxpath_oracle.c) and the reference's own path posteriors and counts;
determinism, no effect on the evaluation, memory, error codes and the CLI's --viterbi."""
import ctypes as C
import gc
import os
import subprocess

import numpy as np
import pytest

import maxpath_oracle as MX
import wfsa_b200 as W
from helpers import load_cases
from oracle import oracle as O
from test_cpu_viterbi import CASES, check_case_against_reference
from test_gpu_rmin import mapped_device, synth_low

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
EXE = os.path.join(os.path.dirname(HERE), "w-fsa_b200", "_build", "wfsa")


@pytest.fixture(scope="module")
def c4():
    return synth_low(256, 64, 8, 4, 31, 600, 64, 128)


def as_paths(off, tr, em):
    return [list(zip(tr[off[s]:off[s + 1]].tolist(), em[off[s]:off[s + 1]].tolist())) for s in range(len(off) - 1)]


def check_valid_path(low, s, steps):
    """The steps start at start, end at end, and their emissions spell string s."""
    tok = low.tokens[low.offsets[s]:low.offsets[s + 1]].tolist()
    cur, pos = low.start, 0
    for i, (t, e) in enumerate(steps):
        assert low.trans_row[cur] <= t < low.trans_row[cur + 1], (s, i)
        v = int(low.trans_dst[t])
        if i == len(steps) - 1:
            assert e == -1 and v == low.end and pos == len(tok), (s, i)
            return
        assert low.emis_row[v] <= e < low.emis_row[v + 1], (s, i)
        lab = low.emis_tok[low.emis_tok_off[e]:low.emis_tok_off[e + 1]].tolist()
        assert tok[pos:pos + len(lab)] == lab, (s, i)
        pos += len(lab)
        cur = v
    assert False, ("empty path", s)


def check_against_oracle(low, trimmed, x, logw, off, tr, em):
    ltw, lew = low.edge_logweights(x, trimmed)
    ref, _ = MX.viterbi(low, ltw, lew)
    paths = as_paths(off, tr, em)
    for s in range(len(ref)):
        if ref[s] == -np.inf:
            assert logw[s] == -np.inf and off[s + 1] == off[s], s
            continue
        check_valid_path(low, s, paths[s])
        assert MX.path_logweight(paths[s], ltw, lew) == logw[s], s              # the summation-order identity, bit for bit
        assert abs(logw[s] - ref[s]) <= 1e-12 * max(1.0, abs(ref[s])), (s, logw[s], ref[s])


@pytest.mark.parametrize("kernel", [1, 2, 3, 4, 6, 7])
@pytest.mark.parametrize("mu,sigma", [(-1.0, 0.3), (-3.0, 1.0)])
def test_every_kernel(c4, kernel, mu, sigma):
    """At x ~ N(-3, 1) path weights of strings of up to 128 symbols fall below 1e-308: only the log domain is right."""
    dev, trimmed, n = mapped_device(c4, force_kernel=kernel, count=300 if kernel == 3 else None)
    assert dev.info()["kernel"] == kernel
    x = np.random.RandomState(kernel).normal(mu, sigma, size=n)
    logw, off, tr, em = dev.viterbi(x)
    low = c4
    if kernel == 3:
        low = W.Lowered.__new__(W.Lowered); low.__dict__.update(c4.__dict__)
        low.set_tokens(c4.offsets[:301], c4.tokens[:c4.offsets[300]], c4.p[:300])
    assert np.isfinite(logw).sum() > len(logw) // 2
    check_against_oracle(low, trimmed, x, logw, off, tr, em)
    again = dev.viterbi(x)                                                      # determinism: the same bits
    assert all(np.array_equal(a.view(np.uint8), b.view(np.uint8)) for a, b in zip((logw, off, tr, em), again))
    dev.close()


@pytest.mark.parametrize("kernel", [2, 3])
@pytest.mark.parametrize("case", CASES, ids=lambda c: c["name"])
def test_golden_posteriors(case, kernel):
    """The reference's own path posteriors and counts (multi-token and empty emissions: the generic kernel's
    MODE_VITERBI); at x = 0 tied paths are all accepted."""
    def decode(low, trimmed, x, ltw, lew):
        dev = W.Device(low, force_kernel=kernel)
        rec, _, _ = dev.structure()
        dev.set_param_map(trimmed, len(x), rec)
        logw, off, tr, em = dev.viterbi(x)
        dev.close()
        return logw, as_paths(off, tr, em)
    low = W.Lowered(W.parse(case["fsa_text"], case["corpus_text"]))
    inner = [s for s in range(low.n_states) if s not in (low.start, low.end)]
    if kernel == 2 and any(low.emis_tok_off[e + 1] - low.emis_tok_off[e] != 1 for s in inner
                           for e in range(low.emis_row[s], low.emis_row[s + 1])):
        pytest.skip("emissions of other than one token: no fast tables")
    check_case_against_reference(case, decode)


def test_config5_true_shape():
    """BASELINE config 5 at its named shape (4096 states / 256 symbols: a CTA per string), several K7 batches: against
    the oracle, and the K7 handle against a forced CTA-per-string handle (same bits)."""
    low = synth_low(4096, 256, 64, 16, 4321, 300, 32, 128)
    os.environ["WFSA_K7_ROWS"] = "9000"
    try:
        dev7, trimmed, n = mapped_device(low, force_kernel=7)
    finally:
        os.environ.pop("WFSA_K7_ROWS", None)
    assert dev7.info()["kernel"] == 7 and dev7.info()["max_candidates"] > 32
    dev2, trimmed2, n2 = mapped_device(low, force_kernel=2)
    assert n2 == n and np.array_equal(trimmed2, trimmed)
    for seed, (mu, sigma) in enumerate([(-1.0, 0.3), (-3.0, 1.0)]):
        x = np.random.RandomState(seed).normal(mu, sigma, size=n)
        r7, r2 = dev7.viterbi(x), dev2.viterbi(x)
        assert all(np.array_equal(a.view(np.uint8), b.view(np.uint8)) for a, b in zip(r7, r2))
        check_against_oracle(low, trimmed, x, *r7)
    dev7.close(); dev2.close()


@pytest.mark.parametrize("kernel", [2, 3, 6, 7])
def test_evaluation_is_unchanged(c4, kernel):
    """A viterbi call between two evaluations, and between eval_launch and eval_fetch (log q on demand on the segmented
    path), changes no bit of what the evaluation returns."""
    dev, trimmed, n = mapped_device(c4, force_kernel=kernel, count=300 if kernel == 3 else None)
    x = np.random.RandomState(11).normal(-1.0, 0.3, size=n)
    y = np.random.RandomState(12).normal(-2.0, 0.5, size=n)
    ll0, lq0, g0 = dev.eval(x)
    dev.viterbi(y)
    ll1, lq1, g1 = dev.eval(x)
    assert ll1 == ll0 and np.array_equal(lq1, lq0) and np.array_equal(g1, g0)
    dev.upload_x(x)
    dev.eval_launch()
    dev.viterbi(y)
    ll2, lq2, g2 = dev.eval_fetch(want_logq=True)
    assert ll2 == ll0 and np.array_equal(lq2, lq0) and np.array_equal(g2, g0)
    dev.close()


def held_bytes():
    gc.collect()
    return W.lib().wfsa_dev_held_bytes()


@pytest.mark.parametrize("kernel", [2, 3, 7])
def test_memory_and_errors(c4, kernel):
    held = held_bytes()
    dev = W.Device(c4, force_kernel=kernel, count=300 if kernel == 3 else None)
    L, h = dev.L, dev.h
    logw = np.zeros(dev.n_strings)
    off = np.zeros(dev.n_strings + 1, dtype=np.int64)
    tr = np.zeros(10, dtype=np.int32)
    x = np.zeros(1)
    assert L.wfsa_dev_viterbi(h, W._p(x, W.F64P), W._p(logw, W.F64P), W._p(off, W.I64P)) == 5        # before set_param_map
    assert L.wfsa_dev_viterbi_paths(h, W._p(tr, W.I32P), W._p(tr, W.I32P)) == 5                      # before any viterbi
    dev.close()
    dev, trimmed, n = mapped_device(c4, force_kernel=kernel, count=300 if kernel == 3 else None)
    L, h = dev.L, dev.h
    x = np.random.RandomState(1).normal(-1.5, 0.8, size=n)
    assert L.wfsa_dev_viterbi(h, None, W._p(logw, W.F64P), W._p(off, W.I64P)) == 1
    assert L.wfsa_dev_viterbi(h, W._p(x, W.F64P), None, W._p(off, W.I64P)) == 1
    assert L.wfsa_dev_viterbi(h, W._p(x, W.F64P), W._p(logw, W.F64P), None) == 1
    assert L.wfsa_dev_viterbi_paths(h, W._p(tr, W.I32P), W._p(tr, W.I32P)) == 5
    dev.eval(x)
    logw, off, tr, em = dev.viterbi(x)
    assert off[-1] > 0
    assert L.wfsa_dev_viterbi_paths(h, None, W._p(em, W.I32P)) == 1
    dev.close()
    assert held_bytes() == held


FIXTURES = [("test3.wfsa", "test.corpus"), ("talk.wfsa", "talk.corpus"), ("test5.wfsa", "test5.corpus"),
            ("test.list.wfsa", "test.corpus"), ("test.loop.wfsa", "test.corpus")]


@pytest.mark.parametrize("fsa,corpus", FIXTURES)
def test_cli_viterbi_paths_are_reference_paths(fsa, corpus, tmp_path):
    """`wfsa -e 0 --viterbi FILE`: one line per corpus string in corpus order; every decoded path is one of the reference
    binary's -pr lines for that word, and w/q is a posterior."""
    name = fsa + "+" + corpus
    case = [c for c in load_cases("fixtures") if c["name"] == name][0]
    (tmp_path / fsa).write_bytes(case["fsa_text"].encode())
    (tmp_path / corpus).write_bytes(case["corpus_text"].encode())
    out = tmp_path / "viterbi.tsv"
    r = subprocess.run([EXE, "-a", str(tmp_path / fsa), "-c", str(tmp_path / corpus), "-e", "0", "-s", "--viterbi", str(out)],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-3000:]
    want = set(load_cases("path_listing")[name])
    lines = out.read_text().split("\n")
    assert lines[-1] == "" and len(lines) - 1 == len(case["corpus"])
    for ln, w in zip(lines, case["corpus"]):
        word, lw, ratio, path = ln.split("\t")
        assert word == w["word"]
        if w["paths"] == 0:
            assert (lw, ratio, path) == ("-inf", "0", "")
            continue
        assert word + ": " + path in want, ln
        assert float(lw) > -np.inf and 0.0 < float(ratio) <= 1.0 + 1e-12
