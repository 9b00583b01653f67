"""N-best decoding on the device (wfsa_dev_nbest / wfsa_dev_viterbi_paths): the k most probable paths of every string on
every kernel, against the CPU reference (tests/nbest_oracle.c) bit for bit and the reference's own path
posteriors and counts; rank 0 and k = 1 against wfsa_dev_viterbi, determinism, no effect on the evaluation, memory, error
codes and the CLI's --nbest."""
import gc
import os
import subprocess

import numpy as np
import pytest

import maxpath_oracle as MX
import nbest_oracle as NB
import wfsa_b200 as W
from helpers import load_cases
from test_cpu_nbest import check_case_nbest
from test_cpu_viterbi import CASES
from test_gpu_rmin import mapped_device, synth_low
from test_gpu_viterbi import as_paths, check_valid_path

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
EXE = os.path.join(os.path.dirname(HERE), "w-fsa_b200", "_build", "wfsa")


@pytest.fixture(scope="module")
def c4():
    return synth_low(256, 64, 8, 4, 31, 600, 64, 128)


def same_bits(a, b):
    return a.shape == b.shape and np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def check_against_oracle(low, trimmed, x, k, res, nthreads=0):
    """Values bit-identical to the CPU reference; every path valid, distinct and the left-to-right sum of its steps."""
    logw, off, tr, em = res
    n = len(logw)
    ltw, lew = low.edge_logweights(x, trimmed)
    ref, _ = NB.nbest(low, ltw, lew, k, nthreads=nthreads)
    assert same_bits(logw, ref), np.argwhere(logw.view(np.uint64) != ref.view(np.uint64))[:5]
    paths = as_paths(off, tr, em)
    assert len(paths) == n * k
    for s in range(n):
        assert all(logw[s, r] >= logw[s, r + 1] for r in range(k - 1)), s
        for r in range(k):
            p = paths[s * k + r]
            if logw[s, r] == -np.inf:
                assert p == [], (s, r)
                continue
            check_valid_path(low, s, p)
            assert MX.path_logweight(p, ltw, lew) == logw[s, r], (s, r)     # the summation-order identity, bit for bit
        found = [tuple(p) for p in paths[s * k:(s + 1) * k] if p]
        assert len(set(found)) == len(found), s


def check_rank0_is_viterbi(dev, x, k, res):
    logw, off, tr, em = res
    vw, voff, vtr, vem = dev.viterbi(x)
    assert same_bits(np.ascontiguousarray(logw[:, 0]), vw)
    paths, vpaths = as_paths(off, tr, em), as_paths(voff, vtr, vem)
    assert all(paths[s * k] == vpaths[s] for s in range(len(vw)))


def sub_corpus(low, count):
    out = W.Lowered.__new__(W.Lowered); out.__dict__.update(low.__dict__)
    out.set_tokens(low.offsets[:count + 1], low.tokens[:low.offsets[count]], low.p[:count])
    return out


@pytest.mark.parametrize("k", [2, 5, 16])
@pytest.mark.parametrize("kernel", [1, 2, 3, 4, 6, 7])
@pytest.mark.parametrize("mu,sigma", [(-1.0, 0.3), (-3.0, 1.0)])
def test_every_kernel(c4, kernel, mu, sigma, k):
    """At x ~ N(-3, 1) path weights of strings of up to 128 symbols fall below 1e-308: only the log domain is right."""
    dev, trimmed, n = mapped_device(c4, force_kernel=kernel, count=300 if kernel == 3 else None)
    assert dev.info()["kernel"] == kernel
    x = np.random.RandomState(kernel).normal(mu, sigma, size=n)
    res = dev.nbest(x, k)
    low = sub_corpus(c4, 300) if kernel == 3 else c4
    assert np.isfinite(res[0][:, 0]).sum() > len(res[0]) // 2 and np.isfinite(res[0][:, k - 1]).any()
    check_against_oracle(low, trimmed, x, k, res)
    check_rank0_is_viterbi(dev, x, k, res)
    again = dev.nbest(x, k)                                                     # determinism: the same bits
    assert all(same_bits(a, b) for a, b in zip(res, again))
    dev.close()


@pytest.mark.parametrize("kernel", [2, 3, 6, 7])
def test_k1_is_viterbi(c4, kernel):
    dev, trimmed, n = mapped_device(c4, force_kernel=kernel, count=300 if kernel == 3 else None)
    x = np.random.RandomState(2).normal(-1.0, 0.3, size=n)
    logw, off, tr, em = dev.nbest(x, 1)
    v = dev.viterbi(x)
    assert same_bits(logw[:, 0], v[0]) and all(same_bits(a, b) for a, b in zip((off, tr, em), v[1:]))
    dev.close()


@pytest.mark.parametrize("k", [2, 4, 16])
@pytest.mark.parametrize("kernel", [2, 3])
@pytest.mark.parametrize("case", CASES, ids=lambda c: c["name"])
def test_golden_posteriors(case, kernel, k):
    """The reference's own path posteriors and counts (multi-token and empty emissions: kg_nbest)."""
    def decode(low, trimmed, x, ltw, lew, k):
        dev = W.Device(low, force_kernel=kernel)
        rec, _, _ = dev.structure()
        dev.set_param_map(trimmed, len(x), rec)
        logw, off, tr, em = dev.nbest(x, k)
        dev.close()
        p = as_paths(off, tr, em)
        return logw, [p[s * k:(s + 1) * k] for s in range(len(logw))]
    low = W.Lowered(W.parse(case["fsa_text"], case["corpus_text"]))
    inner = [s for s in range(low.n_states) if s not in (low.start, low.end)]
    if kernel == 2 and any(low.emis_tok_off[e + 1] - low.emis_tok_off[e] != 1 for s in inner
                           for e in range(low.emis_row[s], low.emis_row[s + 1])):
        pytest.skip("emissions of other than one token: no fast tables")
    check_case_nbest(case, k, decode)


def test_config5_true_shape():
    """BASELINE config 5 at its named shape (4096 states / 256 symbols: a CTA per string), several K7 batches: the K7
    handle against a forced CTA-per-string handle (same bits), both against the oracle."""
    low = synth_low(4096, 256, 64, 16, 4321, 300, 32, 128)
    os.environ["WFSA_K7_ROWS"] = "9000"
    try:
        dev7, trimmed, n = mapped_device(low, force_kernel=7)
    finally:
        os.environ.pop("WFSA_K7_ROWS", None)
    assert dev7.info()["kernel"] == 7 and dev7.info()["max_candidates"] > 32
    dev2, trimmed2, n2 = mapped_device(low, force_kernel=2)
    assert n2 == n and np.array_equal(trimmed2, trimmed)
    for seed, (mu, sigma), k in [(0, (-1.0, 0.3), 16), (1, (-3.0, 1.0), 5)]:
        x = np.random.RandomState(seed).normal(mu, sigma, size=n)
        r7, r2 = dev7.nbest(x, k), dev2.nbest(x, k)
        assert all(same_bits(a, b) for a, b in zip(r7, r2))
        check_against_oracle(low, trimmed, x, k, r7, nthreads=8)
        check_rank0_is_viterbi(dev7, x, k, r7)
    dev7.close(); dev2.close()


@pytest.mark.parametrize("kernel", [2, 3, 6, 7])
def test_evaluation_is_unchanged(c4, kernel):
    """An nbest call between two evaluations, and between eval_launch and eval_fetch (log q on demand on the segmented
    path), changes no bit of what the evaluation returns."""
    dev, trimmed, n = mapped_device(c4, force_kernel=kernel, count=300 if kernel == 3 else None)
    x = np.random.RandomState(11).normal(-1.0, 0.3, size=n)
    y = np.random.RandomState(12).normal(-2.0, 0.5, size=n)
    ll0, lq0, g0 = dev.eval(x)
    dev.nbest(y, 4)
    ll1, lq1, g1 = dev.eval(x)
    assert ll1 == ll0 and np.array_equal(lq1, lq0) and np.array_equal(g1, g0)
    dev.upload_x(x)
    dev.eval_launch()
    dev.nbest(y, 4)
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
    logw = np.zeros(dev.n_strings * 16)
    off = np.zeros(dev.n_strings * 16 + 1, dtype=np.int64)
    x = np.zeros(1)
    assert L.wfsa_dev_nbest(h, W._p(x, W.F64P), 4, W._p(logw, W.F64P), W._p(off, W.I64P)) == 5       # before set_param_map
    dev.close()
    dev, trimmed, n = mapped_device(c4, force_kernel=kernel, count=300 if kernel == 3 else None)
    L, h = dev.L, dev.h
    x = np.random.RandomState(1).normal(-1.5, 0.8, size=n)
    for k in (0, 17, -1):
        assert L.wfsa_dev_nbest(h, W._p(x, W.F64P), k, W._p(logw, W.F64P), W._p(off, W.I64P)) == 1
    assert L.wfsa_dev_nbest(h, None, 4, W._p(logw, W.F64P), W._p(off, W.I64P)) == 1
    assert L.wfsa_dev_nbest(h, W._p(x, W.F64P), 4, None, W._p(off, W.I64P)) == 1
    assert L.wfsa_dev_nbest(h, W._p(x, W.F64P), 4, W._p(logw, W.F64P), None) == 1
    tr = np.zeros(10, dtype=np.int32)
    assert L.wfsa_dev_viterbi_paths(h, W._p(tr, W.I32P), W._p(tr, W.I32P)) == 5                     # before any decode
    dev.eval(x)
    for k in (16, 3):
        lw, off2, tr2, em2 = dev.nbest(x, k)
        assert off2[-1] > 0 and np.isfinite(lw[:, 0]).any()
    dev.close()
    assert held_bytes() == held


def test_limit_when_cta_lists_do_not_fit():
    """A CTA-per-string handle with 1000 candidates per symbol: its lists at k = 16 (2 x 16 x 1024 doubles) exceed the
    shared memory of a CTA, WFSA_ERR_LIMIT with a message; at k = 8 it decodes, against the oracle."""
    low = synth_low(1000, 2, 4, 2, 77, 40, 3, 6)
    dev, trimmed, n = mapped_device(low, force_kernel=2)
    assert dev.info()["max_candidates"] > 768
    x = np.random.RandomState(3).normal(-1.0, 0.5, size=n)
    logw = np.zeros(dev.n_strings * 16)
    off = np.zeros(dev.n_strings * 16 + 1, dtype=np.int64)
    assert dev.L.wfsa_dev_nbest(dev.h, W._p(x, W.F64P), 16, W._p(logw, W.F64P), W._p(off, W.I64P)) == 6
    assert "shared memory" in dev.L.wfsa_dev_last_error(dev.h).decode()
    res = dev.nbest(x, 8)
    check_against_oracle(low, trimmed, x, 8, res)
    check_rank0_is_viterbi(dev, x, 8, res)
    dev.close()


FIXTURES = [("test3.wfsa", "test.corpus"), ("talk.wfsa", "talk.corpus"), ("test5.wfsa", "test5.corpus"),
            ("test.list.wfsa", "test.corpus"), ("test.loop.wfsa", "test.corpus")]


@pytest.mark.parametrize("K", [2, 16])
@pytest.mark.parametrize("fsa,corpus", FIXTURES)
def test_cli_nbest_paths_are_reference_paths(fsa, corpus, K, tmp_path):
    """`wfsa -e 0 -s --viterbi V --nbest K N`: min(K, paths) lines per corpus string in corpus order, every path a distinct
    -pr line of the reference binary for that word, ratios non-increasing and summing to 1 when K >= paths; rank 1 is the
    --viterbi line."""
    name = fsa + "+" + corpus
    case = [c for c in load_cases("fixtures") if c["name"] == name][0]
    (tmp_path / fsa).write_bytes(case["fsa_text"].encode())
    (tmp_path / corpus).write_bytes(case["corpus_text"].encode())
    vit, out = tmp_path / "viterbi.tsv", tmp_path / "nbest.tsv"
    r = subprocess.run([EXE, "-a", str(tmp_path / fsa), "-c", str(tmp_path / corpus), "-e", "0", "-s", "--viterbi", str(vit),
                        "--nbest", str(K), str(out)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-3000:]
    want = set(load_cases("path_listing")[name])
    lines = out.read_text().split("\n")
    assert lines[-1] == ""
    vlines = vit.read_text().split("\n")
    i = 0
    for w, vl in zip(case["corpus"], vlines):
        if w["paths"] == 0:
            assert lines[i].split("\t") == [w["word"], "0", "-inf", "0", ""]
            i += 1
            continue
        m = min(K, w["paths"])
        block = [ln.split("\t") for ln in lines[i:i + m]]
        i += m
        assert [b[0] for b in block] == [w["word"]] * m and [b[1] for b in block] == [str(r + 1) for r in range(m)]
        assert "\t".join([block[0][0]] + block[0][2:]) == vl
        assert len({b[4] for b in block}) == m
        for b in block:
            assert w["word"] + ": " + b[4] in want, b
        ratios = [float(b[3]) for b in block]
        assert all(0.0 < a <= 1.0 + 1e-12 for a in ratios)
        assert all(ratios[j] >= ratios[j + 1] for j in range(m - 1))
        if K >= w["paths"]:
            assert abs(sum(ratios) - 1.0) <= 1e-12, (w["word"], ratios)
    assert i == len(lines) - 1
