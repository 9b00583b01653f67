"""The k most probable paths of every string on the CPU (tests/nbest_oracle.c), against the path
posteriors and path counts the reference itself printed for every evaluation of the golden random cases (multi-token and
empty emissions, dead ends, unrecognised strings), against explicitly enumerated paths, and against the Viterbi reference at
k = 1.  Also the CLI's refusals: --nbest decodes on one GPU, takes K in 1..16, and has no CPU fallback."""
import os
import subprocess

import numpy as np
import pytest

import maxpath_oracle as MX
import nbest_oracle as NB
from helpers import fnum
from oracle import oracle as O
from test_cpu_oracle import perm_golden_to_mine, setup_case
from test_cpu_rmin import _paths
from test_cpu_viterbi import CASES, counts_of

import wfsa_b200 as W

HERE = os.path.dirname(os.path.abspath(__file__))
EXE = os.path.join(os.path.dirname(HERE), "w-fsa_b200", "_build", "wfsa")


def check_case_nbest(case, k, decode):
    """decode(low, trimmed, x, ltw, lew, k) -> (best [n, k], paths [n][k]).  For every stored x and recognised string s:
    exp(best[s, r] - log q_s) for r < min(k, paths) are the reference's posteriors of s in descending order, later ranks are
    -inf without steps, the posteriors sum to 1 when k >= paths, every path's value is the left-to-right sum of its steps,
    the paths are distinct, and each has the counts of a reference path with its posterior (the only one when untied)."""
    d, low, pc, trimmed, n, _ = setup_case(case)
    perm, _ = perm_golden_to_mine(case, low, trimmed)
    golden_of_mine = {int(m): g for g, m in enumerate(perm)}
    P = [{c: v for c, v in zip(case["Pcol"][a:b], case["Pdata"][a:b])} for a, b in zip(case["Prow"], case["Prow"][1:])]
    rec = [s for s in range(len(pc)) if pc[s] > 0]
    for ev in case["evals"]:
        x = np.zeros(n)
        x[perm] = np.array([fnum(v) for v in ev["x"]])
        ltw, lew = low.edge_logweights(x, trimmed)
        best, paths = decode(low, trimmed, x, ltw, lew, k)
        assert best.shape == (len(pc), k)
        _, lq, _ = O.dp_eval(low, ltw, lew, want_grad=False)
        r = [fnum(v) for v in ev["r"]] if ev["r"] else None
        for s in range(len(pc)):
            if pc[s] == 0:
                assert (best[s] == -np.inf).all() and all(p == [] for p in paths[s]), s
        for i, s in enumerate(rec):
            ids = case["Mcol"][case["Mrow"][i]:case["Mrow"][i + 1]]
            post = {p: (r[p] if r else 1.0) for p in ids}       # (unique paths: the reference lists no posteriors, all are 1)
            want = sorted(post.values(), reverse=True)
            m = min(k, len(want))
            assert all(best[s, j] >= best[s, j + 1] for j in range(k - 1)), (s, best[s])
            for rk in range(k):
                if rk >= m or want[rk] == 0.0:
                    assert best[s, rk] == -np.inf and paths[s][rk] == [], (s, rk)
                    continue
                got = np.exp(best[s, rk] - lq[s])
                assert abs(got - want[rk]) <= 1e-12 * want[rk], (s, rk, got, want[rk])
                assert MX.path_logweight(paths[s][rk], ltw, lew) == best[s, rk], (s, rk)
                mine = counts_of(paths[s][rk], low, trimmed, golden_of_mine)
                tied = [p for p in ids if abs(post[p] - want[rk]) <= 1e-12 * want[rk]]
                assert any(P[p] == mine for p in tied), (s, rk, mine, [P[p] for p in tied])
            found = [tuple(p) for p in paths[s] if p]
            assert len(set(found)) == len(found), s
            if k >= len(want):
                assert abs(np.exp(best[s] - lq[s]).sum() - 1.0) <= 1e-12, s


def oracle_nbest(low, trimmed, x, ltw, lew, k):
    return NB.nbest(low, ltw, lew, k, nthreads=2)


@pytest.mark.parametrize("k", [2, 4, 16])
@pytest.mark.parametrize("case", CASES, ids=lambda c: c["name"])
def test_kbest_matches_reference_posteriors(case, k):
    check_case_nbest(case, k, oracle_nbest)


@pytest.mark.parametrize("k", [2, 5, 16])
def test_kbest_is_the_top_of_the_enumerated_paths(k):
    """Per string, the k values are the k largest summed log-weights over the explicitly enumerated paths (the same
    left-to-right sums, so the same bits), and the paths are distinct members of the enumeration."""
    case = [c for c in CASES if c["paths"] > len(c["corpus"])][0]
    d, low, pc, trimmed, n, _ = setup_case(case)
    x = np.random.RandomState(5).normal(-1.0, 1.0, size=n)
    ltw, lew = low.edge_logweights(x, trimmed)
    best, paths = NB.nbest(low, ltw, lew, k, nthreads=1)
    lw = np.concatenate([ltw, lew])
    for s in range(len(pc)):
        sub = W.Lowered.__new__(W.Lowered)
        sub.__dict__.update(low.__dict__)
        sub.set_tokens(low.offsets[s:s + 2] - low.offsets[s], low.tokens[low.offsets[s]:low.offsets[s + 1]], low.p[s:s + 1])
        enum = [p for p in _paths(sub) if np.isfinite(sum(lw[e] for e in p))]
        vals = sorted((sum(lw[e] for e in p) for p in enum), reverse=True)[:k]
        assert best[s, :len(vals)].tolist() == vals, (s, best[s], vals)
        assert (best[s, len(vals):] == -np.inf).all() and all(p == [] for p in paths[s][len(vals):])
        flat = [[a for t, e in paths[s][r] for a in ([t] if e < 0 else [t, low.n_trans + e])] for r in range(len(vals))]
        assert all(f in enum for f in flat)
        assert len(set(map(tuple, flat))) == len(flat)


@pytest.mark.parametrize("case", CASES, ids=lambda c: c["name"])
def test_k1_is_viterbi(case):
    """k = 1 is the Viterbi reference, bit for bit, in values and paths."""
    d, low, pc, trimmed, n, _ = setup_case(case)
    x = np.random.RandomState(3).normal(-1.0, 1.0, size=n)
    ltw, lew = low.edge_logweights(x, trimmed)
    vb, vp = MX.viterbi(low, ltw, lew, nthreads=2)
    nb, npth = NB.nbest(low, ltw, lew, 1, nthreads=2)
    assert np.array_equal(nb[:, 0].view(np.uint64), vb.view(np.uint64))
    assert [p[0] for p in npth] == vp


@pytest.fixture(scope="module")
def small_files(tmp_path_factory):
    case = [c for c in CASES if c["strings"] > 0][0]
    dd = tmp_path_factory.mktemp("nbest")
    fsa, corpus = dd / "a.wfsa", dd / "a.corpus"
    fsa.write_text(case["fsa_text"]); corpus.write_text(case["corpus_text"])
    return str(fsa), str(corpus), str(dd / "out.tsv")


def test_cli_refuses_nbest_on_several_gpus(small_files):
    fsa, corpus, out = small_files
    r = subprocess.run([EXE, "-a", fsa, "-c", corpus, "-e", "0", "-s", "--gpus", "2", "--nbest", "4", out],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 1 and "--nbest" in r.stderr and "--gpus" in r.stderr
    assert not os.path.exists(out)


@pytest.mark.parametrize("K", ["0", "17", "x"])
def test_cli_refuses_nbest_outside_1_to_16(small_files, K):
    fsa, corpus, out = small_files
    r = subprocess.run([EXE, "-a", fsa, "-c", corpus, "-e", "0", "-s", "--nbest", K, out], capture_output=True, text=True, timeout=120)
    assert r.returncode == 1 and "--nbest" in r.stderr
    assert not os.path.exists(out)


def test_cli_nbest_has_no_cpu_fallback(small_files):
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a device is present")
    except ImportError:
        pass
    fsa, corpus, out = small_files
    r = subprocess.run([EXE, "-a", fsa, "-c", corpus, "-e", "0", "-s", "--nbest", "4", out], capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and not os.path.exists(out)
