"""The most probable path of every string on the CPU (tests/maxpath_oracle.c), against the path posteriors and path
counts the reference itself printed for every evaluation of the golden random cases (multi-token and empty emissions,
dead ends, unrecognised strings), and against explicitly enumerated paths.  Also the CLI's refusals: --viterbi decodes on
one GPU, and there is no CPU fallback."""
import os
import subprocess

import numpy as np
import pytest

import maxpath_oracle as MX
from helpers import fnum, good_cases
from oracle import oracle as O
from test_cpu_oracle import perm_golden_to_mine, setup_case
from test_cpu_rmin import _paths

import wfsa_b200 as W

CASES = [c for c in good_cases(("random",)) if c.get("evals")]
HERE = os.path.dirname(os.path.abspath(__file__))
EXE = os.path.join(os.path.dirname(HERE), "w-fsa_b200", "_build", "wfsa")


def counts_of(steps, low, trimmed, golden_of_mine):
    """Trimmed-parameter counts of a path, keyed by the golden case's parameter ids (pinned and unused edges: no entry)."""
    out = {}
    for t, e in steps:
        for r in ([low.trans_param[t]] + ([low.emis_param[e]] if e >= 0 else [])):
            if r >= 0 and trimmed[r] >= 0:
                g = golden_of_mine[trimmed[r]]
                out[g] = out.get(g, 0) + 1
    return out


def check_case_against_reference(case, best_and_paths):
    """For every stored x: exp(best_s - log q_s) is the largest reference posterior among the paths of s, and the path's
    counts are the P row of a path with that posterior."""
    d, low, pc, trimmed, n, _ = setup_case(case)
    perm, _ = perm_golden_to_mine(case, low, trimmed)
    golden_of_mine = {int(m): g for g, m in enumerate(perm)}
    P = [{c: v for c, v in zip(case["Pcol"][a:b], case["Pdata"][a:b])} for a, b in zip(case["Prow"], case["Prow"][1:])]
    rec = [s for s in range(len(pc)) if pc[s] > 0]
    for ev in case["evals"]:
        x = np.zeros(n)
        x[perm] = np.array([fnum(v) for v in ev["x"]])
        ltw, lew = low.edge_logweights(x, trimmed)
        best, paths = best_and_paths(low, trimmed, x, ltw, lew)
        _, lq, _ = O.dp_eval(low, ltw, lew, want_grad=False)
        assert (np.isfinite(best) == (pc > 0)).all()
        assert all((len(paths[s]) > 0) == (pc[s] > 0) for s in range(len(pc)))
        r = [fnum(v) for v in ev["r"]] if ev["r"] else None
        for i, s in enumerate(rec):
            assert MX.path_logweight(paths[s], ltw, lew) == best[s]
            ids = case["Mcol"][case["Mrow"][i]:case["Mrow"][i + 1]]
            post = np.exp(best[s] - lq[s])
            rmax = max(r[p] for p in ids) if r else 1.0        # (unique paths: the reference lists no posteriors, all are 1)
            assert abs(post - rmax) <= 1e-12 * rmax, (s, post, rmax)
            mine = counts_of(paths[s], low, trimmed, golden_of_mine)
            tied = [p for p in ids if not r or abs(r[p] - rmax) <= 1e-12 * rmax]
            assert any(P[p] == mine for p in tied), (s, mine, [P[p] for p in tied])


@pytest.mark.parametrize("case", CASES, ids=lambda c: c["name"])
def test_maxpath_matches_reference_posteriors(case):
    check_case_against_reference(case, lambda low, trimmed, x, ltw, lew: MX.viterbi(low, ltw, lew, nthreads=2))


def test_maxpath_is_the_largest_enumerated_path():
    """Per string, best_s is the largest summed log-weight over the explicitly enumerated paths, and the returned path is
    one of them."""
    case = [c for c in CASES if c["paths"] > len(c["corpus"])][0]
    d, low, pc, trimmed, n, _ = setup_case(case)
    x = np.random.RandomState(5).normal(-1.0, 1.0, size=n)
    ltw, lew = low.edge_logweights(x, trimmed)
    best, paths = MX.viterbi(low, ltw, lew, nthreads=1)
    lw = np.concatenate([ltw, lew])
    for s in range(len(pc)):
        sub = W.Lowered.__new__(W.Lowered)
        sub.__dict__.update(low.__dict__)
        sub.set_tokens(low.offsets[s:s + 2] - low.offsets[s], low.tokens[low.offsets[s]:low.offsets[s + 1]], low.p[s:s + 1])
        enum = _paths(sub)
        if not enum:
            assert best[s] == -np.inf and paths[s] == []
            continue
        assert abs(best[s] - max(sum(lw[e] for e in p) for p in enum)) <= 1e-12 * max(1.0, abs(best[s]))
        flat = [a for t, e in paths[s] for a in ([t] if e < 0 else [t, low.n_trans + e])]
        assert flat in enum


@pytest.fixture(scope="module")
def small_files(tmp_path_factory):
    case = [c for c in CASES if c["strings"] > 0][0]
    dd = tmp_path_factory.mktemp("vit")
    fsa, corpus = dd / "a.wfsa", dd / "a.corpus"
    fsa.write_text(case["fsa_text"]); corpus.write_text(case["corpus_text"])
    return str(fsa), str(corpus), str(dd / "out.tsv")


def test_cli_refuses_viterbi_on_several_gpus(small_files):
    fsa, corpus, out = small_files
    r = subprocess.run([EXE, "-a", fsa, "-c", corpus, "-e", "0", "-s", "--gpus", "2", "--viterbi", out],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 1 and "--viterbi" in r.stderr and "--gpus" in r.stderr
    assert not os.path.exists(out)


def test_cli_viterbi_has_no_cpu_fallback(small_files):
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a device is present")
    except ImportError:
        pass
    fsa, corpus, out = small_files
    r = subprocess.run([EXE, "-a", fsa, "-c", corpus, "-e", "0", "-s", "--viterbi", out], capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and not os.path.exists(out)
