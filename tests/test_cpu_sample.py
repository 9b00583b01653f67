"""Path sampling on the CPU (tests/sample_oracle.c): its Philox4x32-10 and the library's against the Random123 known-answer
vectors, and its draws against the path posteriors and path counts the reference itself printed for every evaluation of
the golden random cases (multi-token and empty emissions, dead ends, unrecognised strings): every draw is a reference path,
its value is the left-to-right sum of its steps, and the draw counts pass a Pearson chi-square test against the
posteriors.  Also the CLI's refusals of --sample."""
import collections
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

import maxpath_oracle as MX
import sample_oracle as SO
from helpers import fnum
from oracle import oracle as O
from test_cpu_oracle import perm_golden_to_mine, setup_case
from test_cpu_viterbi import CASES, counts_of

import wfsa_b200 as W

HERE = os.path.dirname(os.path.abspath(__file__))
EXE = os.path.join(os.path.dirname(HERE), "w-fsa_b200", "_build", "wfsa")
SEEDS = range(16)          # x 256 draws: 4096 draws per string

KAT = [([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
       ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
       ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0],
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1])]


@pytest.mark.parametrize("ctr,key,want", KAT)
def test_philox_known_answers(ctr, key, want):
    assert [int(v) for v in W.philox4x32_10(ctr, key)] == want
    assert SO.philox4x32_10(ctr, key) == want
    assert SO.philox4x32_10_c(ctr, key) == want


def chi2_terms(observed, expected_p, n_draws):
    """Pearson terms of one string: categories with fewer than 5 expected draws are pooled.  (statistic, degrees of freedom)"""
    obs, exp = [], []
    pool_o, pool_e = 0, 0.0
    for k, p in expected_p.items():
        e = p * n_draws
        if e < 5.0:
            pool_o += observed.get(k, 0); pool_e += e
        else:
            obs.append(observed.get(k, 0)); exp.append(e)
    if pool_e > 0.0:
        obs.append(pool_o); exp.append(pool_e)
    if len(obs) < 2:
        return 0.0, 0
    obs, exp = np.array(obs, dtype=float), np.array(exp)
    return float(((obs - exp) ** 2 / exp).sum()), len(obs) - 1


def check_case_sample(case, draw, seeds=SEEDS, n=256):
    """draw(low, trimmed, x, ltw, lew, n, seed) -> (logq [ns], logw [ns, n], steps [ns][n] as tuples of (t, e) pairs).  For
    every stored x: log q is the evaluation's; strings without a path get -inf and no steps; every draw is a path with the
    counts of a reference path of its string and its value is the left-to-right sum of its steps; the draw counts per count
    vector, against the summed reference posteriors of the paths with that vector, pass Pearson's chi-square (p >= 1e-6)
    summed over the strings with at least two paths."""
    d, low, pc, trimmed, n_par, _ = setup_case(case)
    perm, _ = perm_golden_to_mine(case, low, trimmed)
    golden_of_mine = {int(m): g for g, m in enumerate(perm)}
    P = [{c: v for c, v in zip(case["Pcol"][a:b], case["Pdata"][a:b])} for a, b in zip(case["Prow"], case["Prow"][1:])]
    rec = [s for s in range(len(pc)) if pc[s] > 0]
    stat, dof = 0.0, 0
    for ev in case["evals"]:
        x = np.zeros(n_par)
        x[perm] = np.array([fnum(v) for v in ev["x"]])
        ltw, lew = low.edge_logweights(x, trimmed)
        _, lq, _ = O.dp_eval(low, ltw, lew, want_grad=False)
        obs = [collections.Counter() for _ in pc]
        value = {}
        for seed in seeds:
            logq, logw, steps = draw(low, trimmed, x, ltw, lew, n, seed)
            assert logw.shape == (len(pc), n)
            for s in range(len(pc)):
                if pc[s] == 0:
                    assert logq[s] == -np.inf and (logw[s] == -np.inf).all() and all(p == () for p in steps[s]), s
                    continue
                assert abs(logq[s] - lq[s]) <= 1e-12 * max(1.0, abs(lq[s])), (s, logq[s], lq[s])
                for r in range(n):
                    key = (s, steps[s][r])
                    if key not in value:
                        value[key] = MX.path_logweight(steps[s][r], ltw, lew)
                    assert logw[s, r] == value[key], (s, r)
                    obs[s][steps[s][r]] += 1
        r = [fnum(v) for v in ev["r"]] if ev["r"] else None
        for i, s in enumerate(rec):
            ids = case["Mcol"][case["Mrow"][i]:case["Mrow"][i + 1]]
            want = collections.defaultdict(float)
            for p in ids:
                want[frozenset(P[p].items())] += r[p] if r else 1.0
            got = collections.Counter()
            for st, c in obs[s].items():
                k = frozenset(counts_of(list(st), low, trimmed, golden_of_mine).items())
                assert k in want, (s, st)
                got[k] += c
            if len(ids) >= 2:
                t, f = chi2_terms(got, want, len(seeds) * n)
                stat += t; dof += f
    if dof:
        assert stats.chi2.sf(stat, dof) >= 1e-6, (stat, dof)


def oracle_draw(low, trimmed, x, ltw, lew, n, seed):
    logq, logw, paths = SO.sample(low, ltw, lew, n, seed, nthreads=2)
    return logq, logw, [[tuple(p) for p in ps] for ps in paths]


@pytest.mark.parametrize("case", CASES, ids=lambda c: c["name"])
def test_draws_follow_reference_posteriors(case):
    check_case_sample(case, oracle_draw)


def test_draws_are_prefix_stable_and_seeded():
    """The first m draws of n > m are the draws of n = m; another seed changes some draws."""
    case = [c for c in CASES if c["paths"] > 2 * len(c["corpus"])][0]
    d, low, pc, trimmed, n, _ = setup_case(case)
    x = np.random.RandomState(5).normal(-1.0, 1.0, size=n)
    ltw, lew = low.edge_logweights(x, trimmed)
    q4, w4, p4 = SO.sample(low, ltw, lew, 4, 7)
    q32, w32, p32 = SO.sample(low, ltw, lew, 32, 7)
    assert np.array_equal(q4, q32) and np.array_equal(w4, w32[:, :4]) and all(a == b[:4] for a, b in zip(p4, p32))
    _, _, p32b = SO.sample(low, ltw, lew, 32, 8)
    assert p32b != p32


@pytest.fixture(scope="module")
def small_files(tmp_path_factory):
    case = [c for c in CASES if c["strings"] > 0][0]
    dd = tmp_path_factory.mktemp("sample")
    fsa, corpus = dd / "a.wfsa", dd / "a.corpus"
    fsa.write_text(case["fsa_text"]); corpus.write_text(case["corpus_text"])
    return str(fsa), str(corpus), str(dd / "out.tsv")


def test_cli_refuses_sample_on_several_gpus(small_files):
    fsa, corpus, out = small_files
    r = subprocess.run([EXE, "-a", fsa, "-c", corpus, "-e", "0", "-s", "--gpus", "2", "--sample", "4", out],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 1 and "--sample" in r.stderr and "--gpus" in r.stderr
    assert not os.path.exists(out)


@pytest.mark.parametrize("N", ["0", "257", "x"])
def test_cli_refuses_sample_outside_1_to_256(small_files, N):
    fsa, corpus, out = small_files
    r = subprocess.run([EXE, "-a", fsa, "-c", corpus, "-e", "0", "-s", "--sample", N, out], capture_output=True, text=True,
                       timeout=120)
    assert r.returncode == 1 and "--sample" in r.stderr
    assert not os.path.exists(out)


def test_cli_refuses_a_bad_seed(small_files):
    fsa, corpus, out = small_files
    r = subprocess.run([EXE, "-a", fsa, "-c", corpus, "-e", "0", "-s", "--sample", "4", out, "--seed", "-3"],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 1 and "--seed" in r.stderr
    assert not os.path.exists(out)
