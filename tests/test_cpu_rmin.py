"""The smallest path posterior without enumerating paths: exp(m_s - log q_s), m_s from the CPU (min, +) forward pass
(tests/minpath_oracle.c) and log q_s from the CPU forward-backward, against the path posteriors the reference itself printed
for every evaluation of the golden random cases (multi-token and empty emissions, dead ends, unrecognised strings)."""
import numpy as np
import pytest

import wfsa_b200 as W
from helpers import fnum, good_cases
import minpath_oracle as MP
from oracle import oracle as O
from test_cpu_oracle import perm_golden_to_mine, setup_case

CASES = [c for c in good_cases(("random",)) if c.get("evals")]


@pytest.mark.parametrize("case", CASES, ids=lambda c: c["name"])
def test_minpath_rmin_matches_reference_posteriors(case):
    d, low, pc, trimmed, n, _ = setup_case(case)
    perm, _ = perm_golden_to_mine(case, low, trimmed)
    for ev in case["evals"]:
        x = np.zeros(n)
        x[perm] = np.array([fnum(v) for v in ev["x"]])
        ltw, lew = low.edge_logweights(x, trimmed)
        m = MP.dp_minpath(low, ltw, lew, nthreads=2)
        assert (np.isfinite(m) == (pc > 0)).all()              # a smallest path exactly where a path exists
        ref = min((fnum(v) for v in ev["r"]), default=1.0)      # (unique paths: the reference lists no posteriors, all are 1)
        got = MP.rmin(low, ltw, lew, nthreads=2)
        assert abs(got - ref) <= 1e-12 * ref, (got, ref)


def test_minpath_is_the_smallest_enumerated_path():
    """Per string, m_s equals the smallest summed log-weight over the explicitly enumerated paths."""
    case = [c for c in CASES if c["paths"] > len(c["corpus"])][0]
    d, low, pc, trimmed, n, _ = setup_case(case)
    x = np.random.RandomState(5).normal(-1.0, 1.0, size=n)
    ltw, lew = low.edge_logweights(x, trimmed)
    m = MP.dp_minpath(low, ltw, lew, nthreads=1)
    lw = np.concatenate([ltw, lew])
    for s in range(len(pc)):
        sub = W.Lowered.__new__(W.Lowered)
        sub.__dict__.update(low.__dict__)
        sub.set_tokens(low.offsets[s:s + 2] - low.offsets[s], low.tokens[low.offsets[s]:low.offsets[s + 1]], low.p[s:s + 1])
        paths = _paths(sub)
        if not paths:
            assert m[s] == np.inf
        else:
            assert abs(m[s] - min(sum(lw[e] for e in p) for p in paths)) <= 1e-12 * max(1.0, abs(m[s]))


def _paths(low):
    """Every accepting path of the only string of `low`, as edge ids (transitions, then n_trans + emission)."""
    tok = low.tokens
    out = []

    def walk(pos, state, acc):
        for t in range(low.trans_row[state], low.trans_row[state + 1]):
            v = low.trans_dst[t]
            if v == low.end:
                if pos == len(tok):
                    out.append(acc + [t])
                continue
            for e in range(low.emis_row[v], low.emis_row[v + 1]):
                lab = low.emis_tok[low.emis_tok_off[e]:low.emis_tok_off[e + 1]]
                if pos + len(lab) <= len(tok) and list(tok[pos:pos + len(lab)]) == list(lab):
                    walk(pos + len(lab), v, acc + [t, low.n_trans + e])

    walk(0, low.start, [])
    return out
