"""H_f = -sum_s p_s Cov_s(c_j, c_k) on the CPU, against a reference that does not enumerate paths (tests/hessian_oracle.c:
a tangent forward-backward in long double).  The oracle itself is pinned to the enumeration of every path
(oracle/wfsa_oracle.c) where that is feasible; then the path blocks the library derives for the segmented kernel
(wfsa_segmented_compile, the same blocks wfsa_dev_hessian uploads) are checked against it where enumeration is not:
strings that no region type covers (more live lattice nodes than pool slots) and region types of large weight."""
import numpy as np
import pytest

import hessian_oracle as HO
import wfsa_b200 as W
from helpers import good_cases, vec_tol_ok
from oracle import oracle as O
from wfsa_b200 import synth

TALK = "\n^\n$\n^  0\n^ TALK_N 0 TALK_V 0\nTALK_V talk 0\nTALK_V TENSE 0\nTALK_N talk 0\nTALK_N PLUR 0\nPLUR  0 s 0\nPLUR $ 0\nTENSE  0 s 0 ed 0\nTENSE $ 0\n"
# x (yx)^R: one region type (S -> A | B, both emit y, back to S) of weight R; at x = 0, H[S->A, S->A] = -R/4
DIAMOND = "\n^\n$\n^  0\n^ S 0\nS x 0\nS A 0 B 0 $ 0\nA y 0\nA S 0\nB y 0\nB S 0\n"


def trim_all(low):
    zt, ze = np.zeros(low.n_trans), np.zeros(low.n_emis)
    _, _, ee0 = O.dp_eval(low, zt, ze, nthreads=O.max_threads())
    trimmed, n, _ = O.trim(low, ee0 > 0)
    return trimmed, n


def blocks_hv(seg, x, V):
    """H @ V from the path blocks of wfsa_segmented_compile (k5_hessian restated: r = softmax(M x_c), g = M^T r,
    H_b = p (g g^T - M^T diag(r) M))."""
    out = np.zeros_like(V)
    po, co, vo = seg["hb_path_off"], seg["hb_col_off"], seg["hb_val_off"]
    for b in range(len(seg["hb_p"])):
        c = seg["hb_cols"][co[b]:co[b + 1]]
        M = seg["hb_counts"][vo[b]:vo[b + 1]].reshape(po[b + 1] - po[b], len(c))
        s = M @ x[c]
        r = np.exp(s - s.max()); r /= r.sum()
        g = M.T @ r
        MV = M @ V[c]
        out[c] += seg["hb_p"][b] * (np.outer(g, r @ MV) - M.T @ (r[:, None] * MV))
    return out


def enum_h(low, trimmed, x, n, **kw):
    ltw, lew = low.edge_logweights(x, trimmed)
    return O.enum_hessian(low, ltw, lew, HO.edge_param(low, trimmed), n, **kw)


def synth_low(shape, seed, n_strings, lmin, lmax, corpus_seed):
    model = synth.make_model(*shape, seed=seed)
    low = model.lowered()
    offs, toks, w = model.corpus(n_strings, lmin, lmax, seed=corpus_seed)
    low.set_tokens(offs, toks, w / w.sum())
    return low


@pytest.fixture(scope="module")
def medium():
    """The `medium` corpus of test_gpu_parity.py: 3000 strings of 32-128 tokens, two of them not recognised."""
    model = synth.make_model(256, 64, 8, 4, seed=11)
    low = model.lowered()
    offs, toks, w = model.corpus(3000, 32, 128, seed=12)
    toks = toks.copy()
    toks[offs[5]] = -1
    toks[offs[9]:offs[10]] = np.random.RandomState(5).randint(0, 64, size=offs[10] - offs[9])
    low.set_tokens(offs, toks, w / w.sum())
    trimmed, n = trim_all(low)
    x = np.random.RandomState(21).normal(-1.0, 0.5, size=n)
    V = HO.directions(n, 3)
    return low, trimmed, n, x, V, HO.hv(low, trimmed, x, V)


@pytest.mark.parametrize("case", good_cases(("fixtures", "random")), ids=lambda c: c["name"])
def test_oracle_matches_enumeration(case):
    """V = I: the tangent forward-backward against the enumeration of every path of every string.  Relative 1e-12 of
    max|H|; the enumeration forms g g^T - E[c c^T] in double, so it carries ~1e-16 of absolute cancellation error."""
    low = W.Lowered(W.parse(case["fsa_text"], case["corpus_text"]))
    trimmed, n = trim_all(low)
    if n == 0:
        pytest.skip("no parameters")
    x = np.random.RandomState(8).normal(-1.0, 0.7, size=n)
    Href = enum_h(low, trimmed, x, n)
    H = HO.full(low, trimmed, x)
    assert np.abs(H - Href).max() <= 1e-12 * np.abs(Href).max() + 1e-15, np.abs(H - Href).max()
    assert np.abs(H - H.T).max() <= 1e-13 * np.abs(H).max()


def test_oracle_multi_token_and_empty_emissions():
    """Emissions of several tokens and empty ones (a state that emits nothing sits at the same position as its
    predecessor); every string has two paths."""
    low = W.Lowered(W.parse(TALK, "\ntalk 1\ntalks 2\ntalked 1\n"))
    trimmed, n = trim_all(low)
    assert n >= 4
    for seed in range(3):
        x = np.random.RandomState(seed).normal(0.0, 1.5, size=n)
        Href = enum_h(low, trimmed, x, n)
        assert np.abs(Href).max() > 0.01
        H = HO.full(low, trimmed, x)
        assert np.abs(H - Href).max() <= 1e-12 * np.abs(Href).max() + 1e-15


def test_type_blocks_medium(medium):
    """Three independent routes to H_f @ V on `medium` (3000 strings, default 16 slots, no string left out of the region
    types): the blocks of the region types, the tangent oracle and the enumeration of every path."""
    low, trimmed, n, x, V, HV = medium
    seg = W.segmented_compile(low, trimmed, n_slots=16)
    assert len(seg["overflow"]) == 0 and seg["stats"][7] == 0 and len(seg["rejected"]) == 2
    ok, err = vec_tol_ok(blocks_hv(seg, x, V), HV, 1e-10)
    assert ok, err
    Henum = enum_h(low, trimmed, x, n, max_paths=20000000)       # (in double: cancellation in g g^T - E[c c^T])
    ok, err = vec_tol_ok(Henum @ V, HV, 1e-9)
    assert ok, err


def test_overflow_strings_have_blocks(medium):
    """At 4 pool slots some strings of `medium` need more live nodes than slots and belong to no region type: their
    segments are blocks of their own, so the blocks still give H_f of every recognised string."""
    low, trimmed, n, x, V, HV = medium
    seg = W.segmented_compile(low, trimmed, n_slots=4)
    assert len(seg["overflow"]) > 0 and seg["stats"][7] == 0
    assert (seg["hb_slot"] == -1).sum() >= len(seg["overflow"])
    ok, err = vec_tol_ok(blocks_hv(seg, x, V), HV, 1e-10)
    assert ok, err


@pytest.mark.parametrize("lmin,lmax", [(4, 8), (32, 128)])
def test_strings_beyond_the_default_pool(lmin, lmax):
    """make_model(128, 16, 8, 4): most strings need more than the default 16 slots.  Either their blocks give H_f of every
    string, or stats[7] says the blocks are left out (a segment with more than 2^20 paths); never empty or partial
    blocks without the flag."""
    low = synth_low((128, 16, 8, 4), 7, 200, lmin, lmax, 9)
    trimmed, n = trim_all(low)
    seg = W.segmented_compile(low, trimmed, n_slots=16)
    assert len(seg["overflow"]) > 100
    x = np.random.RandomState(2).normal(-1.0, 0.5, size=n)
    if seg["stats"][7]:
        assert len(seg["hb_p"]) == 0 and lmax == 128
        return
    V = HO.directions(n, 4)
    HV = HO.hv(low, trimmed, x, V)
    assert np.abs(HV).max() > 0
    ok, err = vec_tol_ok(blocks_hv(seg, x, V), HV, 1e-10)
    assert ok, err


@pytest.mark.parametrize("R", [40, 70, 100])
def test_heavy_region_type(R):
    """x (yx)^R: one path-form type of weight R (enumeration would need 2^R paths).  The blocks, the oracle and the closed
    form -R/4 agree."""
    low = W.Lowered(W.parse(DIAMOND, "\nx%s 1\n" % ("yx" * R)))
    trimmed, n = trim_all(low)
    seg = W.segmented_compile(low, trimmed, n_slots=16)
    assert len(seg["hb_p"]) == 1 and seg["hb_p"][0] == R
    x = np.zeros(n)
    H = HO.full(low, trimmed, x)
    assert np.allclose(blocks_hv(seg, x, np.eye(n)), H, rtol=1e-13, atol=0)
    ab = [trimmed[low.trans_param[t]] for t in range(low.n_trans) if low.trans_edges[t]["state"] == "S" and low.trans_edges[t]["label"] in "AB"]
    assert len(ab) == 2 and min(ab) >= 0
    i, j = ab
    assert abs(H[i, i] + R / 4) <= 1e-15 * R and abs(H[j, j] + R / 4) <= 1e-15 * R and abs(H[i, j] - R / 4) <= 1e-15 * R
    assert np.abs(H).max() == pytest.approx(R / 4, rel=1e-15)
