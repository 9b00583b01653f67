"""k_eval6, the single-launch evaluation of the segmented kernel, under every schedule of its region phase (P1 in
w-fsa_b200/csrc/kernels_eval6.cuh) and through the host-buffer (graph) call, against the CPU forward-backward.

How a big DAG group is walked depends on the number of big groups (n_big, 32 distinct region types each) against the
persistent grid (one CTA per SM unless WFSA_E6_GRID caps it):
  A  n_big * 4 <= grid: two warps per group (big_fwd / big_bwd<false> / big_red<true>), the owning CTA dedicated to it;
  B  grid / 4 < n_big <= grid: the same two-warp chain, its CTA also taking regular groups;
  C  n_big > grid: one warp per group staged in shared memory (big_one<BigSmem>); with n_big > 16 * grid a warp
     owns several groups and re-stages the later ones;
  D  no staging area (WFSA_E6_NO_STAGING=1): one warp per group, streamed from HBM (big_one<BigGmem>, as kr_regions).
A group longer than the staging area is streamed while the others are staged ("mixed").  Every posterior and every
log-likelihood term is rounded once to 64-bit fixed point and the rounded values are summed as integers, and the two-warp
chain forms the one-warp chain's posteriors bitwise (kernels_seg.cuh, big_sc), so every schedule must return the same bits;
each must also meet the oracle tolerances of test_gpu_parity.py.  Each schedule asserts, through wfsa_dev_info, the regime it claims to run."""
import time

import numpy as np
import pytest

import wfsa_b200 as W
from helpers import vec_tol_ok
from oracle import oracle as O
from wfsa_b200 import synth

pytestmark = pytest.mark.gpu

KNOBS = ("WFSA_E6_GRID", "WFSA_E6_STATIC", "WFSA_E6_DED_DIV", "WFSA_E6_NO_DEDICATE", "WFSA_E6_NO_STAGING", "WFSA_E6_DEBUG",
         "WFSA_E6_PLAIN_LAUNCH", "WFSA_EVAL6_OFF", "WFSA_NO_GRAPH", "WFSA_E2E_COPY_NODE")
OFF = "pipeline"            # WFSA_EVAL6_OFF: the general pipeline, not k_eval6

# name -> (model shape + seed, corpus (strings, lmin, lmax, seed), regime of the default schedule, extra schedules).
# A schedule is (label, environment, regime it must run, True if some warp must own several big groups).  n_big in the
# comments was counted on the host for these seeds; the tests read it from the device.
CORPORA = {
    # config 4, 3 000 strings (and two that are not recognised): n_big 1, 48 rows
    "medium": ((256, 64, 8, 4, 11), (3000, 32, 128, 12), "A", [
        ("no dedicate", {"WFSA_E6_NO_DEDICATE": "1"}, "B", False),
        ("ded div 1", {"WFSA_E6_DED_DIV": "1"}, "A", False),
        ("grid 4", {"WFSA_E6_GRID": "4"}, "A", False),
        ("grid 1", {"WFSA_E6_GRID": "1"}, "B", False)]),
    # 40 strings of 3 500-4 000 tokens: n_big 19, 128 rows
    "long": ((64, 16, 4, 3, 21), (40, 3500, 4000, 22), "A", [
        ("no dedicate", {"WFSA_E6_NO_DEDICATE": "1"}, "B", False),
        ("grid 4", {"WFSA_E6_GRID": "4"}, "C", False),
        ("grid 1", {"WFSA_E6_GRID": "1"}, "C", True),
        ("grid 4, no staging", {"WFSA_E6_GRID": "4", "WFSA_E6_NO_STAGING": "1"}, "D", False)]),
    # five emissions per state, 40 000 strings: n_big 59, 96 rows, two staging areas
    "c5emis": ((256, 64, 8, 5, 1), (40000, 32, 128, 2), "B", [
        ("ded div 1", {"WFSA_E6_DED_DIV": "1"}, "A", False),
        ("grid 2", {"WFSA_E6_GRID": "2"}, "C", True),
        ("grid 1", {"WFSA_E6_GRID": "1"}, "C", True)]),
    # config 4, 200 000 strings: n_big 25, 64 rows
    "c4_200k": ((256, 64, 8, 4, 1234), (200000, 32, 128, 1236), "A", [
        ("no dedicate", {"WFSA_E6_NO_DEDICATE": "1"}, "B", False),
        ("grid 1", {"WFSA_E6_GRID": "1"}, "C", True)]),
    # six emissions per state: n_big 40, one group of 160 rows does not fit the one staging area (144 rows): staged and
    # streamed big groups in one launch
    "mixed": ((256, 64, 8, 6, 3), (6000, 32, 128, 103), "mixed", [
        ("grid 4", {"WFSA_E6_GRID": "4"}, "mixed", False)]),
}


def schedules(name):
    default = CORPORA[name][2]
    return ([("default", {}, default, False),
             ("static 0", {"WFSA_E6_STATIC": "0"}, default, False),
             ("static 100", {"WFSA_E6_STATIC": "100"}, default, False)]
            + CORPORA[name][3]
            + [("no staging", {"WFSA_E6_NO_STAGING": "1"}, "D", False),
               ("eval6 off", {"WFSA_EVAL6_OFF": "1"}, OFF, False)])


def regime(info):
    """The P1 schedule k_eval6 runs, from the conditions in kernels_eval6.cuh (wfsa_dev_info e6_*)."""
    if not info["eval_path"] & 1:
        return OFF
    nb = info["e6_big_groups"]
    if nb == 0:
        return "none"
    if info["e6_two_warp_eligible"] == nb:
        return "A" if info["e6_big_dedicate"] else "B"
    if info["e6_big_slots"] == 0:
        return "D"
    if nb > info["grid"] and info["e6_max_big_rows"] <= info["e6_big_rows"]:
        return "C"
    if info["e6_max_big_rows"] > info["e6_big_rows"]:
        return "mixed"
    return "other"


_lowered = {}


def corpus(name):
    if name not in _lowered:
        (S, A, D, E, seed), (count, lmin, lmax, cseed) = CORPORA[name][:2]
        model = synth.make_model(S, A, D, E, seed=seed)
        low = model.lowered()
        offs, toks, w = model.corpus(count, lmin, lmax, seed=cseed)
        if name == "medium":                  # two strings that are not recognised: an unknown symbol, random junk
            toks = toks.copy()
            toks[offs[5]] = -1
            toks[offs[9]:offs[10]] = np.random.RandomState(5).randint(0, 64, size=offs[10] - offs[9])
        low.set_tokens(offs, toks, w / w.sum())
        _lowered[name] = low
    return _lowered[name]


def build_device(low):
    dev = W.Device(low)
    rec, pc, used = dev.structure()
    params = np.concatenate([low.trans_param, low.emis_param])
    trimmed, n, _ = O.trim(low, np.array([r < 0 or used[r] for r in params]))
    dev.set_param_map(trimmed, n, rec)
    return dev, rec.astype(bool), trimmed, n


def to_params(low, trimmed, n, ee):
    """per-edge values -> per trimmed parameter (the gradient is -sum_s p_s E_s[count])"""
    g = np.zeros(n)
    for e, r in enumerate(np.concatenate([low.trans_param, low.emis_param])):
        if r >= 0 and trimmed[r] >= 0:
            g[trimmed[r]] = ee[e]
    return g


def oracle(low, trimmed, n, x):
    ltw, lew = low.edge_logweights(x, trimmed)
    _, olq, oee = O.dp_eval(low, ltw, lew, nthreads=O.max_threads())
    return olq, -to_params(low, trimmed, n, oee)


def weights_and_oracle(low, trimmed, n, rec):
    """x ~ N(-1, 0.3); N(-12, 3): alpha of a 48-row region falls far below 2^-200 and the CHECK words must rescale it
    (both chains, and sc = scalbn(sc0, Et + F - EQ) for the posteriors); N(+2.5, 1): alpha grows, rescaled the other way;
    the first x with one component at -inf.  That component is the least used parameter (smallest gradient) that lies on
    every path of some recognised string, so that a few strings get q = 0."""
    rng = np.random.RandomState(31)
    xs = [rng.normal(-1.0, 0.3, size=n), rng.normal(-12.0, 3.0, size=n), rng.normal(2.5, 1.0, size=n)]
    refs = [oracle(low, trimmed, n, x) for x in xs]
    g = np.abs(refs[0][1])
    first = None
    for i in [i for i in np.argsort(g) if g[i] > 0][:64]:
        xi = xs[0].copy()
        xi[i] = -np.inf
        ref = oracle(low, trimmed, n, xi)
        first = first or (xi, ref)
        if (rec & np.isneginf(ref[0])).any():
            return xs + [xi], refs + [ref]
    return xs + [first[0]], refs + [first[1]]           # (very ambiguous strings: every string keeps a path, loglik is finite)


def sub_corpus(low, keep):
    sub = type(low).__new__(type(low))
    sub.__dict__.update(low.__dict__)
    offs = np.concatenate([[0], np.cumsum(np.diff(low.offsets)[keep])])
    toks = np.concatenate([low.tokens[low.offsets[i]:low.offsets[i + 1]] for i in keep])
    sub.set_tokens(offs, toks, low.p[keep])
    return sub


def clear_knobs(monkeypatch):
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)


def check_against_oracle(low, trimmed, n, rec, x, out, ref, label):
    ll, logq, grad = out
    olq, og = ref
    p = low.p
    pos = rec & np.isfinite(olq)
    assert np.allclose(logq[pos], olq[pos], rtol=1e-11, atol=1e-10), label
    assert np.isneginf(logq[~pos]).all(), label
    if pos.sum() == rec.sum():
        assert abs(ll - float(np.dot(p[rec], olq[rec]))) <= 1e-11 * abs(ll), label
        ok, err = vec_tol_ok(grad, og, 1e-9)
        assert ok, (label, err)
        return
    # x with a component at -inf: some recognised strings have q = 0.  loglik is -inf.  The oracle's gradient sums over
    # the strings with q > 0; the device's also holds the bridge edges of the q = 0 strings (their posterior, 1, is folded
    # into constant accumulators when the parameter map is set, before any x is known: const_acc in lattice.cpp) and
    # the posteriors of their region types whose q is not 0.  So only the parameters that no q = 0 string touches are
    # compared with the oracle; the rest are pinned by the bitwise agreement of all schedules.
    assert ll == -np.inf, label
    zero = np.where(rec & ~pos)[0]
    zt, ze = low.edge_logweights(np.zeros(n), trimmed)
    _, _, zee = O.dp_eval(sub_corpus(low, zero), zt, ze, nthreads=O.max_threads())
    untouched = to_params(low, trimmed, n, zee) == 0
    assert untouched.any(), label                       # (one 4 000-token string touches nearly every parameter)
    ok, err = vec_tol_ok(grad[untouched], og[untouched], 1e-9)
    assert ok, (label, err)


@pytest.mark.parametrize("name", list(CORPORA))
def test_every_schedule_same_bits_and_oracle(name, monkeypatch):
    t0 = time.perf_counter()
    clear_knobs(monkeypatch)
    low = corpus(name)
    xs = refs = trimmed0 = None
    first = None
    for label, env, want, restage in schedules(name):
        with monkeypatch.context() as m:
            for k, v in env.items():
                m.setenv(k, v)
            dev, rec, trimmed, n = build_device(low)            # (the environment is read when the handle is made and at launches)
            info = dev.info()
            print("\n%-8s %-20s regime %-8s n_big %4d  grid %3d  dedicate %d  big_slots %d  big_rows %3d  longest %3d  two-warp %d"
                  % (name, label, regime(info), info["e6_big_groups"], info["grid"], info["e6_big_dedicate"], info["e6_big_slots"],
                     info["e6_big_rows"], info["e6_max_big_rows"], info["e6_two_warp_eligible"]), end="")
            assert info["kernel"] == 6 and info["n_overflow_strings"] == 0, (label, info["n_overflow_strings"])
            assert regime(info) == want, (label, regime(info), want)
            if restage:
                assert info["e6_big_groups"] > 16 * info["grid"] and info["e6_big_slots"] >= 1, label
            if "WFSA_E6_GRID" in env:
                assert info["grid"] == min(int(env["WFSA_E6_GRID"]), info["sm_count"]), label
            else:
                assert info["grid"] == info["sm_count"], label
            if xs is None:
                trimmed0 = trimmed
                xs, refs = weights_and_oracle(low, trimmed, n, rec)
            assert np.array_equal(trimmed, trimmed0), label
            outs = [dev.eval(x) for x in xs]
            dev.close()
        for x, out, ref in zip(xs, outs, refs):
            check_against_oracle(low, trimmed, n, rec, x, out, ref, label)
        if want == OFF:
            # The general pipeline takes its arc weights as exp(x_t + x_e) (k_arc_weights_log, kernels_seg.cuh: aw[i] = exp(l));
            # k_eval6 as exp(x_t) * exp(x_e) (kernels_eval6.cuh P0: w = ex[tp.x] * ex[tp.y]).  The weights differ in the last
            # bit, so this schedule is held to the oracle tolerances above only.
            continue
        if first is None:
            first = outs
            continue
        for out, ref in zip(outs, first):
            assert out[0] == ref[0], (label, out[0], ref[0])
            assert np.array_equal(out[2], ref[2]), (label, "grad", int(np.sum(out[2] != ref[2])))
            assert np.array_equal(out[1], ref[1]), (label, "log q", int(np.sum(out[1] != ref[1])))
    print("\n%s: %d schedules, %.1f s" % (name, len(schedules(name)), time.perf_counter() - t0))


def eval_resident(dev, x, want_logq=False):
    dev.upload_x(x)
    dev.eval_launch()
    return dev.eval_fetch(want_logq=want_logq)


@pytest.mark.parametrize("name", ["medium", "c5emis"])
def test_host_buffer_call(name, monkeypatch):
    """wfsa_dev_eval without log q replays k_eval6 as a CUDA graph that reads x from mapped host memory and writes its
    results there.  Same bits as upload / launch / fetch, also when the two alternate (epoch parity, ctl[4..6], results on
    the host or on the device) and when log q is fetched after a graph call (k_arc_logw reads the x that CTA 0 copied)."""
    t0 = time.perf_counter()
    clear_knobs(monkeypatch)
    low = corpus(name)
    dev, rec, trimmed, n = build_device(low)
    info = dev.info()
    assert info["eval_path"] & 1 and regime(info) == CORPORA[name][2], regime(info)
    rng = np.random.RandomState(41)
    xs = [rng.normal(*[(-1.0, 0.3), (-12.0, 3.0), (2.5, 1.0)][k % 3], size=n) for k in range(6)]
    ref = [eval_resident(dev, x, want_logq=True) for x in xs]
    # graph, then log q of that same evaluation
    for x, (ll, logq, grad) in zip(xs, ref):
        ll2, none, grad2 = dev.eval(x, want_logq=False)
        assert none is None and ll2 == ll and np.array_equal(grad2, grad)
        ll3, logq3, grad3 = dev.eval_fetch(want_logq=True)
        assert ll3 == ll and np.array_equal(logq3, logq) and np.array_equal(grad3, grad)
    dev.eval(xs[1], want_logq=False)
    dev.eval(xs[0], want_logq=False)
    ll, logq, grad = dev.eval_fetch(want_logq=True)
    olq, og = oracle(low, trimmed, n, xs[0])
    assert np.allclose(logq[rec], olq[rec], rtol=1e-11, atol=1e-10) and np.isneginf(logq[~rec]).all()
    assert abs(ll - float(np.dot(low.p[rec], olq[rec]))) <= 1e-11 * abs(ll)
    ok, err = vec_tol_ok(grad, og, 1e-9)
    assert ok, err
    # graph and launch / fetch alternating, each call with its own x: the epoch goes through both parities many times
    order = [0, 1, 2, 3, 4, 5, 5, 3, 1, 0, 2, 4, 4, 1]
    for k, i in enumerate(order):
        if k % 2 == 0:
            ll, _, grad = dev.eval(xs[i], want_logq=False)
        else:
            ll, grad = eval_resident(dev, xs[i])
        assert ll == ref[i][0] and np.array_equal(grad, ref[i][2]), (k, i)
    dev.close()
    for env in ({"WFSA_NO_GRAPH": "1"}, {"WFSA_E2E_COPY_NODE": "1"}):
        with monkeypatch.context() as m:
            for k, v in env.items():
                m.setenv(k, v)
            d2, _, _, _ = build_device(low)
            assert d2.info()["eval_path"] & 1
            for x, (ll, logq, grad) in zip(xs[:3], ref):
                ll2, _, grad2 = d2.eval(x, want_logq=False)
                assert ll2 == ll and np.array_equal(grad2, grad), env
                ll3, logq3, grad3 = d2.eval_fetch(want_logq=True)
                assert ll3 == ll and np.array_equal(logq3, logq) and np.array_equal(grad3, grad), env
            d2.close()
    print("\nhost-buffer call, %s: %.1f s" % (name, time.perf_counter() - t0))
