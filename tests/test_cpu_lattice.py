"""Host lattice compiler (w-fsa_b200/csrc/lattice.cpp) checked on the CPU: the compiled stream of every
string is interpreted here word by word -- the same forward / backward recurrences the DAG form of region
types runs on the device (big_fwd / big_bwd, w-fsa_b200/csrc/kernels_seg.cuh) -- and must reproduce the
oracle's log q and expected edge counts.  This pins the stream format and the slot / flag / CHECK logic
without a GPU; the device kernels themselves are checked against the oracle in test_gpu_parity.py."""
import ctypes as C

import numpy as np
import pytest

import wfsa_b200 as W
from helpers import good_cases
from oracle import oracle as O
from wfsa_b200 import synth

EDGE, FIN, FIRST_IN, LAST_OUT, BRIDGE = 1 << 31, 1 << 30, 1 << 29, 1 << 28, 1 << 27
CHECK_EVERY = 16


def compile_string(low, trimmed, toks, n_slots=16):
    L = W.lib()
    fd = low.fsa_desc()
    cap = 64 + 40 * (len(toks) + 2) * 16
    words = np.zeros(cap, dtype=np.uint32)
    nw, na = C.c_int64(), C.c_int32()
    acap = 1 << 16
    tid, eid = np.zeros(acap, dtype=np.int32), np.zeros(acap, dtype=np.int32)
    t = np.ascontiguousarray(toks, dtype=np.int32)
    tr = None if trimmed is None else np.ascontiguousarray(trimmed, dtype=np.int32)
    rc = L.wfsa_lattice_compile(C.byref(fd), W._p(tr, W.I32P), W._p(t, W.I32P), len(t), n_slots,
                                words.ctypes.data_as(C.POINTER(C.c_uint32)), cap, C.byref(nw), W._p(tid, W.I32P),
                                W._p(eid, W.I32P), acap, C.byref(na))
    assert rc == 0, L.wfsa_dev_last_error(None)
    return nw.value, words[:max(nw.value, 0)].copy(), tid[:na.value].copy(), eid[:na.value].copy()


def interpret(words, aw):
    """(log q, posterior per arc) of one stream; checks the structural invariants on the way."""
    pool = np.full(16, np.nan)
    pool[0] = 1.0
    xs = np.zeros(len(words))
    live_seen = None
    for i, w in enumerate(words):
        w = int(w)
        if i % CHECK_EVERY == CHECK_EVERY - 1:
            assert not (w & (EDGE | FIN)), "CHECK index must hold a CHECK word"
            live_seen = w & 0xffff
            for s in range(16):
                if live_seen >> s & 1:
                    assert np.isfinite(pool[s]), "live slot without a value"
            continue
        if w & EDGE:
            src, dst, arc = (w >> 19) & 15, (w >> 23) & 15, w & 0xffff
            assert src != dst and np.isfinite(pool[src])
            x = pool[src] * aw[arc]
            xs[i] = x
            pool[dst] = x if w & FIRST_IN else pool[dst] + x
        elif w & FIN:
            assert i == len(words) - 1
            q = pool[w & 15]
    post = np.zeros(len(aw))
    bridge_ok = True
    pool = np.full(16, np.nan)
    for i in range(len(words) - 1, -1, -1):
        w = int(words[i])
        if i % CHECK_EVERY == CHECK_EVERY - 1:
            for s in range(16):
                if (w & 0xffff) >> s & 1:
                    assert np.isfinite(pool[s]), "live slot without a beta"
            continue
        if w & EDGE:
            src, dst, arc = (w >> 19) & 15, (w >> 23) & 15, w & 0xffff
            bd = pool[dst]
            c = aw[arc] * bd
            pool[src] = c if w & LAST_OUT else pool[src] + c
            pst = xs[i] * bd / q
            post[arc] += pst
            if w & BRIDGE:
                bridge_ok = bridge_ok and abs(pst - 1.0) < 1e-12
        elif w & FIN:
            pool[w & 15] = 1.0
    assert bridge_ok, "an edge flagged as bridge has posterior != 1"
    assert abs(pool[0] / q - 1.0) < 1e-12, "beta(start) must equal q"
    return np.log(q), post


def check_against_oracle(low, trimmed, n, x, n_slots=16):
    ltw, lew = low.edge_logweights(x, trimmed)
    pc, olq, oee = O.dp_eval(low, ltw, lew, want_counts=True)
    ee = np.zeros(low.n_trans + low.n_emis)
    n_edges = n_bridge = n_over = 0
    for s in range(len(low.offsets) - 1):
        toks = low.tokens[low.offsets[s]:low.offsets[s + 1]]
        nw, words, tid, eid = compile_string(low, trimmed, toks, n_slots)
        if nw == -1:
            n_over += 1
            continue
        if nw == 0:
            assert not np.isfinite(olq[s]) or pc[s] == 0
            continue
        aw = np.exp(ltw[tid] + np.where(eid >= 0, lew[np.maximum(eid, 0)], 0.0))
        lq, post = interpret(words, aw)
        assert abs(lq - olq[s]) <= 1e-12 * max(1.0, abs(olq[s])), (s, lq, olq[s])
        np.add.at(ee, tid, low.p[s] * post)
        np.add.at(ee, low.n_trans + eid[eid >= 0], low.p[s] * post[eid >= 0])
        n_edges += int(np.sum(words >> 31))
        n_bridge += int(np.sum((words & BRIDGE) != 0))
    return ee, oee, n_edges, n_bridge, n_over


@pytest.mark.parametrize("case", good_cases(("fixtures", "random")), ids=lambda c: c["name"])
def test_compiled_lattice_matches_oracle(case):
    d = W.parse(case["fsa_text"], case["corpus_text"])
    low = W.Lowered(d)
    zt, ze = np.zeros(low.n_trans), np.zeros(low.n_emis)
    pc, _, ee0 = O.dp_eval(low, zt, ze, want_counts=True)
    trimmed, n, _ = O.trim(low, ee0 > 0)
    x = np.random.RandomState(5).normal(-1.0, 0.7, size=n)
    ee, oee, _, _, n_over = check_against_oracle(low, trimmed, n, x)
    assert n_over == 0
    assert np.allclose(ee, oee, rtol=1e-11, atol=1e-14)


def test_config4_shape_streams_bridges_and_overflow():
    model = synth.make_model(64, 16, 4, 3, seed=11)
    low = model.lowered()
    offs, toks, w = model.corpus(300, 8, 40, seed=12)
    low.set_tokens(offs, toks, w / w.sum())
    zt, ze = np.zeros(low.n_trans), np.zeros(low.n_emis)
    _, _, ee0 = O.dp_eval(low, zt, ze)
    trimmed, n, _ = O.trim(low, ee0 > 0)
    x = np.random.RandomState(6).normal(-1.0, 0.5, size=n)
    ee, oee, n_edges, n_bridge, n_over = check_against_oracle(low, trimmed, n, x)
    assert n_over == 0 and n_bridge > 0 and n_edges > n_bridge
    assert np.allclose(ee, oee, rtol=1e-11, atol=1e-14)
    # a pool of 2 slots cannot hold ambiguous strings: they must be reported, never mis-compiled
    _, _, _, _, n_over2 = check_against_oracle(low, trimmed, n, x, n_slots=2)
    assert n_over2 > 0


def test_trimmed_arcs_are_removed():
    model = synth.make_model(32, 8, 3, 2, seed=3)
    low = model.lowered()
    offs, toks, w = model.corpus(50, 5, 20, seed=4)
    low.set_tokens(offs, toks, w / w.sum())
    trimmed = np.arange(low.n_raw, dtype=np.int32)
    trimmed[::5] = -2                                     # weight 0: some strings lose paths or all of them
    n = low.n_raw
    x = np.random.RandomState(1).normal(-1.0, 0.5, size=n)
    ltw, lew = low.edge_logweights(x, trimmed)
    pc, olq, _ = O.dp_eval(low, ltw, lew, want_counts=True)
    for s in range(len(offs) - 1):
        nw, words, tid, eid = compile_string(low, trimmed, toks[offs[s]:offs[s + 1]])
        if not np.isfinite(olq[s]):
            assert nw == 0
        else:
            aw = np.exp(ltw[tid] + np.where(eid >= 0, lew[np.maximum(eid, 0)], 0.0))
            assert np.all(np.isfinite(aw[words[(words >> 31) == 1] & 0xffff]))
            lq, _ = interpret(words, aw)
            assert abs(lq - olq[s]) <= 1e-12 * max(1.0, abs(olq[s]))
