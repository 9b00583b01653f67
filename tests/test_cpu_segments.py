"""Segmented compiled lattices (w-fsa_b200/csrc/lattice.cpp: compile_segments / compile_corpus_segmented)
checked on the CPU.  The arrays the device kernels kr_regions and ks_strings read
(w-fsa_b200/csrc/kernels_seg.cuh) are interpreted here word by word with the same recurrences and must
reproduce the oracle's per-string log q and expected edge counts.  This pins bridges, region words,
type merging, the group layouts and the constant accumulators without a GPU."""
import numpy as np
import pytest

import wfsa_b200 as W
from helpers import good_cases
from oracle import oracle as O
from test_cpu_lattice import compile_string
from wfsa_b200 import synth

EDGE, FIN, FIRST_IN, LAST_OUT = 1 << 31, 1 << 30, 1 << 29, 1 << 28
FX = float(2 ** 40)


def region_fwdbwd(col, aw, big):
    """(log q, {arc: posterior}) of one region given as its column of words."""
    pool = np.full(16, np.nan)
    pool[0] = 1.0
    xs = np.zeros(len(col))
    q, last, n_edges = None, None, 0
    for i, w in enumerate(col):
        w = int(w)
        if big and i % 16 == 15:
            assert not (w & (EDGE | FIN))
            for s in range(16):
                if w >> s & 1:
                    assert np.isfinite(pool[s]), "live slot without a value"
            continue
        if w & EDGE:
            src, dst, arc = (w >> 19) & 15, (w >> 23) & 15, w & 0xffff
            assert src != dst and np.isfinite(pool[src])
            assert bool(w & FIRST_IN) == (not np.isfinite(pool[dst])), "first_in flag must match slot liveness"
            xs[i] = pool[src] * aw[arc]
            pool[dst] = xs[i] if w & FIRST_IN else pool[dst] + xs[i]
            if w & LAST_OUT:
                pool[src] = np.nan                            # the slot is free again
            last = dst
            n_edges += 1
        elif w & FIN:
            assert big
            q = pool[w & 15]
            assert (w & 15) == last
        else:
            assert w == 0, "padding must be zero"
    if not big:
        q = pool[last]
    assert n_edges >= 2
    beta = np.full(16, np.nan)
    beta[last] = 1.0
    post = {}
    for i in range(len(col) - 1, -1, -1):
        w = int(col[i])
        if (big and i % 16 == 15) or not (w & EDGE):
            continue
        src, dst, arc = (w >> 19) & 15, (w >> 23) & 15, w & 0xffff
        c = aw[arc] * beta[dst]
        beta[src] = c if w & LAST_OUT else beta[src] + c
        post[arc] = post.get(arc, 0.0) + xs[i] * beta[dst] / q
    assert abs(beta[0] / q - 1.0) < 1e-12, "beta(entry) must equal q"
    return np.log(q), post


def interpret(seg, aw, n_arcs):
    """lq per type slot, acc per arc (float), log q per string id."""
    rgoff, rgrows, W_ = seg["rgoff"], seg["rgrows"], seg["typeW"]
    n_rg = len(rgrows)
    lq = np.zeros(n_rg * 32 + 1)
    acc = seg["const_acc"].astype(np.float64) / FX
    seen = set()
    n_path_types = n_dag_types = 0
    for g in range(n_rg):
        desc = int(rgrows[g])
        if desc & 0x10000:                                   # path form: PP paths (zero-weight padding) of L edges
            PP, L = (desc >> 8) & 0xff, desc & 0xff
            assert PP in (2, 3, 4, 6, 8) and 1 <= L <= 16
            assert rgoff[g + 1] - rgoff[g] == PP * L * 32
            block = seg["rwords"][rgoff[g]:rgoff[g + 1]].reshape(L, PP, 32).astype(np.int64)
            assert block.max() <= n_arcs
            awz = np.append(aw, 0.0)
            for l in range(32):
                if W_[g * 32 + l] == 0.0:
                    assert (block[:, :, l] == n_arcs).all()
                    continue
                key = (desc, block[:, :, l].tobytes())
                assert key not in seen, "identical regions must be merged into one type"
                seen.add(key)
                r = awz[block[:, :, l]].prod(axis=0)             # product along each path
                real = (block[:, :, l] != n_arcs).all(axis=0)
                assert real.sum() >= 2 and ((block[:, :, l] == n_arcs).all(axis=0) | real).all()
                q = r.sum()
                lq[g * 32 + l] = np.log(q)
                # every edge of path p receives the posterior r_p / q (one RED per (path, edge) on the device)
                for p_ in np.where(real)[0]:
                    for a_ in block[:, p_, l]:
                        acc[a_] += W_[g * 32 + l] * r[p_] / q
                n_path_types += 1
            continue
        rows = desc
        assert rows >= 16 and rows % 16 == 0       # every DAG-form region uses the stream format (CHECK every 16th word, FIN last)
        block = seg["rwords"][rgoff[g]:rgoff[g] + rows * 32].reshape(rows, 32)
        for l in range(32):
            col = block[:, l]
            if not (int(col[0]) & EDGE):
                assert W_[g * 32 + l] == 0.0 and not col.any()
                continue
            key = col.tobytes()
            assert key not in seen, "identical regions must be merged into one type"
            seen.add(key)
            assert W_[g * 32 + l] > 0.0
            lq[g * 32 + l], post = region_fwdbwd(col, aw, True)
            for arc, v in post.items():
                acc[arc] += W_[g * 32 + l] * v
            n_dag_types += 1
    interpret.counts = (n_path_types, n_dag_types)
    sgoff, sgref, ksid, kp = seg["sgoff"], seg["sgref"], seg["ksid"], seg["kp"]
    logq = {}
    with np.errstate(divide="ignore"):
        logaw = np.concatenate([np.log(aw), np.zeros(16)])          # 16 padding entries, one per bank pair
    SUPER, CH = 16, 8                                                # kKsSuper, kKsChunkRows
    assert len(sgref) == (len(sgoff) - 1) * SUPER and len(ksid) == len(sgref) * 32
    n_phase = n_conflict = 0
    for sg in range(len(sgoff) - 1):
        chunks = int((sgoff[sg + 1] - sgoff[sg]) // (SUPER * CH * 32))
        assert chunks >= 1 and sgoff[sg] + chunks * SUPER * CH * 32 == sgoff[sg + 1]
        blk = seg["swords"][sgoff[sg]:sgoff[sg + 1]].reshape(chunks, SUPER, CH, 32)
        for w in range(SUPER):
            g = sg * SUPER + w
            block = blk[:, w].reshape(chunks * CH, 32)                # the rows of group g in order
            pairs = block[sgref[g]:]
            for ids in (pairs & 0xffff, pairs >> 16):                 # one 8-byte table read per lane each
                for half in (ids[:, :16], ids[:, 16:]):               # a 64-bit shared load is served half-warp by half-warp
                    for row in half & 15:
                        cnt = np.bincount(row, minlength=16)
                        assert cnt.max() <= 2, "at most a two-way bank conflict per slot"
                        n_phase += 1
                        n_conflict += int(cnt.max() > 1)
            for l in range(32):
                sid = int(ksid[g * 32 + l])
                refs = block[:sgref[g], l].astype(np.int64)
                arcs = np.concatenate([pairs[:, l] & 0xffff, pairs[:, l] >> 16]).astype(np.int64)
                assert arcs.max(initial=0) < n_arcs + 16 and refs.max(initial=0) <= n_rg * 32
                if sid < 0:
                    assert (refs == n_rg * 32).all() and (arcs >= n_arcs).all() and kp[g * 32 + l] == 0.0
                    continue
                logq[sid] = logaw[arcs].sum() + lq[refs].sum()
    assert n_conflict <= 0.35 * max(n_phase, 1), "the schedule should leave most slots conflict free"
    return lq, acc, logq


def check(low, trimmed, x, n_slots=16):
    ltw, lew = low.edge_logweights(x, trimmed)
    pc, olq, oee = O.dp_eval(low, ltw, lew, want_counts=True)
    _, _, tid, eid = compile_string(low, trimmed, np.zeros(0, dtype=np.int32))
    with np.errstate(divide="ignore"):
        aw = np.exp(ltw[tid] + np.where(eid >= 0, lew[np.maximum(eid, 0)], 0.0))
    seg = W.segmented_compile(low, trimmed, n_slots=n_slots, fx_scale=FX)
    n_strings = len(low.offsets) - 1
    handled = set(int(s) for s in seg["ksid"] if s >= 0)
    assert handled.isdisjoint(seg["overflow"]) and handled.isdisjoint(seg["rejected"])
    assert len(handled) + len(seg["overflow"]) + len(seg["rejected"]) == n_strings
    for s in seg["rejected"]:
        assert pc[s] == 0 or not np.isfinite(olq[s])
    lq, acc, logq = interpret(seg, aw, len(tid))
    for s, v in logq.items():
        assert abs(v - olq[s]) <= 1e-12 * max(1.0, abs(olq[s])), (s, v, olq[s])
    st = seg["stats"]
    assert st[0] == np.count_nonzero(seg["typeW"]) and st[5] == len(handled) and st[0] <= st[1]
    # The objective without a per-string pass (kr_regions + the bridge partials of k_prep6):
    #   sum_s p_s log q_s = sum_arc c[arc] * log w[arc] + sum_types W_type * lq_type,  c = const_acc / fx_scale
    c = seg["const_acc"].astype(np.float64) / FX
    with np.errstate(divide="ignore"):
        ll_bridges = float(sum(c[a] * np.log(aw[a]) for a in np.nonzero(c)[0]))
    Wt = seg["typeW"]
    ll_regions = float(sum(Wt[i] * lq[i] for i in np.nonzero(Wt)[0]))
    ll_strings = float(sum(low.p[s_] * olq[s_] for s_ in handled))
    n_bridge_terms = max(int(st[4]), 1)                     # every bridge adds p_s rounded to the 2^-40 quantum of the test
    assert abs(ll_bridges + ll_regions - ll_strings) <= 1e-11 * max(1.0, abs(ll_strings)) + n_bridge_terms * 2.0 ** -40 * 20, \
        (ll_bridges, ll_regions, ll_strings)
    # expected edge counts of the handled strings only
    ee = np.zeros(low.n_trans + low.n_emis)
    np.add.at(ee, tid, acc)
    np.add.at(ee, low.n_trans + eid[eid >= 0], acc[eid >= 0])
    return seg, ee, oee, olq, handled


@pytest.mark.parametrize("case", good_cases(("fixtures", "random")), ids=lambda c: c["name"])
def test_segmented_form_matches_oracle(case):
    d = W.parse(case["fsa_text"], case["corpus_text"])
    low = W.Lowered(d)
    zt, ze = np.zeros(low.n_trans), np.zeros(low.n_emis)
    _, _, ee0 = O.dp_eval(low, zt, ze, want_counts=True)
    trimmed, n, _ = O.trim(low, ee0 > 0)
    x = np.random.RandomState(5).normal(-1.0, 0.7, size=n)
    seg, ee, oee, _, handled = check(low, trimmed, x)
    assert len(seg["overflow"]) == 0
    # the 2^-40 quantum of the constant accumulators bounds the absolute error per bridge
    assert np.allclose(ee, oee, rtol=1e-10, atol=1e-9)


def test_config4_shape_bridges_regions_and_type_merging():
    model = synth.make_model(64, 16, 4, 3, seed=11)
    low = model.lowered()
    offs, toks, w = model.corpus(600, 8, 60, seed=12)
    low.set_tokens(offs, toks, w / w.sum())
    zt, ze = np.zeros(low.n_trans), np.zeros(low.n_emis)
    _, _, ee0 = O.dp_eval(low, zt, ze)
    trimmed, n, _ = O.trim(low, ee0 > 0)
    x = np.random.RandomState(6).normal(-1.0, 0.5, size=n)
    seg, ee, oee, _, handled = check(low, trimmed, x)
    st = seg["stats"]
    assert len(seg["overflow"]) == 0 and len(handled) == 600
    assert st[4] > 0 and st[1] > st[0] > 0, "expected bridges and merged region types"
    assert st[7] == 0 and len(seg["hb_p"]) > 0, "the H_f path blocks fit"
    assert interpret.counts[0] > 0 and interpret.counts[1] > 0, "expected regions in path form and in DAG form"
    # DAG form only (bit 6 of n_slots): the same numbers, small and big DAG regions
    seg_d, ee_d, _, _, handled_d = check(low, trimmed, x, n_slots=16 | 64)
    assert interpret.counts[0] == 0 and len(handled_d) == 600
    dag_rows = seg_d["rgrows"]
    assert (dag_rows > 16).any() and (dag_rows <= 16).any(), "expected DAG regions of one and of several 16-word blocks"
    assert np.allclose(ee_d, oee, rtol=1e-10, atol=1e-9)
    assert np.allclose(ee, oee, rtol=1e-10, atol=1e-9)
    # a pool of 2 slots cannot hold an ambiguous region: such strings are reported, never mis-compiled
    seg2, _, _, _, handled2 = check(low, trimmed, x, n_slots=2)
    assert len(seg2["overflow"]) > 0 and len(handled2) < 600


def test_trimmed_arcs_are_removed_from_segments():
    model = synth.make_model(32, 8, 3, 2, seed=3)
    low = model.lowered()
    offs, toks, w = model.corpus(80, 5, 20, seed=4)
    low.set_tokens(offs, toks, w / w.sum())
    trimmed = np.arange(low.n_raw, dtype=np.int32)
    trimmed[::5] = -2                                     # weight 0: some strings lose paths or all of them
    x = np.random.RandomState(1).normal(-1.0, 0.5, size=low.n_raw)
    seg, _, _, olq, handled = check(low, trimmed, x)
    for s in range(80):
        assert (s in handled) == bool(np.isfinite(olq[s]))


def test_region_types_beyond_the_path_limit_of_the_hessian_blocks():
    """Eight emissions per state: some region types have more than 2^20 paths, too many for the H_f path blocks.  The
    evaluation does not need those blocks, so the shard still compiles: the region arrays as always, zero path blocks and
    the flag in stats[7].  The region arrays still reproduce the oracle's log q of every string (check)."""
    model = synth.make_model(256, 64, 8, 8, seed=1)
    low = model.lowered()
    offs, toks, w = model.corpus(5000, 32, 128, seed=2)
    low.set_tokens(offs, toks, w / w.sum())
    zt, ze = np.zeros(low.n_trans), np.zeros(low.n_emis)
    _, _, ee0 = O.dp_eval(low, zt, ze, nthreads=O.max_threads())
    trimmed, n, _ = O.trim(low, ee0 > 0)
    x = np.random.RandomState(3).normal(-1.0, 0.3, size=n)
    seg, ee, oee, olq, handled = check(low, trimmed, x)
    assert seg["stats"][7] == 1 and len(handled) > 4000
    assert seg["hb_path_off"].tolist() == [0] and seg["hb_col_off"].tolist() == [0] and seg["hb_val_off"].tolist() == [0]
    assert len(seg["hb_cols"]) == len(seg["hb_counts"]) == len(seg["hb_p"]) == len(seg["hb_slot"]) == 0


def _hessian_from_blocks(seg, x, n):
    """numpy restatement of k5_hessian over the path blocks the library derives from the region types."""
    H = np.zeros((n, n))
    po, co, vo = seg["hb_path_off"], seg["hb_col_off"], seg["hb_val_off"]
    for b in range(len(seg["hb_p"])):
        c = seg["hb_cols"][co[b]:co[b + 1]]
        M = seg["hb_counts"][vo[b]:vo[b + 1]].reshape(po[b + 1] - po[b], len(c))
        s = M @ x[c]
        r = np.exp(s - s.max()); r /= r.sum()
        g = M.T @ r
        H[np.ix_(c, c)] += seg["hb_p"][b] * (np.outer(g, g) - M.T @ (r[:, None] * M))
    return H


@pytest.mark.parametrize("case", good_cases(("fixtures", "random")), ids=lambda c: c["name"])
def test_hessian_blocks_from_region_types(case):
    """H_f = -sum_types W_type Cov_type(c_j, c_k): the path blocks built from the compiled region types (no enumeration per
    string; wfsa_dev.cu make_type_blocks) against the enumeration of every path of every string, which is what
    HessianLearner::ComputeHf does (/root/reference/src/HessianLearner.cpp:498-547; restated in oracle/wfsa_oracle.c)."""
    d = W.parse(case["fsa_text"], case["corpus_text"])
    low = W.Lowered(d)
    zt, ze = np.zeros(low.n_trans), np.zeros(low.n_emis)
    _, _, ee0 = O.dp_eval(low, zt, ze, want_counts=True)
    trimmed, n, _ = O.trim(low, ee0 > 0)
    if n == 0:
        pytest.skip("no parameters")
    x = np.random.RandomState(8).normal(-1.0, 0.7, size=n)
    seg = W.segmented_compile(low, trimmed, n_slots=16, fx_scale=FX)
    assert len(seg["overflow"]) == 0
    H = _hessian_from_blocks(seg, x, n)
    ltw, lew = low.edge_logweights(x, trimmed)
    params = np.concatenate([low.trans_param, low.emis_param])
    edge_param = np.array([trimmed[r] if r >= 0 and trimmed[r] >= 0 else -1 for r in params], dtype=np.int32)
    Href = O.enum_hessian(low, ltw, lew, edge_param, n)
    assert np.allclose(H, Href, rtol=1e-10, atol=1e-13), np.abs(H - Href).max()
