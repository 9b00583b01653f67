"""The reduction plan of the path-form region groups (w-fsa_b200/csrc/lattice.cpp: build_path_plans), interpreted on the
CPU the way kr_paths (w-fsa_b200/csrc/kernels_seg.cuh) walks it: every lane sums the values v[lane', p] its entries
name and adds each sum to the entry's arc.  The per-arc totals must equal those of one addition per cell of the group,
exactly (integers), and the plan must name every non-padding cell once."""
import numpy as np
import pytest

import wfsa_b200 as W
from oracle import oracle as O
from wfsa_b200 import synth

LAST = 1 << 31


@pytest.fixture(scope="module")
def shard():
    """A config-4-shaped shard (the benchmark's automaton and corpus seeds), trimmed as the benchmark trims it."""
    model = synth.make_model(256, 64, 8, 4, seed=1234)
    low = model.lowered()
    offs, toks, w = model.corpus(20000, 32, 128, seed=1235)
    low.set_tokens(offs, toks, w / w.sum())
    zt, ze = np.zeros(low.n_trans), np.zeros(low.n_emis)
    _, _, ee0 = O.dp_eval(low, zt, ze, want_counts=True)
    trimmed, _, _ = O.trim(low, ee0 > 0)
    return W.segmented_compile(low, trimmed, n_slots=16, fx_scale=2.0 ** 40)


def test_plan_sums_equal_cell_sums(shard):
    rw, go, gr, pw, pgo = shard["rwords"], shard["rgoff"], shard["rgrows"], shard["pwords"], shard["pgoff"]
    assert len(pgo) == len(gr) + 1 and pgo[0] == 0 and len(pw) == pgo[-1] + 32
    path = [g for g in range(len(gr)) if gr[g] & 0x10000]
    n_arcs = max(int(rw[go[g]:go[g + 1]].max()) for g in path)    # the padding arc: some cells of the path-form groups are padding
    rng = np.random.RandomState(5)
    n_path = n_cells = n_entries = 0
    for g in range(len(gr)):
        code = int(gr[g])
        plan = pw[pgo[g]:pgo[g + 1]].astype(np.int64).reshape(-1, 32)
        if not code & 0x10000:
            assert len(plan) == 0, "DAG-form groups have no plan"
            continue
        PP, L = (code >> 8) & 0xff, code & 0xff
        blk = rw[go[g]:go[g + 1]].astype(np.int64).reshape(L * PP, 32)
        v = rng.randint(-2 ** 40, 2 ** 40, size=(32, PP)).astype(np.int64)
        # one addition per non-padding cell (what a RED per cell adds)
        k, lane = np.nonzero(blk != n_arcs)
        cell_arc, cell_code = blk[k, lane], lane * 8 + k % PP
        want = np.zeros(n_arcs, np.int64)
        np.add.at(want, cell_arc, v[lane, k % PP])
        # the plan, lane by lane as kr_paths walks it
        got = np.zeros(n_arcs, np.int64)
        plan_code = []
        for ln in range(32):
            col = plan[:, ln]
            ends = np.nonzero(col & LAST)[0]
            used = ends[-1] + 1 if len(ends) else 0
            assert not col[used:].any(), "a stream ends in zero words"
            col = col[:used]
            if used == 0:
                continue
            entry = np.cumsum(col & LAST > 0) - (col & LAST > 0)
            arc, c = col & 0xffff, (col >> 16) & 0xff
            assert ((c & 7) < PP).all()
            first = np.r_[0, ends[:-1] + 1]
            assert (arc == arc[first][entry]).all(), "all words of an entry name one arc"
            s = np.zeros(len(ends), np.int64)
            np.add.at(s, entry, v[c >> 3, c & 7])
            np.add.at(got, arc[first], s)
            plan_code.append(arc * 256 + c)
            n_entries += len(ends)
        assert np.array_equal(got, want), "group %d: per-arc sums differ" % g
        # every non-padding cell once: the multisets of (arc, lane, path) agree
        assert np.array_equal(np.sort(np.concatenate(plan_code)), np.sort(cell_arc * 256 + cell_code)), "group %d: coverage" % g
        # dealt out evenly: no lane walks more than twice the ideal share
        assert len(plan) <= 2 * ((len(k) + 31) // 32), "group %d: %d plan rows for %d cells" % (g, len(plan), len(k))
        n_path += 1
        n_cells += len(k)
    assert n_path > 100 and n_entries < 0.8 * n_cells, (n_path, n_entries, n_cells)
    print("\npath-form groups %d, cells %d, plan entries (REDs) %d" % (n_path, n_cells, n_entries))
