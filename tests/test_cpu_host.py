"""CPU tests (no GPU): the C-ABI library loads and exports what include/*.h declares, the host
parsers reproduce the reference's counts and error behaviour on every golden case, and the
device entry point fails loudly (no CPU fallback) when there is no GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import wfsa_b200 as W
from helpers import all_cases, fnum, key, load_cases

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared(header):
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(wfsa_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = W.lib()
    names = declared("wfsa_dev.h") + declared("wfsa_host.h")
    assert len(names) >= 35
    for n in names:
        assert hasattr(lib, n), "libwfsa_b200.so does not export %s" % n
    assert set(W.DEV_SYMBOLS) <= set(names) and set(W.HOST_SYMBOLS) <= set(names)
    assert b"sm_100a" in lib.wfsa_dev_version()


@pytest.mark.parametrize("case", all_cases(), ids=lambda c: c["name"])
def test_parsers_match_reference_counts(case):
    if "reference_error" in case:
        with pytest.raises(W.WfsaError) as ei:
            W.parse(case["fsa_text"], case["corpus_text"])
        assert ei.value.code == 100 and "Invalid FSA format" in ei.value.message
        return
    d = W.parse(case["fsa_text"], case["corpus_text"])
    for k in ("corpus_size", "states", "transitions", "emissions", "raw_parameters", "raw_constraints"):
        assert d[k] == case[k], k
    assert abs(fnum(d["corpus_sum"]) - fnum(case["corpus_sum"])) < 1e-12
    assert [w["word"] for w in d["corpus"]] == [w["word"] for w in case["corpus"]]
    s = sum(fnum(w["weight"]) for w in d["corpus"])
    for mine, ref in zip(d["corpus"], case["corpus"]):
        assert abs(fnum(mine["weight"]) / s - fnum(ref["p"])) < 1e-15
    mine = {key(e): e for e in d["edges"]}
    assert set(mine) == {key(e) for e in case["edges"]}
    for e in case["edges"]:
        assert (mine[key(e)]["raw"] >= 0) == (e["raw"] >= 0)
        assert fnum(mine[key(e)]["file_logprob"]) == fnum(e["file_logprob"])


def test_parser_error_behaviour():
    ok_corpus = "\na 1\n"
    bad = {
        "start emits": "\n^\n$\n^ x 0\n^ a 0\na a 0\na $ 0\n",
        "duplicate emission": "\n^\n$\n^  0\n^ a 0\na a 0 a 1\na $ 0\n",
        "duplicate transition": "\n^\n$\n^  0\n^ a 0 a 1\na a 0\na $ 0\n",
        "into start": "\n^\n$\n^  0\n^ a 0\na a 0\na ^ 0 $ 0\n",
        "missing transitions": "\n^\n$\n^  0\n^ a 0\na a 0\nb b 0\n",
        "start == end": "\n^\n^\n^  0\n^ a 0\n",
    }
    for what, text in bad.items():
        with pytest.raises(W.WfsaError) as ei:
            W.parse(text, ok_corpus)
        assert ei.value.code == 100, what
    with pytest.raises(W.WfsaError) as ei:
        W.parse("\n^\n$\n^  0\n^ a 0\na a 0\na $ 0\n", "\na 1\na 2\n")
    assert "duplicate" in ei.value.message
    with pytest.raises(W.WfsaError):
        W.parse("\n^\n$\n^  0\n^ a 0\na a 0\na $ 0\n", "\na 0\n")          # weight must be normal
    with pytest.raises(W.WfsaError):
        W.parse("\n^\n$\n^  0\n^ a 0\na a 0\na $ 0\n", "\na -1\n")
    # a trailing separator is tolerated, a multi-character separator works, tokens are concatenated
    d = W.parse("::\n^\n$\n^::::0\n^::a::0\na::a::0::bb::1\na::$::0\n", "::\na::b::b::2::\nx::1\n")
    assert [w["word"] for w in d["corpus"]] == ["abb", "x"] and d["raw_parameters"] == 2


def test_lowering_descriptor_shapes():
    case = [c for c in all_cases() if c["name"] == "talk.wfsa+talk.corpus"][0]
    low = W.Lowered(W.parse(case["fsa_text"], case["corpus_text"]))
    assert low.n_states == 6 and low.n_trans == 6 and low.n_emis == 8 and low.n_raw == 7
    assert low.emis_row[-1] == 8 and low.trans_row[-1] == 6
    lens = np.diff(low.emis_tok_off)
    assert sorted(lens.tolist()) == [0, 0, 0, 1, 1, 2, 4, 4]          # "", "", "", s, s, ed, talk, talk
    assert low.offsets[-1] == sum(len(w) for w in low.words)


def test_no_cpu_fallback_without_gpu():
    """Without a CUDA device the product must fail loudly, not compute somewhere else."""
    case = [c for c in all_cases() if c["name"] == "talk.wfsa+talk.corpus"][0]
    low = W.Lowered(W.parse(case["fsa_text"], case["corpus_text"]))
    try:
        dev = W.Device(low)
    except W.WfsaError as e:
        assert e.code == 3 and "no CPU fallback" in e.message
        with pytest.raises(W.WfsaError):
            W.Session(case["fsa_text"], case["corpus_text"])
        assert W.lib().wfsa_dev_held_bytes() == 0
    else:
        dev.close()
        pytest.skip("a GPU is present")


def test_descriptor_validation():
    case = [c for c in all_cases() if c["name"] == "talk.wfsa+talk.corpus"][0]
    low = W.Lowered(W.parse(case["fsa_text"], case["corpus_text"]))
    low.trans_dst = low.trans_dst.copy()
    low.trans_dst[0] = 99
    with pytest.raises(W.WfsaError) as ei:
        W.Device(low)
    assert ei.value.code == 1                                          # WFSA_ERR_INVALID before any CUDA call


@pytest.mark.parametrize("fsa,corpus", [("test3.wfsa", "test.corpus"), ("talk.wfsa", "talk.corpus"), ("test5.wfsa", "test5.corpus"),
                                        ("test.list.wfsa", "test.corpus"), ("test.loop.wfsa", "test.corpus")])
@pytest.mark.parametrize("order", ["0", "1"])
def test_path_listing_matches_reference_binary(fsa, corpus, order, tmp_path):
    """-pr lists every accepting path of every corpus string (src/main.cpp:178-203).  The listing happens before the
    device is touched, so it can be compared here, without a GPU, against the reference binary's listing of the same
    data fixture (tests/golden/path_listing.json) -- as a set of lines: the reference's order follows its hash-map
    iteration -- and, string by string, against the reference's path counts (tests/golden/fixtures.json)."""
    import subprocess
    from collections import Counter
    name = fsa + "+" + corpus
    case = [c for c in load_cases("fixtures") if c["name"] == name][0]
    (tmp_path / fsa).write_bytes(case["fsa_text"].encode())
    (tmp_path / corpus).write_bytes(case["corpus_text"].encode())
    ours = os.path.join(ROOT, "w-fsa_b200", "_build", "wfsa")
    args = ["-a", str(tmp_path / fsa), "-c", str(tmp_path / corpus), "-pr", "-r", order, "-e", "0", "-s"]
    got = sorted(ln for ln in subprocess.run([ours] + args, capture_output=True, text=True).stderr.splitlines() if " -> " in ln)
    want = load_cases("path_listing")[name]
    assert want and got == want
    paths = Counter(ln.split(": ", 1)[0] for ln in got)
    assert {w["word"]: paths[w["word"]] for w in case["corpus"]} == {w["word"]: w["paths"] for w in case["corpus"]}


def test_cli_gpus_option_without_a_device(tmp_path):
    """`wfsa --gpus N` forks one process per GPU before anything touches CUDA and hands the communicator id down a pipe.
    Without a device every rank must fail loudly (no CPU fallback), rank 0 must collect the children and return 1, and
    out-of-range values must be refused before any fork."""
    import os
    import subprocess
    exe = os.path.join(ROOT, "w-fsa_b200", "_build", "wfsa")
    fsa = tmp_path / "t.wfsa"; corpus = tmp_path / "t.corpus"
    fsa.write_text("\n^\n$\n^  0\n^ A 0\nA a 0\nA A 0 $ 0\n")
    corpus.write_text("\na 1\naa 2\n")
    r = subprocess.run([exe, "-a", str(fsa), "-c", str(corpus), "--gpus", "9"], capture_output=True, text=True, timeout=60)
    assert r.returncode == 1 and "--gpus must be between 1 and 8" in r.stderr
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        pytest.skip("a GPU is present (tests/test_gpu_parity.py::test_cli_two_gpus_same_table covers the working path)")
    r = subprocess.run([exe, "-a", str(fsa), "-c", str(corpus), "-opt", "QuasiNewton", "-i", "7", "-e", "2", "--gpus", "2"],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 1
    assert any(m in r.stderr for m in ("no CPU fallback", "libnccl", "communicator", "a rank ended with an error")), r.stderr[-2000:]


@pytest.mark.parametrize("seed", [0, 1, 2, 3, 30])
def test_kkt_diagonal_schur_complement_against_dense_factorisation(seed):
    """The Newton system of HessianLearner without H_f, [D B; B^T 0] (src/HessianLearner.cpp:622-639; the reference hands it
    to MKL DSS, :100-113): the O(n) solve through the diagonal Schur complement that the optimiser uses must give the
    solution and the inertia of the dense Bunch-Kaufman factorisation -- multipliers of both signs, groups of 1..9
    parameters.  (Seed 30: 340 constraints, ~1 700 parameters -- large enough for the factorisation to run its trailing
    updates on a team of host threads.)"""
    import ctypes as C
    rng = np.random.RandomState(seed)
    k = 40 + 10 * seed
    sizes = rng.randint(1, 10, size=k)
    ccol = np.repeat(np.arange(k), sizes).astype(np.int32)
    n = len(ccol)
    expx = np.exp(rng.normal(-1.0, 1.0, size=n))
    lam = rng.normal(0.0, 1.0, size=k)
    lam[np.abs(lam) < 0.05] = 0.3
    rhs = rng.normal(size=n + k)
    s1, s2 = np.zeros(n + k), np.zeros(n + k)
    inertia = np.zeros(4, dtype=np.int32)
    L = W.lib()
    L.wfsa_host_kkt_solve.argtypes = [C.c_int32, C.c_int32, W.F64P, W.F64P, W.I32P, W.F64P, W.F64P, W.F64P, W.I32P]
    rc = L.wfsa_host_kkt_solve(n, k, W._p(expx, W.F64P), W._p(lam, W.F64P), W._p(ccol, W.I32P), W._p(rhs, W.F64P),
                               W._p(s1, W.F64P), W._p(s2, W.F64P), W._p(inertia, W.I32P))
    assert rc == 0
    K = np.zeros((n + k, n + k))
    K[np.arange(n), np.arange(n)] = expx * lam[ccol]
    K[np.arange(n), n + ccol] = expx
    K[n + ccol, np.arange(n)] = expx
    ref = np.linalg.solve(K, rhs)
    assert np.allclose(s1, ref, rtol=1e-9, atol=1e-9 * np.abs(ref).max())
    assert np.allclose(s2, ref, rtol=1e-8, atol=1e-8 * np.abs(ref).max())
    ev = np.linalg.eigvalsh(K)
    assert (inertia[0], inertia[1]) == (int((ev > 0).sum()), int((ev < 0).sum())) == (inertia[2], inertia[3])
    # a multiplier that is exactly zero: the Schur path declines (the optimiser then factorises densely)
    lam[3] = 0.0
    rc = L.wfsa_host_kkt_solve(n, k, W._p(expx, W.F64P), W._p(lam, W.F64P), W._p(ccol, W.I32P), W._p(rhs, W.F64P),
                               W._p(s1, W.F64P), W._p(s2, W.F64P), W._p(inertia, W.I32P))
    assert rc == 1
