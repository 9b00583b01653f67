"""H_f of the device (wfsa_dev_hessian, Session.hessian) against the tangent forward-backward of tests/hessian_oracle.c,
which does not enumerate paths: so at realistic corpus sizes, at any scale of x, for strings that no region type of the
segmented kernel covers, and for region types whose weight is far above 1.  H @ V is compared for V = 32 Gaussian
directions and 16 unit columns (the full H where n <= 600), 1e-9 relative per component with a floor of 1e-6 * max|.|
(vec_tol_ok: H is summed in 64-bit fixed point)."""
import ctypes as C

import numpy as np
import pytest

import hessian_oracle as HO
import minpath_oracle as MP
import wfsa_b200 as W
from helpers import key, vec_tol_ok
from oracle import oracle as O
from test_cpu_hessian import DIAMOND
from wfsa_b200 import synth

pytestmark = pytest.mark.gpu


def mapped_device(low, **kw):
    dev = W.Device(low, **kw)
    rec, pc, used = dev.structure()
    params = np.concatenate([low.trans_param, low.emis_param])
    trimmed, n, _ = O.trim(low, np.array([r < 0 or used[r] for r in params]))
    dev.set_param_map(trimmed, n, rec)
    return dev, trimmed, n


def device_hessian(dev, x):
    """(H, rmin) of wfsa_dev_hessian."""
    xx = np.ascontiguousarray(x, dtype=np.float64)
    H = np.zeros((dev.n, dev.n))
    rm = C.c_double(-1.0)
    dev._ck(dev.L.wfsa_dev_hessian(dev.h, W._p(xx, W.F64P), W._p(H, W.F64P), C.byref(rm)))
    return H, rm.value


def directions(n, seed):
    return np.eye(n) if n <= 600 else HO.directions(n, seed)


def check_hv(H, low, trimmed, x, seed=0, rtol=1e-9):
    V = directions(len(x), seed)
    ref = HO.hv(low, trimmed, x, V)
    assert np.abs(ref).max() > 0
    ok, err = vec_tol_ok(H @ V, ref, rtol)
    assert ok, err
    assert np.abs(H - H.T).max() <= 1e-15 * max(1.0, np.abs(H).max())


def synth_low(shape, seed, n_strings, lmin, lmax, corpus_seed):
    model = synth.make_model(*shape, seed=seed)
    low = model.lowered()
    offs, toks, w = model.corpus(n_strings, lmin, lmax, seed=corpus_seed)
    low.set_tokens(offs, toks, w / w.sum())
    return model, low


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
    return low


@pytest.mark.parametrize("mu,sigma,rtol", [(-1.0, 0.5, 1e-9), (-12.0, 3.0, 1e-8), (2.5, 1.0, 1e-8)])
def test_segmented_medium(medium, mu, sigma, rtol):
    """Kernel 6 on `medium` across the range of x (the blocks of its region types).  Away from x ~ N(-1, 0.5) most regions
    have one dominant path, and k5_hessian forms Cov = E[c c^T] - g g^T in double, so the small covariances lose a few
    more digits to cancellation (measured on a B200: 2e-9 at N(-12, 3), 1.6e-9 at N(2.5, 1))."""
    dev, trimmed, n = mapped_device(medium, force_kernel=6)
    assert dev.info()["kernel"] == 6
    x = np.random.RandomState(7).normal(mu, sigma, size=n)
    H, _ = device_hessian(dev, x)
    dev.close()
    check_hv(H, medium, trimmed, x, rtol=rtol)


def test_segmented_overflow_strings(medium):
    """Kernel 6 with four pool slots: the strings that need more go to the secondary kernel for the evaluation and have
    blocks of their own segments for H_f.  rmin stays the smallest path posterior of a string."""
    dev, trimmed, n = mapped_device(medium, force_kernel=6, accum_variant=4 << 16)
    assert dev.info()["n_overflow_strings"] > 2
    x = np.random.RandomState(8).normal(-1.0, 0.5, size=n)
    H, rm = device_hessian(dev, x)
    dev.close()
    check_hv(H, medium, trimmed, x)
    ltw, lew = medium.edge_logweights(x, trimmed)
    ref = MP.rmin(medium, ltw, lew)
    assert abs(rm - ref) <= 1e-12 * ref, (rm, ref)


def test_default_pool_overflow():
    """make_model(128, 16, 8, 4), short strings: most strings need more than the default 16 slots, so nearly all of H_f
    comes from the blocks of their segments."""
    _, low = synth_low((128, 16, 8, 4), 7, 200, 4, 8, 9)
    dev, trimmed, n = mapped_device(low)
    info = dev.info()
    assert info["kernel"] == 6 and info["n_overflow_strings"] > 100
    x = np.random.RandomState(9).normal(-1.0, 0.5, size=n)
    H, rm = device_hessian(dev, x)
    dev.close()
    check_hv(H, low, trimmed, x)
    ltw, lew = low.edge_logweights(x, trimmed)
    ref = MP.rmin(low, ltw, lew)
    assert abs(rm - ref) <= 1e-12 * ref, (rm, ref)


@pytest.mark.parametrize("R", [40, 70, 100])
def test_heavy_region_type(R):
    """x (yx)^R: one region type of weight R, H[S->A, S->A] = -R/4 at x = 0: beyond +-16, the range a fixed point sized
    for block weights that sum to 1 would have.  Through the device handle and through the Hessian optimiser's session."""
    corpus = "\nx%s 1\n" % ("yx" * R)
    low = W.Lowered(W.parse(DIAMOND, corpus))
    dev, trimmed, n = mapped_device(low)
    assert dev.info()["kernel"] == 6
    x = np.zeros(n)
    H, _ = device_hessian(dev, x)
    dev.close()
    ref = HO.full(low, trimmed, x)
    assert np.allclose(H, ref, rtol=1e-12, atol=1e-12) and np.abs(H).max() == pytest.approx(R / 4, rel=1e-12)
    s = W.Session(DIAMOND, corpus, "Hessian")
    mine = {key(e): e for e in low.edges}
    perm = np.zeros(n, dtype=np.int64)
    for e in s.describe()["edges"]:
        if e["trimmed"] >= 0:
            perm[trimmed[mine[key(e)]["raw"]]] = e["trimmed"]
    assert s.n == n
    Hs = s.hessian(np.zeros(n))[np.ix_(perm, perm)]
    s.close()
    assert np.allclose(Hs, ref, rtol=1e-12, atol=1e-12)


def test_long_strings():
    """The long-string corpus of test_long_strings_need_rescaling (40 strings of 3500-4000 tokens): the region types
    weigh 237 in all."""
    _, low = synth_low((64, 16, 4, 3), 21, 40, 3500, 4000, 22)
    dev, trimmed, n = mapped_device(low)
    assert dev.info()["kernel"] == 6
    x = np.random.RandomState(4).normal(-1.0, 0.5, size=n)
    H, _ = device_hessian(dev, x)
    dev.close()
    check_hv(H, low, trimmed, x)


@pytest.mark.parametrize("kernel", [1, 2, 3, 4, 7])
def test_route_a_sessions(kernel):
    """The other kernels take the blocks the host enumerates per string (Learner::BuildPathBlocks): the Hessian optimiser's
    session on a synthetic corpus with fewer than 4e6 paths."""
    model = synth.make_model(64, 16, 4, 3, seed=5)
    offs, toks, w = model.corpus(400, 8, 40, seed=6)
    fsa_text, corpus_text = model.text(), model.corpus_text(offs, toks, w)
    low = W.Lowered(W.parse(fsa_text, corpus_text))
    pc, _, ee0 = O.dp_eval(low, np.zeros(low.n_trans), np.zeros(low.n_emis), want_counts=True)
    assert (pc > 0).all() and 1e3 < pc.sum() < 4e6
    trimmed, n, _ = O.trim(low, ee0 > 0)
    s = W.Session(fsa_text, corpus_text, "Hessian", force_kernel=kernel)
    assert s.backend_info()["kernel"] == kernel and s.n == n
    mine = {key(e): e for e in low.edges}
    perm = np.zeros(n, dtype=np.int64)
    for e in s.describe()["edges"]:
        if e["trimmed"] >= 0:
            perm[trimmed[mine[key(e)]["raw"]]] = e["trimmed"]
    x = np.random.RandomState(kernel).normal(-1.0, 0.7, size=n)
    xs = np.zeros(n)
    xs[perm] = x
    H = s.hessian(xs)[np.ix_(perm, perm)]
    s.close()
    check_hv(H, low, trimmed, x)


def test_run_to_run_determinism(medium):
    """Fixed-point sums: the same bits on every call, overflow blocks included."""
    dev, trimmed, n = mapped_device(medium, force_kernel=6, accum_variant=4 << 16)
    x = np.random.RandomState(10).normal(-1.0, 0.5, size=n)
    H1, r1 = device_hessian(dev, x)
    H2, r2 = device_hessian(dev, x)
    dev.close()
    assert np.array_equal(H1, H2) and r1 == r2
