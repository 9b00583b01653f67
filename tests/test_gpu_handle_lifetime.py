"""A device handle gives back all the device and pinned host memory it took, whichever kernel it runs and whichever entry
points it went through.  wfsa_dev_held_bytes counts what the handles of this process hold; cudaMemGetInfo would also see
every other process on the GPU."""
import ctypes as C
import gc

import numpy as np
import pytest

import wfsa_b200 as W
from oracle import oracle as O
from wfsa_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def corpus():
    model = synth.make_model(256, 64, 8, 4, seed=11)
    low = model.lowered()
    offs, toks, w = model.corpus(3000, 32, 128, seed=12)
    low.set_tokens(offs, toks, w / w.sum())
    return low


def held_bytes():
    gc.collect()                         # handles that went out of scope elsewhere are destroyed first
    return W.lib().wfsa_dev_held_bytes()


@pytest.mark.parametrize("kernel", [1, 2, 3, 4, 6, 7])
def test_handle_gives_back_all_it_holds(corpus, kernel):
    low = corpus
    held = held_bytes()
    dev = W.Device(low, force_kernel=kernel, count=300 if kernel == 3 else None)     # (the generic kernel is the slow one)
    assert dev.info()["kernel"] == kernel
    rec, pc, used = dev.structure()
    params = np.concatenate([low.trans_param, low.emis_param])
    trimmed, n, _ = O.trim(low, np.array([r < 0 or used[r] for r in params]))
    dev.set_param_map(trimmed, n, rec)
    mapped = held_bytes()
    assert mapped > held
    if kernel == 7:
        # the batches and the alpha lattice of the first map are replaced, not kept beside the new ones
        dev.set_param_map(trimmed, n, rec)
        assert held_bytes() == mapped
    x = np.random.RandomState(1).normal(-1.5, 0.8, size=n)
    ll, logq, grad = dev.eval(x)
    assert np.isfinite(ll)
    if kernel == 6:
        assert dev.info()["eval_path"] & 1          # single launch: an evaluation without log q is the host-buffer call
        dev.timer_begin()
        dev.eval(x, want_logq=False)
        dev.timer_end()
        dev.timer_kernel_ms(), dev.timer_split_ms(), dev.timer_phase_ms(), dev.timer_step_ms()
        dev.l2_flush()
        ll2, _, grad2 = dev.eval(x, want_logq=False)
        assert ll2 == ll and np.array_equal(grad2, grad)
        H = np.zeros((n, n))
        rmin = C.c_double()
        dev._ck(dev.L.wfsa_dev_hessian(dev.h, W._p(x, W.F64P), W._p(H, W.F64P), C.byref(rmin)))
        assert held_bytes() > mapped                # the Hessian's buffers and the L2 flush buffer are counted as well
    dev.close()
    assert held_bytes() == held
