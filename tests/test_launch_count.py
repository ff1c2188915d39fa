"""Kernel launches are counted where libbgmm makes them (bgmm_launch_count), and the engines' `kernel_launches` is the sum
of the counter's deltas around their library calls.

CPU: every launch in the library goes through the counted helpers, and calls rejected by their argument checks launch
nothing.  GPU: the delta around an engine call equals the libbgmm kernels torch.profiler records for the same call, over
every pass variant with the conditioning guard on and off, the restart batch, the extras and the hidden-Markov paths."""
import glob
import os

import numpy as np
import pytest

from conftest import ROOT
from bayesml_b200 import _lib


def test_every_launch_goes_through_the_counted_helpers():
    sources = glob.glob(os.path.join(ROOT, "bayesml_b200", "csrc", "*.cu*"))
    assert sources
    for path in sources:
        assert "<<<" not in open(path).read(), os.path.basename(path)


def test_rejected_calls_launch_nothing(lib_built):
    lib = _lib.load()
    n0 = lib.bgmm_launch_count()
    assert lib.bgmm_pass(None, 5, 0, 2, 0, None, None, None, None, None, None, 0, 0, None) == -1             # K = 0
    assert lib.bgmm_hmm_pass(None, 10, 3, 2, *([None] * 9), 0, 0, None) == -1                             # NULL buffers
    assert lib.bgmm_hmm_viterbi(10, 3, *([None] * 6), None) == -1
    assert lib.bgmm_small(3, 2, None, 0, 1, 0.0, 2, None, None) == -1
    assert lib.bgmm_colsum(None, 5, 2, 0, None, None, None) == -1
    assert lib.bgmm_pass_batched(None, 5, 3, 2, 1, None, None, None, None, None) == -1                    # R < 2
    assert lib.bgmm_launch_count() == n0


# ---------------------------------------------------------------------------------------------------------------- GPU

def _counted(engines, fn):
    """-> (libbgmm kernels torch.profiler records while fn runs, the engines' kernel_launches delta)."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    before = sum(e.kernel_launches for e in engines)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    kernels = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA and "bgmm" in e.name]
    return kernels, sum(e.kernel_launches for e in engines) - before


def _mixture(k, d, precision="float64", variant=_lib.PASS_AUTO, share=None, n=6000):
    from bayesml_b200 import gaussianmixture
    from bayesml_b200.engine import VBEngine
    rng = np.random.default_rng(k * 100 + d)
    x = rng.normal(size=(n, d)) + 4.0 * rng.integers(0, k, size=(n, 1))
    eng = VBEngine(k, d, precision=precision, variant=variant)
    if share is None:
        eng.load_data(x.astype(np.float32) if precision == "float32" else x)
    else:
        eng.share_data_from(share)
    gaussianmixture.LearnModel(k, d, seed=1)._push_prior(eng)
    eng._alloc_state(8)
    eng.set_params(np.ones(k), x[rng.choice(n, size=k, replace=False)], np.ones(k), np.full(k, float(d)),
                   np.tile(np.eye(d) * d, (k, 1, 1)))
    return eng


@pytest.fixture(params=["guard", "no_guard"])
def guard(request):
    lib = _lib.load()
    old = lib.bgmm_set_robust_threshold(lib.bgmm_robust_threshold() if request.param == "guard" else float("inf"))
    yield request.param
    lib.bgmm_set_robust_threshold(old)


@pytest.mark.gpu
@pytest.mark.parametrize("k,d,precision,want", [
    (4, 3, "float64", _lib.PASS_DMMA), (16, 24, "float64", _lib.PASS_LARGE), (16, 8, "float32", _lib.PASS_TF32),
    (3, 2, "float32", _lib.PASS_F32), (3, 3, "float32", _lib.PASS_F32), (80, 2, "float64", _lib.PASS_SIMPLE)])
def test_mixture_iteration(k, d, precision, want, guard, lib_built):
    eng = _mixture(k, d, precision)
    assert eng.lib.bgmm_pass_resolve(k, d, eng.x_code, _lib.PASS_AUTO, 0) == want

    def iteration():
        eng._pass()
        eng._small(_lib.SMALL_ITERATE, 100, 0.0)

    kernels, delta = _counted([eng], iteration)
    assert delta == len(kernels) > 0, kernels


@pytest.mark.gpu
def test_restart_batch_step(guard, lib_built):
    from bayesml_b200.engine import RestartBatch
    lead = _mixture(5, 24, variant=_lib.PASS_LARGE)
    members = [lead] + [_mixture(5, 24, variant=_lib.PASS_LARGE, share=lead) for _ in range(2)]
    for e in members:
        e.begin(100, 0.0)
    batch = RestartBatch(lead, len(members))
    kernels, delta = _counted(members, lambda: batch.step(members))
    assert delta == len(kernels) > 0, kernels


@pytest.mark.gpu
@pytest.mark.parametrize("call", ["final_pass", "pred_log_density", "draw_dirichlet1"])
def test_mixture_extras(call, lib_built):
    eng = _mixture(4, 3)
    fn = {"final_pass": eng.final_pass,
          "pred_log_density": lambda: eng.pred_log_density(np.ones(4), np.ones(4), np.full(4, 5.0)),
          "draw_dirichlet1": lambda: eng.draw_dirichlet1(seed=7)}[call]
    kernels, delta = _counted([eng], fn)
    assert delta == len(kernels) > 0, kernels


def _hmm(k, d, lengths):
    from bayesml_b200.engine import HMMEngine
    n = int(np.sum(lengths))
    rng = np.random.default_rng(k * 100 + d)
    z = np.repeat(rng.integers(0, k, size=n // 8 + 1), 8)[:n]
    x = 4.0 * rng.normal(size=(k, d))[z] + rng.normal(size=(n, d))
    eng = HMMEngine(k, d)
    eng.load_data(x)
    if len(lengths) > 1:
        eng.set_sequences(np.concatenate([[0], np.cumsum(lengths)[:-1]]))
    eng.set_hmm_prior(np.full(k, .5), np.full((k, k), .5), np.zeros((k, d)), np.ones(k), np.full(k, float(d)),
                      np.tile(np.eye(d), (k, 1, 1)), np.zeros(k), 0.0, 0.0)
    eng._alloc_state(8)
    eng.set_hmm_params(np.full(k, .5), np.full((k, k), .5), x[rng.choice(n, size=k, replace=False)], np.ones(k),
                       np.full(k, float(d)), np.tile(np.eye(d) * d, (k, 1, 1)))
    return eng


# chunks of 32 elements: 24 is one chunk (no sweep), 3200 is 100 chunks (one-level sweep), 20000 is 625 chunks (two-level
# sweep); the several-sequence case has sequences of one chunk, short ones (one segmented sweep) and long ones (two-level)
HMM_LENGTHS = {"one_chunk": [24], "one_level": [3200], "two_level": [20000], "seqs": [10, 500, 8000, 30, 3000, 10000]}


@pytest.mark.gpu
@pytest.mark.parametrize("d", [2, 12])                  # emission: the thread-per-element kernel (D <= 8), the large E kernel
@pytest.mark.parametrize("kind", sorted(HMM_LENGTHS))
def test_hmm_iteration(kind, d, lib_built):
    eng = _hmm(3, d, HMM_LENGTHS[kind])
    if kind == "seqs":
        assert eng.plan[4] >= 1 and eng.plan[5] >= 1           # short and long segments

    def iteration():
        eng._pass()
        eng._small(_lib.SMALL_ITERATE, 100, 0.0)

    kernels, delta = _counted([eng], iteration)
    assert delta == len(kernels) > 0, kernels


@pytest.mark.gpu
@pytest.mark.parametrize("d", [2, 12])
@pytest.mark.parametrize("kind", ["one_level", "seqs"])
def test_hmm_viterbi(kind, d, lib_built):
    eng = _hmm(3, d, HMM_LENGTHS[kind])
    kernels, delta = _counted([eng], lambda: eng.viterbi(np.log(np.full(3, 1 / 3)), np.log(np.full((3, 3), 1 / 3))))
    assert delta == len(kernels) > 0, kernels
