"""GPU: ONE fp64 pass (bgmm_pass) from a GIVEN parameter set against plain references of the same operation, over every
template configuration of the fused DMMA kernel and the shapes of the other fp64 kernels that no full fit in the suite reaches.

The fits in test_gpu_parity.py compare whole trajectories, so a kernel is only checked at the shapes those fits happen to
use.  Here the state is set directly (perturbed parameters on an OracleGMM, as in test_fp32_tensor_core_pass_from_identical_
state) and one `final_pass` is compared with
  (a) ln rho, r and the arg max of OracleGMM.e_step on the same parameters,
  (b) the raw statistics STATS[k][p] against sum_n r_out[n,k] phi_p(x'_n) in long double, from the kernel's OWN r: this
      isolates the statistics GEMM and its reductions (a dropped, duplicated or misplaced row is ~1/n of the sum),
  (c) the tail slots: sum r ln r, the row count, the moment format,
  (d) ctrl.ROBUST == 0: otherwise the conditioning guard would have handed the pass to the DIRECT kernel and the kernel the
      case names would not have run,
  (e) a second pass from the same state gives the same bits.
Each DMMA case is pinned, through torch.profiler, to the pass_dmma_kernel<KB, SP, NPS> instantiation it is meant to cover.
"""
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# pass_dmma_kernel<KB, SP, NPS> as plan_dmma (csrc/bgmm_pass_dmma.cu) picks it: KB = 1, 2, 4 component blocks of 8 for
# K <= 8, 9-16, 17-32; SP = P = 1 + D + D(D+1)/2 rounded up to 32; NPS = 4 Phi stages, 3 where four do not fit in shared
# memory (SP = 192 with KB >= 2).  These are all 18 configurations any (K, D) reaches.  K is not a multiple of 8 where the
# block allows it (padding components), the block maximum elsewhere; odd and even D (the Phi producer has two load paths).
DMMA_CASES = {
    (1, 32, 4): (3, 5), (1, 64, 4): (7, 8), (1, 96, 4): (8, 12), (1, 128, 4): (5, 13), (1, 160, 4): (6, 15),
    (1, 192, 4): (8, 18),
    (2, 32, 4): (13, 4), (2, 64, 4): (10, 9), (2, 96, 4): (16, 11), (2, 128, 4): (11, 14), (2, 160, 4): (15, 16),
    (2, 192, 3): (12, 17),
    (4, 32, 4): (32, 6), (4, 64, 4): (19, 8), (4, 96, 4): (27, 10), (4, 128, 4): (32, 14), (4, 160, 4): (21, 15),
    (4, 192, 3): (32, 18),
}
# one row, a ragged sub-tile, one row past a 32-row sub-tile, several CTAs with a ragged end
ROWS = (1, 31, 33, 4099)
# <= 148 CTAs of 32-row sub-tiles: ~12.7 sub-tiles per CTA, so every CTA cycles its Phi ring (3 or 4 stages) several times
ROWS_RING = 60013
SIMPLE_SHAPES = [(4, 160), (3, 129), (2, 1)]           # (K, D): above D = 128 only these two kernels exist
LARGE_SHAPES = [(7, 19), (33, 20)]                      # padding inside the last 8-component block

_KERNEL = {"simple": r"pass_simple_kernel<double, false>", "direct": r"pass_simple_kernel<double, true>",
           "large": r"e_large_kernel<", "dmma": r"pass_dmma_kernel<"}


def _mixture(n, d, k, seed):
    rng = np.random.default_rng(seed)
    mu = rng.normal(0, 4.0, size=(k, d))
    a = rng.normal(size=(k, d, d))
    chol = np.linalg.cholesky(a @ a.transpose(0, 2, 1) / d + 0.5 * np.eye(d))
    z = rng.integers(0, k, size=n)
    x = mu[z] + np.einsum("nij,nj->ni", chol[z], rng.normal(size=(n, d))) if d <= 32 else \
        mu[z] + np.stack([chol[z[i]] @ rng.normal(size=d) for i in range(n)])
    return rng, x, mu, chol


def _oracle(rng, k, d, mu, chol, tie):
    """Perturbed parameters on an OracleGMM (as test_fp32_tensor_core_pass_from_identical_state); `tie`: component 4 gets
    the bit-identical parameters of component 1."""
    from oracle.gmm_vb_oracle import OracleGMM
    o = OracleGMM(k, d)
    o.hn_m_vecs[:] = mu + 0.2 * rng.normal(size=mu.shape)
    o.hn_nus[:] = d + 2.0 + rng.uniform(0, 50, size=k)
    o.hn_kappas[:] = 1.0 + rng.uniform(0, 50, size=k)
    o.hn_alpha_vec[:] = 0.5 + rng.uniform(0, 100, size=k)
    for j in range(k):
        o.hn_w_mats_inv[j] = (chol[j] @ chol[j].T) * o.hn_nus[j] * rng.uniform(0.7, 1.4)
    if tie:
        for f in (o.hn_m_vecs, o.hn_nus, o.hn_kappas, o.hn_alpha_vec, o.hn_w_mats_inv):
            f[4] = f[1]
    o.hn_w_mats[:] = np.linalg.inv(o.hn_w_mats_inv)
    o.q_pi_features(); o.q_lambda_features()
    return o


def _raw_moments(xc, r, shift, cols):
    """For k in cols: sum_n r[n,k] phi(x'_n - shift_k), phi = [1, x, x_i x_j (i >= j, packed i(i+1)/2 + j)], in long
    double; and sum_n |r[n,k] phi_p| (float64) per entry, the scale of the bar."""
    d = xc.shape[1]
    ii, jj = np.tril_indices(d)
    ref, scale = [], []
    for k in cols:
        y = xc - shift[k]
        yl = xc.astype(np.longdouble) - shift[k].astype(np.longdouble)
        w, wl = r[:, k], r[:, k].astype(np.longdouble)
        m2 = (yl * wl[:, None]).T @ yl
        ref.append(np.concatenate([[wl.sum()], wl @ yl, m2[ii, jj]]))
        ay = np.abs(y)
        a2 = (ay * w[:, None]).T @ ay
        scale.append(np.concatenate([[w.sum()], w @ ay, a2[ii, jj]]))
    return np.array(ref), np.array(scale)


def _kernels_during(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events()}


def _one_pass(k, d, n, variant, seed, tie=False, dmma_cfg=None):
    from bayesml_b200 import _lib
    from bayesml_b200.engine import VBEngine
    code = {"simple": _lib.PASS_SIMPLE, "dmma": _lib.PASS_DMMA, "large": _lib.PASS_LARGE, "direct": _lib.PASS_DIRECT}[variant]
    assert _lib.load().bgmm_pass_supported(k, d, _lib.F64, code)
    rng, x, mu, chol = _mixture(n, d, k, seed)
    o = _oracle(rng, k, d, mu, chol, tie)
    o.alloc(n)
    o.e_step(x)
    eng = VBEngine(k, d, variant=code)
    eng.load_data(x)
    eng.set_prior(o.h0_alpha_vec, o.h0_m_vecs, o.h0_kappas, o.h0_nus, o.h0_w_mats_inv, o.ln_b_h0_w_nus, o.ln_c_h0_alpha)
    load = lambda: eng.set_params(o.hn_alpha_vec, o.hn_m_vecs, o.hn_kappas, o.hn_nus, o.hn_w_mats_inv)  # noqa: E731
    load()
    shift = eng._view("shift", k * d).cpu().numpy().reshape(k, d)         # the DIRECT kernel's moments are about this
    names = _kernels_during(eng.final_pass)
    got = dict(stats=eng.stats.cpu().numpy().copy(), r=eng.r_dev.cpu().numpy(), lnrho=eng.lnrho_dev.cpu().numpy(),
               arg=eng.argmax_dev.cpu().numpy(), ctrl=eng.ctrl.cpu().numpy().copy(), coef=eng.fetch_params()["coef"])
    load()                                                                   # same state again (the pass moved SHIFT)
    eng.final_pass()
    again = dict(stats=eng.stats.cpu().numpy(), r=eng.r_dev.cpu().numpy(), lnrho=eng.lnrho_dev.cpu().numpy(),
                 arg=eng.argmax_dev.cpu().numpy())

    # the kernel the case names ran
    assert any(re.search(_KERNEL[variant], s) for s in names), sorted(names)
    if dmma_cfg is not None:
        ran = {tuple(int(v) for v in m.groups()) for s in names
               for m in [re.search(r"pass_dmma_kernel<\s*(\d+)\s*,\s*(\d+)\s*,\s*(\d+)\s*>", s)] if m}
        assert ran == {dmma_cfg}, f"K={k} D={d}: ran pass_dmma_kernel{sorted(ran)}, expected {dmma_cfg}"
    # (d) the conditioning guard did not hand the pass to the DIRECT kernel
    if variant != "direct":
        assert int(got["ctrl"][_lib.CTRL_ROBUST]) == 0, "the conditioning guard fired: the named kernel did not run"

    # (a) E-step against the oracle's on the same parameters
    r, lnrho, arg = got["r"], got["lnrho"], got["arg"]
    err = np.abs(lnrho - o.ln_rho) / np.maximum(1.0, np.abs(o.ln_rho))
    assert err.max() <= 1e-9, f"ln rho: {err.max():.3e}"
    assert np.allclose(r, o.r_vecs, rtol=1e-9, atol=1e-300), np.max(np.abs(r - o.r_vecs) / np.maximum(o.r_vecs, 1e-300))
    assert np.array_equal(arg, np.argmax(o.r_vecs, axis=1)), np.nonzero(arg != np.argmax(o.r_vecs, axis=1))[0][:10]
    assert np.array_equal(arg, np.argmax(r, axis=1))

    # (b) raw statistics from the kernel's own r; a subset of the components at the largest n (long double is slow)
    pitch = eng.off["pitch"]
    P = 1 + d + d * (d + 1) // 2
    raw = got["stats"][:k * pitch].reshape(k, pitch)
    cols = np.arange(k) if n < 10000 else np.sort(np.random.default_rng(seed).choice(k, size=min(k, 4), replace=False))
    xc = x - eng.center                                                     # the device's x' (one rounding, the same)
    ref, scale = _raw_moments(xc, r, shift if variant == "direct" else np.zeros((k, d)), cols)
    bad = np.abs(raw[cols, :P] - ref) > 1e-12 * scale
    assert not bad.any(), f"STATS[k][p] wrong at (k, p) = {[(int(cols[a]), int(b)) for a, b in zip(*np.nonzero(bad))][:10]}"
    assert np.all(raw[:, P:] == 0.0), "padding columns of STATS are not zero"

    # (c) tail: sum r ln r, rows, format.  1e-12 relative, plus n ulps of 1: each row's term carries an absolute rounding
    # error of about one ulp of 1 on both sides (the kernel takes ln of the softmax denominator, a number in [1, K]; the
    # reference sees r_out rounded to double, and an r near 1 has an absolute error of eps / 2, so has r ln r).  Where
    # nearly every row is certain the sum is ~n * 1e-10 and a purely relative 1e-12 is below what either side can resolve:
    # the kernel's formula evaluated in double on the oracle's ln rho differs from this reference by up to 4e-10 relative.
    tail = got["stats"][k * pitch:]
    rl = r.astype(np.longdouble)
    ent = np.sum(np.where(rl > 0, rl * np.log(np.where(rl > 0, rl, 1)), 0))
    assert abs(tail[_lib.STATS_ENTROPY] - ent) <= 1e-12 * abs(ent) + n * np.finfo(float).eps, \
        (tail[_lib.STATS_ENTROPY], float(ent))
    assert tail[_lib.STATS_ROWS] == n
    assert (tail[_lib.STATS_FORMAT] > 0) if variant == "direct" else (tail[_lib.STATS_FORMAT] == 0)

    # (e) the same bits from the same state
    for f in ("stats", "r", "lnrho", "arg"):
        assert np.array_equal(again[f], got[f]), f"second pass differs in {f}"
    return got, o


@pytest.mark.parametrize("n", ROWS + (ROWS_RING,))
@pytest.mark.parametrize("cfg", sorted(DMMA_CASES), ids=lambda c: "kb%d-sp%d-nps%d" % c)
def test_dmma_pass_against_oracle(cfg, n):
    k, d = DMMA_CASES[cfg]
    _one_pass(k, d, n, "dmma", seed=n + 100 * d + k, dmma_cfg=cfg)


@pytest.mark.parametrize("n", ROWS)
@pytest.mark.parametrize("variant", ["simple", "direct"])
@pytest.mark.parametrize("shape", SIMPLE_SHAPES, ids=lambda s: "k%d-d%d" % s)
def test_simple_and_direct_pass_against_oracle(shape, variant, n):
    k, d = shape
    _one_pass(k, d, n, variant, seed=n + 100 * d + k)


@pytest.mark.parametrize("n", ROWS)
@pytest.mark.parametrize("shape", LARGE_SHAPES, ids=lambda s: "k%d-d%d" % s)
def test_large_pass_against_oracle(shape, n):
    k, d = shape
    _one_pass(k, d, n, "large", seed=n + 100 * d + k)


@pytest.mark.parametrize("variant,k", [("simple", 6), ("direct", 6), ("dmma", 6), ("dmma", 12), ("large", 6)])
def test_exact_ties_give_the_first_index(variant, k):
    """Components 1 and 4 with bit-identical parameters, hence bit-identical coefficient rows: every kernel computes each
    output element with the same instruction sequence, so their r columns must be bit-equal and the arg max must be 1
    (np.argmax: first index on ties) wherever the pair holds the maximum."""
    n, d = 4099, 3
    got, o = _one_pass(k, d, n, variant, seed=7 + k, tie=True)
    assert np.array_equal(got["coef"][1], got["coef"][4])
    r, arg = got["r"], got["arg"]
    assert np.array_equal(r[:, 1], r[:, 4])
    pair = np.isin(np.argmax(o.r_vecs, axis=1), (1, 4))
    assert pair.sum() > n // (2 * k), "too few rows where the tied pair holds the maximum"
    assert np.all(arg[pair] == 1) and not np.any(arg == 4)
