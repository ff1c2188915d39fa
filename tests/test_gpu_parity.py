"""GPU parity tests: the CUDA path (through the C ABI) against the golden fixtures recorded from the real
reference and against the CPU oracle on seeded inputs.

Tolerances (BASELINE.json north_star): fp64 mode — hyperparameters, responsibilities and ELBO within 1e-9
relative; argmax assignments bit-exact.
"""
import contextlib
import io
import re
import warnings

import numpy as np
import pytest

from conftest import ln_rho_rows, load_golden

pytestmark = pytest.mark.gpu

RTOL = 1e-9


def _fit_kwargs(g):
    return eval(str(g["fit_kwargs"]), {"__builtins__": {}}, {"dict": dict})


def _close(a, b, rtol=RTOL, atol=0.0, what="", floor=1e-4):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    scale = np.max(np.abs(b)) if b.size else 0.0
    # element-wise relative error; entries below 1e-4 of the array's largest magnitude (near-zero off-diagonal covariances,
    # values that are ~0 by cancellation) are held to the same ABSOLUTE bound as an entry of that floor size, i.e. the
    # bar is max(rtol * |b|, rtol * 1e-4 * max|b|) — still 1e-13 of the array scale for rtol = 1e-9
    err = np.abs(a - b) / np.maximum(np.abs(b), max(scale * floor, 1e-300))
    worst = float(err.max()) if err.size else 0.0
    assert worst <= rtol or np.allclose(a, b, rtol=rtol, atol=atol), f"{what}: max rel err {worst:.3e}"


def _w_rtol(g, state_idx=None):
    """Bar for hn_w_mats = inv(hn_w_mats_inv): 1e-9, except where hn_w_mats_inv itself is so ill-conditioned (default
    prior mean far from a tight cluster: rank-one term ~ sep^2) that the reference's LAPACK inverse is only defined to
    cond * eps — then 16 * cond * eps."""
    winv = g["final_hn_w_mats_inv"] if state_idx is None else g["traj_hn_w_mats_inv"][state_idx]
    return max(RTOL, 16 * np.finfo(float).eps * float(np.max(np.linalg.cond(winv))))


def _prior_arrays(g):
    from oracle.gmm_vb_oracle import OracleGMM
    prior = {f: g[f] for f in ("h0_alpha_vec", "h0_m_vecs", "h0_kappas", "h0_nus", "h0_w_mats")}
    o = OracleGMM(int(g["K"]), int(g["D"]), **prior)
    return prior, o


def _engine_for(g, variant=0, precision="float64"):
    from bayesml_b200.engine import VBEngine
    prior, o = _prior_arrays(g)
    eng = VBEngine(int(g["K"]), int(g["D"]), variant=variant, precision=precision)
    eng.load_data(g["x"])
    eng.set_prior(o.h0_alpha_vec, o.h0_m_vecs, o.h0_kappas, o.h0_nus, o.h0_w_mats_inv, o.ln_b_h0_w_nus, o.ln_c_h0_alpha)
    return eng, o


TRAJ_CASES = ["traj_d3k4", "traj_d16k8", "traj_offset_d4k3", "traj_prior_d3k2", "traj_k1_d5", "traj_rr_d2k3",
              # conditioning cases (clusters 1e4 .. 1e5 of their own width apart, a far outlier cluster): the feature-map
              # kernels hand over to the DIRECT kernel on the device (ctrl.robust), whatever variant was requested
              "cond_sep1e4_d3k3", "cond_sep1e5_d2k3", "cond_outlier_d4k4", "cond_sep3e4_d16k6", "cond_sub_sep1e4_d3k3"]


@pytest.mark.parametrize("variant", ["simple", "dmma", "large", "direct"])
@pytest.mark.parametrize("name", TRAJ_CASES)
def test_trajectory_from_identical_initial_state(name, variant):
    """Per restart: start the device loop from the reference's recorded initial state, compare every ELBO value of
    the trajectory and the full state at its end (SURVEY.md §7 'hard parts': parity is judged per restart)."""
    from bayesml_b200 import _lib
    g = load_golden(name)
    kw = _fit_kwargs(g)
    code = {"simple": _lib.PASS_SIMPLE, "dmma": _lib.PASS_DMMA, "large": _lib.PASS_LARGE, "direct": _lib.PASS_DIRECT}[variant]
    if not _lib.load().bgmm_pass_supported(int(g["K"]), int(g["D"]), _lib.F64, code):
        pytest.skip(f"{variant} kernel does not cover K={int(g['K'])} D={int(g['D'])}")
    eng, o = _engine_for(g, variant=code)
    restart_of_state = g["restart_of_state"]
    for r in range(kw["num_init"]):
        idx = np.nonzero(restart_of_state == r)[0]
        if "init_r_vecs" in g:
            eng.set_params(o.h0_alpha_vec, o.h0_m_vecs, o.h0_kappas, o.h0_nus, o.h0_w_mats_inv)
            hist, conv = eng.run(kw["max_itr"], kw["tolerance"], r_init=g["init_r_vecs"][r])
        else:
            eng.set_params(o.h0_alpha_vec, g["init_hn_m_vecs"][r], o.h0_kappas, o.h0_nus, g["init_hn_w_mats_inv"][r])
            hist, conv = eng.run(kw["max_itr"], kw["tolerance"])
        assert not conv and len(hist) == len(idx) == kw["max_itr"] + 1
        if name.startswith("cond_") and variant != "direct":
            assert int(eng.ctrl.cpu()[_lib.CTRL_ROBUST]) == 1, "the conditioning guard did not fire"
        elif variant != "direct" and name != "traj_offset_d4k3":
            assert int(eng.ctrl.cpu()[_lib.CTRL_ROBUST]) == 0, "the conditioning guard fired on a well-conditioned case"
        _close(hist, g["traj_vl_terms"][idx, 0], what=f"{name} restart {r} VL history")
        p = eng.fetch_params()
        last = idx[-1]
        for mine, ref in [("alpha", "hn_alpha_vec"), ("m", "hn_m_vecs"), ("kappa", "hn_kappas"), ("nu", "hn_nus"),
                          ("w", "hn_w_mats"), ("winv", "hn_w_mats_inv"), ("e_ln_pi", "_e_ln_pi_vec"),
                          ("e_ln_lambda_dets", "_e_ln_lambda_dets"), ("ln_b", "_ln_b_hn_w_nus"), ("ns", "ns"),
                          ("x_bar", "x_bar_vecs"), ("s_mats", "s_mats")]:
            _close(p[mine], g["traj_" + ref][last], rtol=_w_rtol(g, last) if mine == "w" else RTOL,
                   what=f"{name} restart {r} {ref}")
        # vl_terms order in the fixture: vl, p_x, p_z, p_pi, p_mu_lambda, q_z, q_pi, q_mu_lambda
        _close(p["vl_terms"][:7], g["traj_vl_terms"][last, 1:], what=f"{name} restart {r} ELBO terms")
        _close(p["vl_terms"][7], g["traj_vl_terms"][last, 0], what=f"{name} restart {r} vl")


def _parse_progress(text):
    """-> list per restart of (vl values, converged?, starred?) from the reference's progress text (:861-883)."""
    out = []
    for line in text.split("\n"):
        if not line.strip():
            continue
        vals = [float(v) for v in re.findall(r"VL: (-?[0-9.eE+-]+|nan|inf|-inf)", line)]
        out.append((vals, "(converged)" in line, line.rstrip().endswith("*")))
    return out


E2E_CASES = ["c1_readme", "traj_d3k4", "traj_d16k8", "traj_rr_d2k3", "traj_offset_d4k3", "traj_prior_d3k2",
             "traj_k1_d5", "conv_d2k4", "cond_sub_sep1e4_d3k3"]


@pytest.mark.parametrize("name", E2E_CASES)
def test_learnmodel_end_to_end_matches_reference(name):
    """The drop-in class, same seed and arguments as the recorded reference run: same progress text structure,
    ELBO values, selected restart, final hyperparameters, statistics, responsibilities, assignments."""
    from bayesml_b200 import gaussianmixture
    g = load_golden(name)
    kw = _fit_kwargs(g)
    prior = {f: g[f] for f in ("h0_alpha_vec", "h0_m_vecs", "h0_kappas", "h0_nus", "h0_w_mats")}
    model = gaussianmixture.LearnModel(int(g["K"]), int(g["D"]), seed=int(g["seed"]), **prior)
    live = model.get_hn_params()["hn_m_vecs"]
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf), warnings.catch_warnings(record=True) as wl:
        warnings.simplefilter("always")
        ret = model.update_posterior(g["x"], **kw)
    assert ret is model
    assert live is model.hn_m_vecs                                              # updated in place (SURVEY §3.1)
    assert len([w for w in wl if "not converged" in str(w.message)]) == int(g["n_warnings"])
    mine, ref = _parse_progress(buf.getvalue()), _parse_progress(str(g["stdout"]))
    assert len(mine) == len(ref)
    for r, ((v1, c1, s1), (v2, c2, s2)) in enumerate(zip(mine, ref)):
        assert (len(v1), c1, s1) == (len(v2), c2, s2), f"restart {r}: iterations/converged/selected differ"
        _close(v1, v2, what=f"{name} restart {r} printed VL")
    for f in ("hn_alpha_vec", "hn_m_vecs", "hn_kappas", "hn_nus", "hn_w_mats", "hn_w_mats_inv", "ns", "x_bar_vecs",
              "s_mats", "_e_ln_pi_vec", "_e_ln_lambda_dets", "_ln_b_hn_w_nus"):
        _close(getattr(model, f), g["final_" + f], rtol=_w_rtol(g) if f == "hn_w_mats" else RTOL,
               what=f"{name} final {f}")
    _close(model.vl, g["final_vl_attr"], what="vl attribute (last restart's)")
    r = model.r_vecs
    assert r.shape == g["final_r_vecs"].shape and r.dtype == np.float64
    assert np.allclose(r, g["final_r_vecs"], rtol=RTOL, atol=1e-300), np.abs(r / g["final_r_vecs"] - 1).max()
    assert np.allclose(model._ln_rho[ln_rho_rows(g)], g["final_ln_rho"], rtol=_w_rtol(g), atol=1e-9)   # far components: ln rho ~ d^T (nu W) d
    assert np.array_equal(np.argmax(r, axis=1), np.argmax(g["final_r_vecs"], axis=1))       # bit-exact assignments
    for f in ("p_pi_vec", "p_mu_vecs", "p_nus", "p_lambda_mats"):                            # stale, prior-based
        _close(getattr(model, f), g["stale_" + f], what="stale " + f)
    model.calc_pred_dist()
    for f in ("p_pi_vec", "p_mu_vecs", "p_nus", "p_lambda_mats"):
        _close(getattr(model, f), g["pred_" + f], rtol=_w_rtol(g) if f == "p_lambda_mats" else RTOL, what="pred " + f)
    if "latent_x" in g:
        onehot = model.estimate_latent_vars(g["latent_x"], loss="0-1")
        assert onehot.dtype == g["latent_onehot"].dtype and np.array_equal(onehot, g["latent_onehot"])
        rr = model.estimate_latent_vars(g["latent_x"], loss="squared")
        assert rr is model.r_vecs
        assert np.allclose(rr, g["latent_r"], rtol=RTOL, atol=1e-300)
        _close(model.ns, g["latent_ns_after"], what="ns after estimate_latent_vars")
        from bayesml_b200 import CriteriaError
        with pytest.raises(CriteriaError):
            model.estimate_latent_vars(g["latent_x"], loss="abs")


def test_input_forms_and_edge_sizes():
    """float32 / integer / 3-D inputs are promoted like numpy does in the reference; tiny N; bad init_type."""
    from bayesml_b200 import gaussianmixture
    from oracle.gmm_vb_oracle import OracleGMM, fit
    rng = np.random.default_rng(5)
    base = rng.normal(size=(257, 3)) * 2.0 + rng.integers(0, 3, size=(257, 1)) * 6.0
    for x in (base.astype(np.float32), np.round(base).astype(np.int64), base.reshape(1, 257, 3), base[:1], base[:2]):
        m = gaussianmixture.LearnModel(3, 3, seed=2)
        o = OracleGMM(3, 3, seed=2)
        with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            m.update_posterior(x, max_itr=6, num_init=2, tolerance=0.0)
        fit(o, x, max_itr=6, num_init=2, tolerance=0.0)
        _close(m.hn_m_vecs, o.hn_m_vecs, what="hn_m_vecs")
        _close(m.hn_w_mats_inv, o.hn_w_mats_inv, what="hn_w_mats_inv")
        _close(m.vl, o.vl, what="vl")
        assert np.allclose(m.r_vecs, o.r_vecs, rtol=RTOL, atol=1e-300)
    m = gaussianmixture.LearnModel(3, 3, seed=2)
    with pytest.raises(ValueError, match="init_type"), contextlib.redirect_stdout(io.StringIO()):
        m.update_posterior(base, init_type="kmeans")


def test_sequential_update_wrappers():
    """pred_and_update / estimate_latent_vars_and_update (:1104-1155, :1198-1245) keep working on the new path."""
    from bayesml_b200 import gaussianmixture
    from oracle.ref_loader import reference_available
    rng = np.random.default_rng(8)
    x = rng.normal(size=(200, 2)) + rng.integers(0, 2, size=(200, 1)) * 5.0
    m = gaussianmixture.LearnModel(2, 2, seed=4)
    with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        z = m.estimate_latent_vars_and_update(x, max_itr=20, num_init=2)
        assert z.shape == (200, 2) and np.array_equal(z.sum(axis=1), np.ones(200, dtype=int))
        assert np.allclose(m.h0_alpha_vec, 0.5)            # h0 overwritten by the *pre-update* hn (= prior here)
        pred = m.pred_and_update(x[0], max_itr=5, num_init=1)
        assert pred.shape == (2,) and m.r_vecs.shape == (1, 2)
        assert np.isclose(m.ns.sum(), 1.0)


@pytest.mark.parametrize("variant", ["simple", "auto", "large"])
@pytest.mark.parametrize("shape", [(20000, 16, 32), (50000, 2, 8), (5000, 32, 16), (3000, 7, 5), (4099, 16, 13), (20000, 40, 12)])
def test_larger_shapes_against_oracle_and_elbo_monotone(shape, variant, monkeypatch):
    """Seeded synthetic mixtures at sizes the oracle finishes in seconds: trajectory parity from identical init, and
    the reference's own stated test criterion — the ELBO never decreases (doc/devdoc/vb_method.md:184-194)."""
    from bayesml_b200 import gaussianmixture
    from oracle.gmm_vb_oracle import OracleGMM, fit
    monkeypatch.setenv("BAYESML_B200_PASS_VARIANT", variant)
    n, d, k = shape
    rng = np.random.default_rng(n + d)
    mu = rng.normal(0, 4.0, size=(k, d))
    a = rng.normal(size=(k, d, d))
    chol = np.linalg.cholesky(a @ a.transpose(0, 2, 1) / d + 0.5 * np.eye(d))
    z = rng.integers(0, k, size=n)
    x = mu[z] + np.einsum("nij,nj->ni", chol[z], rng.normal(size=(n, d)))
    m = gaussianmixture.LearnModel(k, d, seed=1)
    o = OracleGMM(k, d, seed=1)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m.update_posterior(x, max_itr=6, num_init=1, tolerance=0.0)
    tr = fit(o, x, max_itr=6, num_init=1, tolerance=0.0)
    vals = _parse_progress(buf.getvalue())[0][0]
    _close(vals, tr.vl_history[0], what="VL history")
    assert all(b >= a - 1e-9 * abs(a) for a, b in zip(vals[1:], vals[2:])), "ELBO decreased"
    for f in ("hn_alpha_vec", "hn_m_vecs", "hn_kappas", "hn_nus", "hn_w_mats_inv", "ns", "x_bar_vecs"):
        _close(getattr(m, f), getattr(o, f), what=f)
    # entry by entry, same bar as everything else.  (D = 40 runs with N = 20000: at 500 samples per 40-dimensional
    # component the fit is so weakly determined that ANY two correct implementations differ by ~5e-10 in the small
    # entries after 6 iterations — measured with every pass on the DIRECT kernel, scratch notes in DESIGN.md §2.)
    _close(m.s_mats, o.s_mats, what="s_mats")
    if variant == "auto":
        _close(m._engine().refine_smats(), o.s_mats, what="two-pass centred s_mats (bgmm_pass DIRECT with r_in)")
    assert np.allclose(m.r_vecs, o.r_vecs, rtol=RTOL, atol=1e-300)
    assert np.array_equal(np.argmax(m.r_vecs, axis=1), np.argmax(o.r_vecs, axis=1))
    assert np.allclose(m.r_vecs.sum(axis=1), 1.0, rtol=0, atol=1e-12)
    assert np.isclose(m.ns.sum(), n, rtol=1e-12)


@pytest.mark.parametrize("packed", ["1", "0"])
@pytest.mark.parametrize("shape", [(60000, 2, 8), (30000, 3, 5), (20000, 1, 3), (4097, 2, 2), (12345, 2, 5)])
def test_fp32_mode_against_fp64_oracle(shape, packed, monkeypatch):
    """precision='float32' (BASELINE config C3's mode): X is rounded to fp32 once and the SAME rounded X is fed to the
    fp64 oracle (the reference promotes float32 input to float64, :780); bar 1e-4 relative, assignments exact.
    packed = 1: D = 2 runs the two-samples-per-thread f32x2 kernel in the loop (odd N: a half-filled last pair);
    packed = 0: the scalar kernel alone."""
    from bayesml_b200 import _lib, gaussianmixture
    from oracle.gmm_vb_oracle import OracleGMM, fit
    n, d, k = shape
    if packed == "0" and d != 2:
        pytest.skip("the packed kernel exists for D = 2 only")
    monkeypatch.setenv("BGMM_F32_PACKED", packed)
    assert _lib.load().bgmm_pass_supported(k, d, _lib.F32, _lib.PASS_F32)
    rng = np.random.default_rng(n + d + k)
    mu = rng.normal(0, 5.0, size=(k, d))
    z = rng.integers(0, k, size=n)
    x32 = (mu[z] + rng.normal(size=(n, d)) * rng.uniform(0.5, 1.5, size=(k, 1))[z]).astype(np.float32)
    m = gaussianmixture.LearnModel(k, d, seed=2, precision="float32")
    o = OracleGMM(k, d, seed=2)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m.update_posterior(x32, max_itr=10, num_init=1, tolerance=0.0)
    tr = fit(o, x32, max_itr=10, num_init=1, tolerance=0.0)
    tol = 1e-4
    vals = _parse_progress(buf.getvalue())[0][0]
    _close(vals, tr.vl_history[0], rtol=tol, what="fp32-mode VL history")
    for f in ("hn_alpha_vec", "hn_m_vecs", "hn_kappas", "hn_nus", "hn_w_mats_inv", "ns", "x_bar_vecs", "s_mats"):
        _close(getattr(m, f), getattr(o, f), rtol=tol, what="fp32-mode " + f)
    big = o.r_vecs > 1e-3                                  # responsibilities that carry weight: relative bar
    assert np.allclose(m.r_vecs[big], o.r_vecs[big], rtol=tol)
    assert np.allclose(m.r_vecs, o.r_vecs, rtol=0, atol=1e-5)
    margin = np.sort(o.r_vecs, axis=1)
    clear = (margin[:, -1] - margin[:, -2]) > 1e-4         # exclude numerical near-ties (SURVEY §7)
    assert np.array_equal(np.argmax(m.r_vecs, axis=1)[clear], np.argmax(o.r_vecs, axis=1)[clear])
    assert clear.mean() > 0.99


@pytest.mark.parametrize("variant", ["auto", "simple"])
def test_high_dimension_shape(variant, monkeypatch):
    """BASELINE config C4's shape class (D=128, K=64) at a size the oracle finishes in seconds: exercises the
    per-component kernel with a 128x128 Cholesky in shared memory and the large-regime (auto) / generic pass kernels."""
    monkeypatch.setenv("BAYESML_B200_PASS_VARIANT", variant)
    from bayesml_b200 import gaussianmixture
    from oracle.gmm_vb_oracle import OracleGMM, fit
    n, d, k = 3000, 128, 64
    rng = np.random.default_rng(9)
    x = rng.normal(size=(n, d)) + 3.0 * rng.normal(size=(k, d))[rng.integers(0, k, size=n)]
    m = gaussianmixture.LearnModel(k, d, seed=1)
    o = OracleGMM(k, d, seed=1)
    with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m.update_posterior(x, max_itr=3, num_init=1, tolerance=0.0)
    fit(o, x, max_itr=3, num_init=1, tolerance=0.0)
    _close(m.vl, o.vl, what="vl")
    for f in ("hn_alpha_vec", "hn_m_vecs", "hn_nus", "hn_w_mats_inv", "ns", "x_bar_vecs"):
        _close(getattr(m, f), getattr(o, f), what=f)
    assert np.array_equal(np.argmax(m.r_vecs, axis=1), np.argmax(o.r_vecs, axis=1))


@pytest.mark.parametrize("shape", [(20000, 16, 32), (20000, 16, 8), (30000, 8, 6), (10000, 5, 3), (9000, 20, 12), (7001, 12, 40),
                                   (4097, 4, 2), (12000, 12, 64)])
def test_fp32_mode_on_tensor_cores_against_fp64_oracle(shape):
    """precision='float32' on shapes the tcgen05 kernels cover (BGMM_PASS_TF32: whitened E-step GEMM + statistics GEMM in
    3xTF32 with TMEM accumulators): the same bar as the streaming fp32 kernel — 1e-4 against the fp64 oracle fed the SAME
    fp32-rounded X, assignments exact away from numerical ties."""
    from bayesml_b200 import _lib, gaussianmixture
    from oracle.gmm_vb_oracle import OracleGMM, fit
    n, d, k = shape
    lib = _lib.load()
    assert lib.bgmm_pass_supported(k, d, _lib.F32, _lib.PASS_TF32)
    assert lib.bgmm_pass_resolve(k, d, _lib.F32, _lib.PASS_AUTO, 0) == _lib.PASS_TF32
    rng = np.random.default_rng(n + d + k)
    mu = rng.normal(0, 4.0, size=(k, d))
    a = rng.normal(size=(k, d, d))
    chol = np.linalg.cholesky(a @ a.transpose(0, 2, 1) / d + 0.5 * np.eye(d))
    z = rng.integers(0, k, size=n)
    x32 = (mu[z] + np.einsum("nij,nj->ni", chol[z], rng.normal(size=(n, d)))).astype(np.float32)
    m = gaussianmixture.LearnModel(k, d, seed=2, precision="float32")
    o = OracleGMM(k, d, seed=2)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m.update_posterior(x32, max_itr=8, num_init=1, tolerance=0.0)
    assert m._engine().x.dtype.is_floating_point and m._engine().x.element_size() == 4
    tr = fit(o, x32, max_itr=8, num_init=1, tolerance=0.0)
    tol = 1e-4
    vals = _parse_progress(buf.getvalue())[0][0]
    _close(vals, tr.vl_history[0], rtol=tol, what="fp32-mode (tf32) VL history")
    # 1e-4 of each array's scale (largest magnitude).  The fp64 tests hold every entry to 1e-9 of its own value with a floor at
    # 1e-4 of the scale; in fp32 mode an entry-wise bar is not meaningful: a float32 X carries 6e-8, one pass differs from
    # the fp64 kernels on the same state by 2e-5 in ln rho, 5e-6 in r and 2e-7 .. 5e-7 of their scale in the statistics, and
    # these test mixtures contain components that SHARE a true cluster, whose soft boundary amplifies that to ~1.5e-5 of the
    # scale of m after 8 iterations (N_k: 5e-6 relative).  The ELBO and the responsibilities keep the 1e-4 relative bar.
    for f in ("hn_alpha_vec", "hn_m_vecs", "hn_kappas", "hn_nus", "hn_w_mats_inv", "ns"):
        _close(getattr(m, f), getattr(o, f), rtol=tol, what="fp32-mode (tf32) " + f, floor=1.0)
    # x_bar_k / S_k enter every update weighted by N_k, and a component that has lost its mass (N_k ~ 1e-30 in fp64, exactly 0
    # in fp32 where r < 1e-38 flushes to zero) has no meaningful mean: compare the weighted statistics
    _close(m.ns[:, None] * m.x_bar_vecs, o.ns[:, None] * o.x_bar_vecs, rtol=tol, what="fp32-mode (tf32) N x_bar", floor=1.0)
    _close(m.ns[:, None, None] * m.s_mats, o.ns[:, None, None] * o.s_mats, rtol=tol, what="fp32-mode (tf32) N S", floor=1.0)
    # responsibilities of the FITTED model: the parameters differ by ~1.5e-5 of their scale (above), which a sample on the soft
    # boundary between two components sharing a cluster turns into a few 1e-4 in r; the kernel-level statement — same state
    # in, r within 1e-4 — is test_fp32_tensor_core_pass_from_identical_state below
    assert np.allclose(m.r_vecs, o.r_vecs, rtol=0, atol=2e-3)
    margin = np.sort(o.r_vecs, axis=1)
    clear = (margin[:, -1] - margin[:, -2]) > 1e-2 if k > 1 else np.ones(n, dtype=bool)
    assert np.array_equal(np.argmax(m.r_vecs, axis=1)[clear], np.argmax(o.r_vecs, axis=1)[clear])


# the last four: fewer rows than one 128-sample tile / 64-sample sub-tile, a single row, one row more than a tile
@pytest.mark.parametrize("shape", [(20000, 16, 32), (30000, 8, 6), (10000, 5, 3), (9000, 20, 12), (7001, 12, 40),
                                   (63, 16, 4), (1, 4, 3), (129, 8, 33), (50, 21, 2)])
def test_fp32_tensor_core_pass_from_identical_state(shape):
    """One E-step + statistics sweep of the tcgen05 kernels from a GIVEN parameter set against the fp64 oracle's E-step from the
    same set on the same fp32-rounded X (north_star: 'identical inputs and identical initial state'): ln rho, r, N_k and the
    weighted statistics within 1e-4, arg max exact away from ties."""
    from bayesml_b200 import _lib, gaussianmixture
    from bayesml_b200.engine import VBEngine
    from oracle.gmm_vb_oracle import OracleGMM
    n, d, k = shape
    rng = np.random.default_rng(n + d + k)
    mu = rng.normal(0, 4.0, size=(k, d))
    a = rng.normal(size=(k, d, d))
    chol = np.linalg.cholesky(a @ a.transpose(0, 2, 1) / d + 0.5 * np.eye(d))
    z = rng.integers(0, k, size=n)
    x32 = (mu[z] + np.einsum("nij,nj->ni", chol[z], rng.normal(size=(n, d)))).astype(np.float32)
    o = OracleGMM(k, d)
    o.hn_m_vecs[:] = mu + 0.2 * rng.normal(size=mu.shape)
    o.hn_nus[:] = d + 2.0 + rng.uniform(0, 50, size=k)
    o.hn_kappas[:] = 1.0 + rng.uniform(0, 50, size=k)
    o.hn_alpha_vec[:] = 0.5 + rng.uniform(0, 100, size=k)
    for j in range(k):
        o.hn_w_mats_inv[j] = (chol[j] @ chol[j].T) * o.hn_nus[j] * rng.uniform(0.7, 1.4)
        o.hn_w_mats[j] = np.linalg.inv(o.hn_w_mats_inv[j])
    o.q_pi_features(); o.q_lambda_features()
    o.alloc(n)
    o.e_step(x32.astype(np.float64))
    model = gaussianmixture.LearnModel(k, d)
    eng = VBEngine(k, d, precision="float32", variant=_lib.PASS_TF32)
    eng.load_data(x32)
    model._push_prior(eng)
    eng.set_params(o.hn_alpha_vec, o.hn_m_vecs, o.hn_kappas, o.hn_nus, o.hn_w_mats_inv)
    st = eng.final_pass()
    r, lnrho, arg = eng.r_dev.cpu().numpy(), eng.lnrho_dev.cpu().numpy(), eng.argmax_dev.cpu().numpy()
    big = o.r_vecs > 1e-3
    assert np.max(np.abs(lnrho - o.ln_rho)[big]) < 1e-4
    assert np.allclose(r[big], o.r_vecs[big], rtol=1e-4)
    assert np.allclose(r, o.r_vecs, rtol=1e-4, atol=1e-6)
    margin = np.sort(o.r_vecs, axis=1)
    clear = (margin[:, -1] - margin[:, -2]) > 1e-4
    assert np.array_equal(arg[clear], np.argmax(o.r_vecs, axis=1)[clear])
    _close(st["ns"], o.ns, rtol=1e-4, what="N_k", floor=1.0)
    _close(st["ns"][:, None] * st["x_bar"], o.ns[:, None] * o.x_bar_vecs, rtol=1e-4, what="N x_bar", floor=1.0)
    _close(st["ns"][:, None, None] * st["s_mats"], o.ns[:, None, None] * o.s_mats, rtol=1e-4, what="N S", floor=1.0)


def test_fp32_precision_request_on_a_shape_without_fp32_kernel_uses_the_fp64_path():
    """precision='float32' with D=40 (neither fp32 kernel covers it): X is promoted on upload and the fp64 kernels run —
    results then meet the fp64 bar against the oracle on the same float32 array."""
    from bayesml_b200 import _lib, gaussianmixture
    from oracle.gmm_vb_oracle import OracleGMM, fit
    rng = np.random.default_rng(3)
    n, d, k = 8000, 40, 6
    x32 = (rng.normal(size=(n, d)) + 4.0 * rng.normal(size=(k, d))[rng.integers(0, k, size=n)]).astype(np.float32)
    m = gaussianmixture.LearnModel(k, d, seed=2, precision="float32")
    o = OracleGMM(k, d, seed=2)
    with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m.update_posterior(x32, max_itr=5, num_init=1, tolerance=0.0)
    fit(o, x32, max_itr=5, num_init=1, tolerance=0.0)
    assert m._engine().x.dtype.is_floating_point and m._engine().x.element_size() == 8
    _close(m.vl, o.vl, what="vl")
    _close(m.hn_m_vecs, o.hn_m_vecs, what="hn_m_vecs")
    assert np.allclose(m.r_vecs, o.r_vecs, rtol=RTOL, atol=1e-300)
