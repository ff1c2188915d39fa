"""GPU: the hidden-Markov (Gaussian emission) VB path (bgmm_hmm_pass / bgmm_hmm_small, SURVEY.md §8 f1) against the
golden trajectories recorded from the real reference and against the CPU oracle.  Tolerance: 1e-9 relative (fp64)."""
import contextlib
import io
import warnings

import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu

RTOL = 1e-9
PRIOR = ("h0_eta_vec", "h0_zeta_vecs", "h0_m_vecs", "h0_kappas", "h0_nus", "h0_w_mats")


def _close(a, b, rtol=RTOL, scale=None):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    scale = np.max(np.abs(b)) if scale is None else scale
    return np.allclose(a, b, rtol=rtol, atol=rtol * 1e-4 * max(scale, 1e-300))


def _fit_kwargs(g):
    return eval(str(g["fit_kwargs"]), {"__builtins__": {}}, {"dict": dict})


def _engine_for(g):
    from bayesml_b200.engine import HMMEngine
    from oracle.hmm_vb_oracle import OracleHMM
    K, D = int(g["K"]), int(g["D"])
    o = OracleHMM(K, D, **{f: g[f] for f in PRIOR})
    eng = HMMEngine(K, D)
    eng.load_data(np.asarray(g["x"]).reshape(-1, D))
    eng.set_hmm_prior(o.h0_eta_vec, o.h0_zeta_vecs, o.h0_m_vecs, o.h0_kappas, o.h0_nus, o.h0_w_mats_inv, o.ln_b_h0_w_nus,
                      o.ln_c_h0_eta_vec, o.ln_c_h0_zeta_vecs_sum)
    return eng, o


@pytest.mark.parametrize("name", ["hmm_traj_d2k3", "hmm_traj_d8k6", "hmm_traj_prior_d3k2", "hmm_traj_offset_d4k3",
                                  "hmm_traj_rr_d2k2", "hmm_len1_d2k3"])
def test_trajectory_from_identical_init(name, lib_built):
    """Every restart starts from the reference's recorded initial state; every ELBO evaluation must agree."""
    g = load_golden(name)
    kw = _fit_kwargs(g)
    eng, o = _engine_for(g)
    K, D = int(g["K"]), int(g["D"])
    restart = np.asarray(g["restart_of_state"])
    for i in range(kw["num_init"]):
        idx = np.nonzero(restart == i)[0]
        if "init_hn_m_vecs" in g.files:
            eng.set_hmm_params(o.h0_eta_vec, o.h0_zeta_vecs, g["init_hn_m_vecs"][i], o.h0_kappas, o.h0_nus,
                               g["init_hn_w_mats_inv"][i])
            hist, _ = eng.run(kw["max_itr"], kw["tolerance"])
        else:
            eng.set_hmm_params(o.h0_eta_vec, o.h0_zeta_vecs, o.h0_m_vecs, o.h0_kappas, o.h0_nus, o.h0_w_mats_inv)
            hist, _ = eng.run(kw["max_itr"], kw["tolerance"],
                              init=(g["init_gamma_vecs"][i], g["init_xi_mats"][i].sum(axis=0)))
        ref_vl = g["traj_vl_terms"][idx, 9]
        assert len(hist) == len(idx)
        assert _close(hist, ref_vl), (name, i, np.max(np.abs(hist - ref_vl) / np.abs(ref_vl)))
        p = eng.fetch_params()
        last = idx[-1]
        for mine, ref in (("alpha", "hn_eta_vec"), ("zeta", "hn_zeta_vecs"), ("m", "hn_m_vecs"), ("kappa", "hn_kappas"),
                          ("nu", "hn_nus"), ("w", "hn_w_mats"), ("winv", "hn_w_mats_inv"), ("ns", "ns"), ("ms", "ms"),
                          ("x_bar", "x_bar_vecs"), ("e_ln_pi", "_ln_pi_tilde_vec"), ("ln_a_tilde", "_ln_a_tilde_mat"),
                          ("e_ln_lambda_dets", "_e_ln_lambda_dets"), ("ln_b", "_ln_b_hn_w_nus")):
            assert _close(p[mine], g["traj_" + ref][last]), (name, i, mine)
        assert _close(p["s_mats"], g["traj_s_mats"][last], rtol=1e-8), (name, i, "s_mats")
        assert _close(p["gamma0"], g["traj_gamma0"][last])
        assert _close(p["sc"][0], g["traj_sum_ln_c"][last], scale=abs(float(g["traj_sum_ln_c"][last])) + 1.0)
        t, vx = p["vl_terms"], p["vlx"]
        mine_terms = np.array([t[0], vx[0], t[2], vx[1], t[3], vx[2], t[5], vx[3], t[6], t[7]])
        ref_terms = g["traj_vl_terms"][last]
        assert np.allclose(mine_terms, ref_terms, rtol=RTOL, atol=RTOL * np.max(np.abs(ref_terms))), (name, i)


@pytest.mark.parametrize("name", ["hmm_traj_d2k3", "hmm_conv_d3k3", "hmm_traj_rr_d2k2", "hmm_len1_d2k3"])
def test_update_posterior_end_to_end(name, lib_built):
    """The drop-in LearnModel from the same seed: same restarts, same progress text structure, same final state."""
    from bayesml_b200 import hiddenmarkovnormal
    g = load_golden(name)
    K, D = int(g["K"]), int(g["D"])
    model = hiddenmarkovnormal.LearnModel(K, D, seed=int(g["seed"]), **{f: g[f] for f in PRIOR})
    out = io.StringIO()
    with contextlib.redirect_stdout(out), warnings.catch_warnings(record=True) as wl:
        warnings.simplefilter("always")
        model.update_posterior(g["x"], **_fit_kwargs(g))
    ref_lines = str(g["stdout"]).split("\n")
    my_lines = out.getvalue().split("\n")
    assert len(my_lines) == len(ref_lines)
    assert [ln.endswith("*") for ln in my_lines] == [ln.endswith("*") for ln in ref_lines]
    assert out.getvalue().count("(converged)") == str(g["stdout"]).count("(converged)")
    assert len([w for w in wl if "not converged" in str(w.message)]) == int(g["n_warnings"])
    for f in ("hn_eta_vec", "hn_zeta_vecs", "hn_m_vecs", "hn_kappas", "hn_nus", "hn_w_mats", "hn_w_mats_inv", "ns", "ms",
              "x_bar_vecs", "_ln_pi_tilde_vec", "_ln_a_tilde_mat", "_e_ln_lambda_dets"):
        assert _close(getattr(model, f), g["final_" + f], rtol=1e-8), f
    assert _close(model.s_mats, g["final_s_mats"], rtol=1e-7)
    assert _close(model.vl, g["final_vl_attr"], rtol=1e-8, scale=abs(float(g["final_vl_attr"])))
    assert _close(model.gamma_vecs, g["final_gamma_vecs"], rtol=1e-8)
    assert _close(model.alpha_vecs, g["final_alpha_vecs"], rtol=1e-8)
    assert _close(model.beta_vecs, g["final_beta_vecs"], rtol=1e-8)
    assert _close(model._cs, g["final_cs"], rtol=1e-8)
    assert _close(model._ln_rho, g["final_ln_rho"], rtol=1e-8)
    if "final_xi_mats" in g.files:
        assert _close(model.xi_mats, g["final_xi_mats"], rtol=1e-8)
    assert _close(model.p_a_mat, g["stale_p_a_mat"])          # predictive params are the prior-based ones until calc_pred_dist
    model.calc_pred_dist()
    assert _close(model.p_lambda_mats, g["pred_p_lambda_mats"], rtol=1e-8)
    assert _close(model.make_prediction("squared"), g["pred_squared"], rtol=1e-8)
    assert _close(model.make_prediction("0-1"), g["pred_01"], rtol=1e-8)
    if "latent_x" in g.files:
        vit = model.estimate_latent_vars(g["latent_x"], loss="0-1", viterbi=True)
        assert np.array_equal(vit, g["latent_viterbi"])
        assert vit.dtype == g["latent_viterbi"].dtype
        assert _close(model.omega_vecs, g["latent_omega"], rtol=1e-8)
        assert model.phi_vecs.shape == model.omega_vecs.shape and np.array_equal(model.phi_vecs[0], np.zeros(K, dtype=int))
        assert _close(model.make_prediction("squared"), g["pred_squared"], rtol=1e-8)     # gamma of the fit is untouched
        onehot = model.estimate_latent_vars(g["latent_x"], loss="0-1", viterbi=False)
        assert np.array_equal(onehot, g["latent_marginal_onehot"])
        gam = model.estimate_latent_vars(g["latent_x"], loss="squared", viterbi=False)
        assert _close(gam, g["latent_gamma"], rtol=1e-8)
        assert _close(model.ms, g["latent_ms_after"], rtol=1e-8)


@pytest.mark.parametrize("shape", [(20000, 4, 5, 3), (9000, 16, 32, 2), (50000, 3, 17, 2), (3000, 40, 9, 2), (777, 2, 1, 3),
                                   # the limits K = 32 and D = 128 (bgmm_hmm_small's 256-thread block kernel with more than 48 KiB
                                   # of shared memory); D = 64 and 33: the last and first D of its 128-thread block kernel.  Enough
                                   # rows that the reference is defined: its subsampling initialisation takes each covariance from
                                   # sqrt(n) rows and it evaluates rho = exp(ln rho) unshifted, so with too few rows some element
                                   # has every component below exp(-745) and its forward recursion is NaN (at (3000, 128, 32),
                                   # (20000, 128, 32) and (4000, 64, 5)).
                                   (40000, 128, 32, 2), (6000, 64, 5, 2), (6000, 33, 17, 2)])
def test_against_oracle_larger_shapes(shape, lib_built):
    """Seeded sticky-chain data at sizes the oracle finishes in seconds; many chunks, K not a power of two."""
    from bayesml_b200.engine import HMMEngine
    from oracle.hmm_vb_oracle import OracleHMM
    n, D, K, iters = shape
    rng = np.random.default_rng(n + D + K)
    mu = rng.normal(0.0, 4.0, size=(K, D))
    z = np.empty(n, dtype=np.int64)
    z[0] = 0
    jump = rng.random(n) > 0.95
    nxt = rng.integers(0, K, size=n)
    for i in range(1, n):
        z[i] = nxt[i] if jump[i] else z[i - 1]
    x = mu[z] + rng.normal(size=(n, D))
    o = OracleHMM(K, D, seed=1)
    o.alloc(n)
    o.init_fb_params()
    o.reset_hn()
    o.init_subsampling(x)
    init_m, init_winv = o.hn_m_vecs.copy(), o.hn_w_mats_inv.copy()
    o.e_step(x)
    o.calc_vl()
    ref = [o.vl]
    for _ in range(iters):
        o.iterate(x)
        ref.append(o.vl)
    eng = HMMEngine(K, D)
    eng.load_data(x)
    eng.set_hmm_prior(o.h0_eta_vec, o.h0_zeta_vecs, o.h0_m_vecs, o.h0_kappas, o.h0_nus, o.h0_w_mats_inv, o.ln_b_h0_w_nus,
                      o.ln_c_h0_eta_vec, o.ln_c_h0_zeta_vecs_sum)
    eng.set_hmm_params(o.h0_eta_vec, o.h0_zeta_vecs, init_m, o.h0_kappas, o.h0_nus, init_winv)
    hist, _ = eng.run(iters, 0.0)
    assert _close(hist, ref), np.max(np.abs(np.asarray(hist) - ref) / np.abs(ref))
    p = eng.fetch_params()
    assert _close(p["ms"], o.ms, rtol=1e-8)
    assert _close(p["ns"], o.ns, rtol=1e-8)
    assert _close(p["zeta"], o.hn_zeta_vecs, rtol=1e-8)
    assert _close(p["m"], o.hn_m_vecs, rtol=1e-8)
    assert np.allclose(eng.gamma_buf.cpu().numpy(), o.gamma_vecs, rtol=1e-7, atol=1e-12)
    assert np.allclose(eng.cs_buf.cpu().numpy(), o.cs, rtol=1e-8)


def test_unsupported_shape_fails_loudly(lib_built):
    from bayesml_b200.engine import HMMEngine
    with pytest.raises(RuntimeError, match="unsupported shape"):
        HMMEngine(40, 4)


def test_window_and_basis_paths_agree(lib_built, monkeypatch):
    """The two ways of getting the chunk boundary vectors — warm-up windows (when the Birkhoff criterion on A~ holds) and
    K basis runs + sequential sweep — must give the same fit; the window path must actually have been taken."""
    from bayesml_b200.engine import HMMEngine
    n, D, K, iters = 1_500_000, 2, 4, 5          # chunks of 368 elements: a window of ~230 steps pays off
    rng = np.random.default_rng(5)
    mu = rng.normal(0.0, 3.0, size=(K, D))
    jump = rng.random(n) > 0.7
    jump[0] = True
    nxt = rng.integers(0, K, size=n)
    z = nxt[np.maximum.accumulate(np.where(jump, np.arange(n), 0))]
    x = mu[z] + rng.normal(size=(n, D))
    eye = np.tile(np.eye(D), (K, 1, 1))
    out = {}
    for cap in ("0", "16384"):
        monkeypatch.setenv("BGMM_HMM_WINDOW_CAP", cap)
        eng = HMMEngine(K, D)
        eng.load_data(x)
        eng.set_hmm_prior(np.full(K, .5), np.full((K, K), .5), np.zeros((K, D)), np.ones(K), np.full(K, float(D)), eye,
                          np.zeros(K), 0.0, 0.0)
        eng.set_hmm_params(np.full(K, .5), np.full((K, K), .5), mu + 0.3, np.ones(K), np.full(K, float(D)), eye * D)
        hist, _ = eng.run(iters, 0.0)
        out[cap] = (hist, eng.fetch_params(), eng.gamma_buf.cpu().numpy(), eng.cs_buf.cpu().numpy())
    assert out["0"][1]["window"] == 0 and out["16384"][1]["window"] >= 8
    assert np.allclose(out["0"][0], out["16384"][0], rtol=1e-11)
    for key in ("ms", "zeta", "m", "winv", "ns"):
        assert np.allclose(out["0"][1][key], out["16384"][1][key], rtol=1e-10, atol=1e-12), key
    assert np.allclose(out["0"][2], out["16384"][2], rtol=1e-9, atol=1e-13)
    assert np.allclose(out["0"][3], out["16384"][3], rtol=1e-11)


@pytest.mark.parametrize("K,D,n", [(32, 3, 120_000), (12, 2, 90_000), (17, 4, 40_000), (8, 2, 200_000), (3, 2, 100_000), (5, 3, 60_000)])
def test_basis_runs_match_the_oracle(K, D, n, lib_built, monkeypatch):
    """Phase A / A' (hmm_basis_mma_kernel: the K basis runs of a chunk as one DMMA matrix recursion, K padded to 8 below 8)
    against the oracle: same fit.  The window shortcut is disabled so the basis path runs."""
    from bayesml_b200.engine import HMMEngine
    from oracle.hmm_vb_oracle import OracleHMM
    rng = np.random.default_rng(K + D)
    mu = rng.normal(0.0, 3.0, size=(K, D))
    jump = rng.random(n) > 0.9
    jump[0] = True
    nxt = rng.integers(0, K, size=n)
    z = nxt[np.maximum.accumulate(np.where(jump, np.arange(n), 0))]
    x = mu[z] + rng.normal(size=(n, D))
    o = OracleHMM(K, D, seed=2)
    o.alloc(n)
    o.init_fb_params()
    o.reset_hn()
    o.init_subsampling(x)
    init_m, init_winv = o.hn_m_vecs.copy(), o.hn_w_mats_inv.copy()
    monkeypatch.setenv("BGMM_HMM_WINDOW_CAP", "0")
    eng = HMMEngine(K, D)
    eng.load_data(x)
    eng.set_hmm_prior(o.h0_eta_vec, o.h0_zeta_vecs, o.h0_m_vecs, o.h0_kappas, o.h0_nus, o.h0_w_mats_inv, o.ln_b_h0_w_nus,
                      o.ln_c_h0_eta_vec, o.ln_c_h0_zeta_vecs_sum)
    eng.set_hmm_params(o.h0_eta_vec, o.h0_zeta_vecs, init_m, o.h0_kappas, o.h0_nus, init_winv)
    hist, _ = eng.run(3, 0.0)
    hist, p = np.asarray(hist), eng.fetch_params()
    assert p["window"] == 0
    o.e_step(x)
    o.calc_vl()
    ref = [o.vl]
    for _ in range(3):
        o.iterate(x)
        ref.append(o.vl)
    assert _close(hist, ref), np.max(np.abs(hist - ref) / np.abs(ref))
    for mine, name in (("ms", "ms"), ("zeta", "hn_zeta_vecs"), ("m", "hn_m_vecs"), ("winv", "hn_w_mats_inv"), ("ns", "ns")):
        assert _close(p[mine], getattr(o, name)), mine
    assert np.allclose(eng.gamma_buf.cpu().numpy(), o.gamma_vecs, rtol=1e-7, atol=1e-12)
    assert _close(eng.cs_buf.cpu().numpy(), o.cs, rtol=1e-8)


def test_viterbi_long_sequence_is_bit_identical_to_the_numpy_recursion(lib_built):
    """bgmm_hmm_viterbi on a 300k-element sequence vs the reference's recursion (numpy, same ln rho): omega, phi and the
    path are bit-identical (same operation order)."""
    import torch
    from bayesml_b200 import _lib
    n, K = 300_000, 7
    rng = np.random.default_rng(11)
    ln_rho = rng.normal(size=(n, K)) * 3.0 - 5.0
    ln_pi = np.log(rng.dirichlet(np.ones(K)))
    ln_a = np.log(rng.dirichlet(np.ones(K), size=K))
    omega = np.zeros((n, K))
    phi = np.zeros((n, K), dtype=np.int64)
    omega[0] = ln_rho[0] + ln_pi
    for i in range(1, n):
        cand = ln_a + omega[i - 1, :, np.newaxis]
        omega[i] = ln_rho[i] + np.max(cand, axis=0)
        phi[i] = np.argmax(cand, axis=0)
    path = np.empty(n, dtype=np.int64)
    path[-1] = np.argmax(omega[-1])
    for i in range(n - 2, -1, -1):
        path[i] = phi[i + 1, path[i + 1]]
    dev = torch.device("cuda:0")
    t = lambda a: torch.as_tensor(a).to(dev)  # noqa: E731
    d_rho, d_pi, d_a = t(ln_rho), t(ln_pi), t(ln_a)
    d_om = torch.empty((n, K), dtype=torch.float64, device=dev)
    d_phi = torch.empty((n, K), dtype=torch.int32, device=dev)
    d_path = torch.empty(n, dtype=torch.int32, device=dev)
    _lib.check(_lib.load().bgmm_hmm_viterbi(n, K, d_rho.data_ptr(), d_pi.data_ptr(), d_a.data_ptr(), d_om.data_ptr(),
                                            d_phi.data_ptr(), d_path.data_ptr(), torch.cuda.current_stream().cuda_stream),
               "bgmm_hmm_viterbi")
    assert np.array_equal(d_om.cpu().numpy(), omega)
    assert np.array_equal(d_phi.cpu().numpy(), phi)
    assert np.array_equal(d_path.cpu().numpy(), path)
