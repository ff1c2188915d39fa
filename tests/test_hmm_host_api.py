"""CPU: host-side contract of the drop-in hiddenmarkovnormal.LearnModel (no GPU): constructor, validation, parameter
plumbing, estimates, predictive parameters — against the real reference where it is present."""
import warnings

import numpy as np
import pytest

from bayesml_b200 import hiddenmarkovnormal
from bayesml_b200._exceptions import CriteriaError, DataFormatError, ParameterFormatError, ResultWarning
from oracle.ref_loader import load_reference_module, reference_available


def test_constructor_defaults_and_live_references():
    m = hiddenmarkovnormal.LearnModel(3, 2, seed=0)
    assert m.get_constants() == {"c_num_classes": 3, "c_degree": 2}
    assert np.array_equal(m.h0_zeta_vecs, np.full((3, 3), 0.5)) and np.array_equal(m.hn_zeta_vecs, m.h0_zeta_vecs)
    assert m.get_hn_params()["hn_zeta_vecs"] is m.hn_zeta_vecs            # live references, as the reference returns
    assert list(m.get_h0_params()) == ["h0_eta_vec", "h0_zeta_vecs", "h0_m_vecs", "h0_kappas", "h0_nus", "h0_w_mats"]
    assert m.alpha_vecs is None and m.gamma_vecs is None and m._cs is None and m.xi_mats is None
    assert np.allclose(m.p_a_mat, 1.0 / 3.0)
    assert m.vl == 0.0 and m._vl_p_a == 0.0


def test_validation_errors():
    with pytest.raises(ParameterFormatError):
        hiddenmarkovnormal.LearnModel(0, 2)
    with pytest.raises(ParameterFormatError):
        hiddenmarkovnormal.LearnModel(2, 2, h0_zeta_vecs=np.array([[1.0, -1.0], [1.0, 1.0]]))
    with pytest.raises(ParameterFormatError):
        hiddenmarkovnormal.LearnModel(2, 3, h0_m_vecs=np.zeros((2, 2)))
    with pytest.raises(ParameterFormatError):
        hiddenmarkovnormal.LearnModel(2, 3, h0_nus=np.array([1.0, 2.0]))
    with pytest.raises(ParameterFormatError):
        hiddenmarkovnormal.LearnModel(2, 2, h0_w_mats=np.array([[1.0, 2.0], [2.0, 1.0]]))
    with pytest.raises(TypeError):
        hiddenmarkovnormal.LearnModel(2, 2, np.ones(2))                  # hyperparameters are keyword-only (:516)
    m = hiddenmarkovnormal.LearnModel(2, 2)
    with pytest.raises(DataFormatError):
        m.update_posterior(np.zeros((5, 3)))
    with pytest.raises(DataFormatError):
        m.estimate_latent_vars(np.zeros((5, 3)))
    with pytest.raises(CriteriaError):
        m.estimate_latent_vars(np.zeros((5, 2)), loss="squared", viterbi=True)
    with pytest.raises(CriteriaError):
        m.estimate_latent_vars(np.zeros((5, 2)), loss="abs", viterbi=False)
    with pytest.raises(CriteriaError):
        m.estimate_params(loss="abs")
    with pytest.raises(DataFormatError):
        m.pred_and_update(np.zeros(3))


def test_broadcast_and_overwrite():
    m = hiddenmarkovnormal.LearnModel(3, 2, h0_eta_vec=2.0, h0_zeta_vecs=np.array([1.0, 2.0, 3.0]), h0_kappas=0.5)
    assert np.array_equal(m.h0_eta_vec, [2.0] * 3)
    assert np.array_equal(m.h0_zeta_vecs, np.tile([1.0, 2.0, 3.0], (3, 1)))
    m.set_hn_params(hn_zeta_vecs=np.full((3, 3), 4.0), hn_m_vecs=np.arange(6.0).reshape(3, 2))
    assert np.allclose(m._ln_a_tilde_mat, m._ln_a_tilde_mat[0, 0])
    m.overwrite_h0_params()
    assert np.array_equal(m.h0_zeta_vecs, np.full((3, 3), 4.0)) and np.array_equal(m.h0_m_vecs, m.hn_m_vecs)
    m.reset_hn_params()
    assert np.array_equal(m.hn_zeta_vecs, m.h0_zeta_vecs)


def test_host_features_and_estimates_equal_reference(tmp_path):
    # stored: priors, final hyperparameters, features and predictive parameters the reference produced (make_golden_hmm.py)
    from conftest import load_golden
    from test_hmm_oracle_golden import CASES, PRIOR
    hn = ("hn_eta_vec", "hn_zeta_vecs", "hn_m_vecs", "hn_kappas", "hn_nus", "hn_w_mats")
    pred = ("p_a_mat", "p_mu_vecs", "p_nus", "p_lambda_mats")
    for name in CASES:
        g = load_golden(name)
        mine = hiddenmarkovnormal.LearnModel(int(g["K"]), int(g["D"]), **{f: g[f] for f in PRIOR})
        for f in pred:                                   # prior-based, as the reference left them after its fit
            assert np.allclose(getattr(mine, f), g["stale_" + f], rtol=1e-13, atol=1e-15), (name, f)
        mine.set_hn_params(**{f: g["final_" + f] for f in hn})
        # hn_w_mats_inv is inv(hn_w_mats) here but the M-step's own matrix in the fixture: it and its log-determinant
        # terms are defined to cond * eps
        w_rtol = max(1e-13, 16 * np.finfo(float).eps * float(np.max(np.linalg.cond(g["final_hn_w_mats"]))))
        for f in ("hn_w_mats_inv", "_e_ln_lambda_dets", "_ln_b_hn_w_nus", "_ln_pi_tilde_vec", "_ln_a_tilde_mat"):
            rtol = w_rtol if f in ("hn_w_mats_inv", "_e_ln_lambda_dets", "_ln_b_hn_w_nus") else 1e-13
            assert np.allclose(getattr(mine, f), g["final_" + f], rtol=rtol, atol=1e-15), (name, f)
        for f in pred:
            assert np.allclose(getattr(mine, f), g["pred_" + f], rtol=1e-13, atol=1e-15), (name, f)
    if not reference_available():
        return
    hm = load_reference_module("hiddenmarkovnormal")
    rng = np.random.default_rng(2)
    a = rng.normal(size=(3, 2, 2))
    kw = dict(h0_eta_vec=np.array([1.5, 2.5, 3.0]), h0_zeta_vecs=rng.uniform(1.1, 4.0, size=(3, 3)),
              h0_m_vecs=rng.normal(size=(3, 2)), h0_kappas=np.array([0.5, 1.0, 2.0]), h0_nus=np.array([3.5, 4.0, 6.0]),
              h0_w_mats=a @ a.transpose(0, 2, 1) + np.eye(2))
    ref, mine = hm.LearnModel(3, 2, **kw), hiddenmarkovnormal.LearnModel(3, 2, **kw)
    for f in ("_ln_c_h0_eta_vec", "_ln_c_h0_zeta_vecs_sum", "_ln_b_h0_w_nus", "_ln_pi_tilde_vec", "_pi_tilde_vec",
              "_ln_a_tilde_mat", "_a_tilde_mat", "_ln_c_hn_zeta_vecs_sum", "_e_lambda_mats", "_e_ln_lambda_dets",
              "_ln_b_hn_w_nus", "p_a_mat", "p_mu_vecs", "p_nus", "p_lambda_mats", "hn_w_mats_inv"):
        assert np.allclose(getattr(mine, f), getattr(ref, f), rtol=1e-13, atol=1e-15), f
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for loss in ("squared", "0-1"):
            for got, want in zip(mine.estimate_params(loss), ref.estimate_params(loss)):
                assert np.allclose(got, want, rtol=1e-13, equal_nan=True)
    kl_m, kl_r = mine.estimate_params("KL"), ref.estimate_params("KL")
    assert np.allclose(kl_m[0].alpha, kl_r[0].alpha) and len(kl_m[1]) == len(kl_r[1]) == 3
    assert np.allclose(kl_m[2][1].shape, kl_r[2][1].shape) and kl_m[3][2].df == kl_r[3][2].df
    path = str(tmp_path / "hn.pkl")
    ref.save_hn_params(path)
    mine.load_hn_params(path)
    assert np.array_equal(mine.hn_zeta_vecs, ref.hn_zeta_vecs)
    low = hiddenmarkovnormal.LearnModel(2, 2)
    with pytest.warns(ResultWarning):
        est = low.estimate_params("0-1")
    assert np.isnan(est[0]).all() and np.isnan(est[1]).all()
