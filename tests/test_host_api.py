"""CPU: the C-ABI library builds, loads and exports every symbol of include/bgmm.h; host-side logic of the drop-in
LearnModel (validation, hyperparameter plumbing, features, RNG stream of the initialisations) matches the oracle."""
import ctypes
import os
import re
import pickle

import numpy as np
import pytest

from conftest import ROOT, load_golden
from bayesml_b200 import _lib, gaussianmixture
from bayesml_b200._exceptions import CriteriaError, DataFormatError, ParameterFormatError
from oracle.gmm_vb_oracle import OracleGMM


def test_library_exports_every_symbol_the_header_declares(lib_built):
    header = open(os.path.join(ROOT, "include", "bgmm.h")).read()
    declared = set(re.findall(r"\b(bgmm_[a-z_]+)\s*\(", header))
    assert {"bgmm_pass", "bgmm_small", "bgmm_layout", "bgmm_colsum", "bgmm_center", "bgmm_workspace_doubles",
            "bgmm_last_error", "bgmm_abi_version", "bgmm_comm_alloc", "bgmm_comm_open", "bgmm_comm_close",
            "bgmm_comm_free", "bgmm_comm_block_doubles", "bgmm_pass_supported"} <= declared
    lib = ctypes.CDLL(lib_built)
    for sym in declared:
        assert hasattr(lib, sym), sym
    assert _lib.load().bgmm_abi_version() == _lib.ABI_VERSION


def test_layout_is_consistent(lib_built):
    for K, D in [(3, 2), (32, 16), (64, 128), (1, 1)]:
        off, poff = _lib.layout(K, D, 101)
        P = 1 + D + D * (D + 1) // 2
        assert off["pitch"] == (P + 7) // 8 * 8
        assert off["stats_len"] == K * off["pitch"] + 8
        keys = ["center", "alpha0", "kappa0", "nu0", "m0", "w0inv", "lnb0", "lnc0", "params0", "params1", "stats", "ns",
                "xbar", "smats", "vlk", "vlterms", "ctrl", "vlhist", "total"]
        vals = [off[k] for k in keys]
        assert vals == sorted(vals) and len(set(vals)) == len(vals)
        assert off["params1"] - off["params0"] == off["params_len"]
        assert all(v % 8 == 0 for v in vals[:-1])
        assert _lib.load().bgmm_workspace_doubles(K, D) >= off["stats_len"]
        off2, _ = _lib.layout(K, D, 7)          # only vlhist's length (and the total) may depend on hist_len
        assert all(off2[k] == off[k] for k in keys[:-1])


def test_host_entry_points_reject_bad_arguments(lib_built):
    lib = _lib.load()
    off = (ctypes.c_int64 * 32)()
    assert lib.bgmm_layout(0, 2, 4, off, off) == -1
    assert b"bgmm_layout" in lib.bgmm_last_error()
    assert lib.bgmm_small(3, 2, None, 0, 1, 0.0, 2, None, None) == -1
    assert lib.bgmm_comm_block_doubles(32, 16) == 2 * (32 * 160 + 8) + 32
    assert lib.bgmm_pass(None, 5, 3, 2, 0, None, None, None, None, None, None, 0, 0, None) == -1
    with pytest.raises(RuntimeError, match="bgmm"):
        _lib.check(-1, "bgmm_pass")


def test_constructor_and_validation():
    m = gaussianmixture.LearnModel(3, 2)
    o = OracleGMM(3, 2)
    for a, b in [("h0_alpha_vec",) * 2, ("h0_w_mats_inv",) * 2, ("hn_w_mats",) * 2, ("_e_ln_pi_vec", "e_ln_pi_vec"),
                 ("_e_ln_lambda_dets", "e_ln_lambda_dets"), ("_ln_b_hn_w_nus", "ln_b_hn_w_nus"),
                 ("_ln_b_h0_w_nus", "ln_b_h0_w_nus"), ("_e_lambda_mats", "e_lambda_mats"), ("p_lambda_mats",) * 2,
                 ("p_nus",) * 2, ("p_pi_vec",) * 2]:
        assert np.array_equal(getattr(m, a), getattr(o, b)), a
    assert m._ln_c_h0_alpha == o.ln_c_h0_alpha
    assert m.r_vecs is None and m._ln_rho is None and m.vl == 0.0
    assert m.get_constants() == {"c_num_classes": 3, "c_degree": 2}
    with pytest.raises(ParameterFormatError):
        gaussianmixture.LearnModel(0, 2)
    with pytest.raises(ParameterFormatError):
        gaussianmixture.LearnModel(3, 2.0)
    with pytest.raises(ParameterFormatError):
        gaussianmixture.LearnModel(3, 2, h0_nus=np.array([0.5, 3.0, 3.0]))       # must exceed D-1
    with pytest.raises(ParameterFormatError):
        gaussianmixture.LearnModel(3, 2, h0_m_vecs=np.zeros((3, 3)))
    with pytest.raises(ParameterFormatError):
        gaussianmixture.LearnModel(3, 2, h0_w_mats=np.array([[1.0, 2.0], [2.0, 1.0]]))  # not positive definite
    with pytest.raises(ParameterFormatError):
        gaussianmixture.LearnModel(3, 2, h0_alpha_vec=np.array([1.0, -1.0, 1.0]))
    assert gaussianmixture.LearnModel(2, gaussianmixture.MAX_DEGREE).c_degree == 160
    with pytest.raises(ParameterFormatError, match="c_degree <= 160"):
        gaussianmixture.LearnModel(2, 161)                                         # bgmm_small's D x D in shared memory
    with pytest.raises(DataFormatError):
        m.update_posterior(np.zeros((5, 3)))
    with pytest.raises(DataFormatError):
        m.update_posterior([[0.0, 1.0]])
    with pytest.raises(DataFormatError):
        m.estimate_latent_vars(np.zeros((5, 3)))
    with pytest.raises(DataFormatError):
        m.pred_and_update(np.zeros((1, 2)))
    with pytest.raises(CriteriaError):
        m.estimate_params(loss="abs")
    with pytest.raises(CriteriaError):
        m.make_prediction(loss="KL")


def test_hyperparameter_plumbing_matches_reference_semantics(tmp_path):
    g = load_golden("traj_prior_d3k2")
    prior = {f: g[f] for f in ("h0_alpha_vec", "h0_m_vecs", "h0_kappas", "h0_nus", "h0_w_mats")}
    m = gaussianmixture.LearnModel(2, 3, **prior)
    o = OracleGMM(2, 3, **prior)
    assert np.array_equal(m._ln_b_h0_w_nus, o.ln_b_h0_w_nus)
    live = m.get_hn_params()["hn_m_vecs"]
    assert live is m.hn_m_vecs                                   # live references, not copies (:655-659)
    # set_hn_params refreshes features and the predictive parameters (:637-640)
    m.set_hn_params(hn_kappas=np.array([4.0, 5.0]), hn_nus=np.array([7.0, 9.5]))
    o.hn_kappas[:] = [4.0, 5.0]; o.hn_nus[:] = [7.0, 9.5]
    o.q_pi_features(); o.q_lambda_features(); o.pred_dist()
    assert np.array_equal(m._e_ln_lambda_dets, o.e_ln_lambda_dets)
    assert np.array_equal(m.p_lambda_mats, o.p_lambda_mats)
    assert np.array_equal(m.make_prediction("squared"), np.sum(o.p_pi_vec[:, None] * o.p_mu_vecs, axis=0))
    # scalar hyperparameters broadcast (:538-540)
    m.set_h0_params(h0_kappas=2.5)
    assert np.array_equal(m.h0_kappas, [2.5, 2.5]) and np.array_equal(m.hn_kappas, [2.5, 2.5])
    # pickle round trip (base.py:148-258): positional load of hn into h0
    path = str(tmp_path / "hn.pkl")
    m.set_hn_params(hn_alpha_vec=np.array([3.0, 4.0]))
    m.save_hn_params(path)
    assert set(pickle.load(open(path, "rb"))) == {"hn_alpha_vec", "hn_m_vecs", "hn_kappas", "hn_nus", "hn_w_mats"}
    m2 = gaussianmixture.LearnModel(2, 3).load_h0_params(path)
    assert np.array_equal(m2.h0_alpha_vec, [3.0, 4.0]) and np.array_equal(m2.hn_alpha_vec, [3.0, 4.0])
    with pytest.raises(ParameterFormatError):
        pickle.dump([1, 2], open(path, "wb"))
        m2.load_hn_params(path)
    m2.overwrite_h0_params()
    pi_hat, mu_hat, lam_hat = m2.estimate_params("0-1")
    assert pi_hat.shape == (2,) and lam_hat.shape == (2, 3, 3)
    dist = m2.estimate_params("KL")
    assert len(dist[1]) == 2 and len(dist[2]) == 2


def test_initialisations_consume_the_reference_rng_stream():
    g = load_golden("traj_d3k4")
    x = g["x"]
    m = gaussianmixture.LearnModel(4, 3, seed=int(g["seed"]))
    for restart in range(2):
        m.reset_hn_params()
        m._init_subsampling(x)
        assert np.array_equal(m.hn_m_vecs, g["init_hn_m_vecs"][restart])
        assert np.array_equal(m.hn_w_mats_inv, g["init_hn_w_mats_inv"][restart])
        assert np.array_equal(m.hn_w_mats, g["init_hn_w_mats"][restart])
    g = load_golden("traj_rr_d2k3")
    m = gaussianmixture.LearnModel(3, 2, seed=int(g["seed"]))
    for restart in range(2):
        assert np.array_equal(m._init_random_responsibility(g["x"].shape[0]), g["init_r_vecs"][restart])


def test_no_cpu_fallback_without_cuda(monkeypatch):
    import torch
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)      # the same check where a GPU is present
    m = gaussianmixture.LearnModel(3, 2, seed=0)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.update_posterior(np.random.default_rng(0).normal(size=(50, 2)))


def test_hmm_entry_points_reject_bad_arguments_without_touching_the_gpu(lib_built):
    """The hidden-Markov C-ABI entry points validate on the host first (no CUDA call is made for these inputs)."""
    lib = _lib.load()
    off = (ctypes.c_int64 * len(_lib.HMM_OFF_NAMES))()
    assert lib.bgmm_hmm_layout(0, off) == -1 and b"bgmm_hmm_layout" in lib.bgmm_last_error()
    assert lib.bgmm_hmm_layout(5, off) == 0
    h = dict(zip(_lib.HMM_OFF_NAMES, off))
    assert h["zeta0"] == 0 and h["set1"] - h["set0"] == 3 * 32 + 8 and h["total"] > h["vlx"] > h["sc"] > h["g0"] > h["ms"]
    assert lib.bgmm_hmm_supported(32, 128) == 1 and lib.bgmm_hmm_supported(33, 4) == 0 and lib.bgmm_hmm_supported(4, 129) == 0
    assert lib.bgmm_hmm_scan_workspace_doubles(40, 1000) == 0 and lib.bgmm_hmm_scan_workspace_doubles(8, 100000) > 100000 * 8
    assert lib.bgmm_hmm_small(3, 2, None, None, 0, 1, 0.0, 2, None) == -1
    assert lib.bgmm_hmm_pass(None, 10, 40, 2, None, None, None, None, None, None, None, None, None, 0, 0, None) == -3
    assert b"unsupported shape" in lib.bgmm_last_error()
    assert lib.bgmm_hmm_pass(None, 10, 4, 2, None, None, None, None, None, None, None, None, None, 0, 0, None) == -1
    assert lib.bgmm_hmm_viterbi(0, 4, None, None, None, None, None, None, None) == -1
    assert lib.bgmm_hmm_viterbi(10, 40, None, None, None, None, None, None, None) == -1
