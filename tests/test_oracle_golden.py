"""CPU: the oracle restatement reproduces every golden fixture recorded from the real reference."""
import numpy as np
import pytest
import scipy

from conftest import ln_rho_rows, load_golden
from oracle.gmm_vb_oracle import OracleGMM, fit

CASES = ["c1_readme", "traj_d3k4", "traj_d16k8", "traj_rr_d2k3", "traj_offset_d4k3", "traj_prior_d3k2", "traj_k1_d5",
         "conv_d2k4", "cond_sep1e4_d3k3", "cond_sep1e5_d2k3", "cond_outlier_d4k4", "cond_sep3e4_d16k6",
         "cond_sub_sep1e4_d3k3"]
# fixtures recorded with the reference's `_init_subsampling` replaced by a given initial state (make_golden.py: init_override)
GIVEN_INIT = {"cond_sep1e4_d3k3", "cond_sep1e5_d2k3", "cond_outlier_d4k4", "cond_sep3e4_d16k6"}
FIELD_MAP = {"ns": "ns", "x_bar_vecs": "x_bar_vecs", "s_mats": "s_mats", "hn_alpha_vec": "hn_alpha_vec",
             "hn_m_vecs": "hn_m_vecs", "hn_kappas": "hn_kappas", "hn_nus": "hn_nus", "hn_w_mats": "hn_w_mats",
             "hn_w_mats_inv": "hn_w_mats_inv", "_e_ln_pi_vec": "e_ln_pi_vec", "_e_ln_lambda_dets": "e_ln_lambda_dets",
             "_ln_b_hn_w_nus": "ln_b_hn_w_nus"}


def _fit_kwargs(g):
    return eval(str(g["fit_kwargs"]), {"__builtins__": {}}, {"dict": dict})


def _same(a, b, exact):
    if exact:
        return np.array_equal(a, b, equal_nan=True)
    return np.allclose(a, b, rtol=1e-10, atol=1e-12, equal_nan=True)


@pytest.mark.parametrize("name", CASES)
def test_oracle_reproduces_reference_trajectory(name):
    g = load_golden(name)
    # bit-exact only on the numpy/scipy the fixtures were recorded with (BLAS / RNG dependence)
    exact = str(g["numpy_version"]) == np.__version__ and str(g["scipy_version"]) == scipy.__version__
    K, D = int(g["K"]), int(g["D"])
    prior = {f: g[f] for f in ("h0_alpha_vec", "h0_m_vecs", "h0_kappas", "h0_nus", "h0_w_mats")}
    model = OracleGMM(K, D, seed=int(g["seed"]), **prior)
    states = []
    if name in GIVEN_INIT:
        restart = [0]

        def given_init(x_):
            model.hn_m_vecs[:] = g["init_hn_m_vecs"][restart[0]]
            model.hn_w_mats_inv[:] = g["init_hn_w_mats_inv"][restart[0]]
            model.hn_w_mats[:] = g["init_hn_w_mats"][restart[0]]
            model.q_lambda_features()
            restart[0] += 1
        model.init_subsampling = given_init

    def record(i, t, m):
        rec = {ref: np.array(getattr(m, mine)) for ref, mine in FIELD_MAP.items()}
        rec["vl_terms"] = np.array([m.vl] + [m.vl_terms[k] for k in
                                             ("p_x", "p_z", "p_pi", "p_mu_lambda", "q_z", "q_pi", "q_mu_lambda")])
        rec["restart"] = i
        states.append(rec)

    trace = fit(model, g["x"], on_state=record, **_fit_kwargs(g))
    assert len(states) == int(g["n_states"])
    assert np.array_equal([s["restart"] for s in states], g["restart_of_state"])
    for ref in FIELD_MAP:
        got = np.stack([s[ref] for s in states])
        assert _same(got, g["traj_" + ref], exact), ref
    assert _same(np.stack([s["vl_terms"] for s in states]), g["traj_vl_terms"], exact)
    for ref, mine in FIELD_MAP.items():
        assert _same(getattr(model, mine), g["final_" + ref], exact), "final " + ref
    assert _same(model.r_vecs, g["final_r_vecs"], exact)
    assert _same(model.ln_rho[ln_rho_rows(g)], g["final_ln_rho"], exact)
    assert _same(model.vl, g["final_vl_attr"], exact)
    assert trace.n_passes == len(states) - (len(trace.vl_history) if "random" in str(g["fit_kwargs"]) else 0) + 1
    # the '*' marks in the reference's progress text are the restarts that became the best so far (:873-874)
    lines = str(g["stdout"]).split("\n")
    starred = [i for i, ln in enumerate(lines) if ln.endswith("*")]
    assert trace.selected == starred[-1]
    assert sum(trace.converged) == str(g["stdout"]).count("(converged)")


def test_c1_anchor_values():
    """SURVEY.md §8c anchor (numpy 2.3.5): restart 0 wins with VL -4028.5489990077567; vl attribute is the last restart's."""
    g = load_golden("c1_readme")
    out = str(g["stdout"])
    assert "0. VL: -7824.254908764117" in out
    assert "VL: -4028.5489990077567" in out
    assert np.allclose(g["final_hn_alpha_vec"], [337.90550798, 334.49481452, 329.0996775])
    assert float(g["final_vl_attr"]) == -4427.637675715983
    assert int(g["n_states"]) == 659  # 649 iterations + 10 post-init evaluations


def test_latent_and_pred_fixture():
    g = load_golden("traj_d3k4")
    K, D = int(g["K"]), int(g["D"])
    model = OracleGMM(K, D, seed=int(g["seed"]))
    fit(model, g["x"], **_fit_kwargs(g))
    model.pred_dist()
    assert np.allclose(model.p_lambda_mats, g["pred_p_lambda_mats"], rtol=1e-12)
    assert np.allclose(model.p_nus, g["pred_p_nus"], rtol=1e-12)
    onehot = model.estimate_latent_vars(g["latent_x"], "0-1")
    assert np.array_equal(onehot, g["latent_onehot"])
    assert np.allclose(model.r_vecs, g["latent_r"], rtol=1e-10, atol=1e-300)
    assert np.allclose(model.ns, g["latent_ns_after"], rtol=1e-12)
