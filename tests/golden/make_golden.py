"""Generate tests/golden/*.npz by running the REAL reference (/root/reference) in the build container.

    python tests/golden/make_golden.py

The reference has no GMM tests or golden vectors of its own (SURVEY.md §4), so these fixtures ARE the
parity pin: the reference's `gaussianmixture.LearnModel` is run on seeded inputs and its state is
recorded after every `_calc_vl` call (post-init and once per VB iteration, _gaussianmixture.py:860,:867)
plus the state right after each initialisation (:851/:854), so that the CUDA path and the oracle can be
started from IDENTICAL initial state and compared iteration by iteration.

Recorded with numpy/scipy versions stored in each file (RNG-dependent values are only valid for them).
"""
import contextlib
import io
import os
import sys
import warnings

import numpy as np
import scipy

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
from conftest import save_golden  # noqa: E402
from oracle.ref_loader import load_reference_gaussianmixture  # noqa: E402

gm = load_reference_gaussianmixture()
ONLY = set(sys.argv[1:])          # optional: names of the cases to (re)generate; default all

STATE_FIELDS = ("ns", "x_bar_vecs", "s_mats", "hn_alpha_vec", "hn_m_vecs", "hn_kappas", "hn_nus",
                "hn_w_mats", "hn_w_mats_inv", "_e_ln_pi_vec", "_e_ln_lambda_dets", "_ln_b_hn_w_nus")
VL_FIELDS = ("vl", "_vl_p_x", "_vl_p_z", "_vl_p_pi", "_vl_p_mu_lambda", "_vl_q_z", "_vl_q_pi", "_vl_q_mu_lambda")


class Recorder:
    """Wraps a reference LearnModel instance and records its trajectory."""

    def __init__(self, model):
        self.model = model
        self.states = []        # one dict per _calc_vl call
        self.inits = []         # one dict per restart
        self.restart_of_state = []
        self._restart = -1
        orig_vl, orig_sub, orig_rr = model._calc_vl, model._init_subsampling, model._init_random_responsibility

        def calc_vl():
            orig_vl()
            rec = {f: np.array(getattr(model, f)) for f in STATE_FIELDS}
            rec["vl_terms"] = np.array([float(getattr(model, f)) for f in VL_FIELDS])
            self.states.append(rec)
            self.restart_of_state.append(self._restart)

        def init_sub(x):
            self._restart += 1
            orig_sub(x)
            self.inits.append({"hn_m_vecs": np.array(model.hn_m_vecs),
                               "hn_w_mats_inv": np.array(model.hn_w_mats_inv),
                               "hn_w_mats": np.array(model.hn_w_mats)})

        def init_rr(x):
            self._restart += 1
            orig_rr(x)
            self.inits.append({"r_vecs": np.array(model.r_vecs)})

        model._calc_vl, model._init_subsampling, model._init_random_responsibility = calc_vl, init_sub, init_rr


def synth(seed, n, d, k, spread=4.0, offset=0.0):
    """Seeded mixture data (numpy only; independent of the reference's slow GenModel.gen_sample)."""
    rng = np.random.default_rng(seed)
    mu = rng.normal(0.0, spread, size=(k, d)) + offset
    a = rng.normal(size=(k, d, d))
    cov = a @ a.transpose(0, 2, 1) / d + 0.5 * np.eye(d)
    chol = np.linalg.cholesky(cov)
    z = rng.integers(0, k, size=n)
    eps = rng.normal(size=(n, d))
    return mu[z] + np.einsum("nij,nj->ni", chol[z], eps)


def run_case(name, x, k, d, seed, fit_kwargs, prior_kwargs=None, latent_x=None, init_override=None):
    if ONLY and name not in ONLY:
        return
    model = gm.LearnModel(k, d, seed=seed, **(prior_kwargs or {}))
    if init_override is not None:
        # the reference's VB iterations from a GIVEN initial state: `_init_subsampling` (:786-796) is replaced by a
        # function that writes hn_m_vecs / hn_w_mats(_inv) and refreshes the features exactly as the original does (:796)
        def patched(x_, _model=model):
            init_override(_model, x_)
            _model._calc_q_lambda_features()
        model._init_subsampling = patched
    rec = Recorder(model)
    out = io.StringIO()
    with contextlib.redirect_stdout(out), warnings.catch_warnings(record=True) as wlist:
        warnings.simplefilter("always")
        model.update_posterior(x, **fit_kwargs)
    payload = {
        "x": x, "K": k, "D": d, "seed": seed,
        "numpy_version": np.__version__, "scipy_version": scipy.__version__,
        "fit_kwargs": repr(fit_kwargs), "stdout": out.getvalue(),
        "n_warnings": len([w for w in wlist if "not converged" in str(w.message)]),
        "restart_of_state": np.array(rec.restart_of_state),
        "n_states": len(rec.states),
        "final_vl_attr": float(model.vl),
        "final_r_vecs": np.array(model.r_vecs), "final_ln_rho": np.array(model._ln_rho),
    }
    for f in STATE_FIELDS:
        payload["traj_" + f] = np.stack([s[f] for s in rec.states])
        payload["final_" + f] = np.array(getattr(model, f))
    payload["traj_vl_terms"] = np.stack([s["vl_terms"] for s in rec.states])
    for key in rec.inits[0]:
        payload["init_" + key] = np.stack([ini[key] for ini in rec.inits])
    for f in ("h0_alpha_vec", "h0_m_vecs", "h0_kappas", "h0_nus", "h0_w_mats"):
        payload[f] = np.array(getattr(model, f))
    for f in ("p_pi_vec", "p_mu_vecs", "p_nus", "p_lambda_mats"):
        payload["stale_" + f] = np.array(getattr(model, f))       # prior-based after update_posterior (SURVEY §3.1)
    model.calc_pred_dist()
    for f in ("p_pi_vec", "p_mu_vecs", "p_nus", "p_lambda_mats"):
        payload["pred_" + f] = np.array(getattr(model, f))
    if latent_x is not None:
        # log predictive density of the rows of latent_x: the mixture of Student-t distributions of
        # bayesml/gaussianmixture/__init__.py:86-97, evaluated with the function the reference itself calls for that
        # density (scipy.stats.multivariate_t, _gaussianmixture.py:1093) on the reference's own p_* parameters
        from scipy.special import logsumexp
        from scipy.stats import multivariate_t
        comp = np.stack([np.log(model.p_pi_vec[j])
                         + multivariate_t.logpdf(latent_x, loc=model.p_mu_vecs[j], shape=np.linalg.inv(model.p_lambda_mats[j]),
                                                 df=model.p_nus[j]) for j in range(k)], axis=1)
        payload["pred_logdens"] = logsumexp(comp, axis=1)
        payload["latent_x"] = latent_x
        payload["latent_onehot"] = model.estimate_latent_vars(latent_x, loss="0-1")
        payload["latent_r"] = np.array(model.estimate_latent_vars(latent_x, loss="squared"))
        payload["latent_ns_after"] = np.array(model.ns)
    path = save_golden(name, payload)
    print(f"{name}: {len(rec.states)} states, {os.path.getsize(path) / 1024:.0f} KiB")


def separated(seed, n, d, k, sep, sigma=1.0, outlier=None):
    """Tight clusters far apart (conditioning cases): unit-scale clusters whose means are `sep` sigma apart; with
    `outlier` the last cluster alone sits that far away and the others are `sep` apart."""
    rng = np.random.default_rng(seed)
    dirs = rng.normal(size=(k, d))
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    mu = dirs * sep * rng.uniform(0.5, 1.0, size=(k, 1))
    if outlier is not None:
        mu[-1] = dirs[-1] * outlier
    a = rng.normal(size=(k, d, d))
    chol = np.linalg.cholesky(a @ a.transpose(0, 2, 1) / d + 0.5 * np.eye(d)) * sigma
    z = rng.integers(0, k, size=n)
    return mu[z] + np.einsum("nij,nj->ni", chol[z], rng.normal(size=(n, d))), mu


def near_truth_init(mu, jitter, seed):
    """Initial state close to the true cluster means (keeps the trajectory out of the symmetry-breaking phase, where any
    two correct implementations diverge): m_k = mu_k + jitter, W_k^-1 = nu_k I."""
    def init(model, x):
        rng = np.random.default_rng(seed)
        model.hn_m_vecs[:] = mu + rng.normal(size=mu.shape) * jitter
        for k in range(mu.shape[0]):
            model.hn_w_mats_inv[k] = np.eye(mu.shape[1]) * model.hn_nus[k]
            model.hn_w_mats[k] = np.linalg.inv(model.hn_w_mats_inv[k])
    return init


def main():
    # conditioning cases (VERDICT r1 weak #1): clusters 1e4 / 1e5 of their own width apart, and one far outlier cluster
    # (prior means h0_m_vecs at the cluster means: with the default m0 = 0 the rank-one term kappa0 N/(kappa0+N) (x_bar-m0)(x_bar-m0)^T
    #  makes hn_w_mats_inv itself ill-conditioned (cond ~ sep^2) and its LAPACK inverse hn_w_mats uncertain at cond * eps —
    #  the default-prior variant is the last case below and is compared with that allowance)
    x, mu = separated(81, 900, 3, 3, 1.0e4)
    run_case("cond_sep1e4_d3k3", x, 3, 3, 6, dict(max_itr=10, num_init=1, tolerance=0.0),
             prior_kwargs=dict(h0_m_vecs=mu), init_override=near_truth_init(mu, 0.5, 1))
    x, mu = separated(82, 800, 2, 3, 1.0e5)
    run_case("cond_sep1e5_d2k3", x, 3, 2, 6, dict(max_itr=10, num_init=1, tolerance=0.0),
             prior_kwargs=dict(h0_m_vecs=mu), init_override=near_truth_init(mu, 0.5, 2))
    x, mu = separated(83, 1200, 4, 4, 8.0, outlier=1.0e5)
    run_case("cond_outlier_d4k4", x, 4, 4, 6, dict(max_itr=10, num_init=1, tolerance=0.0),
             prior_kwargs=dict(h0_m_vecs=mu), init_override=near_truth_init(mu, 0.3, 3))
    x, mu = separated(84, 2000, 16, 6, 3.0e4)
    run_case("cond_sep3e4_d16k6", x, 6, 16, 6, dict(max_itr=6, num_init=1, tolerance=0.0),
             prior_kwargs=dict(h0_m_vecs=mu), init_override=near_truth_init(mu, 0.3, 4))
    # the same geometry through the reference's own subsampling initialisation (all components start near the global mean)
    x, mu = separated(85, 900, 3, 3, 1.0e4)
    run_case("cond_sub_sep1e4_d3k3", x, 3, 3, 6, dict(max_itr=12, num_init=1, tolerance=0.0))

    # C1 — the README-scale config of BASELINE.json configs[0]; anchor values in SURVEY.md §8c
    g = gm.GenModel(c_num_classes=3, c_degree=2, mu_vecs=np.array([[-5., -5.], [0., 0.], [5., 5.]]), seed=0)
    x, _ = g.gen_sample(1000)
    run_case("c1_readme", x, 3, 2, 1, dict(), latent_x=x[:100] + 0.25)

    # fixed-length trajectories (tolerance=0.0 -> exactly max_itr iterations, SURVEY §7)
    run_case("traj_d3k4", synth(11, 600, 3, 4), 4, 3, 5,
             dict(max_itr=15, num_init=2, tolerance=0.0), latent_x=synth(12, 50, 3, 4))
    run_case("traj_d16k8", synth(21, 3000, 16, 8), 8, 16, 7, dict(max_itr=8, num_init=1, tolerance=0.0))
    run_case("traj_rr_d2k3", synth(31, 400, 2, 3), 3, 2, 9,
             dict(max_itr=12, num_init=2, tolerance=0.0, init_type="random_responsibility"))
    # offset data (mean 1000 sigma away from the origin): the centring / shifted-moment hard part of SURVEY §7
    run_case("traj_offset_d4k3", synth(41, 800, 4, 3, offset=1000.0), 3, 4, 3,
             dict(max_itr=10, num_init=1, tolerance=0.0))
    # non-default prior, K=1 (closed-form special case), 3-D input (leading dims flattened, :834)
    d, k = 3, 2
    rng = np.random.default_rng(51)
    a = rng.normal(size=(k, d, d))
    prior = dict(h0_alpha_vec=np.array([1.5, 0.7]), h0_m_vecs=rng.normal(size=(k, d)),
                 h0_kappas=np.array([0.3, 2.0]), h0_nus=np.array([3.5, 6.0]),
                 h0_w_mats=a @ a.transpose(0, 2, 1) + np.eye(d))
    run_case("traj_prior_d3k2", synth(52, 500, 3, 2).reshape(5, 100, 3), 2, 3, 2,
             dict(max_itr=10, num_init=2, tolerance=0.0), prior_kwargs=prior)
    run_case("traj_k1_d5", synth(61, 300, 5, 1), 1, 5, 4, dict(max_itr=4, num_init=1, tolerance=0.0))
    # default-tolerance run with convergence + selection among restarts
    run_case("conv_d2k4", synth(71, 1500, 2, 4, spread=6.0), 4, 2, 8, dict(max_itr=60, num_init=4))


if __name__ == "__main__":
    main()
