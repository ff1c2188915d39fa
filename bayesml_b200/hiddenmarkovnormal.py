"""Drop-in replacement for `bayesml.hiddenmarkovnormal.LearnModel` whose variational-Bayes fit runs on a B200.

Same constructor, methods, attribute names, error types and printed progress text as the reference class
(/root/reference/bayesml/hiddenmarkovnormal/_hiddenmarkovnormal.py:451-1558, cited per method).  The emission
densities, the scaled forward / backward recursions (as chunked parallel scans), gamma, the xi sums, the sufficient
statistics, the M-steps, the ELBO and the convergence test run in hand-written sm_100a kernels (libbgmm.so,
include/bgmm.h: bgmm_hmm_pass / bgmm_hmm_small) through `bayesml_b200.engine.HMMEngine`; there is no CPU fallback
for that path (float64, c_num_classes <= 32, c_degree <= 128; anything else raises).  What stays on the host is
K-sized numpy work outside the iteration loop: argument checks, hyperparameter plumbing, the RNG-consuming
initialisations (so the random stream is the reference's), restart bookkeeping and the predictive parameters.  The
Viterbi path of `estimate_latent_vars` (max-plus recursion + back-tracking) also runs on the device (bgmm_hmm_viterbi).

The per-element arrays (`_ln_rho`, `_rho`, `alpha_vecs`, `beta_vecs`, `gamma_vecs`, `_cs`, `xi_mats`) stay on the
GPU until the attribute is read; `xi_mats` (N x K x K) is formed on the host from them on first access.

Several independent sequences (`lengths=` of `update_posterior` / `estimate_latent_vars`, keyword only): the rows of x
are the sequences concatenated in order, and they share one posterior.  The recursions restart at every sequence start
(forward from pi~, backward from ones at every sequence end), xi is zero at every start (so `ms` counts only transitions
inside a sequence), E ln p(z) / E ln q(z) take gamma summed over the sequence starts, and the Viterbi path is decoded per
sequence.  The per-element arrays keep their (N, K) / (N,) shapes over the concatenated rows.  `lengths=None` and
`lengths=[N]` are the single-sequence path.

`GenModel` is the reference's generative model (pi ~ Dir(h_eta_vec), every row of A ~ Dir(h_zeta_vecs[k]), (mu_k,
Lambda_k) ~ Gauss-Wishart, z a Markov chain, x ~ N(mu_z, Lambda_z^-1)).  `gen_sample(n)` is the reference's per-element
loop with `self.rng`; `gen_sample(n, device="cuda:i")` draws the same distribution on the device (bgmm_hmm_gen_sample:
the chain sampled exactly by composing per-element transition maps over chunks, counter-based Philox, NOT numpy's
stream; c_num_classes <= 32 and c_degree <= 256 there, no CPU fallback).

Additive, defaulted options (they do not exist in the reference): `device`, `device_init` (of `LearnModel`: draw the
'random_responsibility' initial state on the device, bgmm_hmm_init_random: same distribution, NOT numpy's random
stream), `lengths` (of `LearnModel.update_posterior`, `LearnModel.estimate_latent_vars` and `GenModel.gen_sample`),
`as_numpy` (of `GenModel.gen_sample`).
"""
import warnings

import numpy as np
from scipy.special import digamma, gammaln
from scipy.stats import dirichlet as ss_dirichlet
from scipy.stats import multivariate_t as ss_multivariate_t
from scipy.stats import wishart as ss_wishart

from . import _check, base
from ._exceptions import CriteriaError, DataFormatError, ParameterFormatError, ResultWarning
from .gaussianmixture import _LazyDeviceArray

MAX_NUM_CLASSES, MAX_DEGREE = 32, 128        # limits of the device path (bgmm_hmm_supported)

GEN_MAX_NUM_CLASSES, GEN_MAX_DEGREE = 32, 256   # limits of the device sampler (bgmm_hmm_gen_sample)

__all__ = ["GenModel", "LearnModel"]

_HN_NAMES = ("hn_eta_vec", "hn_zeta_vecs", "hn_m_vecs", "hn_kappas", "hn_nus", "hn_w_mats", "hn_w_mats_inv")
_LAZY = ("_ln_rho", "alpha_vecs", "beta_vecs", "gamma_vecs", "_cs")


def _lazy_property(name):
    slot = "_lazy_" + name.lstrip("_")

    def getter(self):
        return getattr(self, slot).get()

    def setter(self, value):
        getattr(self, slot).set_host(value)

    return property(getter, setter)


def _inverse_cdf_table(pi_vec, a_mat):
    """The (K + 1, K) inverse-CDF table of bgmm_hmm_gen_sample: row 0 for pi, row 1 + s for row s of A.  Each row is the
    cumulative sum of its probabilities with the entry of its last positive-probability state set to 2.0; state k is
    drawn for u in (0, 1) as the first k with u <= row[k], so a zero-probability state is never drawn, even when the
    rounded cumulative sum ends below 1 and u falls above it."""
    p = np.vstack([pi_vec[np.newaxis, :], a_mat])
    cdf = np.cumsum(p, axis=1)
    last = p.shape[1] - 1 - np.argmax(p[:, ::-1] > 0, axis=1)
    cdf[np.arange(p.shape[0]), last] = 2.0
    return cdf


class GenModel(base.Generative):
    """The stochastic data generative model of the Bayesian hidden Markov model with Gaussian emissions: pi ~
    Dir(h_eta_vec), a_mat[k] ~ Dir(h_zeta_vecs[k]), (mu_k, Lambda_k) ~ Gauss-Wishart(h_m_vecs, h_kappas, h_nus, h_w_mats),
    z_0 ~ Cat(pi), z_i ~ Cat(a_mat[z_{i-1}]), x_i ~ N(mu_{z_i}, Lambda_{z_i}^-1).  Same constructor, parameters and
    methods as the reference class.

    Parameters
    ----------
    c_num_classes, c_degree : int
        number of hidden states K and data dimension D (positive)
    pi_vec, a_mat, mu_vecs, lambda_mats : optional (keyword only)
        parameters; defaults 1/K, 1/K, 0, I
    h_eta_vec, h_zeta_vecs, h_m_vecs, h_kappas, h_nus, h_w_mats : optional (keyword only)
        hyperparameters of the prior; defaults 1/2, 1/2, 0, 1, D, I (those of LearnModel's h0_*)
    seed : {None, int}
        seed of `numpy.random.default_rng`

    `gen_sample(n)` is the reference's per-element loop (`rng.choice` + `rng.multivariate_normal`); `gen_sample(n,
    device="cuda:0")` draws the same distribution on the device (bgmm_hmm_gen_sample; counter-based Philox, NOT numpy's
    stream) and can leave the sample there (`as_numpy=False`)."""

    def __init__(self, c_num_classes, c_degree, *, pi_vec=None, a_mat=None, mu_vecs=None, lambda_mats=None,
                 h_eta_vec=None, h_zeta_vecs=None, h_m_vecs=None, h_kappas=None, h_nus=None, h_w_mats=None, seed=None):
        self.c_degree = _check.pos_int(c_degree, 'c_degree', ParameterFormatError)
        self.c_num_classes = _check.pos_int(c_num_classes, 'c_num_classes', ParameterFormatError)
        self.rng = np.random.default_rng(seed)
        K, D = self.c_num_classes, self.c_degree
        self.pi_vec = np.ones(K) / K
        self.a_mat = np.ones((K, K)) / K
        self.mu_vecs = np.zeros((K, D))
        self.lambda_mats = np.tile(np.eye(D), (K, 1, 1))
        self.h_eta_vec = np.ones(K) / 2
        self.h_zeta_vecs = np.ones((K, K)) / 2
        self.h_m_vecs = np.zeros((K, D))
        self.h_kappas = np.ones(K)
        self.h_nus = np.ones(K) * D
        self.h_w_mats = np.tile(np.eye(D), (K, 1, 1))
        self.set_params(pi_vec, a_mat, mu_vecs, lambda_mats)
        self.set_h_params(h_eta_vec, h_zeta_vecs, h_m_vecs, h_kappas, h_nus, h_w_mats)

    def get_constants(self):
        """{"c_num_classes", "c_degree"}."""
        return {"c_num_classes": self.c_num_classes, "c_degree": self.c_degree}

    def _shape(self, arr, name, shape):
        if arr.shape != shape:
            raise ParameterFormatError(f"{name}.shape must be {shape} (c_num_classes = {self.c_num_classes}, "
                                       f"c_degree = {self.c_degree}): {name}.shape = {arr.shape}")

    def set_h_params(self, h_eta_vec=None, h_zeta_vecs=None, h_m_vecs=None, h_kappas=None, h_nus=None, h_w_mats=None):
        """Set the hyperparameters of the prior (arrays broadcast to their attribute's shape)."""
        D = self.c_degree
        if h_eta_vec is not None:
            _check.pos_floats(h_eta_vec, 'h_eta_vec', ParameterFormatError)
            self.h_eta_vec[:] = h_eta_vec
        if h_zeta_vecs is not None:
            _check.pos_floats(h_zeta_vecs, 'h_zeta_vecs', ParameterFormatError)
            self.h_zeta_vecs[:] = h_zeta_vecs
        if h_m_vecs is not None:
            _check.float_vecs(h_m_vecs, 'h_m_vecs', ParameterFormatError)
            if h_m_vecs.shape[-1] != D:
                raise ParameterFormatError("h_m_vecs.shape[-1] must coincide with self.c_degree: "
                                           f"h_m_vecs.shape[-1] = {h_m_vecs.shape[-1]}, self.c_degree = {D}")
            self.h_m_vecs[:] = h_m_vecs
        if h_kappas is not None:
            _check.pos_floats(h_kappas, 'h_kappas', ParameterFormatError)
            self.h_kappas[:] = h_kappas
        if h_nus is not None:
            _check.pos_floats(h_nus, 'h_nus', ParameterFormatError)
            if np.any(h_nus <= D - 1):
                raise ParameterFormatError("All the values of h_nus must be greater than self.c_degree - 1: "
                                           f"self.c_degree = {D}, h_nus = {h_nus}")
            self.h_nus[:] = h_nus
        if h_w_mats is not None:
            _check.pos_def_sym_mats(h_w_mats, 'h_w_mats', ParameterFormatError)
            if h_w_mats.shape[-1] != D:
                raise ParameterFormatError("h_w_mats.shape[-1] must coincide with self.c_degree: "
                                           f"h_w_mats.shape[-1] = {h_w_mats.shape[-1]}, self.c_degree = {D}")
            self.h_w_mats[:] = h_w_mats
        return self

    def get_h_params(self):
        """Live references to the hyperparameters."""
        return {"h_eta_vec": self.h_eta_vec, "h_zeta_vecs": self.h_zeta_vecs, "h_m_vecs": self.h_m_vecs,
                "h_kappas": self.h_kappas, "h_nus": self.h_nus, "h_w_mats": self.h_w_mats}

    def gen_params(self):
        """Draw pi ~ Dir(h_eta_vec), then every row of A ~ Dir(h_zeta_vecs[k]), then (Lambda_k, mu_k) for every k as
        `gaussianmixture.GenModel.gen_params` does, all from `self.rng`."""
        self.pi_vec[:] = self.rng.dirichlet(self.h_eta_vec)
        for k in range(self.c_num_classes):
            self.a_mat[k] = self.rng.dirichlet(self.h_zeta_vecs[k])
        for k in range(self.c_num_classes):
            self.lambda_mats[k] = ss_wishart.rvs(df=self.h_nus[k], scale=self.h_w_mats[k], random_state=self.rng)
            self.mu_vecs[k] = self.rng.multivariate_normal(mean=self.h_m_vecs[k],
                                                           cov=np.linalg.inv(self.h_kappas[k] * self.lambda_mats[k]))
        return self

    def set_params(self, pi_vec=None, a_mat=None, mu_vecs=None, lambda_mats=None):
        """Set the parameters of the sampling distribution: pi_vec (K,) and every row of a_mat (K, K) non-negative and
        summing to 1, mu_vecs (K, D), lambda_mats (K, D, D) positive-definite symmetric."""
        K, D = self.c_num_classes, self.c_degree
        if pi_vec is not None:
            _check.float_vec_sum_1(pi_vec, 'pi_vec', ParameterFormatError)
            self._shape(pi_vec, 'pi_vec', (K,))
            if np.any(pi_vec < 0):
                raise ParameterFormatError(f"pi_vec must be non-negative: pi_vec = {pi_vec}")
            self.pi_vec[:] = pi_vec
        if a_mat is not None:
            _check.float_vecs_sum_1(a_mat, 'a_mat', ParameterFormatError)
            self._shape(a_mat, 'a_mat', (K, K))
            if np.any(a_mat < 0):
                raise ParameterFormatError(f"a_mat must be non-negative: a_mat = {a_mat}")
            self.a_mat[:] = a_mat
        if mu_vecs is not None:
            _check.float_vecs(mu_vecs, 'mu_vecs', ParameterFormatError)
            self._shape(mu_vecs, 'mu_vecs', (K, D))
            self.mu_vecs[:] = mu_vecs
        if lambda_mats is not None:
            _check.pos_def_sym_mats(lambda_mats, 'lambda_mats', ParameterFormatError)
            self._shape(lambda_mats, 'lambda_mats', (K, D, D))
            self.lambda_mats[:] = lambda_mats
        return self

    def get_params(self):
        """Live references to pi_vec, a_mat, mu_vecs, lambda_mats."""
        return {"pi_vec": self.pi_vec, "a_mat": self.a_mat, "mu_vecs": self.mu_vecs, "lambda_mats": self.lambda_mats}

    def gen_sample(self, sample_length, *, lengths=None, device=None, as_numpy=True):
        """Generate a sample -> (x (sample_length, c_degree) float64, z (sample_length, c_num_classes) one-hot int).

        device=None: the reference's loop with `self.rng`: z_0 = rng.choice(K, p=pi_vec), then x_0 =
        rng.multivariate_normal(mu[z_0], Lambda[z_0]^-1); for i >= 1, z_i = rng.choice(K, p=a_mat[z_{i-1}]), then that
        element's multivariate_normal.
        lengths : optional (extension, keyword only) 1-D sequence of positive ints summing to sample_length: that many
            independent sequences, concatenated, each starting from pi.  On the host the loop above runs once per
            sequence in order, so lengths=[sample_length] is exactly lengths=None.
        device="cuda:i": one call of bgmm_hmm_gen_sample (same distribution, its own counter-based stream seeded by one
            `self.rng.integers` draw; c_num_classes <= 32, c_degree <= 256, else ParameterFormatError); with
            as_numpy=False, x (float64) and the state indices z (int32, NOT one-hot) stay on the device as torch tensors.
        """
        _check.pos_int(sample_length, 'sample_length', DataFormatError)
        starts = LearnModel._seq_starts(lengths, sample_length)
        K, D = self.c_num_classes, self.c_degree
        cov = np.linalg.inv(self.lambda_mats)
        if device is None:
            z = np.zeros((sample_length, K), dtype=int)
            x = np.empty((sample_length, D))
            first = np.zeros(sample_length, dtype=bool)
            first[0 if starts is None else starts] = True
            k = 0
            for i in range(sample_length):
                k = self.rng.choice(K, p=self.pi_vec if first[i] else self.a_mat[k])
                z[i, k] = 1
                x[i] = self.rng.multivariate_normal(mean=self.mu_vecs[k], cov=cov[k])
            return x, z
        if K > GEN_MAX_NUM_CLASSES or D > GEN_MAX_DEGREE:
            raise ParameterFormatError(
                f"gen_sample on the device supports c_num_classes <= {GEN_MAX_NUM_CLASSES} and c_degree <= "
                f"{GEN_MAX_DEGREE} (got {K}, {D}); there is no CPU fallback")
        import torch
        from . import _lib
        lib = _lib.load()
        dev = torch.device(device)
        seed = int(self.rng.integers(0, 2 ** 63 - 1))
        n_seqs = 1 if starts is None else starts.size
        starts_ptr = None if starts is None else starts.ctypes.data
        with torch.cuda.device(dev):
            consts = [torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).to(dev)
                      for a in (_inverse_cdf_table(self.pi_vec, self.a_mat), self.mu_vecs, np.linalg.cholesky(cov))]
            x_dev = torch.empty((sample_length, D), dtype=torch.float64, device=dev)
            z_dev = torch.empty(sample_length, dtype=torch.int32, device=dev)
            ws = torch.empty(lib.bgmm_hmm_gen_workspace_bytes(K, sample_length, n_seqs, 0), dtype=torch.uint8, device=dev)
            _lib.check(lib.bgmm_hmm_gen_sample(x_dev.data_ptr(), z_dev.data_ptr(), sample_length, K, D,
                                               consts[0].data_ptr(), consts[1].data_ptr(), consts[2].data_ptr(),
                                               starts_ptr, n_seqs, seed, 0, ws.data_ptr(),
                                               torch.cuda.current_stream(dev).cuda_stream), "bgmm_hmm_gen_sample")
            if not as_numpy:
                torch.cuda.current_stream(dev).synchronize()
                return x_dev, z_dev
            return x_dev.cpu().numpy(), np.eye(K, dtype=int)[z_dev.cpu().numpy()]

    def save_sample(self, filename, sample_length):
        """gen_sample, then np.savez_compressed(filename, x=x, z=z)."""
        x, z = self.gen_sample(sample_length)
        np.savez_compressed(filename, x=x, z=z)

    def visualize_model(self, sample_length=200):
        """Print the parameters and plot a sample (x against time for c_degree 1, the plane for c_degree 2, coloured by
        state) for c_degree <= 2; needs matplotlib."""
        if self.c_degree > 2:
            raise ParameterFormatError("if c_degree > 2, it is impossible to visualize the model by this function.")
        print(f"pi_vec:\n {self.pi_vec}")
        print(f"a_mat:\n {self.a_mat}")
        print(f"mu_vecs:\n {self.mu_vecs}")
        print(f"lambda_mats:\n {self.lambda_mats}")
        import matplotlib.pyplot as plt
        sample, z = self.gen_sample(sample_length)
        states = z.argmax(axis=1)
        fig, axes = plt.subplots()
        if self.c_degree == 1:
            axes.plot(np.arange(sample_length), sample[:, 0], color="gray", linewidth=0.5)
            axes.scatter(np.arange(sample_length), sample[:, 0], c=states, cmap="tab10")
            axes.set_xlabel("time"); axes.set_ylabel("x")
        else:
            axes.plot(sample[:, 0], sample[:, 1], color="gray", linewidth=0.5)
            axes.scatter(sample[:, 0], sample[:, 1], c=states, cmap="tab10")
            axes.set_xlabel("x[0]"); axes.set_ylabel("x[1]")
        plt.show()


class LearnModel(base.Posterior, base.PredictiveMixin):
    """Posterior and predictive distribution of the Bayesian hidden Markov model with Gaussian emissions (:451-512).

    Parameters
    ----------
    c_num_classes, c_degree : int
        number of hidden states K and data dimension D (positive)
    h0_eta_vec, h0_zeta_vecs, h0_m_vecs, h0_kappas, h0_nus, h0_w_mats : optional (keyword only)
        Dirichlet (initial state, transition rows) / Gauss-Wishart prior hyperparameters; defaults 1/2, 1/2, 0, 1, D, I
    seed : {None, int}
        seed of `numpy.random.default_rng` used by the initialisations
    device : optional (extension) CUDA device of the fit
    device_init : bool, optional (extension, default False) draw the 'random_responsibility' initial state on the
        device: one `self.rng.integers` value per restart seeds a counter-based generator (bgmm_hmm_init_random).  The
        numbers differ from numpy's; the distribution and the rules of `_init_random_responsibility` are the same
    """

    def __init__(self, c_num_classes, c_degree, *, h0_eta_vec=None, h0_zeta_vecs=None, h0_m_vecs=None, h0_kappas=None,
                 h0_nus=None, h0_w_mats=None, seed=None, device=None, device_init=False):
        self.c_degree = _check.pos_int(c_degree, 'c_degree', ParameterFormatError)
        self.c_num_classes = _check.pos_int(c_num_classes, 'c_num_classes', ParameterFormatError)
        self.rng = np.random.default_rng(seed)
        K, D = self.c_num_classes, self.c_degree
        if K > MAX_NUM_CLASSES or D > MAX_DEGREE:
            # the reference accepts any size; the device scans keep one state vector per lane group (K <= 32) and the
            # per-component kernel factorises W^-1 in shared memory (D <= 128): say so here, not inside update_posterior
            raise ParameterFormatError(
                f"bayesml_b200.hiddenmarkovnormal supports c_num_classes <= {MAX_NUM_CLASSES} and c_degree <= {MAX_DEGREE} "
                f"(got {K}, {D}); there is no CPU fallback")
        self._device = device
        self._device_init = bool(device_init)
        self._engine_obj = None

        # prior hyperparameters and their constants (:531-543)
        self.h0_eta_vec = np.ones(K) / 2.0
        self.h0_zeta_vecs = np.ones([K, K]) / 2.0
        self.h0_m_vecs = np.zeros([K, D])
        self.h0_kappas = np.ones([K])
        self.h0_nus = np.ones(K) * D
        self.h0_w_mats = np.tile(np.eye(D), [K, 1, 1])
        self.h0_w_mats_inv = np.linalg.inv(self.h0_w_mats)
        self._ln_c_h0_eta_vec = 0.0
        self._ln_c_h0_zeta_vecs_sum = 0.0
        self._ln_b_h0_w_nus = np.empty(K)

        # posterior hyperparameters (:546-552)
        self.hn_eta_vec = np.empty(K)
        self.hn_zeta_vecs = np.empty([K, K])
        self.hn_m_vecs = np.empty([K, D])
        self.hn_kappas = np.empty([K])
        self.hn_nus = np.empty(K)
        self.hn_w_mats = np.empty([K, D, D])
        self.hn_w_mats_inv = np.empty([K, D, D])

        # per-element quantities of the forward-backward pass (:554-561), device resident until read
        self._length = 0
        self._starts = None                             # first rows of the sequences (several sequences), else None
        for name in _LAZY:
            setattr(self, "_lazy_" + name.lstrip("_"), _LazyDeviceArray())
        self._rho_host = None
        self._xi_host = None
        self._e_lambda_mats = np.empty([K, D, D])
        self._e_ln_lambda_dets = np.empty(K)
        self._ln_b_hn_w_nus = np.empty(K)
        self._ln_pi_tilde_vec = np.empty(K)
        self._pi_tilde_vec = np.empty(K)
        self._ln_a_tilde_mat = np.empty([K, K])
        self._a_tilde_mat = np.empty([K, K])
        self._ln_c_hn_zeta_vecs_sum = 0.0

        # statistics (:573-576) and ELBO terms (:579-588)
        self.x_bar_vecs = np.empty([K, D])
        self.ns = np.empty(K)
        self.ms = np.empty([K, K])
        self.s_mats = np.empty([K, D, D])
        self.vl = 0.0
        for name in ("_vl_p_x", "_vl_p_z", "_vl_p_pi", "_vl_p_a", "_vl_p_mu_lambda", "_vl_q_z", "_vl_q_pi", "_vl_q_a",
                     "_vl_q_mu_lambda"):
            setattr(self, name, 0.0)

        # predictive parameters (:591-595)
        self.p_a_mat = np.ones([K, K]) / K
        self.p_mu_vecs = np.empty([K, D])
        self.p_nus = np.empty([K])
        self.p_lambda_mats = np.empty([K, D, D])
        self.p_lambda_mats_inv = np.empty([K, D, D])

        # Viterbi work arrays (:598-599), device resident until read
        self._lazy_omega_vecs = _LazyDeviceArray()
        self._lazy_phi_vecs = _LazyDeviceArray()

        self.set_h0_params(h0_eta_vec, h0_zeta_vecs, h0_m_vecs, h0_kappas, h0_nus, h0_w_mats)

    # ------------------------------------------------------------------ big per-element attributes, fetched lazily
    _ln_rho = _lazy_property("_ln_rho")
    alpha_vecs = _lazy_property("alpha_vecs")
    beta_vecs = _lazy_property("beta_vecs")
    gamma_vecs = _lazy_property("gamma_vecs")
    _cs = _lazy_property("_cs")
    omega_vecs = _lazy_property("omega_vecs")

    @property
    def phi_vecs(self):
        """arg-max table of the Viterbi recursion (:1472); int64 as in the reference."""
        v = self._lazy_phi_vecs.get()
        if v is not None and v.dtype != np.int64:
            v = v.astype(np.int64)
            self._lazy_phi_vecs.set_host(v)
        return v

    @phi_vecs.setter
    def phi_vecs(self, value):
        self._lazy_phi_vecs.set_host(value)

    @property
    def _rho(self):
        """exp(_ln_rho) (:997)."""
        if self._rho_host is None and self._ln_rho is not None:
            self._rho_host = np.exp(self._ln_rho)
        return self._rho_host

    @_rho.setter
    def _rho(self, value):
        self._rho_host = value

    @property
    def xi_mats(self):
        """xi_i = alpha_{i-1} rho_i a~ beta_i / c_i, xi_0 = 0 (:1016-1018); formed on the host on first access."""
        if self._xi_host is None and self.alpha_vecs is not None:
            n, K = self._length, self.c_num_classes
            xi = np.zeros([n, K, K])
            if n > 1:
                xi[1:] = (self.alpha_vecs[:-1, :, np.newaxis] * self._rho[1:, np.newaxis, :]
                          * self._a_tilde_mat[np.newaxis, :, :] * self.beta_vecs[1:, np.newaxis, :])
                xi[1:] /= self._cs[1:, np.newaxis, np.newaxis]
            if self._starts is not None:
                xi[self._starts] = 0.0                 # no transition into the first element of a sequence
            self._xi_host = xi
        return self._xi_host

    @xi_mats.setter
    def xi_mats(self, value):
        self._xi_host = value

    def _clear_elementwise(self):
        for name in _LAZY:
            getattr(self, "_lazy_" + name.lstrip("_")).set_host(None)
        self._rho_host = None
        self._xi_host = None

    # ------------------------------------------------------------------ constants / hyperparameter plumbing
    def get_constants(self):
        """{"c_num_classes", "c_degree"} (:608-617)."""
        return {"c_num_classes": self.c_num_classes, "c_degree": self.c_degree}

    def _store_hyper(self, prefix, eta_vec, zeta_vecs, m_vecs, kappas, nus, w_mats):
        """Validate and copy one family (h0 / hn) of hyperparameters in place (:652-691, :754-793)."""
        D = self.c_degree
        if eta_vec is not None:
            _check.pos_floats(eta_vec, prefix + '_eta_vec', ParameterFormatError)
            getattr(self, prefix + '_eta_vec')[:] = eta_vec
        if zeta_vecs is not None:
            _check.pos_floats(zeta_vecs, prefix + '_zeta_vecs', ParameterFormatError)
            getattr(self, prefix + '_zeta_vecs')[:] = zeta_vecs
        if m_vecs is not None:
            _check.float_vecs(m_vecs, prefix + "_m_vecs", ParameterFormatError)
            _check.shape_consistency(m_vecs.shape[-1], prefix + "_m_vecs.shape[-1]", D, "self.c_degree",
                                     ParameterFormatError)
            getattr(self, prefix + '_m_vecs')[:] = m_vecs
        if kappas is not None:
            _check.pos_floats(kappas, prefix + "_kappas", ParameterFormatError)
            getattr(self, prefix + '_kappas')[:] = kappas
        if nus is not None:
            _check.floats(nus, prefix + "_nus", ParameterFormatError)
            if np.all(nus <= D - 1):
                raise ParameterFormatError(
                    f"All the values in {prefix}_nus must be greater than self.c_degree - 1: "
                    + f"self.c_degree = {D}, {prefix}_nus = {nus}")
            getattr(self, prefix + '_nus')[:] = nus
        if w_mats is not None:
            _check.pos_def_sym_mats(w_mats, prefix + '_w_mats', ParameterFormatError)
            _check.shape_consistency(w_mats.shape[-1], f"{prefix}_w_mats.shape[-1] and {prefix}_w_mats.shape[-2]", D,
                                     "self.c_degree", ParameterFormatError)
            getattr(self, prefix + '_w_mats')[:] = w_mats
        getattr(self, prefix + '_w_mats_inv')[:] = np.linalg.inv(getattr(self, prefix + '_w_mats'))

    def set_h0_params(self, h0_eta_vec=None, h0_zeta_vecs=None, h0_m_vecs=None, h0_kappas=None, h0_nus=None,
                      h0_w_mats=None):
        """Set the prior hyperparameters, then reset hn_* to them (:619-699)."""
        self._store_hyper('h0', h0_eta_vec, h0_zeta_vecs, h0_m_vecs, h0_kappas, h0_nus, h0_w_mats)
        self._calc_prior_features()
        self.reset_hn_params()
        return self

    def get_h0_params(self):
        """Live references to h0_* (:701-719)."""
        return {'h0_eta_vec': self.h0_eta_vec, 'h0_zeta_vecs': self.h0_zeta_vecs, 'h0_m_vecs': self.h0_m_vecs,
                'h0_kappas': self.h0_kappas, 'h0_nus': self.h0_nus, 'h0_w_mats': self.h0_w_mats}

    def set_hn_params(self, hn_eta_vec=None, hn_zeta_vecs=None, hn_m_vecs=None, hn_kappas=None, hn_nus=None,
                      hn_w_mats=None):
        """Set the posterior hyperparameters, refresh the E_q features and the predictive parameters (:721-804)."""
        self._store_hyper('hn', hn_eta_vec, hn_zeta_vecs, hn_m_vecs, hn_kappas, hn_nus, hn_w_mats)
        self._calc_q_pi_features()
        self._calc_q_a_features()
        self._calc_q_lambda_features()
        self.calc_pred_dist()
        return self

    def get_hn_params(self):
        """Live references to hn_* (:806-824)."""
        return {'hn_eta_vec': self.hn_eta_vec, 'hn_zeta_vecs': self.hn_zeta_vecs, 'hn_m_vecs': self.hn_m_vecs,
                'hn_kappas': self.hn_kappas, 'hn_nus': self.hn_nus, 'hn_w_mats': self.hn_w_mats}

    # ------------------------------------------------------------------ K-sized host features (outside the loop)
    def _ln_b(self, nus, logdet_w_inv):
        D = self.c_degree
        return (nus * logdet_w_inv - nus * D * np.log(2.0) - D * (D - 1) / 2.0 * np.log(np.pi)
                - 2.0 * gammaln((nus[:, None] - np.arange(D)) / 2.0).sum(axis=1)) / 2.0

    def _calc_prior_features(self):
        """(:826-835)"""
        self._ln_c_h0_eta_vec = gammaln(self.h0_eta_vec.sum()) - gammaln(self.h0_eta_vec).sum()
        self._ln_c_h0_zeta_vecs_sum = np.sum(gammaln(self.h0_zeta_vecs.sum(axis=1)) - gammaln(self.h0_zeta_vecs).sum(axis=1))
        self._ln_b_h0_w_nus = self._ln_b(self.h0_nus, -np.linalg.slogdet(self.h0_w_mats)[1])

    def _calc_q_pi_features(self):
        """(:847-849)"""
        self._ln_pi_tilde_vec[:] = digamma(self.hn_eta_vec) - digamma(self.hn_eta_vec.sum())
        self._pi_tilde_vec[:] = np.exp(self._ln_pi_tilde_vec - self._ln_pi_tilde_vec.max())

    def _calc_q_a_features(self):
        """(:851-854)"""
        self._ln_a_tilde_mat[:] = digamma(self.hn_zeta_vecs) - digamma(self.hn_zeta_vecs.sum(axis=1, keepdims=True))
        self._a_tilde_mat[:] = np.exp(self._ln_a_tilde_mat - self._ln_a_tilde_mat.max())
        self._ln_c_hn_zeta_vecs_sum = np.sum(gammaln(self.hn_zeta_vecs.sum(axis=1)) - gammaln(self.hn_zeta_vecs).sum(axis=1))

    def _calc_q_lambda_features(self):
        """(:856-867)"""
        D = self.c_degree
        logdet = np.linalg.slogdet(self.hn_w_mats_inv)[1]
        self._e_lambda_mats[:] = self.hn_nus[:, None, None] * self.hn_w_mats
        self._e_ln_lambda_dets[:] = (digamma((self.hn_nus[:, None] - np.arange(D)) / 2.0).sum(axis=1)
                                     + D * np.log(2.0) - logdet)
        self._ln_b_hn_w_nus[:] = self._ln_b(self.hn_nus, logdet)

    # ------------------------------------------------------------------ device plumbing
    def _engine(self):
        if self._engine_obj is None:
            from .engine import HMMEngine
            self._engine_obj = HMMEngine(self.c_num_classes, self.c_degree, device=self._device)
        return self._engine_obj

    def _check_x(self, x):
        _check.float_vecs(x, 'x', DataFormatError)
        _check.shape_consistency(x.shape[-1], "x.shape[-1]", self.c_degree, "self.c_degree", DataFormatError)
        return x.reshape(-1, self.c_degree)

    @staticmethod
    def _seq_starts(lengths, n):
        """First rows of the sequences given by `lengths` (int64), or None for one sequence (lengths None or [n])."""
        if lengths is None:
            return None
        arr = np.asarray(lengths)
        if arr.ndim != 1 or arr.size == 0 or arr.dtype.kind not in "iu":
            raise DataFormatError("lengths must be a non-empty 1-dimensional sequence of positive ints.")
        if np.any(arr <= 0):
            raise DataFormatError(f"lengths must be positive: lengths = {arr}")
        if int(arr.sum()) != n:
            raise DataFormatError(f"lengths must sum to the number of rows of x: sum(lengths) = {int(arr.sum())}, rows = {n}")
        if arr.size == 1:
            return None
        starts = np.zeros(arr.size, dtype=np.int64)
        np.cumsum(arr[:-1], out=starts[1:])
        return starts

    def _push_prior(self, eng):
        eng.set_hmm_prior(self.h0_eta_vec, self.h0_zeta_vecs, self.h0_m_vecs, self.h0_kappas, self.h0_nus,
                          self.h0_w_mats_inv, self._ln_b_h0_w_nus, self._ln_c_h0_eta_vec, self._ln_c_h0_zeta_vecs_sum)

    def _push_hn(self, eng):
        eng.set_hmm_params(self.hn_eta_vec, self.hn_zeta_vecs, self.hn_m_vecs, self.hn_kappas, self.hn_nus,
                           self.hn_w_mats_inv)

    def _apply_state(self, p):
        """One restart's device result (parameter set / statistics / ELBO terms) -> the numpy attributes, in place."""
        self.hn_eta_vec[:] = p["alpha"]
        self.hn_zeta_vecs[:] = p["zeta"]
        self.hn_m_vecs[:] = p["m"]
        self.hn_kappas[:] = p["kappa"]
        self.hn_nus[:] = p["nu"]
        self.hn_w_mats[:] = p["w"]
        self.hn_w_mats_inv[:] = p["winv"]
        self._ln_pi_tilde_vec[:] = p["e_ln_pi"]
        self._pi_tilde_vec[:] = np.exp(self._ln_pi_tilde_vec - self._ln_pi_tilde_vec.max())
        self._ln_a_tilde_mat[:] = p["ln_a_tilde"]
        self._a_tilde_mat[:] = p["a_tilde"]
        self._ln_c_hn_zeta_vecs_sum = p["ln_c_zeta_sum"]
        self._e_ln_lambda_dets[:] = p["e_ln_lambda_dets"]
        self._ln_b_hn_w_nus[:] = p["ln_b"]
        self._e_lambda_mats[:] = self.hn_nus[:, None, None] * self.hn_w_mats
        self._pull_stats(p)
        t, vx = p["vl_terms"], p["vlx"]
        # device slots: vlterms = [p_x, -, p_pi, p_mu_lambda, -, q_pi, q_mu_lambda, vl]; vlx = [p_z, p_a, q_z, q_a]
        self._vl_p_x, self._vl_p_pi, self._vl_p_mu_lambda = np.float64(t[0]), np.float64(t[2]), np.float64(t[3])
        self._vl_q_pi, self._vl_q_mu_lambda, self.vl = np.float64(t[5]), np.float64(t[6]), np.float64(t[7])
        self._vl_p_z, self._vl_p_a, self._vl_q_z, self._vl_q_a = (np.float64(v) for v in vx)

    def _pull_stats(self, s):
        self.ns[:] = s["ns"]
        self.ms[:] = s["ms"]
        self.x_bar_vecs[:] = s["x_bar"]
        self.s_mats[:] = s["s_mats"]

    # ------------------------------------------------------------------ initialisations (host: they consume self.rng)
    def _init_random_responsibility(self, n, starts=None):
        """Random xi / gamma (:944-952) -> (gamma [n][K], ms [K][K]); the statistics are computed on the device.

        Several sequences (`starts`, their first rows): the same single draw `rng.dirichlet(np.ones(K**2), n)`; every
        row gets gamma = xi.sum(axis=1), then at every sequence start s, gamma_s = xi_{s+1}.sum(axis=1) (row sums of the
        K x K matrix) when that sequence is longer than 1, or the row sums of its own drawn xi_s for a sequence of
        length 1; then xi_s = 0.  With one sequence this is the reference's rule.

        `device_init=True`: -> one int from `self.rng`, the seed with which the engine draws the same rules on the device
        (bgmm_hmm_init_random) when the restart runs; nothing n-sized is made on the host."""
        if self._device_init:
            return int(self.rng.integers(0, 2 ** 63 - 1))
        K = self.c_num_classes
        gamma = np.ones([n, K]) / K
        xi_sum = np.zeros([K, K])
        if n == 1:
            gamma[0] = self.rng.dirichlet(np.ones(K))
        elif starts is None:
            xi = self.rng.dirichlet(np.ones(K ** 2), n).reshape(n, K, K)
            xi[0] = 0.0
            gamma[:] = xi.sum(axis=1)
            gamma[0] = xi[1].sum(axis=1)
            xi_sum = xi.sum(axis=0)
        else:
            xi = self.rng.dirichlet(np.ones(K ** 2), n).reshape(n, K, K)
            gamma[:] = xi.sum(axis=1)
            ends = np.append(starts[1:], n)
            single = ends - starts == 1
            longer = starts[~single]
            gamma[longer] = xi[longer + 1].sum(axis=2)           # the row sums of xi_{s+1}, as gamma[0] above
            gamma[starts[single]] = xi[starts[single]].sum(axis=2)
            xi[starts] = 0.0
            xi_sum = xi.sum(axis=0)
        return gamma, xi_sum

    def _init_subsampling(self, x):
        """Class-wise sqrt(N)-row subsamples give the initial m_k and W_k (:954-964); host numpy, reference RNG stream."""
        n_sub = int(np.sqrt(x.shape[0]))
        eye_eps = np.eye(self.c_degree) * 1.0E-5
        for k in range(self.c_num_classes):
            sub = self.rng.choice(x, size=n_sub, replace=False, axis=0, shuffle=False)
            self.hn_m_vecs[k] = sub.sum(axis=0) / n_sub
            centred = sub - self.hn_m_vecs[k]
            self.hn_w_mats_inv[k] = centred.T @ centred / n_sub * self.hn_nus[k] + eye_eps
            self.hn_w_mats[k] = np.linalg.inv(self.hn_w_mats_inv[k])
        self._calc_q_lambda_features()

    # ------------------------------------------------------------------ the fit (:1028-1134)
    def update_posterior(self, x, max_itr=100, num_init=10, tolerance=1.0E-8, init_type='subsampling', *, lengths=None):
        """Update the posterior hyperparameters by variational Bayes with `num_init` restarts (:1028-1134).

        Parameters
        ----------
        x : numpy.ndarray, shape (..., c_degree) — one sequence in time order, or the sequences of `lengths` concatenated
        max_itr : int, maximum number of VB iterations per restart (default 100)
        num_init : int, number of restarts (default 10)
        tolerance : float, relative ELBO change that stops a restart (default 1e-8)
        init_type : 'subsampling' | 'random_responsibility'
        lengths : optional (extension, keyword only) 1-D sequence of positive ints summing to the number of rows of x:
            x holds that many independent sequences that share the posterior (see the module docstring).  'subsampling'
            draws rows from all of x, as for one sequence; 'random_responsibility' is described in
            `_init_random_responsibility`.  `make_prediction` / `pred_and_update` continue from the last element of
            the last sequence.

        Nothing else consumes `self.rng` between the restarts (:1087-1100), so all initial states are drawn first (the
        same random stream as the reference's sequential loop) while x is uploaded; the restarts then run one after the
        other on the device and the reference's selection rule (:1114) and progress text are applied in order.  With
        `device_init=True` a 'random_responsibility' restart's initial state is kept as its seed and drawn on the device
        when the restart runs.
        """
        x = self._check_x(x)
        starts = self._seq_starts(lengths, x.shape[0])
        self._length = x.shape[0]
        self._starts = starts
        eng = self._engine()
        eng.load_data_begin(x)
        self._clear_elementwise()

        best_vl = 0.0
        best = {name: np.array(getattr(self, name)) for name in _HN_NAMES}      # :1077-1083
        inits = []
        for i in range(num_init):
            self.reset_hn_params()
            init = None
            if init_type == 'subsampling':
                self._init_subsampling(x)
            elif init_type == 'random_responsibility':
                init = self._init_random_responsibility(x.shape[0], starts)
            else:
                raise ValueError(
                    f'init_type={init_type} is unsupported. '
                    + 'This function supports only '
                    + '"subsampling" and "random_responsibility"')
            inits.append(({name: np.array(getattr(self, name)) for name in _HN_NAMES}, init))
        eng.load_data_finish()
        eng.set_sequences(starts)
        self._push_prior(eng)

        never_converged = True
        for i, (hn, init) in enumerate(inits):
            eng.set_hmm_params(hn["hn_eta_vec"], hn["hn_zeta_vecs"], hn["hn_m_vecs"], hn["hn_kappas"], hn["hn_nus"],
                               hn["hn_w_mats_inv"])
            hist, converged = eng.run(max_itr, tolerance, init=init)
            if eng.failed:
                raise RuntimeError("bgmm_small: a W^-1 matrix was not positive definite (Cholesky failed)")
            print(f'\r{i}. VL: {hist[0]}', end='')                               # :1102, :1110, :1113
            for t in range(len(hist) - 1):
                print(f'\r{i}. VL: {hist[t + 1]} t={t} ', end='')
            if converged:
                never_converged = False
                print('(converged)', end='')
            self._apply_state(eng.fetch_params())
            if i == 0 or self.vl > best_vl:                                      # :1114 (strict: ties keep the earlier)
                print('*')
                best_vl = self.vl
                for name in _HN_NAMES:
                    best[name][:] = getattr(self, name)
            else:
                print('')
        if never_converged:
            warnings.warn("Algorithm has not converged even once.", ResultWarning)

        for name in _HN_NAMES:                                                    # :1125-1131
            getattr(self, name)[:] = best[name]
        self._calc_q_pi_features()
        self._calc_q_a_features()
        self._calc_q_lambda_features()
        self._final_e_step(eng)                                                   # :1133
        return self

    def _final_e_step(self, eng):
        """`_update_q_z` with the current hn_* (:1020-1026): per-element arrays stay on the device until read."""
        self._push_hn(eng)
        self._pull_stats(eng.final_pass())
        self._clear_elementwise()
        self._lazy_ln_rho.set_device(eng.lnrho_buf)
        self._lazy_alpha_vecs.set_device(eng.alpha_buf)
        self._lazy_beta_vecs.set_device(eng.beta_buf)
        self._lazy_gamma_vecs.set_device(eng.gamma_buf)
        self._lazy_cs.set_device(eng.cs_buf)

    # ------------------------------------------------------------------ estimates (:1136-1211)
    def estimate_params(self, loss="squared"):
        """Point estimates (or the posterior itself for loss="KL") of pi, A, mu, Lambda (:1136-1211)."""
        K, D = self.c_num_classes, self.c_degree
        if loss == "squared":
            return (self.hn_eta_vec / self.hn_eta_vec.sum(),
                    self.hn_zeta_vecs / self.hn_zeta_vecs.sum(axis=1, keepdims=True),
                    self.hn_m_vecs, self._e_lambda_mats)
        if loss == "0-1":
            pi_hat = np.empty(K)
            if np.all(self.hn_eta_vec > 1):
                pi_hat[:] = (self.hn_eta_vec - 1) / (np.sum(self.hn_eta_vec) - D)
            else:
                warnings.warn("MAP estimate of pi_vec doesn't exist for the current hn_eta_vec.", ResultWarning)
                pi_hat[:] = np.nan
            a_hat = np.empty([K, K])
            for i in range(K):
                if np.all(self.hn_eta_vec > 1):          # the reference tests hn_eta_vec here too (:1184)
                    a_hat[i] = (self.hn_zeta_vecs[i] - 1) / (np.sum(self.hn_zeta_vecs[i]) - D)
                else:
                    warnings.warn(f"MAP estimate of a_mat[{i}] doesn't exist for the current hn_zeta_vecs[{i}].",
                                  ResultWarning)
                    a_hat[i] = np.nan
            lambda_hat = np.empty([K, D, D])
            for k in range(K):
                if self.hn_nus[k] >= D + 1:
                    lambda_hat[k] = (self.hn_nus[k] - D - 1) * self.hn_w_mats[k]
                else:
                    warnings.warn(f"MAP estimate of lambda_mat doesn't exist for the current hn_nus[{k}].", ResultWarning)
                    lambda_hat[k] = np.nan
            return pi_hat, a_hat, self.hn_m_vecs, lambda_hat
        if loss == "KL":
            dof = self.hn_nus - D + 1
            a_pdfs = [ss_dirichlet(self.hn_zeta_vecs[k]) for k in range(K)]
            mu_pdfs = [ss_multivariate_t(loc=self.hn_m_vecs[k],
                                         shape=self.hn_w_mats_inv[k] / self.hn_kappas[k] / dof[k], df=dof[k])
                       for k in range(K)]
            lambda_pdfs = [ss_wishart(df=self.hn_nus[k], scale=self.hn_w_mats[k]) for k in range(K)]
            return ss_dirichlet(self.hn_eta_vec), a_pdfs, mu_pdfs, lambda_pdfs
        raise CriteriaError(f"loss={loss} is unsupported. "
                            + "This function supports \"squared\", \"0-1\", and \"KL\".")

    def visualize_posterior(self):
        """Print the posterior hyperparameters and plot q(mu), q(Lambda) for D <= 2 (:1213-1314); needs matplotlib."""
        for title, val in (("hn_alpha_vec:", self.hn_eta_vec), ("E[pi_vec]:", self.hn_eta_vec / self.hn_eta_vec.sum()),
                           ("hn_zeta_vecs:", self.hn_zeta_vecs),
                           ("E[a_mat]", self.hn_zeta_vecs / self.hn_zeta_vecs.sum(axis=1, keepdims=True)),
                           ("hn_m_vecs (equivalent to E[mu_vecs]):", self.hn_m_vecs), ("hn_kappas:", self.hn_kappas),
                           ("hn_nus:", self.hn_nus), ("hn_w_mats:", self.hn_w_mats),
                           ("E[lambda_mats]=", self._e_lambda_mats)):
            print(title)
            print(f"{val}")
        if self.c_degree > 2:
            raise ParameterFormatError("if c_degree > 2, it is impossible to visualize the model by this function.")
        import matplotlib.pyplot as plt
        _, _, mu_pdfs, lambda_pdfs = self.estimate_params(loss="KL")
        K = self.c_num_classes
        sd = np.sqrt(np.stack([np.diag(self.hn_w_mats_inv[k] / self.hn_kappas[k] / self.hn_nus[k]) for k in range(K)]))
        if self.c_degree == 1:
            fig, axes = plt.subplots(1, 2)
            axes[0].set_xlabel("mu_vecs"); axes[0].set_ylabel("Density")
            axes[1].set_xlabel("lambda_mats"); axes[1].set_ylabel("Log density")
            for k in range(K):
                grid = np.linspace(self.hn_m_vecs[k, 0] - 4.0 * sd[k, 0], self.hn_m_vecs[k, 0] + 4.0 * sd[k, 0], 100)
                axes[0].plot(grid, mu_pdfs[k].pdf(grid))
                mean_l = self.hn_nus[k] * self.hn_w_mats[k]
                half = 4.0 * np.sqrt(self.hn_nus[k] / 2.0) * (2.0 * self.hn_w_mats[k])
                grid = np.linspace(max(1.0e-8, mean_l - half), mean_l + half, 500)
                axes[1].plot(grid[:, 0, 0], lambda_pdfs[k].logpdf(grid[:, 0, 0]))
            fig.tight_layout()
        else:
            fig, axes = plt.subplots()
            for k in range(K):
                gx = np.linspace(self.hn_m_vecs[k, 0] - 3.0 * sd[k, 0], self.hn_m_vecs[k, 0] + 3.0 * sd[k, 0], 100)
                gy = np.linspace(self.hn_m_vecs[k, 1] - 3.0 * sd[k, 1], self.hn_m_vecs[k, 1] + 3.0 * sd[k, 1], 100)
                xx, yy = np.meshgrid(gx, gy)
                axes.contour(xx, yy, mu_pdfs[k].pdf(np.stack([xx, yy], axis=-1)), cmap='Blues')
                axes.plot(self.hn_m_vecs[k, 0], self.hn_m_vecs[k, 1], marker="x", color='red')
            axes.set_xlabel("mu_vec[0]"); axes.set_ylabel("mu_vec[1]")
        plt.show()

    # ------------------------------------------------------------------ predictive (:1316-1423)
    def get_p_params(self):
        """Live references to p_a_mat, p_mu_vecs, p_nus, p_lambda_mats (:1316-1330)."""
        return {'p_a_mat': self.p_a_mat, 'p_mu_vecs': self.p_mu_vecs, 'p_nus': self.p_nus,
                'p_lambda_mats': self.p_lambda_mats}

    def calc_pred_dist(self):
        """Predictive parameters from hn_* (:1332-1338)."""
        self.p_a_mat[:] = self.hn_zeta_vecs / self.hn_zeta_vecs.sum(axis=1, keepdims=True)
        self.p_mu_vecs[:] = self.hn_m_vecs
        self.p_nus[:] = self.hn_nus - self.c_degree + 1
        scale = self.hn_kappas * self.p_nus / (self.hn_kappas + 1)
        self.p_lambda_mats[:] = scale[:, None, None] * self.hn_w_mats
        return self

    def _gamma_last(self):
        """gamma_vecs[-1] without copying the whole (N, K) array off the device."""
        lazy = self._lazy_gamma_vecs
        if lazy.host is None and lazy.dev is not None:
            return lazy.dev[-1].cpu().numpy()
        return self.gamma_vecs[-1]

    def make_prediction(self, loss="squared"):
        """Predict the next data point: mixture mean ("squared") or the highest weighted mode ("0-1") (:1340-1370)."""
        if loss == "squared":
            return np.sum((self._gamma_last() @ self.p_a_mat)[:, np.newaxis] * self.p_mu_vecs, axis=0)
        if loss == "0-1":
            weights = self._gamma_last() @ self.p_a_mat
            best_val, best_mu = -1.0, np.empty([self.c_degree])
            for k in range(self.c_num_classes):
                dens = ss_multivariate_t.pdf(x=self.p_mu_vecs[k], loc=self.p_mu_vecs[k],
                                             shape=np.linalg.inv(self.p_lambda_mats[k]), df=self.p_nus[k])
                if dens * weights[k] > best_val:
                    best_mu[:] = self.p_mu_vecs[k]
                    best_val = dens * weights[k]
            return best_mu
        raise CriteriaError(f"loss={loss} is unsupported. "
                            + "This function supports \"squared\" and \"0-1\".")

    def pred_and_update(self, x, loss="squared", max_itr=100, num_init=10, tolerance=1.0E-8,
                        init_type='random_responsibility'):
        """Predict one data point, then make the current posterior the prior and learn from x (:1372-1423)."""
        _check.float_vec(x, 'x', DataFormatError)
        if x.shape != (self.c_degree,):
            raise DataFormatError(f"x must be a 1-dimensional float array whose size is c_degree: {self.c_degree}.")
        self.calc_pred_dist()
        prediction = self.make_prediction(loss=loss)
        self.overwrite_h0_params()
        self.update_posterior(x[np.newaxis, :], max_itr=max_itr, num_init=num_init, tolerance=tolerance,
                              init_type=init_type)
        return prediction

    # ------------------------------------------------------------------ latent variables (:1425-1558)
    def estimate_latent_vars(self, x, loss='0-1', viterbi=True, *, lengths=None):
        """Hidden-state estimates of the sequence x (:1425-1499): the jointly most probable path (`viterbi=True`,
        loss "0-1" only) or the per-element marginals gamma ("squared"/"KL") / their arg-max ("0-1").

        `lengths` (extension, keyword only): x holds that many independent sequences, concatenated; the path is decoded
        per sequence (the sequences in parallel on the device), `phi_vecs` is zero at every sequence start, and the
        marginals are those of the multi-sequence model (see the module docstring).

        Everything runs on the device: the emission log densities, the max-plus recursion and back-tracking of the
        Viterbi path (in the reference's operation order), or (for `viterbi=False`) the whole forward-backward pass.
        As in the reference, `viterbi=False` also overwrites ns / ms / x_bar_vecs / s_mats with the statistics of x."""
        _check.float_vecs(x, 'x', DataFormatError)
        if x.shape[-1] != self.c_degree:
            raise DataFormatError(
                "x.shape[-1] must be self.c_degree: "
                + f"x.shape[-1]={x.shape[-1]}, self.c_degree={self.c_degree}")
        x = x.reshape(-1, self.c_degree)
        starts = self._seq_starts(lengths, x.shape[0])
        if viterbi and loss != '0-1':
            raise CriteriaError(f"loss=\"{loss}\" is unsupported. "
                                + "When viterbi == True, this function supports only \"0-1\".")
        if not viterbi and loss not in ("squared", "KL", "0-1"):
            raise CriteriaError(f"loss=\"{loss}\" is unsupported. "
                                + "When viterbi == False, This function supports \"squared\", \"0-1\", and \"KL\".")
        n, K = x.shape[0], self.c_num_classes
        self._length = n
        eng = self._engine()
        eng.load_data(x)
        eng.set_sequences(starts)
        self._push_prior(eng)
        if viterbi:
            # only the emission densities are evaluated (the reference fills _ln_rho / _rho here and nothing else); the
            # max-plus recursion and the back-tracking run on the device in the reference's operation order
            self._push_hn(eng)
            path, omega, phi = eng.viterbi(self._ln_pi_tilde_vec, self._ln_a_tilde_mat)
            self._rho_host = None                   # alpha / beta / gamma / xi keep their values, as in the reference
            # (and so does the sequence split they belong to, `_starts`, which xi_mats uses)
            self._lazy_ln_rho.set_device(eng.lnrho_buf)
            self._lazy_omega_vecs.set_device(omega)
            self._lazy_phi_vecs.set_device(phi)
            z_hat = np.zeros([n, K], dtype=int)
            z_hat[np.arange(n), path] = 1
            return z_hat
        self._starts = starts                       # the per-element arrays below are those of this x and split
        self._final_e_step(eng)
        if loss == "squared" or loss == "KL":
            return self.gamma_vecs
        return np.eye(K, dtype=int)[np.argmax(self.gamma_vecs, axis=1)]

    def estimate_latent_vars_and_update(self, x, loss="0-1", viterbi=True, max_itr=100, num_init=10, tolerance=1.0E-8,
                                        init_type='subsampling'):
        """estimate_latent_vars, then make the current posterior the prior and learn from x (:1501-1558)."""
        _check.float_vec(x, 'x', DataFormatError)
        if x.shape != (self.c_degree,):
            raise DataFormatError(f"x must be a 1-dimensional float array whose size is c_degree: {self.c_degree}.")
        z_hat = self.estimate_latent_vars(x, loss=loss, viterbi=viterbi)
        self.overwrite_h0_params()
        self.update_posterior(x, max_itr=max_itr, num_init=num_init, tolerance=tolerance, init_type=init_type)
        return z_hat
