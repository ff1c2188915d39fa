"""GPU: several independent sequences sharing one posterior (`lengths=`; bgmm_hmm_pass_seqs / bgmm_hmm_viterbi_seqs)
against the multi-sequence oracle (oracle/hmm_multiseq_oracle.py).  Tolerance: 1e-9 relative, 1e-8 for accumulated
per-element arrays, as for one sequence."""
import contextlib
import io
import warnings

import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu

RTOL = 1e-9


def _close(a, b, rtol=RTOL, scale=None):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    scale = np.max(np.abs(b)) if scale is None else scale
    return np.allclose(a, b, rtol=rtol, atol=rtol * 1e-4 * max(scale, 1e-300))


def _lengths(kind, seed):
    rng = np.random.default_rng(seed)
    if kind == "ones":            # many length-1 sequences among a few longer ones
        return [1] * 300 + [2, 3, 40, 1, 64, 1]
    if kind == "short":           # many short ones, below one chunk
        return rng.integers(1, 30, size=200).tolist()
    if kind == "mixed":           # several chunks per sequence, exact chunk multiples, 1 and 2
        return rng.integers(1, 400, size=20).tolist() + [32, 64, 1, 2, 96]
    if kind == "long":            # one long sequence (two-level sweep of its own) among short ones
        return rng.integers(1, 50, size=100).tolist() + [300_000] + rng.integers(1, 50, size=100).tolist()
    raise ValueError(kind)


def _data(n, d, k, seed):
    rng = np.random.default_rng(seed)
    mu = rng.normal(0.0, 3.0, size=(k, d))
    z = np.repeat(rng.integers(0, k, size=n // 3 + 1), 3)[:n]
    return mu[z] + rng.normal(size=(n, d))


def _engine_and_oracle(K, D, x, lengths):
    from bayesml_b200.engine import HMMEngine
    from oracle.hmm_multiseq_oracle import OracleHMMSeqs, seq_starts
    o = OracleHMMSeqs(K, D, seed=3)
    o.alloc(x.shape[0])
    o.set_lengths(lengths)
    eng = HMMEngine(K, D)
    eng.load_data(x)
    eng.set_sequences(seq_starts(lengths))
    eng.set_hmm_prior(o.h0_eta_vec, o.h0_zeta_vecs, o.h0_m_vecs, o.h0_kappas, o.h0_nus, o.h0_w_mats_inv, o.ln_b_h0_w_nus,
                      o.ln_c_h0_eta_vec, o.ln_c_h0_zeta_vecs_sum)
    return eng, o


CASES = [  # K, D, lengths, init, window cap (None: default)
    (1, 1, "short", "subsampling", None),
    (2, 3, "ones", "random_responsibility", "0"),
    (3, 1, "mixed", "subsampling", "0"),
    (3, 3, "mixed", "random_responsibility", None),
    (8, 8, "mixed", "subsampling", "0"),
    (8, 3, "short", "random_responsibility", None),
    (17, 3, "mixed", "subsampling", None),
    (17, 1, "ones", "subsampling", "0"),
    (32, 40, "mixed", "random_responsibility", "0"),
    (32, 8, "mixed", "subsampling", None),
    (3, 3, "long", "subsampling", "0"),
    (2, 1, "long", "random_responsibility", None),
]


@pytest.mark.parametrize("K,D,kind,init_type,cap", CASES)
def test_fit_from_identical_init(K, D, kind, init_type, cap, monkeypatch, lib_built):
    """Every ELBO of every iteration, the 9 terms, hn_*, the statistics against the oracle, from the same initial state."""
    if cap is not None:
        monkeypatch.setenv("BGMM_HMM_WINDOW_CAP", cap)
    lengths = _lengths(kind, K * 100 + D)
    x = _data(sum(lengths), D, K, K + D)
    eng, o = _engine_and_oracle(K, D, x, lengths)
    max_itr = 2 if kind == "long" else 5
    o.init_fb_params()
    o.reset_hn()
    if init_type == "subsampling":
        o.init_subsampling(x)
        eng.set_hmm_params(o.hn_eta_vec, o.hn_zeta_vecs, o.hn_m_vecs, o.hn_kappas, o.hn_nus, o.hn_w_mats_inv)
        o.e_step(x)
        init = None
    else:
        o.init_random_responsibility(x)
        eng.set_hmm_params(o.hn_eta_vec, o.hn_zeta_vecs, o.hn_m_vecs, o.hn_kappas, o.hn_nus, o.hn_w_mats_inv)
        init = (o.gamma_vecs.copy(), o.xi_mats.sum(axis=0))
    o.calc_vl()
    ref = [float(o.vl)]
    for _ in range(max_itr):
        o.iterate(x)
        ref.append(float(o.vl))
    hist, _ = eng.run(max_itr, 0.0, init=init)
    assert _close(hist, ref), np.max(np.abs(np.asarray(hist) - ref) / np.abs(ref))
    p = eng.fetch_params()
    for mine, name in (("alpha", "hn_eta_vec"), ("zeta", "hn_zeta_vecs"), ("m", "hn_m_vecs"), ("kappa", "hn_kappas"),
                       ("nu", "hn_nus"), ("winv", "hn_w_mats_inv"), ("ns", "ns"), ("ms", "ms"), ("x_bar", "x_bar_vecs")):
        assert _close(p[mine], getattr(o, name)), mine
    assert _close(p["s_mats"], o.s_mats, rtol=1e-8)
    assert _close(p["gamma0"], o.gamma_starts())
    t, vx = p["vl_terms"], p["vlx"]
    mine_terms = np.array([t[0], vx[0], t[2], vx[1], t[3], vx[2], t[5], vx[3], t[6]])
    assert np.allclose(mine_terms, o.vl_terms, rtol=RTOL, atol=RTOL * np.max(np.abs(o.vl_terms)))
    # the per-element arrays of one more E-step with the final parameters
    eng.set_hmm_params(o.hn_eta_vec, o.hn_zeta_vecs, o.hn_m_vecs, o.hn_kappas, o.hn_nus, o.hn_w_mats_inv)
    st = eng.final_pass()
    o.e_step(x)
    assert _close(st["ms"], o.ms) and _close(st["ns"], o.ns)
    for buf, name in ((eng.gamma_buf, "gamma_vecs"), (eng.alpha_buf, "alpha_vecs"), (eng.beta_buf, "beta_vecs"),
                      (eng.cs_buf, "cs")):
        assert _close(buf.cpu().numpy(), getattr(o, name), rtol=1e-8), name


def test_windows_are_clamped_to_sequences(lib_built):
    """Mixing mode on the default path with windows that would reach across sequence starts."""
    K, D = 3, 2
    rng = np.random.default_rng(5)
    lengths = rng.integers(40, 200, size=60).tolist()
    x = rng.normal(size=(sum(lengths), D)) * 0.3 + rng.integers(0, 3, size=(sum(lengths), 1))   # fast mixing chain
    eng, o = _engine_and_oracle(K, D, x, lengths)
    o.init_fb_params()
    o.reset_hn()
    o.init_subsampling(x)
    eng.set_hmm_params(o.hn_eta_vec, o.hn_zeta_vecs, o.hn_m_vecs, o.hn_kappas, o.hn_nus, o.hn_w_mats_inv)
    o.e_step(x)
    o.calc_vl()
    ref = [float(o.vl)]
    for _ in range(4):
        o.iterate(x)
        ref.append(float(o.vl))
    hist, _ = eng.run(4, 0.0)
    assert eng.fetch_params()["window"] > 0, "the mixing mode did not run"
    assert _close(hist, ref)


def test_lengths_n_is_the_single_sequence_path(lib_built):
    from bayesml_b200 import hiddenmarkovnormal
    g = load_golden("hmm_traj_d2k3")
    K, D = int(g["K"]), int(g["D"])
    kw = eval(str(g["fit_kwargs"]), {"__builtins__": {}}, {"dict": dict})
    x = np.asarray(g["x"])
    outs, models = [], []
    for lengths in (None, [x.reshape(-1, D).shape[0]]):
        m = hiddenmarkovnormal.LearnModel(K, D, seed=int(g["seed"]))
        out = io.StringIO()
        with contextlib.redirect_stdout(out), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            m.update_posterior(x, lengths=lengths, **kw)
        outs.append(out.getvalue())
        models.append(m)
    assert outs[0] == outs[1]
    for f in ("hn_eta_vec", "hn_zeta_vecs", "hn_m_vecs", "hn_kappas", "hn_nus", "hn_w_mats", "ns", "ms", "x_bar_vecs",
              "s_mats", "gamma_vecs", "alpha_vecs", "beta_vecs", "_cs"):
        assert np.array_equal(getattr(models[0], f), getattr(models[1], f)), f
    assert models[0].vl == models[1].vl


@pytest.mark.parametrize("init_type", ["subsampling", "random_responsibility"])
def test_update_posterior_end_to_end(init_type, lib_built):
    from bayesml_b200 import hiddenmarkovnormal
    from oracle.hmm_multiseq_oracle import OracleHMMSeqs, fit_hmm_seqs
    K, D = 3, 2
    lengths = _lengths("mixed", 7)
    x = _data(sum(lengths), D, K, 8)
    kw = dict(max_itr=20, num_init=3, tolerance=1e-6, init_type=init_type)
    o = OracleHMMSeqs(K, D, seed=21)
    tr = fit_hmm_seqs(o, x, lengths, **kw)
    m = hiddenmarkovnormal.LearnModel(K, D, seed=21)
    out = io.StringIO()
    with contextlib.redirect_stdout(out), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m.update_posterior(x, lengths=lengths, **kw)
    lines = out.getvalue().split("\n")[:-1]
    assert len(lines) == kw["num_init"]
    stars = [i for i, ln in enumerate(lines) if ln.endswith("*")]
    assert stars[-1] == tr.selected
    assert out.getvalue().count("(converged)") == sum(tr.converged)
    for f in ("hn_eta_vec", "hn_zeta_vecs", "hn_m_vecs", "hn_kappas", "hn_nus", "hn_w_mats", "ns", "ms", "x_bar_vecs"):
        assert _close(getattr(m, f), getattr(o, f), rtol=1e-8), f
    for f, of in (("gamma_vecs", "gamma_vecs"), ("alpha_vecs", "alpha_vecs"), ("beta_vecs", "beta_vecs"), ("_cs", "cs")):
        assert _close(getattr(m, f), getattr(o, of), rtol=1e-8), f
    assert _close(m.xi_mats, o.xi_mats, rtol=1e-8)
    assert np.all(m.xi_mats[o.starts] == 0.0)


def _numpy_viterbi(ln_rho, ln_pi, ln_a, starts, n):
    K = ln_rho.shape[1]
    omega = np.zeros([n, K])
    phi = np.zeros([n, K], dtype=int)
    path = np.zeros(n, dtype=int)
    ends = np.append(starts[1:], n)
    for a, b in zip(starts, ends):
        omega[a] = ln_rho[a] + ln_pi
        for i in range(a + 1, b):
            omega[i] = ln_rho[i] + np.max(ln_a + omega[i - 1, :, np.newaxis], axis=0)
            phi[i] = np.argmax(ln_a + omega[i - 1, :, np.newaxis], axis=0)
        k = np.argmax(omega[b - 1])
        path[b - 1] = k
        for i in range(b - 2, a - 1, -1):
            k = phi[i + 1, k]
            path[i] = k
    return omega, phi, path


@pytest.mark.parametrize("K,D", [(1, 2), (3, 2), (8, 3), (32, 4)])
def test_viterbi_per_sequence_bit_identical(K, D, lib_built):
    from bayesml_b200 import hiddenmarkovnormal
    rng = np.random.default_rng(K)
    lengths = rng.integers(1, 25, size=10_000).tolist() + [3000]
    n = sum(lengths)
    x = _data(n, D, K, K + 1)
    m = hiddenmarkovnormal.LearnModel(K, D, seed=2)
    with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m.update_posterior(x[:5000], max_itr=5, num_init=1)
    z = m.estimate_latent_vars(x, lengths=lengths)
    starts = np.concatenate([[0], np.cumsum(lengths)[:-1]])
    omega, phi, path = _numpy_viterbi(m._ln_rho, m._ln_pi_tilde_vec, m._ln_a_tilde_mat, starts, n)
    assert np.array_equal(m.omega_vecs, omega)
    assert np.array_equal(m.phi_vecs, phi)
    assert np.array_equal(np.argmax(z, axis=1), path) and np.all(z.sum(axis=1) == 1)


def test_marginals_and_statistics_per_sequence(lib_built):
    from bayesml_b200 import hiddenmarkovnormal
    from oracle.hmm_multiseq_oracle import OracleHMMSeqs
    K, D = 4, 3
    lengths = _lengths("mixed", 3)
    x = _data(sum(lengths), D, K, 4)
    m = hiddenmarkovnormal.LearnModel(K, D, seed=2)
    with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m.update_posterior(x, max_itr=5, num_init=1, lengths=lengths)
    o = OracleHMMSeqs(K, D)
    o.set_lengths(lengths)
    for f in o.HN:
        getattr(o, f)[:] = getattr(m, f)
    o.q_pi_features(); o.q_a_features(); o.q_lambda_features()
    g = m.estimate_latent_vars(x, loss="squared", viterbi=False, lengths=lengths)
    go = o.estimate_latent_vars(x, loss="squared", viterbi=False)
    assert _close(g, go, rtol=1e-8)
    for f in ("ns", "ms", "x_bar_vecs"):
        assert _close(getattr(m, f), getattr(o, f), rtol=1e-8), f
    assert _close(m.s_mats, o.s_mats, rtol=1e-7)


def test_concatenation_is_not_equivalent(lib_built):
    """Two sequences are not their concatenation: the junction transition must not be counted in ms."""
    from bayesml_b200 import hiddenmarkovnormal
    K, D = 2, 1
    x = np.concatenate([np.zeros(50), np.full(50, 8.0)])[:, None] + np.random.default_rng(0).normal(size=(100, 1)) * 0.1
    res = []
    for lengths in ([50, 50], None):
        m = hiddenmarkovnormal.LearnModel(K, D, seed=4)
        with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            m.update_posterior(x, max_itr=30, num_init=2, lengths=lengths)
        res.append(m.ms.copy())
    assert abs(res[0].sum() - 98.0) < 1e-8 and abs(res[1].sum() - 99.0) < 1e-8
    assert not np.allclose(res[0], res[1])
