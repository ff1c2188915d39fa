"""CPU: hiddenmarkovnormal.GenModel (parameters, validation, the host sample) and the three-phase chain sampler's numpy
model (tools/hmm_gen_model.py) against a plain sequential loop on the same uniforms."""
import numpy as np
import pytest

from bayesml_b200 import DataFormatError, ParameterFormatError, _lib, hiddenmarkovnormal
from tools.hmm_gen_model import draw, phases, sequential

LEFT_RIGHT = np.array([[0.8, 0.2, 0.0, 0.0], [0.0, 0.7, 0.3, 0.0], [0.0, 0.0, 0.9, 0.1], [0.0, 0.0, 0.0, 1.0]])


def _params():
    rng = np.random.default_rng(3)
    a = rng.normal(size=(3, 2, 2))
    return dict(pi_vec=np.array([0.5, 0.3, 0.2]), a_mat=np.array([[0.8, 0.1, 0.1], [0.2, 0.7, 0.1], [0.3, 0.3, 0.4]]),
                mu_vecs=np.array([[-5., -5.], [0., 0.], [5., 5.]]), lambda_mats=a @ a.transpose(0, 2, 1) + np.eye(2))


def test_defaults_constants_and_key_order():
    g = hiddenmarkovnormal.GenModel(3, 2)
    assert g.get_constants() == {"c_num_classes": 3, "c_degree": 2}
    assert list(g.get_params()) == ["pi_vec", "a_mat", "mu_vecs", "lambda_mats"]
    assert list(g.get_h_params()) == ["h_eta_vec", "h_zeta_vecs", "h_m_vecs", "h_kappas", "h_nus", "h_w_mats"]
    assert np.array_equal(g.pi_vec, np.full(3, 1 / 3)) and np.array_equal(g.a_mat, np.full((3, 3), 1 / 3))
    assert np.array_equal(g.mu_vecs, np.zeros((3, 2))) and np.array_equal(g.lambda_mats, np.tile(np.eye(2), (3, 1, 1)))
    learn = hiddenmarkovnormal.LearnModel(3, 2)
    for name in ("eta_vec", "zeta_vecs", "m_vecs", "kappas", "nus", "w_mats"):
        assert np.array_equal(getattr(g, "h_" + name), getattr(learn, "h0_" + name)), name
    assert hiddenmarkovnormal.__all__ == ["GenModel", "LearnModel"]
    big = hiddenmarkovnormal.GenModel(40, 300)                   # the host path has no size limit
    assert big.a_mat.shape == (40, 40)


@pytest.mark.parametrize("kwargs", [
    dict(pi_vec=np.array([0.5, 0.6, 0.2])),                      # does not sum to 1
    dict(pi_vec=np.array([1.2, -0.2, 0.0])),                     # negative entry
    dict(pi_vec=np.array([0.5, 0.5])),                           # wrong shape
    dict(a_mat=np.array([[0.5, 0.5, 0.1], [0.2, 0.7, 0.1], [0.3, 0.3, 0.4]])),
    dict(a_mat=np.array([[1.1, -0.1, 0.0], [0.2, 0.7, 0.1], [0.3, 0.3, 0.4]])),
    dict(a_mat=np.full((2, 3), 1 / 3)),
    dict(mu_vecs=np.zeros((3, 3))),
    dict(mu_vecs=np.zeros((2, 2))),
    dict(lambda_mats=np.tile(np.array([[1.0, 2.0], [2.0, 1.0]]), (3, 1, 1))),    # not positive definite
    dict(lambda_mats=np.tile(np.array([[1.0, 0.5], [0.0, 1.0]]), (3, 1, 1))),    # not symmetric
    dict(lambda_mats=np.tile(np.eye(2), (2, 1, 1))),
    dict(h_eta_vec=np.array([1.0, 0.0, 1.0])),
    dict(h_zeta_vecs=-np.ones((3, 3))),
    dict(h_kappas=np.array([1.0, -1.0, 1.0])),
    dict(h_nus=np.array([0.5, 2.0, 2.0])),                       # <= D - 1
    dict(h_w_mats=np.tile(np.array([[1.0, 2.0], [2.0, 1.0]]), (3, 1, 1))),
    dict(h_m_vecs=np.zeros((3, 3))),
])
def test_invalid_parameters_raise(kwargs):
    with pytest.raises(ParameterFormatError):
        hiddenmarkovnormal.GenModel(3, 2, **kwargs)


def test_sample_argument_errors():
    g = hiddenmarkovnormal.GenModel(3, 2, **_params())
    for bad in (0, -1, 2.0):
        with pytest.raises(DataFormatError):
            g.gen_sample(bad)
    for lengths in ([3, 4], [5, 0, 1], [], np.array([[2, 4]]), [2.0, 4.0]):
        with pytest.raises(DataFormatError):
            g.gen_sample(6, lengths=lengths)
    with pytest.raises(ParameterFormatError):                    # the device sampler's limits, before any device work
        hiddenmarkovnormal.GenModel(33, 2).gen_sample(10, device="cuda:0")
    with pytest.raises(ParameterFormatError):
        hiddenmarkovnormal.GenModel(2, 257).gen_sample(10, device="cuda:0")
    with pytest.raises(ParameterFormatError):
        hiddenmarkovnormal.GenModel(2, 3).visualize_model()


def test_param_roundtrip_and_save_sample(tmp_path):
    g = hiddenmarkovnormal.GenModel(3, 2, h_nus=np.array([3.0, 4.0, 5.0]), h_kappas=np.array([0.5, 1.0, 2.0]), **_params())
    g.save_params(str(tmp_path / "p.pkl"))
    g.save_h_params(str(tmp_path / "h.pkl"))
    h = hiddenmarkovnormal.GenModel(3, 2).load_params(str(tmp_path / "p.pkl")).load_h_params(str(tmp_path / "h.pkl"))
    for name, val in list(g.get_params().items()) + list(g.get_h_params().items()):
        assert np.array_equal(getattr(h, name), val), name
    g.save_sample(str(tmp_path / "s.npz"), 7)
    s = np.load(tmp_path / "s.npz")
    assert s["x"].shape == (7, 2) and s["z"].shape == (7, 3) and np.array_equal(s["z"].sum(axis=1), np.ones(7))


def test_host_sample_is_the_reference_loop():
    g = hiddenmarkovnormal.GenModel(3, 2, seed=7, **_params())
    x, z = g.gen_sample(40)
    # the loop written out: one rng.choice, then one rng.multivariate_normal, per element
    rng, p = np.random.default_rng(7), _params()
    cov = np.linalg.inv(p["lambda_mats"])
    k = rng.choice(3, p=p["pi_vec"])
    for i in range(40):
        if i:
            k = rng.choice(3, p=p["a_mat"][k])
        assert z[i, k] == 1 and z[i].sum() == 1
        assert np.array_equal(x[i], rng.multivariate_normal(mean=p["mu_vecs"][k], cov=cov[k]))
    x2, z2 = hiddenmarkovnormal.GenModel(3, 2, seed=7, **_params()).gen_sample(40, lengths=[40])
    assert np.array_equal(x, x2) and np.array_equal(z, z2)
    x3, z3 = hiddenmarkovnormal.GenModel(3, 2, seed=7, **_params()).gen_sample(40)
    assert np.array_equal(x, x3) and np.array_equal(z, z3)


def test_host_sample_with_lengths_restarts_every_sequence_from_pi():
    lengths = [5, 1, 7]
    g = hiddenmarkovnormal.GenModel(3, 2, seed=11, **_params())
    x, z = g.gen_sample(13, lengths=lengths)
    rng, p = np.random.default_rng(11), _params()
    cov = np.linalg.inv(p["lambda_mats"])
    i = 0
    for length in lengths:                                       # the single-sequence loop once per sequence, in order
        for j in range(length):
            k = rng.choice(3, p=p["pi_vec"] if j == 0 else p["a_mat"][k])
            assert z[i, k] == 1
            assert np.array_equal(x[i], rng.multivariate_normal(mean=p["mu_vecs"][k], cov=cov[k]))
            i += 1


def test_host_sample_respects_structural_zeros():
    g = hiddenmarkovnormal.GenModel(4, 1, seed=2, pi_vec=np.array([0.6, 0.4, 0.0, 0.0]), a_mat=LEFT_RIGHT)
    lengths = [50] * 40
    _, z = g.gen_sample(2000, lengths=lengths)
    s = z.argmax(axis=1)
    starts = np.cumsum([0] + lengths[:-1])
    assert np.all(s[starts] <= 1)
    inner = np.ones(2000, dtype=bool)
    inner[starts] = False
    prev, cur = s[np.flatnonzero(inner) - 1], s[inner]
    assert np.all(LEFT_RIGHT[prev, cur] > 0)


def test_gen_params_draw_order():
    g = hiddenmarkovnormal.GenModel(3, 2, seed=4, h_zeta_vecs=np.array([[1.0, 2.0, 3.0], [0.5, 0.5, 0.5], [4.0, 1.0, 1.0]]))
    g.gen_params()
    rng = np.random.default_rng(4)
    assert np.array_equal(g.pi_vec, rng.dirichlet(g.h_eta_vec))
    for k in range(3):
        assert np.array_equal(g.a_mat[k], rng.dirichlet(g.h_zeta_vecs[k]))
    from scipy.stats import wishart
    for k in range(3):
        lam = wishart.rvs(df=g.h_nus[k], scale=g.h_w_mats[k], random_state=rng)
        assert np.array_equal(g.lambda_mats[k], lam)
        assert np.array_equal(g.mu_vecs[k], rng.multivariate_normal(mean=g.h_m_vecs[k], cov=np.linalg.inv(lam)))


def test_against_the_reference_genmodel():
    from oracle.ref_loader import load_reference_module, reference_available
    if not reference_available():
        pytest.skip("the reference BayesML is not available")
    try:
        ref = load_reference_module("hiddenmarkovnormal")
    except ImportError:
        pytest.skip("the reference BayesML has no hiddenmarkovnormal here")
    for seed in (0, 5):
        a = hiddenmarkovnormal.GenModel(3, 2, seed=seed, **_params())
        b = ref.GenModel(3, 2, seed=seed, **_params())
        xa, za = a.gen_sample(50)
        xb, zb = b.gen_sample(50)
        assert np.array_equal(xa, xb) and np.array_equal(za, zb) and za.dtype == zb.dtype
        a.gen_params()
        b.gen_params()
        for f in ("pi_vec", "a_mat", "mu_vecs", "lambda_mats"):
            assert np.array_equal(getattr(a, f), getattr(b, f)), f
    assert a.get_constants() == b.get_constants()
    assert list(a.get_params()) == list(b.get_params()) and list(a.get_h_params()) == list(b.get_h_params())


# ---------------------------------------------------------------- the inverse-CDF rule and the three-phase model
def test_cdf_rule_never_draws_a_zero_probability_state():
    # a row whose rounded cumulative sum ends below 1 (0.1 * 10 in floating point is 0.9999999999999999)
    p = np.array([0.1] * 10 + [0.0, 0.0])
    assert np.cumsum(p)[-1] < 1.0
    pi = np.array([0.0, 0.5, 0.0, 0.5] + [0.0] * 8)
    table = hiddenmarkovnormal._inverse_cdf_table(pi, np.tile(p, (12, 1)))
    below_one = np.nextafter(1.0, 0.0)
    for u in (below_one, 1.0 - 2 ** -53, 0.99999999999999995, 0.5, 1e-300, np.cumsum(p)[-1]):
        assert p[draw(table[1], u)] > 0 and pi[draw(table[0], u)] > 0, u
    for u in np.random.default_rng(0).random(20000):
        assert p[draw(table[1], u)] > 0 and pi[draw(table[0], u)] > 0
    assert draw(table[0], 0.5) == 1 and draw(table[0], 0.5000001) == 3 and draw(table[1], below_one) == 9
    # the last positive entry is 2.0, and everything before it is the plain cumulative sum
    assert table[1, 9] == 2.0 and np.array_equal(table[1, :9], np.cumsum(p)[:9])
    assert table[0, 3] == 2.0


def _random_model(K, rng, zeros):
    pi = rng.dirichlet(np.ones(K))
    a = rng.dirichlet(np.ones(K) * 0.5, size=K)
    if zeros and K > 1:
        pi[rng.integers(0, K)] = 0.0
        a[rng.random((K, K)) < 0.3] = 0.0
        a[np.arange(K), np.arange(K)] += 0.1
        pi, a = pi / pi.sum(), a / a.sum(axis=1, keepdims=True)
    return hiddenmarkovnormal._inverse_cdf_table(pi, a)


@pytest.mark.parametrize("K", [1, 2, 3, 5])
@pytest.mark.parametrize("lengths", [None, [1, 1, 1, 30, 1, 2], [7, 7, 7, 7, 12], [1] * 40, [13, 27]])
def test_phase_model_equals_the_sequential_loop(K, lengths):
    rng = np.random.default_rng(K * 100 + (0 if lengths is None else len(lengths)))
    n = 40
    starts = None if lengths is None else np.cumsum([0] + lengths[:-1])
    u = 1.0 - rng.random(n)                                      # (0, 1]
    u[::9] = np.nextafter(1.0, 0.0)
    for zeros in (False, True):
        cdf = _random_model(K, rng, zeros)
        ref = sequential(cdf, u, starts)
        for L in (1, 2, 7, 13, 64, n):
            assert np.array_equal(phases(cdf, u, starts, L), ref), (L, zeros)


def test_gen_entry_points_load_and_reject_bad_arguments(lib_built):
    lib = _lib.load()
    assert lib.bgmm_hmm_gen_workspace_bytes(8, 4_000_000, 1, 0) > 0
    assert lib.bgmm_hmm_gen_workspace_bytes(8, 4_000_000, 1, 976) == 0           # 4099 chunks
    assert lib.bgmm_hmm_gen_workspace_bytes(8, 4_000_000, 1, 977) > 0            # 4095 chunks
    assert lib.bgmm_hmm_gen_workspace_bytes(33, 100, 1, 0) == 0
    fake = 256                                                   # never dereferenced: the checks come first
    starts = np.array([0, 3, 4], dtype=np.int64)

    def call(n=10, K=3, D=2, seq=None, n_seqs=1, chunk_len=0):
        return lib.bgmm_hmm_gen_sample(fake, fake, n, K, D, fake, fake, fake, seq, n_seqs, 1, chunk_len, fake, None)

    for kwargs in (dict(K=33), dict(K=0), dict(D=257), dict(D=0), dict(n=-1), dict(n=5000, chunk_len=1),
                   dict(chunk_len=-1), dict(seq=starts.ctypes.data, n_seqs=3, n=4),
                   dict(seq=np.array([1, 3], dtype=np.int64).ctypes.data, n_seqs=2),
                   dict(seq=np.array([0, 3, 3], dtype=np.int64).ctypes.data, n_seqs=3),
                   dict(seq=np.array([0, 5, 3], dtype=np.int64).ctypes.data, n_seqs=3)):
        assert call(**kwargs) == -1, kwargs
        assert b"bgmm_hmm_gen_sample" in lib.bgmm_last_error()
    assert call(n=0) == 0
