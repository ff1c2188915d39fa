"""GenModel: host path = the reference's random stream (CPU, needs the reference); device path = same distribution (GPU)."""
import numpy as np
import pytest


def _params():
    rng = np.random.default_rng(3)
    a = rng.normal(size=(3, 2, 2))
    return dict(pi_vec=np.array([0.5, 0.3, 0.2]), mu_vecs=np.array([[-5., -5.], [0., 0.], [5., 5.]]),
                lambda_mats=a @ a.transpose(0, 2, 1) + np.eye(2))


def test_host_gen_sample_and_gen_params_follow_the_reference_stream():
    from bayesml_b200 import gaussianmixture
    from conftest import load_golden
    from oracle.ref_loader import load_reference_gaussianmixture, reference_available
    # stored: the c1_readme fixture's input rows are the reference GenModel's own sample (make_golden.py)
    g = load_golden("c1_readme")
    x, z = gaussianmixture.GenModel(c_num_classes=3, c_degree=2, mu_vecs=np.array([[-5., -5.], [0., 0.], [5., 5.]]),
                                    seed=0).gen_sample(1000)
    assert np.array_equal(x, g["x"]) and z.shape == (1000, 3)
    if not reference_available():
        return
    ref = load_reference_gaussianmixture()
    for seed in (0, 5):
        a, b = gaussianmixture.GenModel(3, 2, seed=seed, **_params()), ref.GenModel(3, 2, seed=seed, **_params())
        xa, za = a.gen_sample(50)
        xb, zb = b.gen_sample(50)
        assert np.array_equal(xa, xb) and np.array_equal(za, zb) and za.dtype == zb.dtype
        a.gen_params(); b.gen_params()
        for f in ("pi_vec", "mu_vecs", "lambda_mats"):
            assert np.array_equal(getattr(a, f), getattr(b, f)), f
    assert a.get_constants() == b.get_constants()
    assert list(a.get_params()) == list(b.get_params()) and list(a.get_h_params()) == list(b.get_h_params())


def test_argument_errors_and_param_roundtrip(tmp_path):
    from bayesml_b200 import DataFormatError, ParameterFormatError, gaussianmixture
    g = gaussianmixture.GenModel(3, 2, **_params())
    with pytest.raises(ParameterFormatError):
        g.set_params(pi_vec=np.array([0.5, 0.6, 0.2]))
    with pytest.raises(ParameterFormatError):
        g.set_params(mu_vecs=np.zeros((3, 3)))
    with pytest.raises(ParameterFormatError):
        g.set_h_params(h_nus=np.array([0.5, 2.0, 2.0]))
    with pytest.raises(DataFormatError):
        g.gen_sample(0)
    g.save_params(str(tmp_path / "p.pkl")); g.save_h_params(str(tmp_path / "h.pkl"))
    h = gaussianmixture.GenModel(3, 2).load_params(str(tmp_path / "p.pkl")).load_h_params(str(tmp_path / "h.pkl"))
    assert np.array_equal(h.mu_vecs, g.mu_vecs) and np.array_equal(h.lambda_mats, g.lambda_mats)
    g.save_sample(str(tmp_path / "s.npz"), 7)
    s = np.load(tmp_path / "s.npz")
    assert s["x"].shape == (7, 2) and s["z"].shape == (7, 3)


@pytest.mark.gpu
def test_device_gen_sample_has_the_model_distribution():
    from bayesml_b200 import gaussianmixture
    g = gaussianmixture.GenModel(3, 2, seed=1, **_params())
    n = 400000
    x, z = g.gen_sample(n, device="cuda:0")
    assert x.shape == (n, 2) and z.shape == (n, 3) and z.dtype == int and np.array_equal(z.sum(axis=1), np.ones(n, dtype=int))
    frac = z.mean(axis=0)
    assert np.allclose(frac, g.pi_vec, atol=4 * np.sqrt(0.25 / n))
    cov = np.linalg.inv(g.lambda_mats)
    for k in range(3):
        xs = x[z[:, k] == 1]
        se = np.sqrt(np.diag(cov[k]) / xs.shape[0])
        assert np.all(np.abs(xs.mean(axis=0) - g.mu_vecs[k]) < 5 * se)
        assert np.allclose(np.cov(xs.T), cov[k], rtol=0.03, atol=0.01)
    x2, z2 = gaussianmixture.GenModel(3, 2, seed=1, **_params()).gen_sample(n, device="cuda:0")
    assert np.array_equal(x, x2) and np.array_equal(z, z2)                      # reproducible from the seed
    xd, zd = gaussianmixture.GenModel(5, 40, seed=2).gen_sample(1000, device="cuda:0", as_numpy=False)
    assert xd.is_cuda and tuple(xd.shape) == (1000, 40) and zd.dtype.is_floating_point is False
