"""GPU: hiddenmarkovnormal.GenModel.gen_sample(device=...) — bgmm_hmm_gen_sample samples the chain exactly (bit-identical
for every chunking), honours structural zeros, has the model's distribution, and a LearnModel fit recovers A."""
import contextlib
import io
import warnings

import numpy as np
import pytest

from bayesml_b200 import ParameterFormatError, _lib, hiddenmarkovnormal

pytestmark = pytest.mark.gpu

LEFT_RIGHT = np.array([[0.8, 0.2, 0.0, 0.0], [0.0, 0.7, 0.3, 0.0], [0.0, 0.0, 0.9, 0.1], [0.0, 0.0, 0.0, 1.0]])


def _model(K, D, seed, zeros=False):
    rng = np.random.default_rng(seed)
    pi = rng.dirichlet(np.ones(K))
    a = rng.dirichlet(np.ones(K) * 0.3, size=K)
    if zeros and K > 1:
        a[rng.random((K, K)) < 0.3] = 0.0
        a[np.arange(K), np.arange(K)] += 0.05
        a /= a.sum(axis=1, keepdims=True)
        pi[0] = 0.0
        pi /= pi.sum()
    b = rng.normal(size=(K, D, D))
    return hiddenmarkovnormal.GenModel(K, D, seed=seed, pi_vec=pi, a_mat=a, mu_vecs=rng.normal(size=(K, D)) * 3,
                                       lambda_mats=b @ b.transpose(0, 2, 1) + np.eye(D))


def _sample(g, n, starts, chunk_len, seed):
    """One bgmm_hmm_gen_sample call with a forced chunk length -> (x, z) on the host."""
    import torch
    lib = _lib.load()
    K, D = g.c_num_classes, g.c_degree
    dev = torch.device("cuda:0")
    cdf, mu, chol = (torch.as_tensor(np.ascontiguousarray(a)).to(dev) for a in (
        hiddenmarkovnormal._inverse_cdf_table(g.pi_vec, g.a_mat), g.mu_vecs,
        np.linalg.cholesky(np.linalg.inv(g.lambda_mats))))
    n_seqs = 1 if starts is None else starts.size
    x = torch.empty((n, D), dtype=torch.float64, device=dev)
    z = torch.empty(n, dtype=torch.int32, device=dev)
    ws = torch.empty(lib.bgmm_hmm_gen_workspace_bytes(K, n, n_seqs, chunk_len), dtype=torch.uint8, device=dev)
    _lib.check(lib.bgmm_hmm_gen_sample(x.data_ptr(), z.data_ptr(), n, K, D, cdf.data_ptr(), mu.data_ptr(), chol.data_ptr(),
                                       None if starts is None else starts.ctypes.data, n_seqs, seed, chunk_len,
                                       ws.data_ptr(), torch.cuda.current_stream(dev).cuda_stream), "bgmm_hmm_gen_sample")
    return x.cpu().numpy(), z.cpu().numpy()


def _mixed_lengths(n, rng):
    out = []
    while sum(out) < n:
        out.append(int(rng.choice([1, 1, 2, 5, 37, 300, 4000])))
    out[-1] -= sum(out) - n
    return [v for v in out if v > 0]


@pytest.mark.parametrize("K", [1, 2, 3, 8, 17, 32])
@pytest.mark.parametrize("D", [1, 2, 8])
def test_sample_is_bit_identical_for_every_chunking(K, D):
    rng = np.random.default_rng(K * 31 + D)
    for n in (1, 97, 5000, 300_000):
        g = _model(K, D, seed=K + D, zeros=True)
        for lengths in (None, _mixed_lengths(n, rng)):
            starts = None if lengths is None or len(lengths) == 1 else np.cumsum([0] + lengths[:-1]).astype(np.int64)
            ref = _sample(g, n, starts, n, 12345)                      # one chunk: the sequential recursion
            for L in (0, -(-n // 4096), 1009):
                x, z = _sample(g, n, starts, L, 12345)
                assert np.array_equal(z, ref[1]) and np.array_equal(x, ref[0]), (n, L, lengths is None)
            assert z.min() >= 0 and z.max() < K


def test_structural_zeros_at_four_million():
    n = 4_000_000
    g = hiddenmarkovnormal.GenModel(4, 1, seed=5, pi_vec=np.array([0.0, 0.7, 0.3, 0.0]), a_mat=LEFT_RIGHT)
    lengths = [1, 2, 997] + [1000] * 3999
    starts = np.cumsum([0] + lengths[:-1])
    _, z = g.gen_sample(n, lengths=lengths, device="cuda:0", as_numpy=False)
    s = z.cpu().numpy()
    assert np.all((s[starts] == 1) | (s[starts] == 2))
    inner = np.ones(n, dtype=bool)
    inner[starts] = False
    assert np.all(LEFT_RIGHT[s[np.flatnonzero(inner) - 1], s[inner]] > 0)


def test_transition_and_start_frequencies():
    K, n = 5, 4_000_000
    g = _model(K, 2, seed=9)
    _, z = g.gen_sample(n, device="cuda:0", as_numpy=False)
    s = z.cpu().numpy().astype(np.int64)
    counts = np.zeros((K, K))
    np.add.at(counts, (s[:-1], s[1:]), 1.0)
    rows = counts.sum(axis=1, keepdims=True)
    sigma = np.sqrt(rows * g.a_mat * (1 - g.a_mat))
    assert np.all(np.abs(counts - rows * g.a_mat) <= 5 * sigma + 1e-9)
    # start states over 2e5 sequences with a sticky A: the starts still follow pi
    sticky = np.full((K, K), 0.01 / (K - 1)) + np.eye(K) * (0.99 - 0.01 / (K - 1))
    g2 = hiddenmarkovnormal.GenModel(K, 1, seed=3, pi_vec=np.array([0.4, 0.3, 0.15, 0.1, 0.05]), a_mat=sticky)
    m = 200_000
    _, z2 = g2.gen_sample(m * 3, lengths=[3] * m, device="cuda:0", as_numpy=False)
    first = np.bincount(z2.cpu().numpy()[::3], minlength=K)
    assert np.all(np.abs(first - m * g2.pi_vec) <= 5 * np.sqrt(m * g2.pi_vec * (1 - g2.pi_vec)))


def test_emission_distribution():
    g = _model(3, 2, seed=1)
    n = 600_000
    x, z = g.gen_sample(n, device="cuda:0")
    assert x.shape == (n, 2) and z.shape == (n, 3) and z.dtype == int and np.array_equal(z.sum(axis=1), np.ones(n, dtype=int))
    cov = np.linalg.inv(g.lambda_mats)
    for k in range(3):
        xs = x[z[:, k] == 1]
        se = np.sqrt(np.diag(cov[k]) / xs.shape[0])
        assert np.all(np.abs(xs.mean(axis=0) - g.mu_vecs[k]) < 5 * se)
        assert np.allclose(np.cov(xs.T), cov[k], rtol=0.03, atol=0.01)


def test_api_behaviour():
    import torch
    x1, z1 = _model(4, 3, seed=2).gen_sample(10_000, device="cuda:0")
    x2, z2 = _model(4, 3, seed=2).gen_sample(10_000, device="cuda:0")
    assert np.array_equal(x1, x2) and np.array_equal(z1, z2)                    # reproducible from the seed
    x3, z3 = _model(4, 3, seed=2).gen_sample(10_000, lengths=[10_000], device="cuda:0")
    assert np.array_equal(x1, x3) and np.array_equal(z1, z3)
    xd, zd = _model(4, 3, seed=2).gen_sample(1000, device="cuda:0", as_numpy=False)
    assert xd.is_cuda and zd.is_cuda and xd.dtype == torch.float64 and zd.dtype == torch.int32
    assert tuple(xd.shape) == (1000, 3) and tuple(zd.shape) == (1000,)
    with pytest.raises(ParameterFormatError):
        hiddenmarkovnormal.GenModel(33, 2).gen_sample(10, device="cuda:0")
    with pytest.raises(ParameterFormatError):
        hiddenmarkovnormal.GenModel(2, 257).gen_sample(10, device="cuda:0")
    xb, _ = hiddenmarkovnormal.GenModel(2, 256, seed=0).gen_sample(300, device="cuda:0")     # the largest D
    assert xb.shape == (300, 256) and np.all(np.isfinite(xb))


def test_fit_recovers_the_transition_matrix():
    K, D, n = 4, 3, 1_000_000
    a = np.array([[0.90, 0.05, 0.03, 0.02], [0.04, 0.85, 0.06, 0.05], [0.10, 0.05, 0.80, 0.05], [0.02, 0.03, 0.05, 0.90]])
    mu = np.array([[-6.0, 0.0, 0.0], [6.0, 0.0, 0.0], [0.0, 6.0, 0.0], [0.0, 0.0, 6.0]])
    g = hiddenmarkovnormal.GenModel(K, D, seed=0, pi_vec=np.full(K, 0.25), a_mat=a, mu_vecs=mu,
                                    lambda_mats=np.tile(np.eye(D), (K, 1, 1)))
    x, _ = g.gen_sample(n, device="cuda:0")
    learn = hiddenmarkovnormal.LearnModel(K, D, seed=1, device="cuda:0")
    with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        learn.update_posterior(x, max_itr=50, num_init=2)
    _, a_hat, mu_hat, _ = learn.estimate_params()
    order = [int(np.argmin(np.linalg.norm(mu_hat - m, axis=1))) for m in mu]
    assert sorted(order) == list(range(K))
    assert np.max(np.abs(a_hat[np.ix_(order, order)] - a)) < 0.02
