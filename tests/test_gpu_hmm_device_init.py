"""`hiddenmarkovnormal.LearnModel(device_init=True)`: the 'random_responsibility' initial state drawn on the device
(bgmm_hmm_init_random) against its numpy model (tools/hmm_init_model.py: Philox4x32-10 in uint64 arithmetic with the
counter mapping of include/bgmm.h, then the rules of `_init_random_responsibility`), the fit from that state against the
CPU oracle from the same state, the distribution of the draw, its determinism, and the class end to end.

The CPU tests (unmarked) check the Philox model against the published known-answer vectors, the model's rules against
the host rule, and the argument checks of the C entry point."""
import contextlib
import inspect
import io
import warnings

import numpy as np
import pytest

from tools import hmm_init_model as model

RTOL = 1e-9


def _close(a, b, rtol=RTOL, scale=None):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    scale = np.max(np.abs(b)) if scale is None else scale
    return np.allclose(a, b, rtol=rtol, atol=rtol * 1e-4 * max(scale, 1e-300))


def _lengths(kind, seed):
    """The `lengths` kinds of tests/test_gpu_hmm_seqs.py."""
    rng = np.random.default_rng(seed)
    if kind == "ones":
        return [1] * 300 + [2, 3, 40, 1, 64, 1]
    if kind == "short":
        return rng.integers(1, 30, size=200).tolist()
    if kind == "mixed":
        return rng.integers(1, 400, size=20).tolist() + [32, 64, 1, 2, 96]
    if kind == "long":
        return rng.integers(1, 50, size=100).tolist() + [300_000] + rng.integers(1, 50, size=100).tolist()
    raise ValueError(kind)


def _starts(lengths):
    from oracle.hmm_multiseq_oracle import seq_starts
    return None if lengths is None else seq_starts(lengths)


# ---------------------------------------------------------------------------------------------------------------- CPU

def test_philox_model_known_answers():
    """Random123's known-answer vectors for philox4x32-10."""
    cases = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
             ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
             ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
              (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for ctr, key, want in cases:
        got = model.philox4x32_10(*[np.array([c], dtype=np.uint64) for c in ctr], *key)
        assert [int(w[0]) for w in got] == list(want)


class _FixedDirichlet:
    """Stands in for `LearnModel.rng`: `dirichlet` returns the given draw."""

    def __init__(self, flat):
        self.flat = flat

    def dirichlet(self, alpha, size=None):
        assert size is None or size == self.flat.shape[0]
        return self.flat.copy()


@pytest.mark.parametrize("K,n,kind", [(3, 1, None), (1, 40, None), (3, 50, None), (4, 700, "ones"), (5, 900, "mixed"),
                                      (2, 600, "short")])
def test_model_rules_are_the_host_rules(K, n, kind):
    """tools/hmm_init_model.py applies `_init_random_responsibility`'s rules: fed the model's xi, the host rule gives the
    model's gamma and sum xi."""
    from bayesml_b200 import hiddenmarkovnormal
    lengths = None if kind is None else _lengths(kind, 3)
    n = n if lengths is None else sum(lengths)
    starts = _starts(lengths)
    gamma, ms, g0, _ = model.init_state(n, K, 77, starts)
    m = hiddenmarkovnormal.LearnModel(K, 2, seed=0)
    if n == 1:
        t = model.draw([0], K, 77)[0, 0]
        m.rng = _FixedDirichlet(t / t.sum())
    else:
        m.rng = _FixedDirichlet(model.xi(np.arange(n), K, 77).reshape(n, K * K))
    g_host, ms_host = m._init_random_responsibility(n, starts)
    assert np.allclose(g_host, gamma, rtol=1e-14, atol=0) and np.allclose(ms_host, ms, rtol=1e-13, atol=0)
    assert np.allclose(g0, g_host[0 if starts is None else starts].reshape(-1, K).sum(axis=0), rtol=1e-14, atol=0)


def test_device_init_is_keyword_only():
    from bayesml_b200 import hiddenmarkovnormal
    p = inspect.signature(hiddenmarkovnormal.LearnModel.__init__).parameters["device_init"]
    assert p.kind == inspect.Parameter.KEYWORD_ONLY and p.default is False


def test_rejected_arguments_launch_nothing(lib_built):
    from bayesml_b200 import _lib
    lib = _lib.load()
    buf = np.zeros(64)
    ptr = buf.ctypes.data                       # never dereferenced: every call below fails its host checks
    good = np.array([0, 3, 7], dtype=np.int64)
    n0 = lib.bgmm_launch_count()
    for n, K, hs, ds, ns, g, h, w in [
            (10, 0, None, None, 1, ptr, ptr, ptr), (10, 33, None, None, 1, ptr, ptr, ptr),
            (0, 3, None, None, 1, ptr, ptr, ptr), (10, 3, None, None, 0, ptr, ptr, ptr),
            (10, 3, None, None, 1, None, ptr, ptr), (10, 3, None, None, 1, ptr, None, ptr),
            (10, 3, None, None, 1, ptr, ptr, None), (10, 3, good.ctypes.data, None, 3, ptr, ptr, ptr),
            (10, 3, None, ptr, 3, ptr, ptr, ptr), (2, 3, good.ctypes.data, ptr, 3, ptr, ptr, ptr)]:
        assert lib.bgmm_hmm_init_random(n, K, 1, hs, ds, ns, g, h, w, None) == -1, (n, K, ns)
    for bad in ([1, 3, 7], [0, 3, 3], [0, 7, 3], [0, 3, 10]):
        arr = np.array(bad, dtype=np.int64)
        assert lib.bgmm_hmm_init_random(10, 3, 1, arr.ctypes.data, ptr, 3, ptr, ptr, ptr, None) == -1, bad
        assert "seq_starts" in lib.bgmm_last_error().decode()
    assert lib.bgmm_launch_count() == n0
    assert lib.bgmm_hmm_init_random_workspace_doubles(33, 10) == 0 and lib.bgmm_hmm_init_random_workspace_doubles(3, 0) == 0


# ---------------------------------------------------------------------------------------------------------------- GPU

def _engine(K, D, x, lengths):
    from bayesml_b200.engine import HMMEngine
    eng = HMMEngine(K, D)
    eng.load_data(x)
    eng.set_sequences(_starts(lengths))
    return eng


def _device_state(eng, seed):
    """(gamma, ms, g0, sc) of one device draw."""
    K = eng.K
    eng.draw_random_init(seed)
    h = eng.hst.cpu().numpy()
    o = eng.hoff
    return (eng.gamma_buf.cpu().numpy(), h[o["ms"]:o["ms"] + K * K].reshape(K, K), h[o["g0"]:o["g0"] + K].copy(),
            h[o["sc"]:o["sc"] + 8].copy())


def _check_against_model(K, n, lengths, seed):
    eng = _engine(K, 1, np.zeros((n, 1)), lengths)
    eng.hst.fill_(np.nan)
    gamma, ms, g0, sc = _device_state(eng, seed)
    mg, mms, mg0, _ = model.init_state(n, K, seed, _starts(lengths))
    assert np.allclose(gamma, mg, rtol=1e-14, atol=0), np.max(np.abs(gamma - mg) / mg)
    assert np.allclose(ms, mms, rtol=1e-13, atol=0), np.max(np.abs(ms - mms) / np.maximum(mms, 1e-300))
    assert np.allclose(g0, mg0, rtol=1e-13, atol=0)
    assert np.all(sc == 0.0)
    assert np.allclose(gamma.sum(axis=1), 1.0, rtol=0, atol=1e-13)
    assert abs(ms.sum() - (n - (1 if lengths is None else len(lengths)))) < 1e-9 * n


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 1000, 50_000])
@pytest.mark.parametrize("K", [1, 2, 3, 8, 17, 32])
def test_draw_matches_the_numpy_model_one_sequence(K, n, lib_built):
    _check_against_model(K, n, None, 1234 + K + n)


# the numpy model of the 3e5-element "long" kind takes minutes at K > 8
SEQ_CASES = [(kind, K) for kind in ("ones", "short", "mixed", "long") for K in (1, 2, 3, 8, 17, 32)
             if kind != "long" or K <= 8]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,K", SEQ_CASES)
def test_draw_matches_the_numpy_model_sequences(kind, K, lib_built):
    lengths = _lengths(kind, K * 100 + 1)
    _check_against_model(K, sum(lengths), lengths, 2 ** 63 - 5 - K)


def _data(n, d, k, seed):
    rng = np.random.default_rng(seed)
    mu = rng.normal(0.0, 3.0, size=(k, d))
    z = np.repeat(rng.integers(0, k, size=n // 3 + 1), 3)[:n]
    return mu[z] + rng.normal(size=(n, d))


FIT_CASES = [  # K, D, n or lengths kind, window cap (None: default; "0": the basis + sweep path)
    (3, 2, 3000, None), (3, 2, 3000, "0"), (4, 3, 1, None), (2, 1, 2, "0"), (8, 3, "mixed", None), (8, 3, "mixed", "0"),
    (2, 3, "ones", "0"), (17, 2, "short", None), (32, 4, "mixed", "0"), (5, 2, 40_000, None),
]


@pytest.mark.gpu
@pytest.mark.parametrize("K,D,size,cap", FIT_CASES)
def test_fit_equals_the_oracle_from_the_same_state(K, D, size, cap, monkeypatch, lib_built):
    """Every ELBO, the 9 terms, hn_* and the statistics of the device fit from the device-drawn state equal the oracle's
    from the model's state (the same numbers)."""
    from oracle.hmm_multiseq_oracle import OracleHMMSeqs
    if cap is not None:
        monkeypatch.setenv("BGMM_HMM_WINDOW_CAP", cap)
    lengths = _lengths(size, K + D) if isinstance(size, str) else None
    n = sum(lengths) if lengths is not None else size
    x = _data(n, D, K, K * D)
    seed = 99 + K
    o = OracleHMMSeqs(K, D)
    o.alloc(n)
    o.set_lengths(lengths)
    o.init_fb_params()
    o.reset_hn()
    gamma, _, _, xi = model.init_state(n, K, seed, _starts(lengths), want_xi=True)
    o.gamma_vecs[:] = gamma
    o.xi_mats[:] = xi
    o.calc_n_m_x_bar_s(x)
    o.calc_vl()
    max_itr = 5
    ref = [float(o.vl)]
    for _ in range(max_itr):
        o.iterate(x)
        ref.append(float(o.vl))
    eng = _engine(K, D, x, lengths)
    eng.set_hmm_prior(o.h0_eta_vec, o.h0_zeta_vecs, o.h0_m_vecs, o.h0_kappas, o.h0_nus, o.h0_w_mats_inv, o.ln_b_h0_w_nus,
                      o.ln_c_h0_eta_vec, o.ln_c_h0_zeta_vecs_sum)
    eng.set_hmm_params(o.h0_eta_vec, o.h0_zeta_vecs, o.h0_m_vecs, o.h0_kappas, o.h0_nus, o.h0_w_mats_inv)
    hist, _ = eng.run(max_itr, 0.0, init=seed)
    assert _close(hist, ref), np.max(np.abs(np.asarray(hist) - ref) / np.abs(ref))
    p = eng.fetch_params()
    if cap == "0" and n > 1:
        assert p["window"] == 0
    for mine, name in (("alpha", "hn_eta_vec"), ("zeta", "hn_zeta_vecs"), ("m", "hn_m_vecs"), ("kappa", "hn_kappas"),
                       ("nu", "hn_nus"), ("winv", "hn_w_mats_inv"), ("ns", "ns"), ("ms", "ms"), ("x_bar", "x_bar_vecs")):
        assert _close(p[mine], getattr(o, name)), mine
    assert _close(p["s_mats"], o.s_mats, rtol=1e-8)
    assert _close(p["gamma0"], o.gamma_starts())
    t, vx = p["vl_terms"], p["vlx"]
    mine_terms = np.array([t[0], vx[0], t[2], vx[1], t[3], vx[2], t[5], vx[3], t[6]])
    assert np.allclose(mine_terms, o.vl_terms, rtol=RTOL, atol=RTOL * np.max(np.abs(o.vl_terms)))


@pytest.mark.gpu
def test_distribution(lib_built):
    """K = 3: xi entries ~ Beta(1, K^2 - 1) (the model's draw, which the device equals above), gamma inside a sequence and at
    sequence starts ~ Beta(K, K^2 - K) (sums of K entries of a Dirichlet(1_{K^2})), gamma_0 of n = 1 ~ Beta(1, K - 1)."""
    from scipy import stats
    K, n = 3, 400_000
    xi = model.xi(np.arange(n), K, 5)
    for j in range(K):
        for k in range(K):
            assert stats.kstest(xi[:, j, k], stats.beta(1, K * K - 1).cdf).pvalue > 1e-4, (j, k)
    rng = np.random.default_rng(8)
    lengths = rng.integers(1, 5, size=n // 2)
    lengths = lengths[np.cumsum(lengths) <= n].tolist()
    if sum(lengths) < n:
        lengths.append(n - sum(lengths))
    starts = _starts(lengths)
    gamma = _device_state(_engine(K, 1, np.zeros((n, 1)), lengths), 6)[0]
    inner = np.ones(n, dtype=bool)
    inner[starts] = False
    assert inner.sum() > 1e5 and starts.size > 1e5
    for k in range(K):
        assert stats.kstest(gamma[inner, k], stats.beta(K, K * K - K).cdf).pvalue > 1e-4, k
        assert stats.kstest(gamma[starts, k], stats.beta(K, K * K - K).cdf).pvalue > 1e-4, k
    eng = _engine(K, 1, np.zeros((1, 1)), None)
    g1 = np.array([_device_state(eng, s)[0][0] for s in range(3000)])
    for k in range(K):
        assert stats.kstest(g1[:, k], stats.beta(1, K - 1).cdf).pvalue > 1e-4, k


@pytest.mark.gpu
def test_determinism_and_split_independence(lib_built):
    K, n = 5, 200_000
    lengths = _lengths("mixed", 4)
    lengths.append(n - sum(lengths))
    starts = _starts(lengths)
    one = _engine(K, 1, np.zeros((n, 1)), None)
    split = _engine(K, 1, np.zeros((n, 1)), lengths)
    a = _device_state(one, 11)
    b = _device_state(one, 11)
    for u, v in zip(a, b):
        assert np.array_equal(u, v)
    c = _device_state(one, 12)
    assert not np.array_equal(a[0], c[0]) and not np.array_equal(a[1], c[1])
    s1, s2 = _device_state(split, 11), _device_state(split, 11)
    for u, v in zip(s1, s2):
        assert np.array_equal(u, v)
    inner = np.ones(n, dtype=bool)
    inner[starts] = False
    assert np.array_equal(a[0][inner], s1[0][inner])
    assert not np.array_equal(a[0][starts[1:]], s1[0][starts[1:]])


def _fit(m, x, **kw):
    out = io.StringIO()
    with contextlib.redirect_stdout(out), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m.update_posterior(x, **kw)
    return out.getvalue()


class _OracleDeviceInit:
    """Mixed into the oracle: 'random_responsibility' takes one integer from the oracle's rng per restart and loads the
    model's state for that seed, as LearnModel(device_init=True) does."""

    def init_random_responsibility(self, x):
        seed = int(self.rng.integers(0, 2 ** 63 - 1))
        gamma, _, _, xi = model.init_state(self.length, self.K, seed, self.starts, want_xi=True)
        self.gamma_vecs[:] = gamma
        self.xi_mats[:] = xi
        self.calc_n_m_x_bar_s(x)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [None, "mixed"])
def test_update_posterior_end_to_end(kind, lib_built):
    from bayesml_b200 import hiddenmarkovnormal
    from oracle.hmm_multiseq_oracle import OracleHMMSeqs, fit_hmm_seqs
    K, D, s = 3, 2, 21
    lengths = None if kind is None else _lengths(kind, 7)
    x = _data(4000 if lengths is None else sum(lengths), D, K, 8)
    kw = dict(max_itr=20, num_init=3, tolerance=1e-6, init_type="random_responsibility")
    m = hiddenmarkovnormal.LearnModel(K, D, seed=s, device_init=True)
    text = _fit(m, x, lengths=lengths, **kw)
    rng = np.random.default_rng(s)
    for _ in range(kw["num_init"]):
        rng.integers(0, 2 ** 63 - 1)
    assert m.rng.bit_generator.state == rng.bit_generator.state          # one integer per restart, nothing else
    o = type("Oracle", (_OracleDeviceInit, OracleHMMSeqs), {})(K, D, seed=s)
    tr = fit_hmm_seqs(o, x, lengths, **kw)
    lines = text.split("\n")[:-1]
    assert len(lines) == kw["num_init"]
    best = [i for i in range(len(tr.vl_history)) if i == 0 or tr.vl_history[i][-1] > max(h[-1] for h in tr.vl_history[:i])]
    assert [i for i, ln in enumerate(lines) if ln.endswith("*")] == best and best[-1] == tr.selected
    assert text.count("(converged)") == sum(tr.converged)
    for f in ("hn_eta_vec", "hn_zeta_vecs", "hn_m_vecs", "hn_kappas", "hn_nus", "hn_w_mats", "ns", "ms", "x_bar_vecs"):
        assert _close(getattr(m, f), getattr(o, f), rtol=1e-8), f
    assert _close(m.gamma_vecs, o.gamma_vecs, rtol=1e-8)


@pytest.mark.gpu
@pytest.mark.parametrize("lengths", [None, [700, 1, 299]])
def test_subsampling_is_unchanged(lengths, lib_built):
    from bayesml_b200 import hiddenmarkovnormal
    x = _data(1000, 2, 3, 3)
    res = []
    for flag in (False, True):
        m = hiddenmarkovnormal.LearnModel(3, 2, seed=4, device_init=flag)
        res.append((_fit(m, x, max_itr=10, num_init=2, lengths=lengths), m))
    assert res[0][0] == res[1][0]
    for f in ("hn_eta_vec", "hn_zeta_vecs", "hn_m_vecs", "hn_kappas", "hn_nus", "hn_w_mats", "ns", "ms", "gamma_vecs"):
        assert np.array_equal(getattr(res[0][1], f), getattr(res[1][1], f)), f
    assert res[0][1].rng.bit_generator.state == res[1][1].rng.bit_generator.state


@pytest.mark.gpu
def test_pred_and_update_draws_one_element_on_the_device(lib_built):
    """pred_and_update learns from one element with 'random_responsibility' (the n = 1 rule) through update_posterior."""
    from bayesml_b200 import hiddenmarkovnormal
    x = _data(500, 2, 3, 5)
    m = hiddenmarkovnormal.LearnModel(3, 2, seed=6, device_init=True)
    _fit(m, x, max_itr=5, num_init=1, init_type="random_responsibility")
    state = m.rng.bit_generator.state
    with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m.pred_and_update(x[0], max_itr=3, num_init=2)
    rng = np.random.default_rng()
    rng.bit_generator.state = state
    for _ in range(2):
        rng.integers(0, 2 ** 63 - 1)
    assert m.rng.bit_generator.state == rng.bit_generator.state
    assert np.all(np.isfinite(m.hn_eta_vec)) and m.gamma_vecs.shape == (1, 3)


_LAUNCH_CHECK = """
import json, sys
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
from test_launch_count import _counted, _hmm
out = []
for K in (3, 32):
    for lengths in ([20000], [10, 500, 1, 8000, 30, 3000]):
        eng = _hmm(K, 2, lengths)
        kernels, delta = _counted([eng], lambda: eng.draw_random_init(7))
        out.append([K, len(lengths), delta, kernels])
print(json.dumps(out))
"""


@pytest.mark.gpu
def test_every_launch_is_counted(lib_built):
    """The draw passes tests/test_launch_count.py's `_counted` check (the library's launch count equals the libbgmm
    kernels torch.profiler records) for one sequence and several, at K = 3 and 32.  It runs in a child process: profiler
    sessions opened in the pytest process before tests/test_launch_count.py runs can make the first session of that
    module record fewer kernels than were launched, so this file leaves the pytest process unprofiled."""
    import json
    import os
    import subprocess
    import sys
    from conftest import ROOT
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", _LAUNCH_CHECK, ROOT]
    res = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT, env=dict(os.environ), timeout=600)
    assert res.returncode == 0, res.stderr[-4000:]
    cases = json.loads(res.stdout.strip().splitlines()[-1])
    assert len(cases) == 4
    for K, n_seqs, delta, kernels in cases:
        assert delta == len(kernels) == 2, (K, n_seqs, kernels)
