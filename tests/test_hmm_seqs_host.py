"""CPU: several independent sequences (`lengths=`) of the hidden-Markov model — the multi-sequence oracle against the
reference-pinned single-sequence oracle, `lengths` validation of the public API, and argument checks of the new C entry
points (the library loads without a GPU)."""
import ctypes

import numpy as np
import pytest

from bayesml_b200 import _lib, hiddenmarkovnormal
from bayesml_b200._exceptions import DataFormatError
from oracle.hmm_multiseq_oracle import OracleHMMSeqs, fit_hmm_seqs, seq_starts
from oracle.hmm_vb_oracle import OracleHMM, fit_hmm

# lengths with 1, 2, sequences shorter than one device chunk (32 elements at these sizes) and exact chunk multiples
LENGTH_SETS = [[1, 2, 5, 1, 40], [32, 64, 1, 31, 33], [2, 2, 2, 96, 1, 1, 7]]


def _data(n, d, seed):
    rng = np.random.default_rng(seed)
    return rng.normal(size=(n, d)) + np.repeat(rng.normal(0, 3, size=(n // 4 + 1, d)), 4, axis=0)[:n]


def _fixed(model, seed):
    """Deterministic, non-trivial parameters (the same for every model built with this seed)."""
    K, D = model.K, model.D
    rng = np.random.default_rng(seed)
    model.reset_hn()
    model.hn_eta_vec[:] = rng.uniform(0.5, 3.0, K)
    model.hn_zeta_vecs[:] = rng.uniform(0.5, 3.0, (K, K))
    model.hn_m_vecs[:] = rng.normal(0, 2, (K, D))
    model.q_pi_features()
    model.q_a_features()
    model.q_lambda_features()


@pytest.mark.parametrize("lengths", LENGTH_SETS)
def test_oracle_per_sequence_is_single_sequence_oracle(lengths):
    K, D = 3, 2
    x = _data(sum(lengths), D, 1)
    m = OracleHMMSeqs(K, D)
    m.alloc(x.shape[0])
    m.set_lengths(lengths)
    _fixed(m, 7)
    m.e_step(x)
    ns = np.zeros(K)
    ms = np.zeros((K, K))
    xs = np.zeros((K, D))
    for a, b in m._spans():
        o = OracleHMM(K, D)
        o.alloc(b - a)
        o.init_fb_params()
        _fixed(o, 7)
        o.e_step(x[a:b])
        for name in ("alpha_vecs", "beta_vecs", "cs", "gamma_vecs", "ln_rho"):
            assert np.array_equal(getattr(m, name)[a:b], getattr(o, name)), name
        assert np.array_equal(m.xi_mats[a:b], o.xi_mats)
        ns += o.ns
        ms += o.ms
        xs += o.gamma_vecs.T @ x[a:b]
    assert np.allclose(m.ns, ns, rtol=1e-13)
    assert np.allclose(m.ms, ms, rtol=1e-13)
    assert np.allclose(m.x_bar_vecs * m.ns[:, None], xs, rtol=1e-12)
    assert np.allclose(m.gamma_starts(), m.gamma_vecs[m.starts].sum(axis=0))
    assert np.all(m.xi_mats[m.starts] == 0.0)


@pytest.mark.parametrize("init_type", ["subsampling", "random_responsibility"])
def test_oracle_one_sequence_is_oracle(init_type):
    K, D = 3, 2
    x = _data(60, D, 2)
    a, b = OracleHMM(K, D, seed=5), OracleHMMSeqs(K, D, seed=5)
    ta = fit_hmm(a, x, max_itr=6, num_init=2, tolerance=1e-12, init_type=init_type)
    tb = fit_hmm_seqs(b, x, [60], max_itr=6, num_init=2, tolerance=1e-12, init_type=init_type)
    assert ta.vl_history == tb.vl_history and ta.selected == tb.selected
    for name in OracleHMM.HN + ("gamma_vecs", "alpha_vecs", "beta_vecs", "cs", "ms", "ns", "vl_terms"):
        assert np.array_equal(getattr(a, name), getattr(b, name)), name


def test_oracle_viterbi_per_sequence():
    K, D = 3, 2
    lengths = LENGTH_SETS[2]
    x = _data(sum(lengths), D, 3)
    m = OracleHMMSeqs(K, D)
    m.set_lengths(lengths)
    _fixed(m, 9)
    z = m.estimate_latent_vars(x)
    for a, b in m._spans():
        o = OracleHMM(K, D)
        _fixed(o, 9)
        zo = o.estimate_latent_vars(x[a:b])
        assert np.array_equal(z[a:b], zo)
        assert np.array_equal(m.omega_vecs[a:b], o.omega_vecs) and np.array_equal(m.phi_vecs[a:b], o.phi_vecs)


def test_random_responsibility_rule_matches_oracle():
    """The public class's host initialisation draws the same stream and applies the same rule as the oracle."""
    K, D = 3, 2
    lengths = [1, 4, 1, 2, 9]
    x = _data(sum(lengths), D, 4)
    model = hiddenmarkovnormal.LearnModel(K, D, seed=11)
    gamma, ms = model._init_random_responsibility(x.shape[0], seq_starts(lengths))
    o = OracleHMMSeqs(K, D, seed=11)
    o.alloc(x.shape[0])
    o.set_lengths(lengths)
    o.init_random_responsibility(x)
    assert np.array_equal(gamma, o.gamma_vecs) and np.array_equal(ms, o.ms)
    assert np.all(o.xi_mats[o.starts] == 0.0)
    assert np.allclose(gamma.sum(axis=1), 1.0)


@pytest.mark.parametrize("bad", [[10, 9], [0, 20], [-1, 21], [2.5, 17.5], [[5, 15]], [], "20"])
def test_lengths_validation(bad):
    model = hiddenmarkovnormal.LearnModel(2, 2)
    x = np.zeros((20, 2)) + np.arange(20)[:, None]
    with pytest.raises(DataFormatError):
        model.update_posterior(x, lengths=bad)
    with pytest.raises(DataFormatError):
        model.estimate_latent_vars(x, lengths=bad)


def test_lengths_starts():
    assert hiddenmarkovnormal.LearnModel._seq_starts(None, 5) is None
    assert hiddenmarkovnormal.LearnModel._seq_starts([5], 5) is None
    assert hiddenmarkovnormal.LearnModel._seq_starts(np.array([2, 3]), 5).tolist() == [0, 2]


def test_seq_entry_points_reject_bad_arguments(lib_built):
    lib = _lib.load()
    starts = np.array([0, 3, 4], dtype=np.int64)
    p = starts.ctypes.data
    assert lib.bgmm_hmm_seq_plan(10, 0, p, None, 0) == -1 and b"bgmm_hmm_seq_plan" in lib.bgmm_last_error()
    assert lib.bgmm_hmm_seq_plan(10, 3, None, None, 0) == -1
    assert lib.bgmm_hmm_seq_plan(4, 3, p, None, 0) == -1                          # a start at or past n
    bad = np.array([0, 3, 3], dtype=np.int64)
    assert lib.bgmm_hmm_seq_plan(10, 3, bad.ctypes.data, None, 0) == -1           # an empty sequence
    size = lib.bgmm_hmm_seq_plan(10, 3, p, None, 0)
    assert size == 8 + 3 * 3 + 1 + 3
    plan = np.zeros(size, dtype=np.int64)
    assert lib.bgmm_hmm_seq_plan(10, 3, p, plan.ctypes.data, size) == size
    assert plan[:6].tolist() == [10, 3, 32, 3, 0, 0]
    assert plan[8:12].tolist() == [0, 3, 4, 10] and plan[-3:].tolist() == [0, 3, 4]
    assert lib.bgmm_hmm_seq_workspace_doubles(3, 10, 0) == 0 and lib.bgmm_hmm_seq_workspace_doubles(40, 10, 2) == 0
    assert lib.bgmm_hmm_seq_workspace_doubles(3, 10, 3) >= lib.bgmm_hmm_scan_workspace_doubles(3, 10)
    nul = [None] * 9
    assert lib.bgmm_hmm_pass_seqs(None, 10, 4, 2, *nul, 0, 0, None, None, None) == -1
    assert lib.bgmm_hmm_pass_seqs(None, 11, 4, 2, *nul, 0, 0, plan.ctypes.data, plan.ctypes.data, None) == -1   # n mismatch
    assert lib.bgmm_hmm_viterbi_seqs(10, 4, *([None] * 6), None, 0, None) == -1
    assert lib.bgmm_hmm_viterbi_seqs(10, 4, *([ctypes.c_void_p(8)] * 6), p, 0, None) == -1
    assert lib.bgmm_hmm_viterbi_seqs(10, 4, *([ctypes.c_void_p(8)] * 6), None, 3, None) == -1


def test_long_sequences_get_the_two_level_sweep(lib_built):
    lib = _lib.load()
    n = 400_000
    starts = np.array([0, 10, 11, 380_000], dtype=np.int64)
    size = lib.bgmm_hmm_seq_plan(n, 4, starts.ctypes.data, None, 0)
    plan = np.zeros(size, dtype=np.int64)
    lib.bgmm_hmm_seq_plan(n, 4, starts.ctypes.data, plan.ctypes.data, size)
    L, nch, nshort, nlong = plan[2], plan[3], plan[4], plan[5]
    assert L == 104 and nlong == 1 and nshort == 1
    coff = plan[8:8 + nch + 1]
    assert coff[0] == 0 and coff[-1] == n and np.all(np.diff(coff) >= 1) and np.all(np.diff(coff) <= L)
    sst = plan[8 + nch + 1:8 + 2 * nch + 1]
    assert set(sst.tolist()) == set(starts.tolist())
    segs = plan[8 + 3 * nch + 1:8 + 3 * nch + 1 + 2 * (nshort + nlong)].reshape(-1, 2)
    assert segs[0, 1] == -(-20_000 // L) and segs[1, 1] == -(-(380_000 - 11) // L)      # short one first, then the long one
