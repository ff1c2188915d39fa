"""CPU: the chunked scan over several sequences (tools/hmm_scan_model.py, the algorithm bgmm_hmm_pass_seqs runs: chunks
aligned to sequence starts, segmented sweep, windows clamped to their sequence) equals the multi-sequence oracle."""
import numpy as np
import pytest

from oracle.hmm_multiseq_oracle import OracleHMMSeqs
from tools.hmm_scan_model import (backward_boundaries_window_seqs, backward_seqs, forward_boundaries_window_seqs,
                                  forward_seqs, seq_chunks, window)

# lengths with 1, 2, sequences shorter than one chunk, exact chunk multiples and sequences of several chunks
LENGTH_SETS = [([1, 2, 5, 1, 40], 8), ([32, 64, 1, 31, 33], 16), ([2, 2, 2, 96, 1, 1, 7, 50], 16), ([3], 8)]


def _model(lengths, K, spread, seed):
    rng = np.random.default_rng(seed)
    n, D = sum(lengths), 2
    m = OracleHMMSeqs(K, D, seed=0)
    m.set_lengths(lengths)
    x = rng.normal(size=(n, D)) * 2.0
    m.alloc(n)
    m.init_fb_params()
    m.hn_m_vecs[:] = rng.normal(size=(K, D)) * 2.0
    m.hn_zeta_vecs[:] = rng.uniform(1.0, 1.0 + spread, size=(K, K))
    m.hn_eta_vec[:] = rng.uniform(0.2, 5.0, size=K)
    m.q_pi_features(); m.q_a_features(); m.q_lambda_features()
    m.e_step(x)
    starts = m.starts if m.starts is not None else np.zeros(1, dtype=np.int64)
    return m, starts


@pytest.mark.parametrize("lengths,L", LENGTH_SETS)
@pytest.mark.parametrize("K", [1, 3, 5])
def test_segmented_scan_matches_oracle(lengths, L, K):
    m, starts = _model(lengths, K, 4.0, len(lengths) + K)
    chunks = seq_chunks(list(starts), m.length, L)
    assert all(s0 <= i0 < i1 <= s1 and i1 - i0 <= L for i0, i1, s0, s1 in chunks)
    alpha, cs, _ = forward_seqs(m.rho, m.pi_tilde_vec, m.a_tilde_mat, chunks)
    assert np.allclose(alpha, m.alpha_vecs, rtol=1e-11, atol=1e-300)
    assert np.allclose(cs, m.cs, rtol=1e-11)
    beta, gamma, S, G0, _ = backward_seqs(m.rho, m.cs, m.alpha_vecs, m.a_tilde_mat, chunks)
    assert np.allclose(beta, m.beta_vecs, rtol=1e-10, atol=1e-300)
    assert np.allclose(gamma, m.gamma_vecs, rtol=1e-10, atol=1e-300)
    assert np.allclose(m.a_tilde_mat * S, m.ms, rtol=1e-10, atol=1e-13)
    assert np.allclose(G0, m.gamma_starts(), rtol=1e-12)


@pytest.mark.parametrize("lengths,L", [([150, 3, 200, 90, 1, 160], 16), ([64] * 8, 16)])
def test_windows_clamped_to_sequences(lengths, L):
    """In the mixing regime the window boundary vectors equal the exact ones; a window that would reach across a sequence
    start (end) starts from pi~ (ones) there instead."""
    K = 4
    m, starts = _model(lengths, K, 1.0, 7)
    W = window(m.a_tilde_mat, 10 ** 6)
    assert 8 <= W and W > L                            # windows longer than a chunk: they would cross sequence starts
    chunks = seq_chunks(list(starts), m.length, L)
    v = forward_boundaries_window_seqs(m.rho, m.pi_tilde_vec, m.a_tilde_mat, chunks, W)
    w = backward_boundaries_window_seqs(m.rho, m.cs, m.a_tilde_mat, chunks, W)
    for c, (i0, i1, s0, s1) in enumerate(chunks):
        if i0 > s0:
            assert np.allclose(v[c], m.alpha_vecs[i0 - 1], rtol=1e-13, atol=1e-300), c
        assert np.allclose(w[c], m.beta_vecs[i1 - 1], rtol=1e-12, atol=1e-300), c
    # the same boundary vectors come out of the segmented sweep
    _, _, v_exact = forward_seqs(m.rho, m.pi_tilde_vec, m.a_tilde_mat, chunks)
    _, _, _, _, w_exact = backward_seqs(m.rho, m.cs, m.alpha_vecs, m.a_tilde_mat, chunks)
    assert np.allclose(v, v_exact, rtol=1e-12, atol=1e-300) and np.allclose(w, w_exact, rtol=1e-12, atol=1e-300)
