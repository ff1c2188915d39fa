"""CPU oracle: the VB hidden-Markov fit of oracle/hmm_vb_oracle.py over several independent sequences that share one
posterior (`lengths=` of `hiddenmarkovnormal.LearnModel.update_posterior` / `estimate_latent_vars`).

TEST INFRASTRUCTURE — NOT PRODUCT CODE, like oracle/hmm_vb_oracle.py.

The reference has no multi-sequence mode, so this module is the specification.  All of the model's statistics are sums
over elements, so only three things differ from one sequence:
  - the recursions restart at every sequence start: forward from pi~, backward from ones at every sequence end;
  - xi is zero at every sequence start, so ms counts only the transitions inside a sequence;
  - gamma_0 in E ln p(z) and E ln q(z) becomes the sum over sequence starts of gamma there.
Per sequence, the forward / backward / gamma / xi expressions are OracleHMM's, applied to that sequence's rows, so with
fixed parameters they are bit-identical to `OracleHMM.e_step` on that sequence alone; with one sequence (lengths None or
[n]) every method is OracleHMM's own.
"""
from __future__ import annotations

import numpy as np

from oracle.hmm_vb_oracle import OracleHMM, fit_hmm

__all__ = ["OracleHMMSeqs", "fit_hmm_seqs", "seq_starts"]


def seq_starts(lengths):
    """First rows of the sequences (int64), or None for one sequence."""
    if lengths is None or len(lengths) == 1:
        return None
    lengths = np.asarray(lengths, dtype=np.int64)
    starts = np.zeros(lengths.size, dtype=np.int64)
    np.cumsum(lengths[:-1], out=starts[1:])
    return starts


class OracleHMMSeqs(OracleHMM):
    """OracleHMM over the sequences of `set_lengths` (concatenated rows)."""

    starts = None

    def set_lengths(self, lengths):
        self.starts = seq_starts(lengths)

    def _spans(self):
        if self.starts is None:
            return [(0, self.length)]
        ends = np.append(self.starts[1:], self.length)
        return list(zip(self.starts.tolist(), ends.tolist()))

    def forward(self):
        if self.starts is None:
            return super().forward()
        for a, b in self._spans():
            al, rho, cs = self.alpha_vecs[a:b], self.rho[a:b], self.cs[a:b]
            al[0] = rho[0] * self.pi_tilde_vec
            cs[0] = al[0].sum()
            al[0] /= cs[0]
            for i in range(1, b - a):
                al[i] = rho[i] * (al[i - 1] @ self.a_tilde_mat)
                cs[i] = al[i].sum()
                al[i] /= cs[i]

    def backward(self):
        if self.starts is None:
            return super().backward()
        for a, b in self._spans():
            be, rho, cs = self.beta_vecs[a:b], self.rho[a:b], self.cs[a:b]
            be[b - a - 1] = 1.0
            for i in range(b - a - 2, -1, -1):
                be[i] = self.a_tilde_mat @ (rho[i + 1] * be[i + 1])
                be[i] /= cs[i + 1]

    def e_step(self, x):
        if self.starts is None:
            return super().e_step(x)
        self.calc_rho(x)
        self.forward()
        self.backward()
        self.gamma_vecs[:] = self.alpha_vecs * self.beta_vecs
        self.xi_mats[1:, :, :] = (self.alpha_vecs[:-1, :, np.newaxis] * self.rho[1:, np.newaxis, :]
                                  * self.a_tilde_mat[np.newaxis, :, :] * self.beta_vecs[1:, np.newaxis, :])
        self.xi_mats[1:, :, :] /= self.cs[1:, np.newaxis, np.newaxis]
        self.xi_mats[self.starts] = 0.0
        self.calc_n_m_x_bar_s(x)

    def gamma_starts(self):
        """G0: gamma summed over the sequence starts."""
        if self.starts is None:
            return self.gamma_vecs[0]
        return self.gamma_vecs[self.starts].sum(axis=0)

    def calc_vl(self):
        super().calc_vl()
        if self.starts is None:
            return
        g0 = self.gamma_starts()
        p_x, _, p_pi, p_a, p_mu_lambda, _, q_pi, q_a, q_mu_lambda = self.vl_terms
        p_z = (g0 * self.ln_pi_tilde_vec).sum() + (self.ms * self.ln_a_tilde_mat).sum()
        q_z = (-(self.gamma_vecs * self.ln_rho).sum()
               - (self.ms * (self.ln_a_tilde_mat - self.ln_a_tilde_mat.max())).sum()
               - (g0 * (self.ln_pi_tilde_vec - self.ln_pi_tilde_vec.max())).sum()
               + np.log(self.cs).sum())
        self.vl_terms[1], self.vl_terms[5] = p_z, q_z
        self.vl = (p_x + p_z + p_pi + p_a + p_mu_lambda + q_z + q_pi + q_a + q_mu_lambda)

    def init_random_responsibility(self, x):
        if self.starts is None:
            return super().init_random_responsibility(x)
        K, n = self.K, self.length
        xi = self.rng.dirichlet(np.ones(K ** 2), n).reshape(n, K, K)
        self.gamma_vecs[:] = xi.sum(axis=1)
        ends = np.append(self.starts[1:], n)
        single = ends - self.starts == 1
        longer = self.starts[~single]
        self.gamma_vecs[longer] = xi[longer + 1].sum(axis=2)
        self.gamma_vecs[self.starts[single]] = xi[self.starts[single]].sum(axis=2)
        xi[self.starts] = 0.0
        self.xi_mats[:] = xi
        self.calc_n_m_x_bar_s(x)

    def estimate_latent_vars(self, x, loss="0-1", viterbi=True):
        if self.starts is None:
            return super().estimate_latent_vars(x, loss=loss, viterbi=viterbi)
        K = self.K
        x = x.reshape(-1, self.D)
        n = x.shape[0]
        self.length = n
        if not viterbi:
            return super().estimate_latent_vars(x, loss=loss, viterbi=False)     # e_step is this class's
        if loss != "0-1":
            raise ValueError(loss)
        self.ln_rho = np.zeros([n, K])
        self.rho = np.ones([n, K])
        self.calc_rho(x)
        z_hat = np.zeros([n, K], dtype=int)
        omega = np.zeros([n, K])
        phi = np.zeros([n, K], dtype=int)
        for a, b in self._spans():
            om, ph, lr = omega[a:b], phi[a:b], self.ln_rho[a:b]
            om[0] = lr[0] + self.ln_pi_tilde_vec
            for i in range(1, b - a):
                om[i] = lr[i] + np.max(self.ln_a_tilde_mat + om[i - 1, :, np.newaxis], axis=0)
                ph[i] = np.argmax(self.ln_a_tilde_mat + om[i - 1, :, np.newaxis], axis=0)
            k = np.argmax(om[-1])
            z_hat[b - 1, k] = 1
            for i in range(b - a - 2, -1, -1):
                k = ph[i + 1, k]
                z_hat[a + i, k] = 1
        self.omega_vecs, self.phi_vecs = omega, phi
        return z_hat


def fit_hmm_seqs(model: OracleHMMSeqs, x, lengths, **kw):
    """`fit_hmm` (update_posterior without the prints) over the sequences of `lengths`."""
    model.set_lengths(lengths)
    return fit_hmm(model, x, **kw)
