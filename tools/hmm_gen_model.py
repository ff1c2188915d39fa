"""numpy model of the three-phase Markov-chain sampler that csrc/bgmm_extras.cu runs on the device (bgmm_hmm_gen_sample).

Design aid + executable specification: tests/test_hmm_genmodel.py checks it against a plain sequential loop on the same
uniforms.  Element i of a chain is z_i = f_i(z_{i-1}): f_i(s) = the inverse CDF of row s of A at u_i, or at a sequence
start the constant map "inverse CDF of pi at u_i".  Maps on {0..K-1} compose associatively, so for chunks of L elements:
phase A composes every chunk's maps (run the chunk from each start state s), phase B sweeps the chunk maps to the state
entering every chunk, and phase C reruns every chunk from that state.  The table is `hiddenmarkovnormal._inverse_cdf_table`.
"""
import numpy as np


def draw(row, u):
    """The first k with u <= row[k] (K - 1 when there is none): the device's inverse-CDF rule."""
    k = int(np.argmax(u <= row))
    return k if u <= row[k] else row.size - 1


def _is_start(n, starts):
    first = np.zeros(n, dtype=bool)
    first[0] = True
    if starts is not None:
        first[np.asarray(starts)] = True
    return first


def sequential(cdf, u, starts=None):
    """The chain drawn one element after another: row 0 of `cdf` at a sequence start, else row 1 + z_{i-1}."""
    first = _is_start(u.size, starts)
    z = np.empty(u.size, dtype=np.int64)
    s = 0
    for i in range(u.size):
        s = draw(cdf[0] if first[i] else cdf[1 + s], u[i])
        z[i] = s
    return z


def phases(cdf, u, starts, L):
    """The same chain from phases A / B / C over chunks of L elements."""
    n, K = u.size, cdf.shape[1]
    first = _is_start(n, starts)
    nch = (n + L - 1) // L

    def run(c, s, out=None):
        for i in range(c * L, min(n, (c + 1) * L)):
            s = draw(cdf[0] if first[i] else cdf[1 + s], u[i])
            if out is not None:
                out[i] = s
        return s

    maps = np.array([[run(c, s) for s in range(K)] for c in range(nch)], dtype=np.int64)    # phase A
    incoming = np.zeros(nch, dtype=np.int64)                                                 # phase B
    for c in range(1, nch):
        incoming[c] = maps[c - 1, incoming[c - 1]]
    z = np.empty(n, dtype=np.int64)                                                          # phase C
    for c in range(nch):
        run(c, incoming[c], z)
    return z
