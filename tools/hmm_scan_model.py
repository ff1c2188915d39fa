"""numpy model of the chunked (three-phase) forward-backward scan that csrc/bgmm_hmm.cu runs on the device.

Design aid + executable specification: tests/test_hmm_scan_model.py checks it against the sequential recursions of
the oracle.  Phase A: per chunk, the recursion is run from the K unit vectors (normalised, log scale kept) -> chunk
transfer matrix.  Phase B: one sequential sweep over chunk matrices -> the vector at every chunk boundary.
Phase C: per chunk, the exact recursion from its boundary vector (what the reference computes, up to rounding).
The *_seqs functions model several independent sequences (bgmm_hmm_pass_seqs): chunks aligned to sequence starts,
phase B segmented per sequence, windows clamped to their sequence (tests/test_hmm_seqs_scan_model.py).
"""
import numpy as np


def forward(rho, pi_t, a_t, L):
    n, K = rho.shape
    nch = (n + L - 1) // L
    # phase A
    T = np.zeros((nch, K, K)); ls = np.zeros((nch, K))
    for c in range(nch - 1):
        for j in range(K):
            t = np.zeros(K); t[j] = 1.0; s_log = 0.0
            for i in range(c * L, min((c + 1) * L, n)):
                t = (t if i == 0 else t @ a_t) * rho[i]
                s = t.sum(); t = t / s; s_log += np.log(s)
            T[c, j], ls[c, j] = t, s_log
    # phase B
    v = np.zeros((nch, K)); v[0] = pi_t
    for c in range(nch - 1):
        w = v[c] * np.exp(ls[c] - ls[c].max())
        nv = w @ T[c]
        v[c + 1] = nv / nv.sum()
    # phase C
    alpha = np.empty((n, K)); cs = np.empty(n)
    for c in range(nch):
        a = v[c]
        for i in range(c * L, min((c + 1) * L, n)):
            u = (a if i == 0 else a @ a_t) * rho[i]
            cs[i] = u.sum(); a = u / cs[i]; alpha[i] = a
    return alpha, cs


def backward(rho, cs, alpha, a_t, L):
    """-> beta, gamma, S = sum_i alpha_{i-1} (x) (rho_i beta_i / c_i)   (xi summed over time = a_t * S)."""
    n, K = rho.shape
    nch = (n + L - 1) // L
    U = np.zeros((nch, K, K)); ls = np.zeros((nch, K))
    for c in range(1, nch):
        s0, e0 = c * L, min((c + 1) * L, n) - 1
        for j in range(K):
            b = np.zeros(K); b[j] = 1.0; s_log = 0.0
            for i in range(e0, s0 - 1, -1):
                b = a_t @ (rho[i] * b / cs[i])
                s = b.sum(); b = b / s; s_log += np.log(s)
            U[c, j], ls[c, j] = b, s_log
    w = np.zeros((nch, K)); w[nch - 1] = 1.0
    for c in range(nch - 1, 0, -1):
        acc = np.zeros(K)
        for j in range(K):
            if w[c, j] > 0:
                acc += np.exp(ls[c, j] + np.log(w[c, j])) * U[c, j]
        w[c - 1] = acc
    beta = np.empty((n, K)); gamma = np.empty((n, K)); S = np.zeros((K, K))
    for c in range(nch):
        s0, e0 = c * L, min((c + 1) * L, n) - 1
        b = w[c]
        for i in range(e0, s0 - 1, -1):
            beta[i] = b; gamma[i] = alpha[i] * b
            wv = rho[i] * b / cs[i]
            if i >= 1:
                S += np.outer(alpha[i - 1], wv)
            b = a_t @ wv
    return beta, gamma, S


# ---- mixing mode: when W steps provably forget the start vector, a warm-up window per chunk replaces phases A and B ----
def hilbert_diameter(a_t):
    """Projective diameter of the positive matrix a_t: max_{j,j'} [max_k d_k - min_k d_k], d = ln a_j - ln a_j'."""
    la = np.log(a_t)
    d = la[:, None, :] - la[None, :, :]
    return float((d.max(axis=2) - d.min(axis=2)).max())


def window(a_t, chunk_len, eps_log=-41.5):
    """Smallest W with tau^(W-1) Delta < 1e-18, tau = tanh(Delta / 4) (Birkhoff); 0 when it is not worth it."""
    K = a_t.shape[0]
    delta = hilbert_diameter(a_t)
    if delta == 0.0:
        return 8
    lntau = np.log1p(-2.0 / (np.exp(0.5 * delta) + 1.0))
    if not lntau < 0.0:
        return 0
    w = np.ceil((eps_log - np.log(delta)) / lntau) + 1.0
    if not w <= min(16384.0, 0.5 * chunk_len * K):
        return 0
    return max(8, int(w))


def forward_boundaries_window(rho, pi_t, a_t, L, W):
    """v[c] = normalised alpha at element cL-1 from a run over the W elements before chunk c."""
    n, K = rho.shape
    nch = (n + L - 1) // L
    v = np.zeros((nch, K)); v[0] = pi_t
    for c in range(1, nch):
        end, first = c * L - 1, c * L - W
        t = np.array(pi_t) if first <= 0 else np.ones(K)
        for i in range(max(first, 0), end + 1):
            t = (t if i == 0 else t @ a_t) * rho[i]
            t = t / t.sum()
        v[c] = t
    return v


def backward_boundaries_window(rho, cs, a_t, L, W):
    """w[c] = beta at the last element of chunk c from an un-normalised run from ones over the W elements after it."""
    n, K = rho.shape
    nch = (n + L - 1) // L
    w = np.zeros((nch, K))
    for c in range(nch):
        e = min((c + 1) * L, n) - 1
        b = np.ones(K)
        for i in range(min(e + W, n - 1), e, -1):
            b = a_t @ (rho[i] * b / cs[i])
        w[c] = b
    return w


# ---- several independent sequences (bgmm_hmm_pass_seqs): every sequence is cut into its own chunks ----------------------
def seq_chunks(starts, n, L):
    """[(i0, i1, s0, s1)]: chunk [i0, i1) of the sequence [s0, s1); chunks of L elements, the last of a sequence shorter."""
    ends = list(starts[1:]) + [n]
    return [(i0, min(i0 + L, b), a, b) for a, b in zip(starts, ends) for i0 in range(a, b, L)]


def forward_seqs(rho, pi_t, a_t, chunks):
    """Phase A only for chunks followed by a chunk of the same sequence; phase B segmented per sequence (a chunk that
    starts a sequence takes pi~); phase C restarts (no transition) at every sequence start.  -> alpha, cs, v."""
    n, K = rho.shape
    nch = len(chunks)
    T = np.zeros((nch, K, K)); ls = np.zeros((nch, K))
    for c, (i0, i1, s0, s1) in enumerate(chunks):
        if i1 == s1:
            continue
        for j in range(K):
            t = np.zeros(K); t[j] = 1.0; s_log = 0.0
            for i in range(i0, i1):
                t = (t if i == s0 else t @ a_t) * rho[i]
                s = t.sum(); t = t / s; s_log += np.log(s)
            T[c, j], ls[c, j] = t, s_log
    v = np.zeros((nch, K))
    for c, (i0, i1, s0, s1) in enumerate(chunks):
        if i0 == s0:
            v[c] = pi_t
        else:
            w = v[c - 1] * np.exp(ls[c - 1] - ls[c - 1].max())
            nv = w @ T[c - 1]
            v[c] = nv / nv.sum()
    alpha = np.empty((n, K)); cs = np.empty(n)
    for c, (i0, i1, s0, s1) in enumerate(chunks):
        a = v[c]
        for i in range(i0, i1):
            u = (a if i == s0 else a @ a_t) * rho[i]
            cs[i] = u.sum(); a = u / cs[i]; alpha[i] = a
    return alpha, cs, v


def backward_seqs(rho, cs, alpha, a_t, chunks):
    """Phase A' only for chunks preceded by a chunk of the same sequence; phase B' segmented (a chunk that ends a sequence
    takes ones); phase C' with xi = 0 at every sequence start.  -> beta, gamma, S, G0 (gamma summed over the starts), w."""
    n, K = rho.shape
    nch = len(chunks)
    U = np.zeros((nch, K, K)); ls = np.zeros((nch, K))
    for c, (i0, i1, s0, s1) in enumerate(chunks):
        if i0 == s0:
            continue
        for j in range(K):
            b = np.zeros(K); b[j] = 1.0; s_log = 0.0
            for i in range(i1 - 1, i0 - 1, -1):
                b = a_t @ (rho[i] * b / cs[i])
                s = b.sum(); b = b / s; s_log += np.log(s)
            U[c, j], ls[c, j] = b, s_log
    w = np.zeros((nch, K))
    for c in range(nch - 1, -1, -1):
        i0, i1, s0, s1 = chunks[c]
        if i1 == s1:
            w[c] = 1.0
        else:
            acc = np.zeros(K)
            for j in range(K):
                if w[c + 1, j] > 0:
                    acc += np.exp(ls[c + 1, j] + np.log(w[c + 1, j])) * U[c + 1, j]
            w[c] = acc
    beta = np.empty((n, K)); gamma = np.empty((n, K)); S = np.zeros((K, K)); G0 = np.zeros(K)
    for c, (i0, i1, s0, s1) in enumerate(chunks):
        b = w[c]
        for i in range(i1 - 1, i0 - 1, -1):
            beta[i] = b; gamma[i] = alpha[i] * b
            wv = rho[i] * b / cs[i]
            if i > s0:
                S += np.outer(alpha[i - 1], wv)
            else:
                G0 += gamma[i]
            b = a_t @ wv
    return beta, gamma, S, G0, w


def forward_boundaries_window_seqs(rho, pi_t, a_t, chunks, W):
    """v[c] from a run over the W elements before chunk c, clamped to its sequence (from pi~ when it reaches the start)."""
    K = rho.shape[1]
    v = np.zeros((len(chunks), K))
    for c, (i0, i1, s0, s1) in enumerate(chunks):
        if i0 == s0:
            v[c] = pi_t
            continue
        end, first = i0 - 1, i0 - W
        t = np.array(pi_t) if first <= s0 else np.ones(K)
        for i in range(max(first, s0), end + 1):
            t = (t if i == s0 else t @ a_t) * rho[i]
            t = t / t.sum()
        v[c] = t
    return v


def backward_boundaries_window_seqs(rho, cs, a_t, chunks, W):
    """w[c] from an un-normalised run from ones over the W elements after chunk c, clamped to its sequence."""
    K = rho.shape[1]
    w = np.zeros((len(chunks), K))
    for c, (i0, i1, s0, s1) in enumerate(chunks):
        e = i1 - 1
        b = np.ones(K)
        for i in range(min(e + W, s1 - 1), e, -1):
            b = a_t @ (rho[i] * b / cs[i])
        w[c] = b
    return w
