"""numpy model of the hidden-Markov 'random_responsibility' initial state that csrc/bgmm_extras.cu draws on the device
(bgmm_hmm_init_random, `hiddenmarkovnormal.LearnModel(device_init=True)`).

Executable specification of the counter mapping in include/bgmm.h: element i's K x K matrix xt_i of standard
exponentials -ln u, where pair p = r * K + k gives entries (2r, k) and (2r + 1, k) from Philox4x32-10 (Salmon et al.
2011) of counter (i lo, i hi, p, TAG) under key (seed lo, seed hi).  The rules applied to xi_i = xt_i / sum(xt_i) are
those of `LearnModel._init_random_responsibility`.  Philox runs in uint64 arithmetic, so the uniforms are the device's
bit for bit and only `log` and the order of the sums can differ.
"""
import numpy as np

TAG = 0x484D4D49                    # "HMMI"
_M0, _M1, _W0, _W1, _MASK = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85, 0xFFFFFFFF


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Ten Philox4x32 rounds on uint64 arrays holding 32-bit words -> the four output words."""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) for c in (c0, c1, c2, c3))
    k0, k1 = np.uint64(k0), np.uint64(k1)
    for _ in range(10):
        p0, p1 = np.uint64(_M0) * c0, np.uint64(_M1) * c2
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & np.uint64(_MASK),
                          (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & np.uint64(_MASK))
        k0, k1 = (k0 + np.uint64(_W0)) & np.uint64(_MASK), (k1 + np.uint64(_W1)) & np.uint64(_MASK)
    return c0, c1, c2, c3


def uniform_open(hi, lo):
    """(0, 1) from two words: the top 53 bits of hi:lo plus one half, over 2^53 (never 0 or 1)."""
    u = (hi << np.uint64(32)) | lo
    return ((u >> np.uint64(11)).astype(np.float64) + 0.5) * (1.0 / 9007199254740992.0)


def draw(idx, K, seed):
    """xt of the elements `idx` -> [len(idx), K, K] (unnormalised)."""
    idx = np.asarray(idx, dtype=np.uint64)
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    k0, k1 = seed & _MASK, seed >> 32
    out = np.empty((idx.size, K, K))
    c0 = np.repeat((idx & np.uint64(_MASK))[:, None], K, axis=1)
    c1 = np.repeat((idx >> np.uint64(32))[:, None], K, axis=1)
    c3 = np.full(c0.shape, TAG, dtype=np.uint64)
    for r in range((K + 1) // 2):
        c2 = np.broadcast_to(np.arange(r * K, r * K + K, dtype=np.uint64), c0.shape)
        w0, w1, w2, w3 = philox4x32_10(c0, c1, c2, c3, k0, k1)
        out[:, 2 * r, :] = -np.log(uniform_open(w0, w1))
        if 2 * r + 1 < K:
            out[:, 2 * r + 1, :] = -np.log(uniform_open(w2, w3))
    return out


def xi(idx, K, seed):
    """Normalised draws xi of the elements `idx` (each a Dirichlet(1_{K^2}) as a K x K matrix)."""
    t = draw(idx, K, seed)
    return t / t.sum(axis=(1, 2), keepdims=True)


def init_state(n, K, seed, starts=None, want_xi=False, block=8192):
    """-> (gamma [n][K], ms [K][K], g0 [K], xi [n][K][K] with xi = 0 at the starts, or None): the rules of
    `_init_random_responsibility` on the device's draws.  `starts`: first rows of the sequences (None: one sequence)."""
    starts = np.zeros(1, dtype=np.int64) if starts is None else np.asarray(starts, dtype=np.int64)
    if n == 1:
        t = draw([0], K, seed)[0, 0]
        g = t / t.sum()
        return g[None, :], np.zeros((K, K)), g.copy(), (np.zeros((1, K, K)) if want_xi else None)
    ends = np.append(starts[1:], n)
    gamma, ms = np.empty((n, K)), np.zeros((K, K))
    xi_all = np.empty((n, K, K)) if want_xi else None
    for b0 in range(0, n, block):
        b1 = min(n, b0 + block)
        x = xi(np.arange(b0, b1), K, seed)
        gamma[b0:b1] = x.sum(axis=1)
        here = (starts >= b0) & (starts < b1)
        for s, e in zip(starts[here], ends[here]):
            gamma[s] = (xi([s + 1], K, seed)[0] if e - s > 1 else x[s - b0]).sum(axis=1)
        x[starts[here] - b0] = 0.0
        ms += x.sum(axis=0)
        if want_xi:
            xi_all[b0:b1] = x
    return gamma, ms, gamma[starts].sum(axis=0), xi_all
