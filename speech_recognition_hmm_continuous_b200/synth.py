"""Synthetic 39-dim "MFCC-shaped" data and model generator (SURVEY.md section 8d).

Per-dimension scale s_d: 13 static coefficients 10*0.8^k, 13 deltas at 0.3x, 13 delta-deltas at
0.1x.  Word v / state i / mixture m has centre mu = s * N(0,1) and standard deviation s.  An
utterance of word v walks the states left to right (uniform segmentation with +-20 % jitter),
T ~ U{250..350}.  Class separation stays around 1.4 sigma per dimension, which keeps the
reference's linear-domain arithmetic finite (SURVEY.md section 7).
"""
import numpy as np


def dim_scales(D=39):
    k = np.arange(D)
    third = max(1, (D + 2) // 3)
    base = 10.0 * 0.8 ** (k % third)
    mult = np.where(k < third, 1.0, np.where(k < 2 * third, 0.3, 0.1))
    return base * mult


def make_centres(V, N, M, D=39, seed=1234):
    """Generating centres [V][N][M][D] and the per-dimension sigma [D]."""
    rng = np.random.default_rng(seed)
    s = dim_scales(D)
    return s * rng.standard_normal((V, N, M, D)), s


def make_utterances(centres, s, labels, seed=1234, tmin=250, tmax=350, lengths=None):
    """-> x float64 [F][D], off int64 [U+1].  labels[u] = word of utterance u; its length is lengths[u] when given,
    otherwise drawn from U{tmin..tmax}."""
    rng = np.random.default_rng(seed + 1)
    V, N, M, D = centres.shape
    U = len(labels)
    T = rng.integers(tmin, tmax + 1, size=U) if lengths is None else np.asarray(lengths, dtype=np.int64)
    off = np.zeros(U + 1, dtype=np.int64)
    np.cumsum(T, out=off[1:])
    F = int(off[-1])
    # state of every frame: uniform segmentation with +-20 % jitter on the segment lengths
    state = np.empty(F, dtype=np.int64)
    word = np.repeat(np.asarray(labels, dtype=np.int64), T)
    for u in range(U):
        w = 1.0 + 0.4 * (rng.random(N) - 0.5)
        cuts = np.floor(np.cumsum(w) / w.sum() * T[u]).astype(np.int64)
        cuts[-1] = T[u]
        seg = np.diff(np.concatenate([[0], cuts]))
        state[off[u]:off[u + 1]] = np.repeat(np.arange(N), seg)
    mix = rng.integers(0, M, size=F)
    x = centres[word, state, mix] + s * rng.standard_normal((F, D))
    return np.ascontiguousarray(x), off


def make_models(centres, s, seed=99):
    """Models drawn from the generator (not trained): left-to-right A with self-loop p, uniform
    weights, variance s^2.  Returned as dict of stacked float64 arrays in the reference's
    semantics (iv = inverse variance, det = product of variances)."""
    V, N, M, D = centres.shape
    A = np.zeros((V, N, N))
    for i in range(N):
        if i + 1 < N:
            A[:, i, i] = 0.98
            A[:, i, i + 1] = 0.02
        else:
            A[:, i, i] = 1.0
    c = np.full((V, N, M), 1.0 / M)
    var = np.broadcast_to(s * s, (V, N, M, D)).copy()
    return dict(A=A, c=c, mu=centres.copy(), iv=1.0 / var, det=np.prod(var, axis=-1))
