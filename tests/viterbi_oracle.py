"""Viterbi-training E-step restated on the oracle's primitives (TEST INFRASTRUCTURE): oracle.viterbi on the
double-precision oracle.emissions, the path turned into counts and one-hot occupancies, and the mixture sums
accumulated with the in-state posteriors around the old mean, as oracle.estep_streams does for Baum-Welch."""
import numpy as np

from oracle import oracle as o


def log_emissions(m, x):
    with np.errstate(divide="ignore"):
        return np.log(o.emissions(m, x, want_post=False)[0])


def path_counts(path, N):
    """(num_trans[N][N], den_trans[N], den_mix[N]) of one utterance's state sequence."""
    path = np.asarray(path, dtype=np.int64)
    num = np.zeros((N, N))
    np.add.at(num, (path[:-1], path[1:]), 1.0)
    return num, np.bincount(path[:-1], minlength=N).astype(float), np.bincount(path, minlength=N).astype(float)


def decision_margin(m, logb, path):
    """The smallest gap, over the back-pointer decisions along the oracle's best path, between the winning and the
    runner-up predecessor (termination is fixed in state N-1).  Where it is below the error of single-precision
    log-emissions, the device may legitimately take the other path."""
    T, N = logb.shape
    with np.errstate(divide="ignore"):
        la = np.log(m.A)
    delta = np.full((T, N), -np.inf)
    delta[0, 0] = logb[0, 0]
    gap = np.inf
    for t in range(1, T):
        cand = delta[t - 1][:, None] + la  # [i][j]
        delta[t] = cand.max(0) + logb[t]
        c = np.sort(cand[:, path[t]])[::-1]
        if N > 1 and np.isfinite(c[0]):
            gap = min(gap, c[0] - c[1]) if np.isfinite(c[1]) else gap
    return gap


def estep_viterbi(m, x, off, paths=None):
    """E-step of Viterbi training of one model over utterances x[off[u]:off[u+1]] -> (oracle.Stats, scores, paths).
    paths[u] replaces the oracle's own alignment of utterance u when given (statistics for the device's path)."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    U = len(off) - 1
    st = o.Stats(m.N, m.M, m.D)
    scores, out = np.zeros(U), []
    for u in range(U):
        xu = x[off[u]:off[u + 1]]
        b, post = o.emissions(m, xu)
        s, p = o.viterbi(m, b)
        if paths is not None:
            p = np.asarray(paths[u], dtype=np.int32)
        scores[u] = s
        out.append(p)
        st.sum_logp += s
        st.n_utt += 1
        if not np.isfinite(s):  # no path to the final state: no occupancy, no counts
            continue
        num, dt, dm = path_counts(p, m.N)
        st.num_trans += num
        st.den_trans += dt
        st.den_mix += dm
        w = post[np.arange(len(p)), p]  # [T][M] in-state posteriors of the aligned state
        for i in range(m.N):
            sel = p == i
            if not sel.any():
                continue
            wi, xi = w[sel], xu[sel]
            st.S0[i] += wi.sum(0)
            st.S1[i] += wi.T @ xi
            dev = xi[:, None, :] - m.mu[i][None]
            st.S2c[i] += np.einsum("tm,tmd->md", wi, dev * dev)
    return st, scores, out
