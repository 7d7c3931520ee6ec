"""Numpy restatement of MMI training (TEST INFRASTRUCTURE): the hypotheses and weights of hmmcu_estep_mmi from a matrix of
forward scores, the [2][V][stats_size] statistics buffer formed from oracle.estep, and the extended Baum-Welch update of
hmmh_mstep_ebw / hmmcu_mstep_ebw."""
import numpy as np

from oracle import oracle as o

MIN_POST = 1e-5   # HMMCU_MMI_MIN_POST
FLOOR = 1e-5      # FINITE_PROBAB, T-FS:39


def stats_vec(st):
    return np.concatenate([st.num_trans.ravel(), st.den_trans, st.den_mix, st.S0.ravel(), st.S1.ravel(), st.S2c.ravel(),
                           [st.sum_logp, st.n_utt]])


def model(ms, v):
    return o.Model(ms.A[v], ms.c[v], ms.mu[v], ms.iv[v], ms.det[v], ms.words[v])


def hypotheses(S, label, kappa, H):
    """-> (hyps, term): hyps[u] = [(word, weight), ..] (the label first; empty for a left-out utterance),
    term[u] = logsumexp - kappa S[u][label] (NaN when left out), and the log-posteriors a[U][V]."""
    U, V = S.shape
    a = np.full((U, V), -np.inf)
    hyps, term = [], np.full(U, np.nan)
    for u in range(U):
        lab = label[u]
        if lab < 0 or not np.isfinite(S[u, lab]):
            hyps.append([])
            continue
        k = kappa * S[u]
        m = k.max()
        lse = m + np.log(np.exp(k - m).sum())
        a[u] = k - lse
        term[u] = lse - k[lab]
        others = sorted((w for w in range(V) if w != lab and np.exp(a[u, w]) >= MIN_POST), key=lambda w: (-a[u, w], w))
        hyps.append([(lab, np.exp(a[u, lab]))] + [(w, np.exp(a[u, w])) for w in others[:H - 1]])
    return hyps, term, a


def mmi_buffer(ms, x, off, label, S, kappa, H, us=None):
    """The statistics of hmmcu_estep_mmi over utterances `us` (default: all): [2][V][stats_size]."""
    V = ms.V
    us = range(len(off) - 1) if us is None else us
    hyps, term, _ = hypotheses(S, label, kappa, H)
    ss = ms.N * ms.N + 2 * ms.N + ms.N * ms.M + 2 * ms.N * ms.M * ms.D + 2
    out = np.zeros((2, V, ss))
    for v in range(V):
        uv = [u for u in us if label[u] == v]
        if uv:
            xv = np.concatenate([x[off[u]:off[u + 1]] for u in uv])
            offv = np.concatenate([[0], np.cumsum([off[u + 1] - off[u] for u in uv])]).astype(np.int64)
            out[0, v] = stats_vec(o.estep(model(ms, v), xv, offv)[0])
    for u in us:
        xu = x[off[u]:off[u + 1]]
        offu = np.array([0, len(xu)], dtype=np.int64)
        for h, w in hyps[u]:
            st = o.estep(model(ms, h), xu, offu)[0]
            out[1, h, :-2] += w * stats_vec(st)[:-2]
        if hyps[u]:
            out[1, label[u], -2] += term[u]
            out[1, label[u], -1] += 1
    return out


def ebw(ms, num, den, E, tau, branch=None):
    """The extended Baum-Welch update of means and variances, in place on ms.  branch (optional dict) receives per
    Gaussian which constant was used: 'dmin' (2 D_min), 'e' (E S0_den) or 'none' (unchanged)."""
    N, M, D = ms.N, ms.M, ms.D
    G = N * M
    o0 = N * N + 2 * N
    for v in range(ms.V):
        s0n, s0d = num[v, o0:o0 + G], den[v, o0:o0 + G]
        s1n, s1d = num[v, o0 + G:o0 + G + G * D].reshape(G, D), den[v, o0 + G:o0 + G + G * D].reshape(G, D)
        s2n, s2d = num[v, o0 + G + G * D:o0 + G + 2 * G * D].reshape(G, D), den[v, o0 + G + G * D:o0 + G + 2 * G * D].reshape(G, D)
        mu, iv, det = ms.mu[v].reshape(G, D), ms.iv[v].reshape(G, D), ms.det[v].reshape(G)
        for k in range(G):
            m, var = mu[k].copy(), 1.0 / iv[k]
            sc = 1.0 + tau / s0n[k] if s0n[k] > 0 else 1.0
            qn = s2n[k] + 2.0 * m * s1n[k] - m * m * s0n[k]
            qd = s2d[k] + 2.0 * m * s1d[k] - m * m * s0d[k]
            dg = s0n[k] * sc - s0d[k]
            ds = s1n[k] * sc - s1d[k]
            dq = qn * sc - qd
            b = dq + dg * (var + m * m) - 2.0 * m * ds
            c = dq * dg - ds * ds
            disc = b * b - 4.0 * var * c
            roots = np.where(disc >= 0, (-b + np.sqrt(np.maximum(disc, 0))) / (2.0 * var), 0.0)
            dmin = max(0.0, float(roots.max()))
            Dc = max(2.0 * dmin, E * s0d[k])
            if not dg + Dc > 0:
                if branch is not None:
                    branch[(v, k)] = "none"
                continue
            if branch is not None:
                branch[(v, k)] = "dmin" if 2.0 * dmin >= E * s0d[k] else "e"
            mn = (ds + Dc * m) / (dg + Dc)
            vn = np.maximum((dq + Dc * (var + m * m)) / (dg + Dc) - mn * mn, FLOOR)
            mu[k] = mn
            iv[k] = 1.0 / vn
            det[k] = np.prod(vn)
    return ms
