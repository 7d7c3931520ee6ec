"""MMI training where its statistics are small: the hypotheses of k_mmi_post read back one utterance at a time, words that
only competitors reach (block 1 without block 0) on every accumulate path, every state count of the weighted
forward-backward, the production batch shapes of k_fb_res with the per-word objective tail, and the extended Baum-Welch
update on those statistics.

A word's block-1 total is dominated by its label round (weight near 1); competitor rounds weigh 1e-5 .. 0.1, below the
Baum-Welch bar of that total.  So every check here isolates the small statistics: a word that no utterance is labelled
with, compared against its own occupancy, or one utterance at a time, where a round's weight is read back exactly."""
import types

import numpy as np
import pytest

from mmi_oracle import MIN_POST, ebw, hypotheses, mmi_buffer
from speech_recognition_hmm_continuous_b200 import api, synth
from test_fb_res_batches import _batching, _corpus
from test_mmi_training import _assert_separated, _kappa
from test_viterbi_training import RTOL, _assert_mixture_stats, _dispatches

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = api.Context(0)
    yield c
    c.close()


def _unreachable(A):
    """A with every transition into the final state removed (rows renormalised): that word scores -inf."""
    N = A.shape[0]
    A = A.copy()
    A[:N - 1, N - 1] = 0.0
    return A / A.sum(-1, keepdims=True)


def _split(vec, ms):
    return api.split_stats(vec, ms.N, ms.M, ms.D)


# ------------------------------------------------------------------ k_mmi_post, read back exactly ----
def _twin_set():
    """V = 70 (lanes 0..31 take 2 or 3 words each), N = 3, M = 2, U = 19 (three CTAs of 8 rows, the last one partial).
    Words 35 (the lane of word 3) and 36 (the next lane) are bit-identical copies of word 3; word 69 cannot reach its
    final state.  Utterances 0, 8 and 18 are drawn from word 3, the others from the words that are neither twins nor 69."""
    V, N, M, U = 70, 3, 2, 19
    cen, s = synth.make_centres(V, N, M, 39, seed=7070)
    cen[35] = cen[3]
    cen[36] = cen[3]
    rng = np.random.default_rng(7071)
    gen = rng.choice([v for v in range(69) if v not in (3, 35, 36)], size=U)
    gen[[0, 8, 18]] = 3
    x, off = synth.make_utterances(cen, s, gen, seed=7072, tmin=20, tmax=40)
    d = synth.make_models(cen, s)
    d["A"][69] = _unreachable(d["A"][69])
    return api.ModelSet.from_dict(d), x, off


def _competitors(a, lab):
    """Posteriors of the words other than the label, descending."""
    return np.sort(np.exp(np.delete(a, lab)))[::-1]


def _assert_ties_exact(a, lab):
    """Two competitors have either the same posterior (the twins: bit-equal scores) or posteriors more than 1e-9 apart
    (relative), and none lies within 1e-9 of the floor: the device and numpy then select the same words."""
    p = _competitors(a, lab)
    p = p[p > 0]
    d = np.abs(np.diff(p))
    assert ((d == 0) | (d > 1e-9 * p[1:])).all()
    assert (np.abs(p - MIN_POST) > 1e-9 * MIN_POST).all()


def test_posteriors_and_hypotheses_read_back_exactly(ctx):
    """With one utterance u labelled and all others -1, block 1 of word h is w(u, h) times the plain E-step of u against
    h, so w(u, h) = den_mix total of block 1[h] / den_mix total of that E-step (both sums of the same gamma, in double).
    Checked: the set of words with mass equals numpy's selection on the device's own scores, every weight to 1e-12, the
    objective term and n_utt = 1, the number of rounds.  Cases: rows 0, 8 and 18 (first, second and partial third CTA),
    H in {1, 2, 4, 16}, a kappa at which every case has >= 15 competitors above the floor and one at which the floor cuts
    the list short; labels 3 (the twins 35, 36 tie with the label), 35 (word 3 has exactly the label's posterior and ties
    with 36 across lanes) and 10 (3 and 35 tie within a lane, 36 across lanes)."""
    ms, x, off = _twin_set()
    V, U = ms.V, len(off) - 1
    ctx.set_features(x, off)
    ctx.set_models(ms)
    S = ctx.forward_scores()
    assert np.array_equal(S[:, 3], S[:, 35]) and np.array_equal(S[:, 3], S[:, 36])
    assert (S[:, 69] == -np.inf).all() and np.isfinite(S[:, :69]).all()
    cases = {0: 3, 8: 35, 18: 10}
    for u in cases:
        assert S[u, 3] == S[u].max(), u  # the twins lead: every rank cut below H = 4 falls among them

    ref = {}

    def unweighted_den(u, h):
        if (u, h) not in ref:
            m = np.full(U, -1, dtype=np.int32)
            m[u] = h
            st, _ = ctx.estep(m)
            assert (np.delete(st, h, axis=0) == 0).all()
            ref[(u, h)] = _split(st[h], ms)["den_mix"].sum()
        return ref[(u, h)]

    def n_comp(kappa, u):
        lab = np.full(U, -1)
        lab[u] = cases[u]
        _, _, a = hypotheses(S, lab, kappa, 1)
        return int((_competitors(a[u], cases[u]) >= MIN_POST).sum())

    k_small = k_floor = _kappa(S, S.argmax(1), 3.0)
    while min(n_comp(k_small, u) for u in cases) < 15:
        k_small /= 2
    while min(n_comp(k_floor, u) for u in cases) >= 15:
        k_floor *= 2
    seen_rounds = set()
    for kappa in (k_small, k_floor):
        for u, lab in cases.items():
            label = np.full(U, -1, dtype=np.int32)
            label[u] = lab
            for H in (1, 2, 4, 16):
                stats = ctx.estep_mmi(label, kappa, H)
                hyps, term, a = hypotheses(S, label, kappa, H)
                _assert_ties_exact(a[u], lab)
                want = dict(hyps[u])
                assert want[lab] > 0
                got = {h for h in range(V) if (stats[1, h, :-2] != 0).any()}
                assert got == set(want), (u, H, sorted(got), sorted(want))
                assert ctx.kernel_ms("mmi_rounds") == len(want)
                seen_rounds.add(len(want))
                for h, w in want.items():
                    wd = _split(stats[1, h], ms)["den_mix"].sum() / unweighted_den(u, h)
                    assert abs(wd - w) <= 1e-12 * w, (u, H, h, wd, w)
                assert stats[1, lab, -1] == 1 and abs(stats[1, lab, -2] - term[u]) <= 1e-12 * abs(term[u]), (u, H)
                assert (np.delete(stats[1, :, -2:], lab, axis=0) == 0).all()
                assert (stats[:, 69] == 0).all()
                if H == 2 and lab != 3:
                    assert set(want) == {lab, 3}  # the cut between the twins: word 3 (the lower index) only
                if lab == 35:
                    assert H == 1 or want[3] == want[35]
            if kappa == k_small:
                assert ctx.kernel_ms("mmi_rounds") == 16
    assert {1, 2, 4, 16} <= seen_rounds and len(seen_rounds) > 4, seen_rounds


# ------------------------------------------------------------------ competitor-only words ----
def _competitor_set(N, M, D=39, V=40, n_lab=20, U=120, seed=0, dense=False):
    """Words 0 .. n_lab-1 label the utterances (20 .. 60 frames); words n_lab .. V-2 are close copies of words
    0 .. V-2-n_lab (the last state's centres moved by 0.3 sigma), which only ever receive denominator mass; word V-1
    cannot reach its final state (N > 1)."""
    cen, s = synth.make_centres(V, N, M, D, seed=seed)
    rng = np.random.default_rng(seed + 1)
    for k in range(n_lab, V - 1):
        cen[k] = cen[k - n_lab]
        cen[k, N - 1] += 0.3 * s * rng.standard_normal((M, D))
    labels = np.arange(U) % n_lab
    x, off = synth.make_utterances(cen, s, labels, seed=seed + 2, tmin=20, tmax=60)
    d = synth.make_models(cen, s)
    if dense:
        A = 0.9 * d["A"] + 0.1 / N
        d["A"] = A / A.sum(-1, keepdims=True)
    if N > 1:
        d["A"][V - 1] = _unreachable(d["A"][V - 1])
    return api.ModelSet.from_dict(d), x, off, labels


def _hard(S, labels):
    """A kappa at which the median utterance's best competitor has posterior 1e-4, and the labels with the utterances whose
    best competitor would exceed 1e-3 left out (-1): every competitor posterior then lies in [1e-5, 1e-3]."""
    gaps = np.array([S[u, labels[u]] - np.max(np.delete(S[u], labels[u])) for u in range(len(labels))])
    kappa = np.log(1e4) / np.median(gaps)
    return kappa, np.where(kappa * gaps >= 1.001 * np.log(1e3), labels, -1)


def _check_competitor_words(ms, x, stats, want, words):
    """Block 1 of `words` (no utterance is labelled with them) against the oracle, at bars relative to each word's own
    occupancy; their block 0 and their tail exactly 0.  -> the words that received mass."""
    fed = []
    for v in words:
        sp, wp = _split(stats[1, v], ms), _split(want[1, v], ms)
        assert (stats[0, v] == 0).all(), v
        assert stats[1, v, -2] == 0 and stats[1, v, -1] == 0, v
        if wp["S0"].sum() == 0:
            assert (stats[1, v] == 0).all(), v
            continue
        fed.append(v)
        _assert_mixture_stats(sp, types.SimpleNamespace(S0=wp["S0"], S1=wp["S1"], S2c=wp["S2c"]), x)
        for name in ("num_trans", "den_trans", "den_mix"):
            assert np.allclose(sp[name], wp[name], rtol=RTOL, atol=1e-6 * np.abs(wp[name]).max()), (v, name)
    return fed


ACC_PATHS = [  # option, accumulate kernel, (tc_active, acc_h_active)
    (None, "k_accum_h", (1.0, 1.0)),
    ("h_acc", "k_accum_ws", (1.0, 0.0)),
    ("ws_acc", "k_accum_tc", (1.0, 0.0)),
    ("tc_emis", "CUDA cores", (0.0, 0.0)),
]


@pytest.mark.parametrize("M", [3, 16])
def test_competitor_only_words_on_every_accumulate_path(ctx, M):
    """V = 40, N = 5: words 20..38 receive denominator mass only, word 39 none.  Two kappas: soft (the median best
    competitor 1 nat below the label) and hard (every competitor posterior in [1e-5, 1e-3], where the accumulators'
    weights are posterior x gamma x mixture posterior), each on the four accumulate paths."""
    ms, x, off, labels = _competitor_set(5, M, seed=3100 + M)
    ctx.set_features(x, off)
    ctx.set_models(ms)
    S = ctx.forward_scores()
    assert (S[:, 39] == -np.inf).all()
    H = 4
    for kname, (kappa, lab) in (("soft", (_kappa(S, labels, 1.0), labels)), ("hard", _hard(S, labels))):
        hyps, _, a = hypotheses(S, lab, kappa, H)
        _assert_separated(a, lab, H)
        comp = [w for h in hyps for _, w in h[1:]]
        if kname == "hard":
            assert comp and all(MIN_POST <= w <= 1e-3 for w in comp), (min(comp), max(comp))
        want = mmi_buffer(ms, x, off, lab, S, kappa, H)
        for opt, kernel, active in ACC_PATHS:
            if opt:
                ctx.set_option(opt, 0)
            try:
                stats = ctx.estep_mmi(lab, kappa, H)
                assert (ctx.kernel_ms("tc_active"), ctx.kernel_ms("acc_h_active")) == active, kernel
            finally:
                if opt:
                    ctx.set_option(opt, 1)
            fed = _check_competitor_words(ms, x, stats, want, range(20, 39))
            assert (stats[:, 39] == 0).all()
            print("M=%d %s kappa=%.3g %s: %d competitor rounds, %d of 19 competitor-only words fed"
                  % (M, kname, kappa, kernel, len(comp), len(fed)))
            assert len(fed) >= (15 if kname == "soft" else 3), fed


# ------------------------------------------------------------------ weighted forward-backward, every N ----
@pytest.mark.parametrize("N", [1, 2, 4, 6, 7])
def test_weighted_forward_backward_every_state_count(ctx, N):
    """k_fb_res<N, true> (banded A, res_fb 1) and k_fb<N, *, true> (banded and dense A, res_fb 0) at the state counts
    the MMI tests do not otherwise reach, checked on words 6..10, which only competitors reach."""
    for dense in ((False, True) if N > 1 else (False,)):
        ms, x, off, labels = _competitor_set(N, 3, V=12, n_lab=6, U=36, seed=3200 + 10 * N + dense, dense=dense)
        ctx.set_features(x, off)
        ctx.set_models(ms)
        try:
            for res_fb in _dispatches(dense):
                ctx.set_option("res_fb", res_fb)
                S = ctx.forward_scores()
                kappa = _kappa(S, labels, 1.0)
                hyps, _, a = hypotheses(S, labels, kappa, 4)
                _assert_separated(a, labels, 4)
                stats = ctx.estep_mmi(labels, kappa, 4)
                want = mmi_buffer(ms, x, off, labels, S, kappa, 4)
                fed = _check_competitor_words(ms, x, stats, want, range(6, 11))
                assert len(fed) == 5, fed
                if N > 1:
                    assert (stats[:, 11] == 0).all()
        finally:
            ctx.set_option("res_fb", 1)


# ------------------------------------------------------------------ production batch shapes, objective tail ----
def _round_sizes(S, labels, kappa, H):
    hyps, _, _ = hypotheses(S, labels, kappa, H)
    return [sum(len(h) > r for h in hyps) for r in range(H)], hyps


@pytest.mark.parametrize("N", [2, 8])
def test_production_batches_and_objective_tail(N):
    """The short-word corpus of test_fb_res_batches (20,000 utterances over 64 words, T < N and T = 1 in words 0 and 1):
    the label map runs full batches of k_fb_res, the 15 competitor rounds run smaller batches on the reused batch counter
    (round 1 with >= 1,000 live utterances, the last with under 1,000 and at most 1 / 1.3 of round 1: competitors of
    this corpus come in groups, so the rounds shrink slowly), and k_mmi_tail sums about 312 terms per word over 8 CTAs,
    leaving out the utterances whose label score is -inf.  Block 1 of every word against the oracle, the tail to 1e-12, n_utt exactly, two calls bit-identical."""
    x, off, labels, ms, _ = _corpus(N, short_words=True)
    U, V = len(labels), ms.V
    T = np.diff(off)
    c = api.Context(0)
    try:
        c.set_features(x, off)
        c.set_models(ms)
        c.estep(labels, download=False)
        nb, bmax, teams = _batching(c)
        assert bmax == 16, (nb, bmax)
        S = c.forward_scores()
        H = 16
        # the smallest kappa on a log grid at which the last round has at most 1,000 live utterances
        kappa = _kappa(S, labels, 3.0)
        sizes, _ = _round_sizes(S, labels, kappa, H)
        while sizes[-1] > 1000:
            kappa *= 2 ** 0.125
            sizes, _ = _round_sizes(S, labels, kappa, H)
        assert sizes[1] >= 1000 and sizes[1] >= 1.3 * sizes[-1] >= 1.3 * 150, sizes
        hyps, term, a = hypotheses(S, labels, kappa, H)
        _assert_separated(a, labels, H)
        stats = c.estep_mmi(labels, kappa, H)
        assert c.kernel_ms("mmi_rounds") == H
        nb_last, bmax_last, _ = _batching(c)
        assert bmax_last < 16, (nb_last, bmax_last)
        again = c.estep_mmi(labels, kappa, H)
        assert np.array_equal(stats, again)
    finally:
        c.close()
    print("N=%d kappa=%.3g live utterances per round %s, label map %d batches of <= %d, last round %d of <= %d"
          % (N, kappa, sizes, nb, bmax, nb_last, bmax_last))
    want = mmi_buffer(ms, x, off, labels, S, kappa, H)
    for v in range(V):
        sp, wp = _split(stats[1, v], ms), _split(want[1, v], ms)
        _assert_mixture_stats(sp, types.SimpleNamespace(S0=wp["S0"], S1=wp["S1"], S2c=wp["S2c"]), x)
        for name in ("num_trans", "den_trans", "den_mix"):
            assert np.allclose(sp[name], wp[name], rtol=RTOL, atol=1e-6 * np.abs(wp[name]).max()), (v, name)
        inc = [u for u in np.nonzero(labels == v)[0] if np.isfinite(term[u])]
        assert sp["n_utt"] == len(inc), v
        t = float(np.sum(term[inc]))
        assert abs(sp["sum_logp"] - t) <= 1e-12 * abs(t), (v, sp["sum_logp"], t)
        if v < 2:  # utterances shorter than the chain are left out
            assert len(inc) < (labels == v).sum() and len(inc) == ((labels == v) & (T >= N)).sum(), v
        else:
            assert len(inc) == (labels == v).sum(), v


# ------------------------------------------------------------------ extended Baum-Welch ----
@pytest.mark.parametrize("D", [13, 39])
def test_ebw_on_competitor_only_words(ctx, D):
    """k_mstep_ebw (G = 15, not a multiple of its 8 warps) on the statistics of the competitor-only set: device against
    host to 1e-12 on mu, iv and det; the unreachable word unchanged bit for bit; and all three branches of the update
    (D = 2 D_min, D = E S0_den, no occupancy at all: unchanged) taken, per the numpy restatement on the same statistics."""
    ms, x, off, labels = _competitor_set(5, 3, D=D, seed=3300 + D)
    ctx.set_features(x, off)
    ctx.set_models(ms)
    S = ctx.forward_scores()
    branches = {}
    for kappa, lab in ((_kappa(S, labels, 1.0), labels), _hard(S, labels)):
        for E, tau in ((2.0, 100.0), (1.5, 0.0)):
            ctx.set_models(ms)
            stats = ctx.estep_mmi(lab, kappa, 4)
            before = ctx.get_models(D)
            want = api.mstep_ebw(before.copy(), stats[0], stats[1], E, tau)
            ctx.mstep_ebw(E, tau)
            got = ctx.get_models(D)
            for name in ("mu", "iv", "det"):
                g, w = getattr(got, name), getattr(want, name)
                assert np.allclose(g, w, rtol=1e-12, atol=0), (name, np.abs(g - w).max())
                assert np.array_equal(g[39], getattr(before, name)[39]), name
            br = {}
            ebw(before.copy(), stats[0], stats[1], E, tau, branch=br)
            for k, b in br.items():
                branches.setdefault(b, set()).add(k[0])
    print("D=%d: words per branch %s" % (D, {b: len(v) for b, v in branches.items()}))
    assert set(branches) == {"dmin", "e", "none"}, sorted(branches)
    assert any(v >= 20 for v in branches["dmin"] | branches["e"])  # competitor-only words were updated
