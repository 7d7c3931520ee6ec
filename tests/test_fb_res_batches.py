"""k_fb_res, the default training recursion, at the batch shapes a corpus of short words gives it.

The batching rule (set_train_map) cuts the live utterances, longest first, into batches of at most
min(16, ceil(live / teams)) utterances that also fit one team's quarter of the shared memory; the teams (4 per CTA, one
CTA per SM) claim batches from a counter that the last claim of every launch sets back to 0.  With 20,000 utterances of
mostly 2..30 frames every batch is full (16 utterances: all 32 lanes of the chain warp busy, each warp of the staging and
gamma phases takes four utterances), the longest ones are cut by shared memory, and every team takes about two batches
(the idle warp claims and prefetches the next one while the chains run).  The tests read the batching back through
hmmcu_last_kernel_ms ("res_batches", "res_batch_max", "res_teams") and fail when the rule or the device no longer gives
this regime, rather than silently testing something else."""
import numpy as np
import pytest

from oracle import oracle as o
from speech_recognition_hmm_continuous_b200 import api, synth

pytestmark = pytest.mark.gpu
RTOL = 1e-4  # north_star tolerance for floating-point results
V, M, D, U = 64, 3, 39, 20000


def _corpus(N, short_words):
    """V words of U / V utterances each (labels u % V).  T ~ U{N..30}, about 2 % of them T ~ U{100..300}; with
    short_words, words 0 and 1 take T ~ U{1..30} instead, so that only they have utterances with T < N (log P = -inf,
    no occupancy) and T = 1.  Models: the generating ones with the means moved by 0.3 sigma."""
    rng = np.random.default_rng(4100 + N)
    labels = np.arange(U) % V
    T = rng.integers(N, 31, size=U)
    long_ = rng.random(U) < 0.02
    T[long_] = rng.integers(100, 301, size=int(long_.sum()))
    short = rng.integers(1, 31, size=U)
    if short_words:
        T[labels < 2] = short[labels < 2]
    cen, s = synth.make_centres(V, N, M, D, seed=4200 + N)
    x, off = synth.make_utterances(cen, s, labels, seed=4300 + N, lengths=T)
    ms = api.ModelSet.from_dict(synth.make_models(cen + 0.3 * s * rng.standard_normal(cen.shape), s))
    return x, off, labels, ms, s


@pytest.fixture(scope="module")
def corpus():
    cache = {}

    def get(N, short_words=True):
        if (N, short_words) not in cache:
            cache[(N, short_words)] = _corpus(N, short_words)
        return cache[(N, short_words)]
    return get


def _oracle_model(ms, v):
    return o.Model(ms.A[v], ms.c[v], ms.mu[v], ms.iv[v], ms.det[v], ms.words[v])


def _word(x, off, us):
    """The frames and offsets of utterances us, concatenated."""
    xv = np.concatenate([x[off[u]:off[u + 1]] for u in us])
    offv = np.concatenate([[0], np.cumsum(off[us + 1] - off[us])])
    return xv, offv


def _batching(c):
    return tuple(int(c.kernel_ms(k)) for k in ("res_batches", "res_batch_max", "res_teams"))


def _assert_kernels_agree(st, lp, st0, lp0):
    """k_fb_res (st, lp) against the windowed k_fb (st0, lp0) at the bars of test_forward_backward_kernels_agree."""
    fin, sf = np.isfinite(lp0), np.isfinite(st0)  # sum_logp is -inf for a word with an utterance shorter than its state chain
    assert (np.isfinite(lp) == fin).all() and (lp[~fin] == lp0[~fin]).all()
    assert np.allclose(lp[fin], lp0[fin], rtol=1e-8, atol=0)
    assert (np.isfinite(st) == sf).all() and (st[~sf] == st0[~sf]).all()
    assert np.allclose(st[sf], st0[sf], rtol=2e-5, atol=1e-6 * np.abs(st0[sf]).max())


@pytest.mark.parametrize("N", [2, 5, 8])  # odd and even row strides; N = 8 has the least shared memory per frame
def test_full_batches_match_oracle(corpus, N):
    """One E-step over the whole corpus in full and shared-memory-cut batches, several per team: log P of EVERY
    utterance (exactly -inf for T < N) and the statistics of EVERY word against the oracle at the bars of the C2 test.
    With about 300 utterances per word, one wrong short utterance moves its word's S0 well beyond 1e-4.  Then the
    windowed kernel (no batches, no counter) on the same corpus."""
    x, off, labels, ms, _ = corpus(N)
    T = np.diff(off)
    assert (T == 1).any() and set(labels[T < N]) <= {0, 1}
    c = api.Context(0)
    c.set_features(x, off)
    c.set_models(ms)
    stats, lpu = c.estep(labels)
    nb, bmax, teams = _batching(c)
    c.close()
    assert bmax == 16 and nb > -(-U // 16), (nb, bmax)        # full batches, and some cut by shared memory
    assert nb >= 2 * teams, (nb, teams)                         # teams take a second batch
    for v in range(V):
        us = np.nonzero(labels == v)[0]
        st, lp = o.estep(_oracle_model(ms, v), *_word(x, off, us))
        sp = api.split_stats(stats[v], N, M, D)
        fin = np.isfinite(lp)
        assert (fin == (T[us] >= N)).all(), v
        got = lpu[us]
        assert (got[~fin] == -np.inf).all() and (np.abs(got[fin] - lp[fin]) <= RTOL * np.abs(lp[fin])).all(), v
        if np.isfinite(st.sum_logp):
            assert abs(sp["sum_logp"] - st.sum_logp) <= RTOL * abs(st.sum_logp), v
        else:
            assert sp["sum_logp"] == st.sum_logp, v
        assert sp["n_utt"] == len(us), v
        for name in ("num_trans", "den_trans", "den_mix", "S0"):
            want = getattr(st, name)
            assert np.allclose(sp[name], want, rtol=RTOL, atol=1e-6 * np.abs(want).max()), (v, name)
        S0 = np.maximum(st.S0, 1e-300)[..., None]
        sd = np.sqrt(st.S2c / S0)
        assert (np.abs(sp["S1"] / S0 - st.S1 / S0) <= RTOL * np.maximum(np.abs(st.S1 / S0), sd)).all(), (v, "S1")
        assert np.allclose(sp["S2c"] / S0, st.S2c / S0, rtol=RTOL), (v, "S2c")
    w = api.Context(0)
    w.set_option("res_fb", 0)
    w.set_features(x, off)
    w.set_models(ms)
    st0, lp0 = w.estep(labels)
    assert _batching(w) == (0, 0, 0)
    w.close()
    _assert_kernels_agree(stats, lpu, st0, lp0)


def test_batch_composition_leaves_each_utterance_unchanged(corpus):
    """DESIGN section 5: no utterance's arithmetic depends on the batch it lands in.  The full map and a map with every
    third utterance masked both give full batches, of different utterances: every live utterance's log P is bit-identical
    between the two, and every masked one reads exactly 0."""
    x, off, labels, ms, _ = corpus(5)
    masked = labels.copy()
    masked[::3] = -1
    c = api.Context(0)
    c.set_features(x, off)
    c.set_models(ms)
    _, lp_full = c.estep(labels, download=False)
    b_full = _batching(c)
    _, lp_mask = c.estep(masked, download=False)
    b_mask = _batching(c)
    c.close()
    assert b_full[1] == b_mask[1] == 16 and b_full[0] > b_mask[0], (b_full, b_mask)
    live = masked >= 0
    assert (lp_mask[~live] == 0).all()
    assert np.array_equal(lp_mask[live], lp_full[live])


def test_batch_counter_across_launches_and_graph_replay(corpus):
    """The self-resetting batch counter: a launch that found it non-zero would process no batch and leave the previous
    call's results in place.  Every E-step of the tested context (graphs on: the first two calls under one map launch
    directly, the third captures, the fourth replays) is checked against the windowed kernel on the same models, and no
    two consecutive E-steps share both the models and the map, so a launch that did nothing cannot pass.  Maps in turn:
    full; every third utterance masked; 100 live utterances (fewer CTAs than SMs, so a different last claim); none;
    full again."""
    x, off, labels, ms, s = corpus(5, short_words=False)
    c = api.Context(0)
    ref = api.Context(0)
    ref.set_option("res_fb", 0)
    ref.set_option("graphs", 0)
    for ctx in (c, ref):
        ctx.set_features(x, off)
        ctx.set_models(ms)
    c.em_reset()
    rng = np.random.default_rng(4400)

    def estep(u2m):
        ref.set_models(c.get_models(D))
        st, lp = c.estep(u2m)
        st0, lp0 = ref.estep(u2m)
        _assert_kernels_agree(st, lp, st0, lp0)
        assert (lp[u2m < 0] == 0).all()
        return st, lp, _batching(c)

    def mstep():  # every word has live utterances
        _, nu, upd = c.mstep(threshold=-1.0)
        assert upd.all() and (nu > 0).all()

    masked = labels.copy()
    masked[::3] = -1
    few = np.full(U, -1, dtype=labels.dtype)
    few[::200] = labels[::200]
    none = np.full(U, -1, dtype=labels.dtype)
    for k in range(4):
        _, _, (nb, bmax, teams) = estep(labels)
        assert bmax == 16 and nb >= 2 * teams, (k, nb, teams)
        mstep()
    for k in range(4):  # the first call follows a full-map call that left finite log P at the masked utterances
        _, _, (nb, bmax, _) = estep(masked)
        assert bmax == 16, (k, nb, bmax)
        mstep()
    for k in range(2):  # 8 of the 64 words have live utterances: new models through set_models
        _, _, (nb, bmax, t) = estep(few)
        assert nb == 100 and bmax == 1 and t == 4 * min(100, teams // 4) and t < teams, (nb, bmax, t)
        m = c.get_models(D)
        m.mu += 0.05 * s * rng.standard_normal(m.mu.shape)
        c.set_models(m)
    st, lp, b = estep(none)
    assert (st == 0).all() and (lp == 0).all() and b == (0, 0, 0)
    for k in range(4):
        _, _, (nb, bmax, t) = estep(labels)
        assert bmax == 16 and t == teams, (k, nb, t)
        mstep()
    c.close()
    ref.close()
