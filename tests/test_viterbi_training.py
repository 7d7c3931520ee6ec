"""Viterbi (segmental k-means) training: hmmcu_estep_viterbi, the E-step whose state occupancies come from the best
state sequence instead of forward-backward, and hmmh_train_viterbi, the EM loop around it.

The device aligns on the single-precision training log-emissions, the oracle on double-precision ones, so a path may
legitimately differ where the oracle's decision between two predecessors is a near-tie.  Utterances whose smallest
decision margin along the oracle's path is below MARGIN are left out of the path comparison; on the seeded sets here
that excludes none (asserted, so that a change of the sets cannot quietly weaken the test)."""
import numpy as np
import pytest

from oracle import oracle as o
from speech_recognition_hmm_continuous_b200 import api, synth
from test_fb_res_batches import _corpus
from viterbi_oracle import decision_margin, estep_viterbi, log_emissions, path_counts

pytestmark = pytest.mark.gpu
RTOL = 1e-4     # the Baum-Welch E-step's bar against the oracle (test_estep_statistics_match_oracle)
SRTOL = 1e-6    # Viterbi scores against the oracle's
MARGIN = 1e-3   # near-tie bound of the path comparison


@pytest.fixture(scope="module")
def ctx():
    c = api.Context(0)
    yield c
    c.close()


def _oracle_model(ms, v):
    return o.Model(ms.A[v], ms.c[v], ms.mu[v], ms.iv[v], ms.det[v], ms.words[v])


def _synth(V, N, M, U, seed, tmin=40, tmax=120, dense=False):
    cen, s = synth.make_centres(V, N, M, 39, seed=seed)
    labels = np.arange(U) % V
    x, off = synth.make_utterances(cen, s, labels, seed=seed + 1, tmin=tmin, tmax=tmax)
    d = synth.make_models(cen, s)
    if dense:  # every transition allowed: the path may skip states and go back
        A = 0.9 * d["A"] + 0.1 / N
        d["A"] = A / A.sum(-1, keepdims=True)
    return api.ModelSet.from_dict(d), x, off, labels


def _dispatches(dense):
    """res_fb values to run: the per-utterance rows + k_fb_reduce (banded A only) and the atomics of the windowed path."""
    return [0] if dense else [1, 0]


def _host_counts(path, off, us, N):
    num, dt, dm = np.zeros((N, N)), np.zeros(N), np.zeros(N)
    for u in us:
        a, b, c = path_counts(path[off[u]:off[u + 1]], N)
        num += a
        dt += b
        dm += c
    return num, dt, dm


def _assert_mixture_stats(sp, st, x):
    """S0 / S1 / S2c at the bars of test_estep_statistics_match_oracle (x: all the context's features, whose centre the
    device's second-order sums are formed about)."""
    want = st.S0
    assert np.allclose(sp["S0"], want, rtol=RTOL, atol=1e-6 * np.abs(want).max()), "S0"
    S0 = np.maximum(st.S0, 1e-300)[..., None]
    occ = st.S0 > 1e-3 * st.S0.max()
    sd = np.sqrt(st.S2c / S0)
    assert (np.abs(sp["S1"] / S0 - st.S1 / S0)[occ] <= RTOL * np.maximum(np.abs(st.S1 / S0), sd)[occ]).all(), "S1"
    want2 = st.S2c / S0
    scale2 = want2 + (st.S1 / S0 - x.mean(0)) ** 2
    assert (np.abs(sp["S2c"] / S0 - want2)[occ] <= (RTOL * want2 + 2e-6 * scale2 + 1e-8)[occ]).all(), "S2c"


def _check_against_oracle(ms, x, off, labels, stats, lpu, path):
    """Paths (outside near-ties), scores, exact counts and mixture statistics of every word.  -> utterances excluded."""
    N, M, D = ms.N, ms.M, ms.D
    excluded = 0
    for v in range(ms.V):
        us = np.nonzero(labels == v)[0]
        mo = _oracle_model(ms, v)
        sp = api.split_stats(stats[v], N, M, D)
        for u in us:
            xu = x[off[u]:off[u + 1]]
            s, p = o.viterbi(mo, o.emissions(mo, xu, want_post=False)[0])
            if decision_margin(mo, log_emissions(mo, xu), p) > MARGIN:
                assert (path[off[u]:off[u + 1]] == p).all(), u
            else:
                excluded += 1
            if np.isfinite(s):
                assert abs(lpu[u] - s) <= SRTOL * abs(s), (u, lpu[u], s)
            else:
                assert lpu[u] == s, u
        # the counts are the device's path, exactly
        num, dt, dm = _host_counts(path, off, us, N)
        assert np.array_equal(sp["num_trans"], num) and np.array_equal(sp["den_trans"], dt) and np.array_equal(sp["den_mix"], dm)
        # the mixture sums of that path, and the scores' sum
        xv = np.concatenate([x[off[u]:off[u + 1]] for u in us])
        offv = np.concatenate([[0], np.cumsum(off[us + 1] - off[us])])
        st, sc, _ = estep_viterbi(mo, xv, offv, paths=[path[off[u]:off[u + 1]] for u in us])
        assert sp["n_utt"] == st.n_utt == len(us)
        assert abs(sp["sum_logp"] - st.sum_logp) <= RTOL * abs(st.sum_logp)
        _assert_mixture_stats(sp, st, x)
    return excluded


# ------------------------------------------------------------------ alignment, counts, statistics ----
CASES = [(N, M, dense) for N in (1, 3, 5, 8) for M in (1, 3, 16) for dense in (False, True) if not (N == 1 and dense)]


@pytest.mark.parametrize("N,M,dense", CASES)
def test_alignment_counts_and_statistics_match_oracle(ctx, N, M, dense):
    ms, x, off, labels = _synth(2, N, M, 6, seed=500 + 10 * N + M + (5 if dense else 0), dense=dense)
    ctx.set_features(x, off)
    ctx.set_models(ms)
    got = []
    for res_fb in _dispatches(dense):
        ctx.set_option("res_fb", res_fb)
        stats, lpu, path = ctx.estep_viterbi(labels, want_path=True)
        excluded = _check_against_oracle(ms, x, off, labels, stats, lpu, path)
        print("N=%d M=%d %s res_fb=%d: %d of %d utterances excluded as near-ties" % (N, M, "dense" if dense else "banded", res_fb, excluded, len(labels)))
        assert excluded == 0
        got.append((stats, lpu, path))
    ctx.set_option("res_fb", 1)
    if len(got) == 2:  # both dispatches: the same alignment, scores and counts; sum_logp only to rounding
        (s1, l1, p1), (s0, l0, p0) = got
        assert np.array_equal(p1, p0) and np.array_equal(l1, l0)
        tail = api.stats_size(N, M, ms.D) - 2
        assert np.array_equal(np.delete(s1, tail, axis=1), np.delete(s0, tail, axis=1))
        assert np.allclose(s1[:, tail], s0[:, tail], rtol=1e-12)


# ------------------------------------------------------------------------------------ edge cases ----
@pytest.mark.parametrize("res_fb", [1, 0])
def test_masked_short_and_single_frame_utterances(ctx, res_fb):
    """Masked utterances: no statistics, score 0, path -1.  T = 1 and T < N: score -inf, no occupancy, no counts, and
    sum_logp / n_utt as the Baum-Welch E-step gives them for the same utterances."""
    ctx.set_option("res_fb", res_fb)
    ms, x, off, labels = _synth(2, 5, 3, 6, seed=55)
    ctx.set_features(x, off)
    ctx.set_models(ms)
    full, _, fpath = ctx.estep_viterbi(labels, want_path=True)
    masked = labels.copy()
    masked[labels == 1] = -1
    part, lpu, path = ctx.estep_viterbi(masked, want_path=True)
    assert np.allclose(part[0], full[0], rtol=1e-12) and (part[1] == 0).all() and (lpu[labels == 1] == 0).all()
    for u in range(len(labels)):
        want = fpath[off[u]:off[u + 1]] if labels[u] == 0 else -1
        assert (path[off[u]:off[u + 1]] == want).all(), u
    # T = 1, T = 3 < N = 5, then a normal utterance
    off2 = np.array([0, 1, 4, off[1]], dtype=np.int64)
    ctx.set_features(x[:off[1]], off2)
    u2m = np.zeros(3, dtype=np.int32)
    stats, lpu, path = ctx.estep_viterbi(u2m, want_path=True)
    bw, bw_lp = ctx.estep(u2m)
    assert lpu[0] == -np.inf and lpu[1] == -np.inf and np.isfinite(lpu[2])
    sp, sb = api.split_stats(stats[0], 5, 3, 39), api.split_stats(bw[0], 5, 3, 39)
    assert sp["sum_logp"] == sb["sum_logp"] == -np.inf and sp["n_utt"] == sb["n_utt"] == 3
    num, dt, dm = _host_counts(path, off2, [2], 5)
    assert np.array_equal(sp["num_trans"], num) and np.array_equal(sp["den_trans"], dt) and np.array_equal(sp["den_mix"], dm)
    assert dm.sum() == off2[3] - off2[2]
    assert abs(sp["S0"].sum() - dm.sum()) <= 1e-4 * dm.sum()  # only the aligned frames carry mixture weight
    mo = _oracle_model(ms, 0)
    s, p = o.viterbi(mo, o.emissions(mo, x[off2[2]:off2[3]], want_post=False)[0])
    assert (path[off2[2]:off2[3]] == p).all() and abs(lpu[2] - s) <= SRTOL * abs(s)
    # an empty map and a map that masks everything
    allm = np.full(3, -1, dtype=np.int32)
    stats, lpu, path = ctx.estep_viterbi(allm, want_path=True)
    assert (stats == 0).all() and (lpu == 0).all() and (path == -1).all()
    ctx.set_features(np.zeros((0, 39)), np.zeros(1, dtype=np.int64))
    stats, lpu, path = ctx.estep_viterbi(np.zeros(0, dtype=np.int32), want_path=True)
    assert (stats == 0).all() and len(lpu) == 0 and len(path) == 0
    ctx.set_option("res_fb", 1)


@pytest.mark.parametrize("N", [2, 5, 8])
def test_short_utterance_corpus(N):
    """The corpus of test_fb_res_batches (20,000 utterances of 64 words, mostly 2..30 frames, words 0 and 1 with T = 1
    and T < N): per-utterance rows summed by k_fb_reduce at the batch shapes that corpus gives, against the windowed
    atomics and against the oracle (every utterance's path outside near-ties and score, every word's counts)."""
    x, off, labels, ms, _s = _corpus(N, True)
    c = api.Context(0)
    c.set_features(x, off)
    c.set_models(ms)
    stats, lpu, path = c.estep_viterbi(labels, want_path=True)
    assert c.kernel_ms("res_batch_max") == 16  # full batches of rows, as the Baum-Welch E-step cuts this corpus
    c.set_option("res_fb", 0)
    s0, l0, p0 = c.estep_viterbi(labels, want_path=True)
    c.close()
    assert np.array_equal(path, p0) and np.array_equal(lpu, l0)
    tail = api.stats_size(N, ms.M, ms.D) - 2
    assert np.array_equal(np.delete(stats, tail, axis=1), np.delete(s0, tail, axis=1))
    fin = np.isfinite(stats[:, tail])
    assert (np.isfinite(s0[:, tail]) == fin).all() and np.allclose(stats[fin, tail], s0[fin, tail], rtol=1e-12)
    T = np.diff(off)
    assert (lpu[T < N] == -np.inf).all() and np.isfinite(lpu[T >= N]).all()
    excluded = 0
    for u in range(len(labels)):
        mo = _oracle_model(ms, labels[u])
        xu = x[off[u]:off[u + 1]]
        s, p = o.viterbi(mo, o.emissions(mo, xu, want_post=False)[0])
        if not np.isfinite(s):
            assert lpu[u] == -np.inf
            continue
        assert abs(lpu[u] - s) <= SRTOL * abs(s), u
        if decision_margin(mo, log_emissions(mo, xu), p) > MARGIN:
            assert (path[off[u]:off[u + 1]] == p).all(), u
        else:
            excluded += 1
    print("N=%d: %d of %d utterances excluded as near-ties" % (N, excluded, len(labels)))
    assert excluded == 0
    # counts of every word from the path: frame pairs inside an utterance, frames of utterances with a finite score
    live = np.repeat(np.isfinite(lpu), T)
    word = np.repeat(labels, T)
    inner = np.ones(len(path), dtype=bool)
    inner[off[1:] - 1] = False
    inner &= live
    for v in range(ms.V):
        sp = api.split_stats(stats[v], N, ms.M, ms.D)
        fv, pv = live & (word == v), inner & (word == v)
        num = np.zeros((N, N))
        idx = np.nonzero(pv)[0]
        np.add.at(num, (path[idx], path[idx + 1]), 1.0)
        assert np.array_equal(sp["num_trans"], num), v
        assert np.array_equal(sp["den_trans"], np.bincount(path[pv], minlength=N).astype(float)), v
        assert np.array_equal(sp["den_mix"], np.bincount(path[fv], minlength=N).astype(float)), v
        assert sp["n_utt"] == (labels == v).sum()


# ---------------------------------------------------------------------------------- interleaving ----
def test_interleaved_with_baum_welch_graphs():
    """hmmcu_estep -> hmmcu_estep_viterbi -> hmmcu_estep -> hmmcu_estep_viterbi on one context, four calls each, so that
    both launch sequences are captured as graphs and replayed: every Baum-Welch result is bit-identical to a fresh
    context's, every Viterbi result to its own first call."""
    ms, x, off, labels = _synth(3, 5, 3, 9, seed=808)

    def fresh():
        c = api.Context(0)
        c.set_features(x, off)
        c.set_models(ms)
        return c
    f = fresh()
    bw_ref = f.estep(labels)
    f.close()
    c = fresh()
    vit_ref = None
    for block in range(4):
        for _ in range(4):
            if block % 2 == 0:
                st, lp = c.estep(labels)
                assert np.array_equal(st, bw_ref[0]) and np.array_equal(lp, bw_ref[1]), block
            else:
                got = c.estep_viterbi(labels, want_path=True)
                if vit_ref is None:
                    vit_ref = got
                for a, b in zip(got, vit_ref):
                    assert np.array_equal(a, b), block
    c.close()


# --------------------------------------------------------------------------------- training loop ----
def _py_train_viterbi(c, ms, labels, max_iter, threshold=1e-3):
    """hmmh_train_viterbi restated: estep_viterbi + the device M-step, the per-word stopping rule checked on the host."""
    c.set_models(ms)
    c.em_reset()
    V = ms.V
    active, old = np.ones(V, dtype=bool), np.ones(V)
    its, mean = np.zeros(V, dtype=np.int32), np.zeros(V)
    it = 0
    while active.any() and (max_iter <= 0 or it < max_iter):
        it += 1
        c.estep_viterbi(np.where(active[labels], labels, -1).astype(np.int32), download=False, want_logp=False)
        lp, nu, upd = c.mstep(threshold)
        for v in np.nonzero(active)[0]:
            assert bool(upd[v]) == (abs((old[v] - lp[v]) / old[v]) > threshold), (it, v)
            old[v] = lp[v]
            its[v], mean[v] = it, lp[v] / nu[v]
            if not upd[v]:
                active[v] = False
    return its, mean, c.get_models(ms.D)


def test_train_viterbi_equals_python_loop_and_host_mstep():
    ms0, x, off, labels = _synth(3, 5, 3, 12, seed=909, tmin=60, tmax=120)
    c = api.Context(0)
    c.set_features(x, off)
    ms0 = c.init_models(labels, 3, 5, 3)  # the reference's initial models: Viterbi training has something to move
    ms = ms0.copy()
    its, mean = c.train_viterbi(ms, labels, max_iter=20)
    its_p, mean_p, got = _py_train_viterbi(c, ms0, labels, 20)
    print("iterations", its, "mean", mean)
    assert np.array_equal(its, its_p) and np.array_equal(mean, mean_p)
    for name in ("A", "c", "mu", "iv", "det"):
        assert np.array_equal(getattr(ms, name), getattr(got, name)), name
    # three iterations against the host M-step on the downloaded statistics
    c.set_models(ms0)
    c.em_reset()
    want = ms0.copy()
    for it in range(3):
        stats, _, _ = c.estep_viterbi(labels)
        c.mstep(threshold=-1.0)
        api.mstep(want, stats)
        now = c.get_models(ms0.D)
        for name in ("A", "c", "mu", "iv", "det"):
            assert np.allclose(getattr(now, name), getattr(want, name), rtol=1e-9, atol=0), (it, name)
        want = now.copy()
    c.close()


def test_viterbi_then_baum_welch_recognises_held_out_set():
    """train_viterbi(max_iter=3) then train, against train alone, from the same initial models; both accuracies are
    printed."""
    V, N, M = 5, 5, 3
    cen, s = synth.make_centres(V, N, M, 39, seed=1701)
    lab = np.arange(10 * V) % V
    x, off = synth.make_utterances(cen, s, lab, seed=1702, tmin=60, tmax=120)
    xt, offt = synth.make_utterances(cen, s, lab, seed=1703, tmin=60, tmax=120)
    c = api.Context(0)
    c.set_features(x, off)
    ms0 = c.init_models(lab, V, N, M)
    bw = ms0.copy()
    c.train(bw, lab)
    vb = ms0.copy()
    its_v, _ = c.train_viterbi(vb, lab, max_iter=3)
    c.train(vb, lab)
    assert (its_v >= 1).all() and (its_v <= 3).all()
    c.set_features(xt, offt)
    acc = []
    for m in (bw, vb):
        c.set_models(m)
        label, _ = c.rank(c.forward_scores())
        acc.append(float((label == lab).mean()))
    c.close()
    print("held-out accuracy: Baum-Welch %.3f, Viterbi x3 then Baum-Welch %.3f" % tuple(acc))
    assert acc[1] >= acc[0]


# ------------------------------------------------------------------------------------- two ranks ----
def test_two_ranks_sum_viterbi_statistics():
    """Two contexts of one process as two ranks: peer_allreduce sums their Viterbi statistics in rank order, and the
    M-step on the sum equals the M-step after one Viterbi E-step over the union."""
    ms, x, off, labels = _synth(3, 5, 4, 12, seed=1313, tmin=60, tmax=120)
    U = len(labels)
    halves = [(0, U // 2), (U // 2, U)]
    ctxs = []
    for u0, u1 in halves:
        c = api.Context(0)
        c.set_features(x[off[u0]:off[u1]], off[u0:u1 + 1] - off[u0])
        c.set_models(ms)
        c.peer_export(2)
        ctxs.append(c)
    areas = [c.peer_area() for c in ctxs]
    for r_, c in enumerate(ctxs):
        c.peer_import_pointers(r_, 2, areas)
    local = [c.estep_viterbi(labels[u0:u1])[0] for c, (u0, u1) in zip(ctxs, halves)]
    for c in ctxs:
        c.peer_allreduce()
    got = [c.stats_download() for c in ctxs]
    assert not ctxs[0].peer_error() and not ctxs[1].peer_error()
    assert np.array_equal(got[0], got[1]) and np.array_equal(got[0], local[0] + local[1])
    for c in ctxs:
        c.em_reset()
        c.mstep(threshold=-1.0)
    m0, m1 = ctxs[0].get_models(ms.D), ctxs[1].get_models(ms.D)
    for name in ("A", "c", "mu", "iv", "det"):
        assert np.array_equal(getattr(m0, name), getattr(m1, name)), name
    for c in ctxs:
        c.close()
    c = api.Context(0)
    c.set_features(x, off)
    c.set_models(ms)
    full, _, _ = c.estep_viterbi(labels)
    counts = ms.N * ms.N + 2 * ms.N
    assert np.array_equal(full[:, :counts], got[0][:, :counts])  # integer counts: exact in any order
    assert np.allclose(full, got[0], rtol=1e-5, atol=1e-6 * np.abs(full).max())
    c.em_reset()
    c.mstep(threshold=-1.0)
    one = c.get_models(ms.D)
    c.close()
    # the parameters to the bars of test_golden_synth_c1_training (means relative to their standard deviation)
    assert np.array_equal(one.A, m0.A)
    assert np.allclose(one.c, m0.c, rtol=RTOL, atol=1e-9)
    assert np.allclose(1.0 / one.iv, 1.0 / m0.iv, rtol=RTOL)
    assert (np.abs(one.mu - m0.mu) <= RTOL * np.maximum(np.abs(m0.mu), np.sqrt(1.0 / m0.iv))).all()
    assert np.allclose(np.log(one.det), np.log(m0.det), rtol=RTOL, atol=1e-3)


def test_linked_primary_is_refused():
    """Viterbi training of multi-stream models is not supported: a linked primary fails with a message."""
    ms, x, off, labels = _synth(2, 5, 3, 4, seed=77)
    a, b = api.Context(0), api.Context(0)
    for c in (a, b):
        c.set_features(x, off)
        c.set_models(ms)
    a.link_streams([b])
    with pytest.raises(api.HmmCudaError, match="multi-stream"):
        a.estep_viterbi(labels)
    a.link_streams([])
    assert a.estep_viterbi(labels)[0] is not None
    a.close()
    b.close()
