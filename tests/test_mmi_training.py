"""MMI training on the device: hmmcu_estep_mmi (numerator and posterior-weighted denominator statistics),
hmmcu_mstep_ebw (the extended Baum-Welch update) and hmmh_train_mmi, against the numpy restatement in mmi_oracle.py.

The hypotheses and weights are recomputed in numpy from the device's own forward scores; on the seeded sets no
posterior lies within 1e-9 (relative) of the floor or of a rank cut (asserted), so both sides pick the same words."""
import types

import numpy as np
import pytest

from mmi_oracle import MIN_POST, ebw, hypotheses, mmi_buffer, model
from oracle import oracle as o
from speech_recognition_hmm_continuous_b200 import api, synth
from test_viterbi_training import RTOL, _assert_mixture_stats, _dispatches, _synth

pytestmark = pytest.mark.gpu


def _kappa(S, label, spread=3.0):
    """An acoustic scale at which the median utterance's best competitor sits `spread` nats below its label."""
    gaps = []
    for u in range(S.shape[0]):
        if label[u] >= 0 and np.isfinite(S[u, label[u]]):
            gaps.append(abs(S[u, label[u]] - np.max(np.delete(S[u], label[u]))))
    return spread / max(float(np.median(gaps)), 1e-9)


@pytest.fixture(scope="module")
def ctx():
    c = api.Context(0)
    yield c
    c.close()


def _assert_separated(a, label, H):
    """No posterior within 1e-9 relative of the floor or of the rank cut after H - 1 competitors."""
    for u in range(a.shape[0]):
        if label[u] < 0 or not np.isfinite(a[u]).any():
            continue
        p = np.sort(np.exp(np.delete(a[u], label[u])))[::-1]
        assert (np.abs(p - MIN_POST) > 1e-9 * MIN_POST).all(), u
        if len(p) >= H and p[H - 2] >= MIN_POST:
            assert abs(p[H - 2] - p[H - 1]) > 1e-9 * p[H - 2], u


def _check_buffer(ctx, ms, x, off, label, S, kappa, H, stats, exact=True):
    """Block 0 against hmmcu_estep bit for bit; block 1 against the oracle at the Baum-Welch bars, its tail to 1e-12.
    exact=False: the forward-backward of k_fb adds its transition sums and log P by atomics, so two E-steps on that path
    agree up to the order of those sums (1e-12) rather than bit for bit."""
    N, M, D = ms.N, ms.M, ms.D
    hyps, term, a = hypotheses(S, label, kappa, H)
    _assert_separated(a, label, H)
    want = mmi_buffer(ms, x, off, label, S, kappa, H)
    ss = api.stats_size(N, M, D)
    for v in range(ms.V):
        sp, wp = api.split_stats(stats[1, v], N, M, D), api.split_stats(want[1, v], N, M, D)
        if wp["S0"].sum() > 0:
            _assert_mixture_stats(sp, types.SimpleNamespace(S0=wp["S0"], S1=wp["S1"], S2c=wp["S2c"]), x)
        for name in ("num_trans", "den_trans", "den_mix"):
            assert np.allclose(sp[name], wp[name], rtol=RTOL, atol=1e-6 * max(np.abs(wp[name]).max(), 1.0)), (v, name)
        inc = [u for u in range(len(label)) if label[u] == v and np.isfinite(term[u])]
        assert stats[1, v, ss - 1] == len(inc)
        t = float(np.sum(term[inc])) if inc else 0.0
        assert abs(stats[1, v, ss - 2] - t) <= 1e-12 * max(abs(t), 1e-300), (v, stats[1, v, ss - 2], t)
    num, _ = ctx.estep(label)
    if exact:
        assert np.array_equal(stats[0], num)  # the numerator is hmmcu_estep's statistics, bit for bit
    else:
        assert np.allclose(stats[0], num, rtol=1e-12, atol=0)
    return hyps


CASES = [(N, M, dense) for N in (3, 5, 8) for M in (1, 3, 16) for dense in (False, True)]


@pytest.mark.parametrize("N,M,dense", CASES)
def test_mmi_statistics_match_oracle(ctx, N, M, dense):
    ms, x, off, labels = _synth(3, N, M, 9, seed=900 + 10 * N + M + (5 if dense else 0), tmin=20, tmax=60, dense=dense)
    ctx.set_features(x, off)
    ctx.set_models(ms)
    try:
        for res_fb in _dispatches(dense):
            ctx.set_option("res_fb", res_fb)
            S = ctx.forward_scores()
            kappa = _kappa(S, labels)
            stats = ctx.estep_mmi(labels, kappa, 4)
            assert stats.shape == (2, ms.V, api.stats_size(N, M, ms.D))
            assert np.array_equal(ctx.forward_scores(), S)
            hyps = _check_buffer(ctx, ms, x, off, labels, S, kappa, 4, stats, exact=res_fb == 1 and not dense)
            rounds = max(len(h) for h in hyps)
            assert rounds >= 2
            assert ctx.kernel_ms("mmi_rounds") == rounds
            print("N=%d M=%d %s res_fb=%d: %d rounds" % (N, M, "dense" if dense else "banded", res_fb, rounds))
    finally:
        ctx.set_option("res_fb", 1)


def test_mmi_edge_cases(ctx):
    """max_hyp = 1, a kappa small enough for several rounds, masked labels, an utterance with T < N (left out of block 1),
    and two calls that are bit-identical."""
    V, N, M = 4, 5, 3
    cen, s = synth.make_centres(V, N, M, 39, seed=4242)
    labels = np.arange(13) % V
    lengths = np.full(13, 30)
    lengths[5] = 3  # T < N: no path to the final state
    x, off = synth.make_utterances(cen, s, labels, seed=4243, lengths=lengths)
    ms = api.ModelSet.from_dict(synth.make_models(cen, s))
    ctx.set_features(x, off)
    ctx.set_models(ms)
    S = ctx.forward_scores()
    lab = labels.astype(np.int32).copy()
    lab[[2, 7]] = -1
    k0 = _kappa(S, lab)
    for kappa, H in ((k0, 1), (k0 / 10, 6), (k0, 16)):
        first = ctx.estep_mmi(lab, kappa, H)
        hyps = _check_buffer(ctx, ms, x, off, lab, S, kappa, H, first)
        assert hyps[5] == [] and hyps[2] == [] and hyps[7] == []
        assert ctx.kernel_ms("mmi_rounds") == max(len(h) for h in hyps)
        if H == 1:
            assert ctx.kernel_ms("mmi_rounds") == 1
        if H == 6:
            assert ctx.kernel_ms("mmi_rounds") >= 3
        again = ctx.estep_mmi(lab, kappa, H)
        assert np.array_equal(first, again)


def test_device_ebw_matches_host_and_repacks(ctx):
    ms, x, off, labels = _synth(3, 5, 4, 9, seed=5151, tmin=20, tmax=60)
    ctx.set_features(x, off)
    ctx.set_models(ms)
    kappa = _kappa(ctx.forward_scores(), labels)
    for E, tau in ((2.0, 100.0), (1.5, 0.0)):
        stats = ctx.estep_mmi(labels, kappa, 4)
        want = api.mstep_ebw(ctx.get_models(ms.D), stats[0], stats[1], E, tau)
        ctx.mstep_ebw(E, tau)
        got = ctx.get_models(ms.D)
        for name in ("mu", "iv", "det"):
            a, b = getattr(got, name), getattr(want, name)
            assert np.allclose(a, b, rtol=1e-12, atol=0), (name, np.abs(a - b).max())
        assert np.array_equal(got.A, ms.A) and np.array_equal(got.c, ms.c)
        fresh = api.Context(0)
        fresh.set_features(x, off)
        fresh.set_models(got)
        assert np.array_equal(ctx.forward_scores(), fresh.forward_scores())
        fresh.close()


def test_train_mmi_matches_the_python_loop_and_the_oracle(ctx):
    ms, x, off, labels = _synth(3, 5, 3, 9, seed=6161, tmin=20, tmax=50)
    ctx.set_features(x, off)
    ctx.set_models(ms)
    kappa = _kappa(ctx.forward_scores(), labels)
    # Bit for bit against the same loop from the Context pieces.  The EBW update shrinks some variances far enough that
    # the accuracy guard sends the second iteration's E-steps to the CUDA-core path, whose accumulators add by double
    # atomics (not reproducible in the last bit).  So both loops run with the tensor-core path pinned ("tc_emis" 2), whose
    # sums meet in a fixed order.
    ctx.set_option("tc_emis", 2)
    try:
        a = ms.copy()
        obj = ctx.train_mmi(a, labels, kappa, 4, E=2.0, tau=100.0, iterations=2)
        ctx.set_models(ms)
        want = []
        for _ in range(2):
            st = ctx.estep_mmi(labels, kappa, 4)
            assert ctx.kernel_ms("tc_active") == 1.0
            want.append(-st[1, :, -2].sum() / st[1, :, -1].sum())
            ctx.mstep_ebw(2.0, 100.0)
        b = ctx.get_models(ms.D)
    finally:
        ctx.set_option("tc_emis", 1)
    assert np.array_equal(obj, np.array(want))
    for name in ("mu", "iv", "det", "A", "c"):
        assert np.array_equal(getattr(a, name), getattr(b, name)), name
    # the oracle (double-precision scores and statistics, the numpy update) against the default, guarded path
    a = ms.copy()
    obj = ctx.train_mmi(a, labels, kappa, 4, E=2.0, tau=100.0, iterations=2)
    c = ms.copy()
    G, o0 = ms.N * ms.M, ms.N * ms.N + 2 * ms.N
    occ = np.ones((ms.V, G), dtype=bool)
    for k in range(2):
        S = np.array([[o.forward_score(model(c, v), x[off[u]:off[u + 1]]) for v in range(c.V)] for u in range(len(labels))])
        buf = mmi_buffer(c, x, off, labels, S, kappa, 4)
        assert abs(-buf[1, :, -2].sum() / buf[1, :, -1].sum() - obj[k]) <= 1e-4 * abs(obj[k])
        s0 = buf[0, :, o0:o0 + G] + buf[1, :, o0:o0 + G]
        occ &= s0 > 1e-3 * s0.max()  # (a Gaussian with next to no occupancy amplifies the emissions' rounding)
        ebw(c, buf[0], buf[1], 2.0, 100.0)
    sd = np.sqrt(1.0 / c.iv).reshape(ms.V, G, -1)[occ]
    dmu = np.abs(a.mu - c.mu).reshape(ms.V, G, -1)[occ]
    dvar = np.abs(1.0 / a.iv - 1.0 / c.iv).reshape(ms.V, G, -1)[occ] / sd ** 2
    print("oracle loop: %d of %d Gaussians compared, max |dmu| / sd %.2e, |dvar| / var median %.2e max %.2e"
          % (occ.sum(), occ.size, (dmu / sd).max(), np.median(dvar), dvar.max()))
    # The device's statistics come from single-precision emissions (1e-6 relative).  A dimension whose constant D is
    # its own 2 D_min gets a new variance that is a difference of nearly equal terms, which amplifies that noise: the
    # bar on the largest variance deviation is wide, the typical one is held at 1e-5.
    assert (dmu <= 1e-3 * sd).all() and np.median(dvar) <= 1e-5 and (dvar <= 5e-2).all()


def _confusable(seed, sets, tmin=8, tmax=16):
    """Word pairs 2k, 2k + 1 that share every state but the last, whose centres lie close (0.15 sigma per dimension);
    short utterances -> [(x, off, labels)] for every count in `sets`, all from the same words."""
    V, N, Mg = 6, 4, 4
    cen, s = synth.make_centres(V, N, Mg, 39, seed=seed)
    rng = np.random.default_rng(seed + 1)
    for k in range(0, V, 2):
        cen[k + 1, :N - 1] = cen[k, :N - 1]
        cen[k + 1, N - 1] = cen[k, N - 1] + 0.15 * s * rng.standard_normal(cen[k, N - 1].shape)
    out = []
    for i, U in enumerate(sets):
        labels = np.arange(U) % V
        out.append(synth.make_utterances(cen, s, labels, seed=seed + 7 + 100 * i, tmin=tmin, tmax=tmax) + (labels,))
    return out


def test_mmi_raises_the_objective_on_a_confusable_corpus(ctx):
    V, N, M = 6, 4, 1
    (x, off, labels), (xt, offt, labt) = _confusable(777, (240, 120))
    ctx.set_features(x, off)
    ms = ctx.init_models(labels, V, N, M)
    ctx.train(ms, labels, max_iter=20)
    acc = lambda c: float((np.argmax(c.forward_scores(), axis=1) == (labels if c is ctx else labt)).mean())
    held = api.Context(0)
    held.set_features(xt, offt)
    held.set_models(ms)
    acc_ml, held_ml = acc(ctx), acc(held)
    ctx.set_models(ms)
    kappa = _kappa(ctx.forward_scores(), labels, 1.0)
    mm = ms.copy()
    obj = list(ctx.train_mmi(mm, labels, kappa, 8, E=2.0, tau=100.0, iterations=4))
    ctx.set_models(mm)
    st = ctx.estep_mmi(labels, kappa, 8)
    obj.append(-st[1, :, -2].sum() / st[1, :, -1].sum())
    acc_mmi = acc(ctx)
    held.set_models(mm)
    held_mmi = acc(held)
    held.close()
    print("ML: train %.3f held-out %.3f   MMI x4: train %.3f held-out %.3f   objective %s" % (acc_ml, held_ml, acc_mmi, held_mmi, obj))
    assert acc_ml < 1.0
    assert all(b > a for a, b in zip(obj, obj[1:])), obj
    assert acc_mmi >= acc_ml


def test_refusals(ctx):
    ms, x, off, labels = _synth(2, 5, 3, 4, seed=77)
    ctx.set_features(x, off)
    ctx.set_models(ms)
    kappa = 0.01
    for kappa, H in ((0.0, 4), (-1.0, 4), (1.0, 0), (1.0, 17)):
        with pytest.raises(api.HmmCudaError):
            ctx.estep_mmi(labels, kappa, H)
    ctx.estep(labels)
    with pytest.raises(api.HmmCudaError, match="estep_mmi"):
        ctx.mstep_ebw(2.0, 100.0)  # after a plain E-step
    ctx.estep_mmi(labels, kappa, 4)
    for E in (1.0, 0.5):
        with pytest.raises(api.HmmCudaError):
            ctx.mstep_ebw(E, 100.0)
    with pytest.raises(api.HmmCudaError):
        ctx.mstep_ebw(2.0, -1.0)
    ctx.em_reset()
    with pytest.raises(api.HmmCudaError, match="mstep"):
        ctx.mstep()  # the MMI buffer is not a Baum-Welch statistics vector
    p = api.Context(0)
    p.set_features(x, off)
    p.set_models(ms)
    p.peer_export(1)
    p.peer_import_pointers(0, 1, [p.peer_area()])
    p.estep_mmi(labels, kappa, 4)
    with pytest.raises(api.HmmCudaError, match="changed size"):
        p.peer_allreduce()
    p.close()
    a, b = api.Context(0), api.Context(0)
    for c in (a, b):
        c.set_features(x, off)
        c.set_models(ms)
    a.link_streams([b])
    with pytest.raises(api.HmmCudaError, match="multi-stream"):
        a.estep_mmi(labels, kappa, 4)
    a.link_streams([])
    assert a.estep_mmi(labels, kappa, 4) is not None
    a.close()
    b.close()


def test_baum_welch_after_mmi_matches_a_fresh_context(ctx):
    """Graph and map caches: a Baum-Welch E-step + M-step after MMI iterations equals the same on a fresh context.
    Transition sums, log P and the counts are compared bit for bit; the mixture sums to 1e-12: after the EBW updates the
    accuracy guard can send these E-steps to the CUDA-core accumulators, which add by double atomics (5e-16 seen)."""
    ms, x, off, labels = _synth(3, 5, 4, 9, seed=8181, tmin=20, tmax=60)
    ctx.set_features(x, off)
    ctx.set_models(ms)
    for _ in range(3):  # long enough for the Baum-Welch graph to be captured before the MMI iterations
        ctx.estep(labels, download=False)
    mm = ms.copy()
    ctx.train_mmi(mm, labels, _kappa(ctx.forward_scores(), labels), 4, iterations=2)
    fresh = api.Context(0)
    fresh.set_features(x, off)
    for c in (ctx, fresh):
        c.set_models(mm)
    head = ms.N * ms.N + 2 * ms.N
    for _ in range(4):  # plain launches, then the captured graph, then its replay
        got, lg = ctx.estep(labels)
        want, lw = fresh.estep(labels)
        assert np.array_equal(got[:, :head], want[:, :head]) and np.array_equal(got[:, -2:], want[:, -2:]) and np.array_equal(lg, lw)
        assert np.allclose(got, want, rtol=1e-12, atol=0)
    for c in (ctx, fresh):
        c.em_reset()
        c.mstep(threshold=-1.0)
    g, w = ctx.get_models(ms.D), fresh.get_models(ms.D)
    assert np.array_equal(g.A, w.A)
    for name in ("c", "mu", "iv", "det"):
        assert np.allclose(getattr(g, name), getattr(w, name), rtol=1e-12, atol=0), name
    fresh.close()
