"""Parity of the CUDA path (through the C ABI, libhmmcu.so) against the CPU oracle and the golden
vectors the reference produced.  Tolerances are BASELINE.json's: labels and Viterbi state sequences
bit-exact; log-likelihoods and re-estimated parameters within 1e-4 relative."""
import glob
import json
import os
import re
import subprocess

import numpy as np
import pytest

from oracle import oracle as o
from oracle import ref as r
from speech_recognition_hmm_continuous_b200 import api, synth
from cli_lists import write_list

pytestmark = pytest.mark.gpu
RTOL = 1e-4  # north_star tolerance for floating-point results


@pytest.fixture(scope="module", params=["tc", "simt"])
def ctx(request):
    """Every parity test runs twice: emissions on the tcgen05 tensor-core kernel (the default path) and
    on the CUDA-core kernel (hmmcu_set_option "tc_emis" = 0)."""
    c = api.Context(0)
    c.set_option("tc_emis", 1 if request.param == "tc" else 0)
    c.path = request.param
    yield c
    c.close()


def _oracle_model(ms, v):
    return o.Model(ms.A[v], ms.c[v], ms.mu[v], ms.iv[v], ms.det[v], ms.words[v])


def _synth(V, N, M, U, seed, tmin=60, tmax=120, D=39):
    cen, s = synth.make_centres(V, N, M, D, seed=seed)
    labels = np.arange(U) % V
    x, off = synth.make_utterances(cen, s, labels, seed=seed + 1, tmin=tmin, tmax=tmax)
    ms = api.ModelSet.from_dict(synth.make_models(cen, s))
    return ms, x, off, labels


def _assert_params_close(ms, v, mo, tol=RTOL):
    var_g, var_o = 1.0 / ms.iv[v], 1.0 / mo.iv
    assert np.allclose(ms.A[v], mo.A, rtol=tol, atol=1e-12), "transitions"
    assert np.allclose(ms.c[v], mo.c, rtol=tol, atol=1e-9), "weights"
    assert np.allclose(var_g, var_o, rtol=tol), "variances"
    assert (np.abs(ms.mu[v] - mo.mu) <= tol * np.maximum(np.abs(mo.mu), np.sqrt(var_o))).all(), "means"


# ------------------------------------------------------------------------------- emissions ----
@pytest.mark.parametrize("N,M", [(5, 3), (5, 16), (3, 128), (6, 1), (1, 1), (8, 2)])
def test_emissions_match_oracle(ctx, N, M):
    ms, x, off, labels = _synth(2, N, M, 3, seed=100 + N * M, tmin=50, tmax=130)
    ctx.set_features(x, off)
    ctx.set_models(ms)
    for u, v in ((0, 0), (1, 1), (2, 1)):
        logb, post = ctx.emissions(u, v)
        b, p = o.emissions(_oracle_model(ms, v), x[off[u]:off[u + 1]])
        with np.errstate(divide="ignore"):
            lb = np.log(b)
        fin = np.isfinite(lb)
        assert np.allclose(logb[fin], lb[fin], rtol=2e-6, atol=2e-4)
        assert np.abs(post - p).max() < 2e-4


# ------------------------------------------------------------------------- forward scoring ----
def test_forward_scores_and_labels_match_oracle(ctx):
    ms, x, off, labels = _synth(7, 5, 3, 21, seed=7)
    ctx.set_features(x, off)
    ctx.set_models(ms)
    got = ctx.forward_scores()
    assert ctx.kernel_ms("tc_active") == (1 if ctx.path == "tc" else 0)
    want = np.array([[o.forward_score(_oracle_model(ms, v), x[off[u]:off[u + 1]]) for v in range(ms.V)] for u in range(len(labels))])
    assert np.allclose(got, want, rtol=RTOL, atol=0)
    assert np.abs(got / want - 1).max() < 1e-6  # in practice far inside the bar
    label, second = ctx.rank(got)
    order = np.stack([o.rank(w) for w in want])
    assert (label == order[:, 0]).all() and (second == order[:, 1]).all()
    assert (label == labels).all()


def test_golden_synth_c1_recognition(ctx, golden_dir):
    g = np.load(os.path.join(golden_dir, "synth_c1.npz"))
    V, N, M, D = int(g["V"]), int(g["N"]), int(g["M"]), int(g["D"])
    cen, s = synth.make_centres(V, N, M, D, seed=1234)
    xt, offt = synth.make_utterances(cen, s, g["test_labels"], seed=4321, tmin=70, tmax=110)
    ms = api.ModelSet(g["trained_A"], g["trained_c"], g["trained_mu"], g["trained_iv"], g["trained_det"])
    ctx.set_features(xt, offt)
    ctx.set_models(ms)
    got = ctx.forward_scores()
    assert np.allclose(got, g["score"], rtol=RTOL, atol=0)
    label, second = ctx.rank(got)
    assert (label == g["order"][:, 0]).all() and (second == g["order"][:, 1]).all()


def test_rank_rule_with_nan_and_inf(ctx):
    rng = np.random.default_rng(3)
    sc = rng.standard_normal((200, 9))
    sc[rng.random(sc.shape) < 0.25] = np.nan
    sc[rng.random(sc.shape) < 0.1] = -np.inf
    sc[:, 4] = sc[:, 2]
    sc[0] = np.nan
    label, second = ctx.rank(sc)
    want = np.stack([o.rank(row) for row in sc])
    assert (label == want[:, 0]).all() and (second == want[:, 1]).all()
    l1, s1 = ctx.rank(sc[:, :1])
    assert (l1 == 0).all()


def test_shipped_fixtures_degenerate_regime(ctx, golden_dir):
    """The reference's own 13 feature files against its 13 diagonal models: most cells underflow to
    NaN / -inf in the reference.  With emulate_underflow the recognised labels must be the same."""
    kat = json.load(open(os.path.join(golden_dir, "kat_diag.json")))
    km = np.load(os.path.join(golden_dir, "kat_models.npz"))
    words = [str(w) for w in km["words"]]
    ms = api.ModelSet(km["A"], km["c"], km["mu"], km["iv"], km["det"], words)
    files = sorted(glob.glob(os.path.join(golden_dir, "perfil", "*.perfil")))
    xs = [api.read_features(f) for f in files]
    off = np.concatenate([[0], np.cumsum([len(a) for a in xs])])
    ctx.set_features(np.concatenate(xs), off)
    ctx.set_models(ms)
    got = ctx.forward_scores(emulate_underflow=True)
    assert ctx.kernel_ms("kappa") > 1e4 and ctx.kernel_ms("tc_active") == 0  # raw-Hz data: the accuracy guard picks the direct form
    label, second = ctx.rank(got)
    for u, rec in enumerate(kat["recognition"]):
        ref_score = {w: float(v.replace("-nan", "nan")) for w, v in rec["sorted"]}
        assert words[label[u]] == rec["sorted"][0][0], rec["spoken"]
        for v, w in enumerate(words):
            rs = ref_score[w]
            if np.isfinite(rs):
                assert np.isfinite(got[u, v]) and abs(got[u, v] - rs) <= RTOL * abs(rs), (rec["spoken"], w)
            else:
                assert not np.isfinite(got[u, v]), (rec["spoken"], w, got[u, v], rs)


# --------------------------------------------------------------------------------- E-step ----
@pytest.mark.parametrize("N,M,V,U", [(5, 3, 3, 9), (5, 16, 2, 6), (3, 128, 1, 2), (6, 1, 2, 4), (1, 2, 1, 2), (8, 2, 2, 4)])
def test_estep_statistics_match_oracle(ctx, N, M, V, U):
    ms, x, off, labels = _synth(V, N, M, U, seed=31 + N + M)
    ctx.set_features(x, off)
    ctx.set_models(ms)
    stats, lpu = ctx.estep(labels)
    for v in range(V):
        us = np.nonzero(labels == v)[0]
        xv = np.concatenate([x[off[u]:off[u + 1]] for u in us])
        offv = np.concatenate([[0], np.cumsum([off[u + 1] - off[u] for u in us])])
        st, lp = o.estep(_oracle_model(ms, v), xv, offv)
        sp = api.split_stats(stats[v], N, M, ms.D)
        assert np.allclose(lpu[us], lp, rtol=RTOL)
        assert abs(sp["sum_logp"] - st.sum_logp) <= RTOL * abs(st.sum_logp) and sp["n_utt"] == len(us)
        for name in ("num_trans", "den_trans", "den_mix", "S0"):
            want = getattr(st, name)
            assert np.allclose(sp[name], want, rtol=RTOL, atol=1e-6 * np.abs(want).max()), name
        # first / second order sums: compare through the quantities the M-step forms from them
        S0 = np.maximum(st.S0, 1e-300)[..., None]
        occ = st.S0 > 1e-3 * st.S0.max()
        sd = np.sqrt(st.S2c / S0)
        assert (np.abs(sp["S1"] / S0 - st.S1 / S0)[occ] <= RTOL * np.maximum(np.abs(st.S1 / S0), sd)[occ]).all(), "S1"
        # second-order sums.  The tensor-core path forms sum w (x - mu)^2 from raw moments about the data
        # centre (in double, from FP32-accurate sums), so its error is absolute in the moment's own scale
        # E_w[(x - centre)^2], not relative to a variance that happens to be tiny because a one-frame
        # Gaussian sits on its mean (such variances are floored at 1e-5 by the M-step anyway, T-FS:1942).
        want2 = st.S2c / S0
        scale2 = want2 + (st.S1 / S0 - x.mean(0)) ** 2
        assert (np.abs(sp["S2c"] / S0 - want2)[occ] <= (RTOL * want2 + 2e-6 * scale2 + 1e-8)[occ]).all(), "S2c"


def test_estep_masked_utterances_and_empty(ctx):
    ms, x, off, labels = _synth(2, 5, 3, 6, seed=55)
    ctx.set_features(x, off)
    ctx.set_models(ms)
    full, _ = ctx.estep(labels)
    masked = labels.copy()
    masked[labels == 1] = -1
    part, lpu = ctx.estep(masked)
    assert np.allclose(part[0], full[0], rtol=1e-12) and (part[1] == 0).all() and (lpu[labels == 1] == 0).all()
    ctx.set_features(np.zeros((0, 39)), np.zeros(1, dtype=np.int64))
    st, lp = ctx.estep(np.zeros(0, dtype=np.int32))
    assert (st == 0).all() and len(lp) == 0


def test_short_and_single_frame_utterances(ctx):
    """T = 1 and T < N: the final state is unreachable -> logP = -inf and no occupancy, as in the
    reference (log(0) at T-FS:1549)."""
    ms, x, off, labels = _synth(1, 5, 2, 3, seed=66, tmin=40, tmax=50)
    off2 = np.array([0, 1, 4, off[1]], dtype=np.int64)
    ctx.set_features(x[: off[1]], off2)
    ctx.set_models(ms)
    stats, lpu = ctx.estep(np.zeros(3, dtype=np.int32))
    mo = _oracle_model(ms, 0)
    with np.errstate(all="ignore"):
        want = [o.forward_score(mo, x[off2[u]:off2[u + 1]]) for u in range(3)]
    assert lpu[0] == -np.inf and lpu[1] == -np.inf and want[0] == -np.inf and want[1] == -np.inf
    assert abs(lpu[2] - want[2]) <= RTOL * abs(want[2])
    sc = ctx.forward_scores()
    assert sc[0, 0] == -np.inf and sc[1, 0] == -np.inf


def test_device_mstep_matches_host_mstep(ctx):
    """hmmcu_mstep (M-step + stopping rule on the device) against hmmh_mstep, the host restatement that is
    bit-exact with the compiled reference (tests/test_host_cpu.py): same parameters to rounding."""
    ms, x, off, labels = _synth(3, 5, 3, 9, seed=77)
    ctx.set_features(x, off)
    ctx.set_models(ms)
    ctx.em_reset()
    want = ms.copy()
    for it in range(2):
        stats, _ = ctx.estep(labels)
        lp, nu, upd = ctx.mstep()
        api.mstep(want, stats)
        got = ctx.get_models(ms.D)
        assert upd.all() and (nu == 3).all()
        assert np.allclose(lp, [api.split_stats(stats[v], 5, 3, ms.D)["sum_logp"] for v in range(3)], rtol=1e-15)
        for name in ("A", "c", "mu", "iv", "det"):
            assert np.allclose(getattr(got, name), getattr(want, name), rtol=1e-12, atol=0), (it, name)
        want = got.copy()  # continue both from the same point
    # a model whose log-probability no longer moves is frozen, and stays frozen
    lp, nu, upd = ctx.mstep(threshold=1e9)
    assert not upd.any()
    frozen = ctx.get_models(ms.D)
    ctx.estep(labels)
    lp, nu, upd = ctx.mstep(threshold=-1.0)
    assert not upd.any() and np.array_equal(ctx.get_models(ms.D).mu, frozen.mu)


# ------------------------------------------------------------------------------- training ----
def test_golden_synth_c1_training(ctx, golden_dir):
    """Whole EM loop on the GPU from the reference's own initial models; iteration counts equal, mean
    log-probabilities and every re-estimated parameter within 1e-4 of what the reference wrote."""
    g = np.load(os.path.join(golden_dir, "synth_c1.npz"))
    V, N, M, D = int(g["V"]), int(g["N"]), int(g["M"]), int(g["D"])
    cen, s = synth.make_centres(V, N, M, D, seed=1234)
    x, off = synth.make_utterances(cen, s, g["train_labels"], seed=1234, tmin=70, tmax=110)
    ms = api.ModelSet(g["init_A"], g["init_c"], g["init_mu"], g["init_iv"], g["init_det"])
    ctx.set_features(x, off)
    ctx.set_models(ms)
    stats, _ = ctx.estep(g["train_labels"])
    for v in range(V):
        sp = api.split_stats(stats[v], N, M, D)
        for name in ("num_trans", "den_trans", "den_mix", "S0"):
            want = g["stat_" + name][v]
            assert np.allclose(sp[name], want, rtol=RTOL, atol=1e-6 * np.abs(want).max()), name
        assert abs(sp["sum_logp"] - g["stat_sum_logp"][v]) <= RTOL * abs(g["stat_sum_logp"][v])
    its, mean = ctx.train(ms, g["train_labels"])
    assert (its == g["iterations"]).all()
    assert np.allclose(mean, g["mean_logp"], rtol=RTOL)
    for v in range(V):
        mo = o.Model(g["trained_A"][v], g["trained_c"][v], g["trained_mu"][v], g["trained_iv"][v], g["trained_det"][v])
        _assert_params_close(ms, v, mo)
        assert np.allclose(np.log(ms.det[v]), np.log(mo.det), rtol=RTOL, atol=1e-3)


def test_shipped_kats_training(ctx, golden_dir):
    """The 13 shipped feature files, N=6 M=1 (SURVEY 4.5): host init + GPU EM loop reproduces the
    reference's mean log-probability and iteration count."""
    kat = json.load(open(os.path.join(golden_dir, "kat_diag.json")))
    for word, rec in kat["train"].items():
        x = api.read_features(os.path.join(golden_dir, "perfil", rec["file"]))
        off = np.array([0, len(x)], dtype=np.int64)
        ms = api.init_model(6, 1, x, off, word)
        ctx.set_features(x, off)
        its, mean = ctx.train(ms, np.zeros(1, dtype=np.int32))
        assert its[0] == rec["iterations"], word
        assert abs(mean[0] - rec["mean_logp"]) <= RTOL * abs(rec["mean_logp"]), word


# -------------------------------------------------------------------------------- Viterbi ----
def test_viterbi_paths_bit_exact_and_scores(ctx):
    ms, x, off, labels = _synth(4, 5, 3, 12, seed=91)
    ctx.set_features(x, off)
    ctx.set_models(ms)
    score, path = ctx.viterbi(labels)
    allsc = ctx.viterbi_scores()
    fwd = ctx.forward_scores()
    for u in range(len(labels)):
        mo = _oracle_model(ms, labels[u])
        b, _ = o.emissions(mo, x[off[u]:off[u + 1]], want_post=False)
        s, p = o.viterbi(mo, b)
        assert (path[off[u]:off[u + 1]] == p).all(), u
        assert abs(score[u] - s) <= 1e-9 * abs(s)
        assert abs(allsc[u, labels[u]] - s) <= 1e-5 * abs(s)
    assert (allsc <= fwd + 1e-6 * np.abs(fwd)).all()
    assert (np.argmax(allsc, axis=1) == labels).all()


# ---------------------------------------------------------------------- drop-in programs ----
def test_cli_train_then_test_matches_reference_outputs(golden_dir, tmp_path, monkeypatch):
    """bin/hmm_continuous_fs and bin/recognition_continuous_fs with the reference's argv on the
    synth_c1 case: reports agree with the reference's (iterations, mean probability to 1e-4, labels)."""
    monkeypatch.chdir(tmp_path)
    g = np.load(os.path.join(golden_dir, "synth_c1.npz"))
    V, N, M, D = int(g["V"]), int(g["N"]), int(g["M"]), int(g["D"])
    cen, s = synth.make_centres(V, N, M, D, seed=1234)
    x, off = synth.make_utterances(cen, s, g["train_labels"], seed=1234, tmin=70, tmax=110)
    xt, offt = synth.make_utterances(cen, s, g["test_labels"], seed=4321, tmin=70, tmax=110)
    bindir = os.path.join(os.path.dirname(api.LIB_PATH), "bin")
    models = []
    for v in range(V):
        files = []
        for u in np.nonzero(g["train_labels"] == v)[0]:
            f = str(tmp_path / ("tr%d.bin" % u))
            api.write_features(f, x[off[u]:off[u + 1]])
            files.append(f)
        lst = str(tmp_path / ("list%d.txt" % v))
        write_list(lst, files)
        hmm = str(tmp_path / ("w%d.hmm" % v))
        subprocess.run([os.path.join(bindir, "hmm_continuous_fs"), "word%d" % v, str(N), "1", str(M), lst, os.path.basename(hmm)],
                       check=True, stdout=subprocess.DEVNULL)
        mean, its = r.parse_train_report(hmm[:-4] + ".txt")
        assert its == g["iterations"][v] and abs(mean - g["mean_logp"][v]) <= RTOL * abs(g["mean_logp"][v])
        models.append(hmm)
    tf = []
    for u in range(len(offt) - 1):
        f = str(tmp_path / ("te%d.bin" % u))
        api.write_features(f, xt[offt[u]:offt[u + 1]])
        tf.append(f)
    write_list(tmp_path / "models.txt", models)
    write_list(tmp_path / "feat.txt", tf)
    open(str(tmp_path / "words.txt"), "w").write("\n".join("word%d" % v for v in g["test_labels"]) + "\n")
    res = str(tmp_path / "res.txt")
    subprocess.run([os.path.join(bindir, "recognition_continuous_fs"), "1", str(tmp_path / "models.txt"), "1",
                    str(tmp_path / "feat.txt"), str(tmp_path / "words.txt"), res], check=True, stdout=subprocess.DEVNULL)
    txt = open(res).read()
    assert "Algorithm used for recognition: Forward" in txt
    assert "Correct words: %d\nErrors: 0" % len(g["test_labels"]) in txt.split("Considering all the words:")[1]
    if r.available("d39m16"):
        # V != NUMBER_WORDS of the prebuilt reference binary only affects its stdout, not the result file
        ref_res = str(tmp_path / "ref_res.txt")
        r.run_test_cli("d39m16", str(tmp_path / "models.txt"), str(tmp_path / "feat.txt"), str(tmp_path / "words.txt"), ref_res)
        strip = lambda t: [l for l in t.splitlines() if not l.startswith(("Date and time", "Average recognition time"))]
        assert strip(txt) == strip(open(ref_res).read())


def test_cli_two_model_sets_weighted_sum(tmp_path, monkeypatch):
    """recognition_continuous_fs with models_number = 2 (R-FS:326-364): two model sets of different topology and
    feature width, each with its own feature list; the score of a word is sum_j coef_j * logP_j and the label its
    argmax.  Expected values from the oracle's forward scorer on every (utterance, word, set)."""
    monkeypatch.chdir(tmp_path)
    V, labels = 4, [0, 1, 2, 3, 2, 0]
    sets = []
    for j, (N, M, D) in enumerate(((5, 3, 39), (3, 2, 13))):
        cen, sc = synth.make_centres(V, N, M, D, seed=21 + j)
        ms = api.ModelSet.from_dict(synth.make_models(cen, sc), ["word%d" % v for v in range(V)])
        x, off = synth.make_utterances(cen, sc, labels, seed=31 + j, tmin=40, tmax=70)
        mp = [str(tmp_path / ("s%dw%d.hmm" % (j, v))) for v in range(V)]
        api.write_model_set(mp, ms)
        fp = []
        for u in range(len(labels)):
            fp.append(str(tmp_path / ("s%du%d.bin" % (j, u))))
            api.write_features(fp[-1], x[off[u]:off[u + 1]])
        write_list(tmp_path / ("models%d.txt" % j), mp)
        write_list(tmp_path / ("feat%d.txt" % j), fp)
        sets.append((ms, x, off))
    open(str(tmp_path / "words.txt"), "w").write("\n".join("word%d" % v for v in labels) + "\n")
    coef = (0.75, 0.25)
    want = np.zeros((len(labels), V))
    for j, (ms, x, off) in enumerate(sets):
        for u in range(len(labels)):
            for v in range(V):
                mo = o.Model(ms.A[v], ms.c[v], ms.mu[v], ms.iv[v], ms.det[v])
                want[u, v] += coef[j] * o.forward_score(mo, x[off[u]:off[u + 1]])
    res = str(tmp_path / "res.txt")
    bindir = os.path.join(os.path.dirname(api.LIB_PATH), "bin")
    out = subprocess.run([os.path.join(bindir, "recognition_continuous_fs"), "2", str(tmp_path / "models0.txt"), str(tmp_path / "models1.txt"),
                          str(coef[0]), str(coef[1]), str(tmp_path / "feat0.txt"), str(tmp_path / "feat1.txt"), str(tmp_path / "words.txt"), res],
                         check=True, stdout=subprocess.PIPE).stdout.decode()
    got = re.findall(r"Spoken word: (\S+) -> (\S+) : (\S+)", out)
    assert len(got) == len(labels)
    for u, (spoken, rec, score) in enumerate(got):
        assert spoken == "word%d" % labels[u] and rec == "word%d" % int(np.argmax(want[u]))
        assert abs(float(score) - want[u].max()) <= RTOL * abs(want[u].max())
    txt = open(res).read()
    assert "Number of models: 2" in txt and "Model name 2: %s" % (tmp_path / "models1.txt") in txt
    assert "Correct words: %d\nErrors: 0" % len(labels) in txt.split("Considering all the words:")[1]


# ------------------------------------------------------------- multi-stream models (P = 2) ----
def test_two_stream_model_matches_reference(golden_dir):
    """param_number = 2 (SURVEY 8f-4): two linked contexts against the reference trainer / recogniser run with two
    feature streams (tests/golden/synth_p2.npz) and against the multi-stream oracle: first E-step statistics of both
    streams, the EM loop (iterations, mean log-probability, every trained parameter), forward scores, Viterbi."""
    g = np.load(os.path.join(golden_dir, "synth_p2.npz"))
    V, N, labels, off = int(g["V"]), int(g["N"]), g["train_labels"], g["off"]
    cs = [api.Context(0), api.Context(0)]
    init = []
    for p, c in enumerate(cs):
        c.set_features(g["x%d" % p], off)
        init.append(c.init_models(labels, V, N, int(g["M"][p])))
    assert np.array_equal(init[0].A, init[1].A)
    cs[0].link_streams([cs[1]])
    st0, lpu = cs[0].estep(labels)
    stats = [st0, cs[1].stats_download()]
    for v in range(V):
        us = np.nonzero(labels == v)[0]
        offv = np.concatenate([[0], np.cumsum([off[u + 1] - off[u] for u in us])])
        xs = [np.concatenate([g["x%d" % p][off[u]:off[u + 1]] for u in us]) for p in range(2)]
        want, lp = o.estep_streams([_oracle_model(init[p], v) for p in range(2)], xs, offv)
        assert np.allclose(lpu[us], lp, rtol=RTOL)
        for p in range(2):
            sp = api.split_stats(stats[p][v], N, int(g["M"][p]), int(g["D"][p]))
            assert abs(sp["sum_logp"] - want[p].sum_logp) <= RTOL * abs(want[p].sum_logp) and sp["n_utt"] == len(us)
            for name in ("num_trans", "den_trans", "den_mix", "S0"):
                w = getattr(want[p], name)
                assert np.allclose(sp[name], w, rtol=RTOL, atol=1e-6 * np.abs(w).max()), (v, p, name)
    # the EM loop, every word with the reference's stopping rule (T-FS:238-361)
    for c in cs:
        c.em_reset()
    active, its, mean = np.ones(V, bool), np.zeros(V, int), np.zeros(V)
    for it in range(1, 50):
        cs[0].estep(np.where(active[labels], labels, -1), download=False, want_logp=False)
        lp0, nu0, upd0 = cs[0].mstep()
        lp1, nu1, upd1 = cs[1].mstep()
        assert np.array_equal(upd0, upd1) and np.array_equal(lp0[active], lp1[active])
        its[active], mean[active] = it, (lp0 / np.maximum(nu0, 1))[active]
        active &= upd0.astype(bool)
        if not active.any():
            break
    assert (its == g["iterations"]).all(), (its, g["iterations"])
    assert np.allclose(mean, g["mean_logp"], rtol=RTOL)
    trained = [cs[p].get_models(int(g["D"][p])) for p in range(2)]
    assert np.array_equal(trained[0].A, trained[1].A)
    for p in range(2):
        for v in range(V):
            mo = o.Model(*[g["trained_s%d_%s" % (p, k)][v] for k in ("A", "c", "mu", "iv", "det")])
            _assert_params_close(trained[p], v, mo)
    # recognition with the reference-trained models: product of the streams' densities (R-FS:341-364)
    offt, tl = g["offt"], g["test_labels"]
    ref_ms = [api.ModelSet(*[g["trained_s%d_%s" % (p, k)] for k in ("A", "c", "mu", "iv", "det")]) for p in range(2)]
    for p, c in enumerate(cs):
        c.set_features(g["xt%d" % p], offt)
        c.set_models(ref_ms[p])
    fw = cs[0].forward_scores()
    assert np.allclose(fw, g["score"], rtol=RTOL)
    assert (cs[0].rank(fw)[0] == tl).all()
    vs = cs[0].viterbi_scores()
    score, path = cs[0].viterbi(tl)
    for u in range(len(tl)):
        b = None
        for p in range(2):
            bp = o.emissions(_oracle_model(ref_ms[p], tl[u]), g["xt%d" % p][offt[u]:offt[u + 1]], want_post=False)[0]
            b = bp if b is None else b * bp
        s, pth = o.viterbi(_oracle_model(ref_ms[0], tl[u]), b)
        assert (path[offt[u]:offt[u + 1]] == pth).all() and abs(score[u] - s) <= 1e-9 * abs(s)
        assert abs(vs[u, tl[u]] - s) <= 1e-5 * abs(s)
    # a linked stream refuses to run on its own; unlinking restores the single-stream behaviour
    with pytest.raises(api.HmmCudaError, match="linked stream"):
        cs[1].forward_scores()
    cs[0].link_streams([])
    single = cs[1].forward_scores()
    assert np.isfinite(single).all() and not np.allclose(single, fw)
    for c in cs:
        c.close()


def test_cli_two_streams_match_reference_outputs(golden_dir, tmp_path, monkeypatch):
    """The drop-in programs with param_number = 2 on the case the reference itself was run on (synth_p2.npz): training
    report (iterations, mean probability), the two-stream .hmm files, and the recogniser's result file line by line."""
    monkeypatch.chdir(tmp_path)
    g = np.load(os.path.join(golden_dir, "synth_p2.npz"))
    V, N, off, offt = int(g["V"]), int(g["N"]), g["off"], g["offt"]
    bindir = os.path.join(os.path.dirname(api.LIB_PATH), "bin")
    hmms = []
    for v in range(V):
        lists = []
        for p in range(2):
            files = []
            for u in np.nonzero(g["train_labels"] == v)[0]:
                files.append(str(tmp_path / ("tr_s%d_%d.bin" % (p, u))))
                api.write_features(files[-1], g["x%d" % p][off[u]:off[u + 1]])
            lists.append(str(tmp_path / ("list_s%d_w%d.txt" % (p, v))))
            write_list(lists[-1], files)
        hmms.append(str(tmp_path / ("w%d.hmm" % v)))
        subprocess.run([os.path.join(bindir, "hmm_continuous_fs"), "word%d" % v, str(N), "2", str(g["M"][0]), str(g["M"][1]), lists[0], lists[1], os.path.basename(hmms[-1])],
                       check=True, stdout=subprocess.DEVNULL)
        mean, its = r.parse_train_report(hmms[-1][:-4] + ".txt")
        assert its == g["iterations"][v] and abs(mean - g["mean_logp"][v]) <= RTOL * abs(g["mean_logp"][v])
        rep = open(hmms[-1][:-4] + ".txt").read()
        assert "number of parameters: 2 \nnumber of mixtures 1: %d \nnumber of mixtures 2: %d \n" % (g["M"][0], g["M"][1]) in rep
        streams = r.read_model_streams(hmms[-1])
        assert len(streams) == 2 and streams[0].word == "word%d" % v
        for p in range(2):
            got = api.ModelSet(*[getattr(streams[p], k)[None] for k in ("A", "c", "mu", "iv", "det")])
            _assert_params_close(got, 0, o.Model(*[g["trained_s%d_%s" % (p, k)][v] for k in ("A", "c", "mu", "iv", "det")]))
    feats = []
    for p in range(2):
        files = []
        for u in range(len(g["test_labels"])):
            files.append(str(tmp_path / ("te_s%d_%d.bin" % (p, u))))
            api.write_features(files[-1], g["xt%d" % p][offt[u]:offt[u + 1]])
        feats.append(str(tmp_path / ("feat_s%d.txt" % p)))
        write_list(feats[-1], files)
    write_list(tmp_path / "models.txt", hmms)
    open(str(tmp_path / "words.txt"), "w").write("\n".join("word%d" % v for v in g["test_labels"]) + "\n")
    res = str(tmp_path / "res.txt")
    out = subprocess.run([os.path.join(bindir, "recognition_continuous_fs"), "1", str(tmp_path / "models.txt"), "1", feats[0], feats[1],
                          str(tmp_path / "words.txt"), res], check=True, stdout=subprocess.PIPE).stdout.decode()
    got = re.findall(r"Spoken word: (\S+) -> (\S+) : (\S+)", out)
    for u, (spoken, rec, score) in enumerate(got):
        assert rec == spoken == "word%d" % g["test_labels"][u]
        assert abs(float(score) - g["score"][u].max()) <= RTOL * abs(g["score"][u].max())
    strip = lambda t: [l for l in t.splitlines() if not l.startswith(("Date and time", "Average recognition time", "Model name"))]
    assert strip(open(res).read()) == strip(str(g["result_file"]))


def test_two_stream_estep_on_the_tensor_core_path():
    """Linked streams at MFCC-sized widths (D = 39 and D = 13, M = 4 and 2): both contexts take the tcgen05 kernels, the
    second one accumulates with the first one's state posteriors.  Against the multi-stream oracle."""
    V, N, U = 2, 5, 24
    labels = np.arange(U) % V
    sets = []
    for p, (M, D) in enumerate(((4, 39), (2, 13))):
        cen, sc = synth.make_centres(V, N, M, D, seed=900 + p)
        x, off = synth.make_utterances(cen, sc, labels, seed=55, tmin=90, tmax=140)
        sets.append((api.ModelSet.from_dict(synth.make_models(cen, sc)), x, off))
    assert np.array_equal(sets[0][2], sets[1][2])
    off = sets[0][2]
    cs = [api.Context(0), api.Context(0)]
    for c, (ms, x, _) in zip(cs, sets):
        c.set_features(x, off)
        c.set_models(ms)
    cs[0].link_streams([cs[1]])
    st0, lpu = cs[0].estep(labels)
    stats = [st0, cs[1].stats_download()]
    for v in range(V):
        us = np.nonzero(labels == v)[0]
        offv = np.concatenate([[0], np.cumsum([off[u + 1] - off[u] for u in us])])
        xs = [np.concatenate([sets[p][1][off[u]:off[u + 1]] for u in us]) for p in range(2)]
        want, lp = o.estep_streams([_oracle_model(sets[p][0], v) for p in range(2)], xs, offv)
        assert np.allclose(lpu[us], lp, rtol=RTOL)
        for p in range(2):
            ms = sets[p][0]
            sp = api.split_stats(stats[p][v], N, ms.M, ms.D)
            for name in ("num_trans", "den_trans", "den_mix", "S0"):
                w = getattr(want[p], name)
                assert np.allclose(sp[name], w, rtol=RTOL, atol=1e-6 * np.abs(w).max()), (v, p, name)
            got, mo = ms.copy(), _oracle_model(ms, v)
            api.mstep(got, stats[p])
            o.mstep(mo, want[p])
            _assert_params_close(got, v, mo)
    for c in cs:
        c.close()


# ------------------------------------------------- full-size, size-independent properties ----
def test_two_stream_underflow_is_flushed_per_stream():
    """The reference flushes every stream's density on its own before it multiplies them (R-FS:341-367): a cell in which
    one stream's density underflows to exactly 0 is dead even when the SUM of the streams' log-densities is
    representable.  Stream 0 of the wrong word sits 40 sigma off (log density -802 < log DBL_TRUE_MIN = -744.4),
    stream 1 has a sharp, perfectly matching Gaussian (log density +61): sum = -741."""
    V, N, T, U = 2, 2, 12, 2
    A = np.tile(np.array([[0.6, 0.4], [0.0, 1.0]]), (V, 1, 1))
    c1 = np.ones((V, N, 1))
    mu0 = np.zeros((V, N, 1, 2)); mu0[1, :, :, 0] += 40.0
    ms0 = api.ModelSet(A, c1, mu0, np.ones((V, N, 1, 2)), np.ones((V, N, 1)))
    var1 = 1e-14
    mu1 = np.zeros((V, N, 1, 4))
    ms1 = api.ModelSet(A, c1, mu1, np.full((V, N, 1, 4), 1.0 / var1), np.full((V, N, 1), var1 ** 4))
    off = np.arange(U + 1, dtype=np.int64) * T
    x0 = np.zeros((U * T, 2)); x0[T:, 0] += 40.0          # utterance 0 = word 0, utterance 1 = word 1
    x1 = np.zeros((U * T, 4))
    cs = [api.Context(0), api.Context(0)]
    cs[0].set_features(x0, off); cs[0].set_models(ms0)
    cs[1].set_features(x1, off); cs[1].set_models(ms1)
    cs[0].link_streams([cs[1]])
    got = cs[0].forward_scores(emulate_underflow=True)
    plain = cs[0].forward_scores()
    with np.errstate(all="ignore"):
        want = np.array([[o.forward_score_streams([_oracle_model(ms0, v), _oracle_model(ms1, v)], [x0[off[u]:off[u + 1]], x1[off[u]:off[u + 1]]])
                          for v in range(V)] for u in range(U)])
    assert np.isfinite(want[0, 0]) and np.isfinite(want[1, 1]) and not np.isfinite(want[0, 1]) and not np.isfinite(want[1, 0])
    assert (np.isfinite(got) == np.isfinite(want)).all(), (got, want)
    fin = np.isfinite(want)
    assert np.allclose(got[fin], want[fin], rtol=RTOL)
    assert np.isfinite(plain).all()                    # without the emulation the log-domain score of the dead cells exists
    for c in cs:
        c.close()


def test_c2_size_properties(ctx):
    """BASELINE config 2 (N=5, M=16, 1000 utterances of ~300 frames): too big for the CPU oracle in a
    test, so check identities that hold at any size: sum_m S0 = den_mix; band row sums of num_trans =
    den_trans; den_mix - den_trans = last-frame occupancy >= 0; sum_i den_mix = sum_u w_u T_u <= F;
    and E-step log-probabilities equal the decode path's forward scores."""
    V, N, M, U = 10, 5, 16, 1000
    cen, s = synth.make_centres(V, N, M, 39, seed=1234)
    labels = np.arange(U) % V
    x, off = synth.make_utterances(cen, s, labels, seed=1234)
    ms = api.ModelSet.from_dict(synth.make_models(cen, s))
    ctx.set_features(x, off)
    ctx.set_models(ms)
    stats, lpu = ctx.estep(labels)
    assert np.isfinite(lpu).all()
    T = np.diff(off)
    for v in range(V):
        sp = api.split_stats(stats[v], N, M, 39)
        assert np.allclose(sp["S0"].sum(axis=1), sp["den_mix"], rtol=1e-5)
        assert np.allclose(sp["num_trans"].sum(axis=1)[:-1], sp["den_trans"][:-1], rtol=1e-6)
        assert (sp["den_mix"] - sp["den_trans"] >= -1e-9).all()
        assert sp["den_mix"].sum() <= T[labels == v].sum() * (1 + 1e-9)
        assert sp["n_utt"] == (labels == v).sum()
        assert abs(sp["sum_logp"] - lpu[labels == v].sum()) <= 1e-9 * abs(sp["sum_logp"])
    sub = np.arange(0, U, 50)
    offs = np.concatenate([[0], np.cumsum(T[sub])])
    ctx.set_features(np.concatenate([x[off[u]:off[u + 1]] for u in sub]), offs)
    sc = ctx.forward_scores()
    assert np.allclose(sc[np.arange(len(sub)), labels[sub]], lpu[sub], rtol=1e-6)
    lab, _ = ctx.rank(sc)
    assert (lab == labels[sub]).all()
    # a spot check against the oracle on two utterances
    for k in (0, 7):
        u = sub[k]
        want = o.forward_score(o.Model(ms.A[labels[u]], ms.c[labels[u]], ms.mu[labels[u]], ms.iv[labels[u]], ms.det[labels[u]]), x[off[u]:off[u + 1]])
        assert abs(lpu[u] - want) <= RTOL * abs(want)


def test_c2_full_size_estep_and_decode_match_oracle(ctx):
    """BASELINE configs[1] in full -- 10 words, N=5, M=16, D=39, 1,000 utterances, ~300,000 frames, the workload of the
    headline bench line -- against the oracle (the C restatement finishes it in seconds): log P of every utterance, the
    statistics of EVERY word (T-FS:244-321) and the parameters the M-step makes of them within 1e-4; then the forward
    scores of every tenth utterance against all 10 models and the labels (R-FS:341-390).  The models are the generating
    ones moved by 0.3 sigma, so that the posteriors are not trivially sharp."""
    V, N, M, U = 10, 5, 16, 1000
    cen, s = synth.make_centres(V, N, M, 39, seed=1234)
    labels = np.arange(U) % V
    x, off = synth.make_utterances(cen, s, labels, seed=1234)
    rng = np.random.default_rng(99)
    ms = api.ModelSet.from_dict(synth.make_models(cen + 0.3 * s * rng.standard_normal(cen.shape), s))
    ctx.set_features(x, off)
    ctx.set_models(ms)
    stats, lpu = ctx.estep(labels)
    assert np.isfinite(lpu).all()
    for v in range(V):
        us = np.nonzero(labels == v)[0]
        xv = np.concatenate([x[off[u]:off[u + 1]] for u in us])
        offv = np.concatenate([[0], np.cumsum([off[u + 1] - off[u] for u in us])])
        st, lp = o.estep(_oracle_model(ms, v), xv, offv)
        sp = api.split_stats(stats[v], N, M, ms.D)
        assert np.allclose(lpu[us], lp, rtol=RTOL), v
        assert abs(sp["sum_logp"] - st.sum_logp) <= RTOL * abs(st.sum_logp) and sp["n_utt"] == len(us)
        for name in ("num_trans", "den_trans", "den_mix", "S0"):
            want = getattr(st, name)
            assert np.allclose(sp[name], want, rtol=RTOL, atol=1e-6 * np.abs(want).max()), (v, name)
        S0 = np.maximum(st.S0, 1e-300)[..., None]
        sd = np.sqrt(st.S2c / S0)
        assert (np.abs(sp["S1"] / S0 - st.S1 / S0) <= RTOL * np.maximum(np.abs(st.S1 / S0), sd)).all(), (v, "S1")
        assert np.allclose(sp["S2c"] / S0, st.S2c / S0, rtol=RTOL), (v, "S2c")
        mo = _oracle_model(ms, v)
        o.mstep(mo, st)
        one = api.ModelSet(ms.A[v:v + 1].copy(), ms.c[v:v + 1].copy(), ms.mu[v:v + 1].copy(), ms.iv[v:v + 1].copy(), ms.det[v:v + 1].copy())
        _assert_params_close(api.mstep(one, stats[v:v + 1]), 0, mo)
    sc = ctx.forward_scores()
    vsc = ctx.viterbi_scores()
    lab, sec = ctx.rank(sc)
    assert (lab == labels).all()
    for u in range(0, U, 10):
        xu = x[off[u]:off[u + 1]]
        want = np.array([o.forward_score(_oracle_model(ms, v), xu) for v in range(V)])
        assert np.allclose(sc[u], want, rtol=RTOL, atol=0), u
        order = o.rank(want)
        assert lab[u] == order[0] and sec[u] == order[1]
        assert (vsc[u] <= sc[u] + 1e-6 * np.abs(sc[u])).all()      # the best path is one of the paths the forward score sums
    assert np.allclose(sc[np.arange(U), labels], lpu, rtol=1e-6)   # the E-step's log P and the decode path's score of the own model


# ------------------------------------------------------ new code paths of this round's kernels ----
def test_graph_replay_gives_the_same_em_iterations():
    """The E-step / M-step launch sequences are replayed as CUDA graphs from the third call on: five EM
    iterations with and without graphs must produce the same models and log-likelihoods (the scratch-slot
    reduction makes the statistics order-deterministic, so the comparison is tight)."""
    ms, x, off, labels = _synth(3, 5, 4, 12, seed=808)
    out = []
    for graphs in (1, 0):
        c = api.Context(0)
        c.set_option("graphs", graphs)
        c.set_features(x, off)
        c.set_models(ms)
        c.em_reset()
        lps = []
        for _ in range(5):
            c.estep(labels, download=False, want_logp=False)
            lp, nu, upd = c.mstep(threshold=-1.0)
            lps.append(lp.copy())
        out.append((np.array(lps), c.get_models(ms.D)))
        c.close()
    (lp_g, m_g), (lp_p, m_p) = out
    assert np.allclose(lp_g, lp_p, rtol=1e-9)
    for name in ("A", "c", "mu", "iv"):
        assert np.allclose(getattr(m_g, name), getattr(m_p, name), rtol=1e-7, atol=1e-12), name
    assert (np.diff(lp_g.sum(1)) > -1e-6 * np.abs(lp_g.sum(1)[:-1])).all()  # EM does not decrease the likelihood


def test_chunked_upload_matches_device_resident_features():
    """hmmcu_set_features (chunked copy pipelined with packing, centre formed on the host) and
    hmmcu_set_features_device (k_center on the device) must give the same packed features."""
    torch = pytest.importorskip("torch")
    ms, x, off, labels = _synth(2, 5, 3, 40, seed=909, tmin=200, tmax=300)   # > 4096 frames: several chunks
    c = api.Context(0)
    c.set_features(x, off)
    c.set_models(ms)
    st_h, lp_h = c.estep(labels)
    xd = torch.from_numpy(x).cuda()
    c.set_features_device(xd.data_ptr(), off, x.shape[1])
    st_d, lp_d = c.estep(labels)
    c.close()
    assert np.allclose(lp_h, lp_d, rtol=1e-12) and np.allclose(st_h, st_d, rtol=1e-9, atol=1e-9)


def test_ingest_pipeline_and_streamed_upload_match_set_features(tmp_path):
    """SURVEY 8f-2: feature files -> pinned staging -> HBM through hmmh_ingest, and the streaming C ABI under it with
    ranges appended out of order, leave the context in the same state as hmmcu_set_features on the host buffer."""
    ms, x, off, labels = _synth(2, 5, 3, 40, seed=909, tmin=200, tmax=300)
    paths = []
    for u in range(len(off) - 1):
        p = str(tmp_path / ("u%03d.bin" % u))
        api.write_features(p, x[off[u]:off[u + 1]])
        paths.append(p)
    c = api.Context(0)
    c.set_features(x, off)
    c.set_models(ms)
    st_h, lp_h = c.estep(labels)
    fw_h = c.forward_scores()
    off_i, D, st = c.ingest(paths, threads=4)
    assert D == x.shape[1] and np.array_equal(off_i, off) and st.bytes == x.nbytes and st.batches >= 1
    st_i, lp_i = c.estep(labels)
    fw_i = c.forward_scores()
    F = int(off[-1])
    cuts = [0, 1000, 1001, 4096, F]
    order = [2, 0, 3, 1]
    c.features_stream(off, x.shape[1], [(cuts[k], x[cuts[k]:cuts[k + 1]]) for k in order])
    st_s, lp_s = c.estep(labels)
    with pytest.raises(api.HmmCudaError, match="frames appended"):
        c.features_stream(off, x.shape[1], [(0, x[:100])])
    c.close()
    assert np.allclose(lp_h, lp_i, rtol=1e-12) and np.allclose(st_h, st_i, rtol=1e-9, atol=1e-9)
    assert np.allclose(lp_i, lp_s, rtol=1e-12), np.abs(lp_i - lp_s).max()
    assert np.allclose(st_i, st_s, rtol=1e-9, atol=1e-9, equal_nan=True)
    assert np.allclose(fw_h, fw_i, rtol=1e-12), np.abs(fw_h - fw_i).max()


def test_many_small_models_take_the_atomic_flush_path(ctx):
    """A CTA of the accumulate kernel that walks through more than two (model, Gaussian block) images flushes
    the later ones with atomics instead of scratch slots; both must add up to the oracle's statistics."""
    V, U = 24, 48
    ms, x, off, labels = _synth(V, 3, 2, U, seed=1010, tmin=6, tmax=14)
    ctx.set_features(x, off)
    ctx.set_models(ms)
    stats, lpu = ctx.estep(labels)
    for v in (0, 7, V - 1):
        us = np.nonzero(labels == v)[0]
        xv = np.concatenate([x[off[u]:off[u + 1]] for u in us])
        offv = np.concatenate([[0], np.cumsum([off[u + 1] - off[u] for u in us])])
        st, lp = o.estep(_oracle_model(ms, v), xv, offv)
        sp = api.split_stats(stats[v], 3, 2, ms.D)
        assert np.allclose(lpu[us], lp, rtol=RTOL)
        assert np.allclose(sp["S0"], st.S0, rtol=RTOL, atol=1e-6 * st.S0.max())
        assert np.allclose(sp["num_trans"], st.num_trans, rtol=RTOL, atol=1e-6 * st.num_trans.max())


@pytest.mark.parametrize("N,M,D,spread", [(5, 16, 39, 0.0), (5, 3, 39, 2.0), (3, 128, 39, 0.0), (4, 4, 15, 1.0), (5, 2, 9, 0.0)])
def test_half_precision_accumulate_operands(N, M, D, spread):
    """k_accum_h (half-precision operands, frame tiles packed once per feature set; the default for feature widths with
    D + 1 rounded to a multiple of 8) against k_accum_ws (3xTF32) and against the oracle's calc_mix_param sums
    (T-FS:1691-1727), also with feature dimensions decades apart (every dimension gets its own power-of-two scales) and
    through a second E-step after new models (the tiles stay, the W images follow the models).  D = 9 (DP = 12) has no
    half-precision form: the option must fall back to k_accum_ws by itself."""
    V, U = 2, 8
    ms, x, off, labels = _synth(V, N, M, U, seed=5200 + N * M, tmin=50, tmax=110, D=D)
    if spread > 0:
        g = 10.0 ** np.random.default_rng(23).uniform(-spread, spread, size=x.shape[1])
        x = x * g
        ms = api.ModelSet(ms.A, ms.c, ms.mu * g, ms.iv / g ** 2, ms.det * np.prod(g ** 2))
    want = []
    for v in range(V):
        us = np.nonzero(labels == v)[0]
        xv = np.concatenate([x[off[u]:off[u + 1]] for u in us])
        offv = np.concatenate([[0], np.cumsum([off[u + 1] - off[u] for u in us])])
        want.append(o.estep(_oracle_model(ms, v), xv, offv)[0])
    got = {}
    for h in (1, 0):
        c = api.Context(0)
        c.set_option("h_acc", h)
        c.set_features(x, off)
        c.set_models(ms)
        for rep in range(2):  # the second E-step reuses the packed tiles
            stats, _ = c.estep(labels)
        assert c.kernel_ms("tc_active") == 1 and c.kernel_ms("acc_h_active") == (1 if h and (D + 1 + 3) // 4 * 4 % 8 == 0 else 0)
        got[h] = [api.split_stats(stats[v], N, M, D) for v in range(V)]
        # new models (every mean moved, variances changed), same features: only the W images are repacked
        ms2 = api.ModelSet(ms.A, ms.c, ms.mu + 0.05 / np.sqrt(ms.iv), ms.iv * 0.8, ms.det / 0.8 ** D)
        c.set_models(ms2)
        st2, _ = c.estep(labels)
        got[(h, 2)] = [api.split_stats(st2[v], N, M, D) for v in range(V)]
        c.close()
    def close(sp, st, mean_x):
        S0 = np.maximum(st.S0, 1e-300)[..., None]
        occ = st.S0 > 1e-3 * st.S0.max()
        sd = np.sqrt(st.S2c / S0)
        assert np.allclose(sp["S0"], st.S0, rtol=RTOL, atol=1e-6 * st.S0.max()), "S0"
        assert (np.abs(sp["S1"] / S0 - st.S1 / S0)[occ] <= RTOL * np.maximum(np.abs(st.S1 / S0), sd)[occ]).all(), "S1"
        want2 = st.S2c / S0
        scale2 = want2 + (st.S1 / S0 - mean_x) ** 2
        assert (np.abs(sp["S2c"] / S0 - want2)[occ] <= (RTOL * want2 + 2e-6 * scale2)[occ]).all(), "S2c"
    for v in range(V):
        close(got[1][v], want[v], x.mean(0))
        close(got[0][v], want[v], x.mean(0))
        us = np.nonzero(labels == v)[0]
        xv = np.concatenate([x[off[u]:off[u + 1]] for u in us])
        offv = np.concatenate([[0], np.cumsum([off[u + 1] - off[u] for u in us])])
        st2 = o.estep(_oracle_model(ms2, v), xv, offv)[0]
        close(got[(1, 2)][v], st2, x.mean(0))


@pytest.mark.parametrize("N,M,D", [(4, 2, 13), (5, 32, 39), (2, 160, 39)])
def test_decode_paths_other_shapes(ctx, N, M, D):
    """Forward scores / labels and Viterbi paths for feature widths other than 39 (generic k_logb64), for a
    state that spans several 16-column chunks (M = 32) and for a wide state (M = 160: single operand stage)."""
    ms, x, off, labels = _synth(3, N, M, 6, seed=1111 + M, D=D)
    ctx.set_features(x, off)
    ctx.set_models(ms)
    sc = ctx.forward_scores()
    vs, path = ctx.viterbi(labels)
    for u in range(6):
        for v in range(3):
            want = o.forward_score(_oracle_model(ms, v), x[off[u]:off[u + 1]])
            assert abs(sc[u, v] - want) <= RTOL * abs(want)
        mo = _oracle_model(ms, labels[u])
        b, _ = o.emissions(mo, x[off[u]:off[u + 1]], want_post=False)
        s_o, p_o = o.viterbi(mo, b)
        assert (path[off[u]:off[u + 1]] == p_o).all() and abs(vs[u] - s_o) <= 1e-9 * abs(s_o)
    lab, _ = ctx.rank(sc)
    assert (lab == labels).all()


@pytest.mark.parametrize("N,M,D", [(1, 1, 39), (8, 2, 39), (3, 8, 39), (6, 16, 39), (2, 5, 39), (7, 3, 39), (5, 3, 7), (4, 4, 12)])
def test_decode_kernel_variants_match_oracle(N, M, D):
    """Every image layout k_emis_dec is built for (1, 2, 3, 4, 5, 8, 16 mixtures per state; 1 to 8 states; feature widths
    whose padded row is not a multiple of 8 floats) with the interleaved layout and both cell scorers behind it: forward
    scores within 1e-4 of the oracle (R-FS:341-369, 739-836), Viterbi scores within 1e-4 of the oracle's, labels equal."""
    ms, x, off, labels = _synth(5, N, M, 10, seed=900 + 10 * N + M, tmin=max(N, 9), tmax=70, D=D)
    c = api.Context(0)
    c.set_features(x, off)
    c.set_models(ms)
    sc, vs = c.forward_scores(), c.viterbi_scores()
    assert c.kernel_ms("dec_grid") > 0          # k_emis_dec ran
    for u in range(len(labels)):
        xu = x[off[u]:off[u + 1]]
        for v in range(ms.V):
            mo = _oracle_model(ms, v)
            want = o.forward_score(mo, xu)
            b, _ = o.emissions(mo, xu, want_post=False)
            wv, _ = o.viterbi(mo, b)
            assert abs(sc[u, v] - want) <= RTOL * abs(want), (u, v)
            assert abs(vs[u, v] - wv) <= RTOL * abs(wv), (u, v)
    lab, _ = c.rank(sc)
    assert (lab == labels).all()
    c.close()


@pytest.mark.parametrize("N,M,spread", [(5, 3, 0.0), (5, 16, 0.0), (3, 8, 2.0), (5, 3, 3.0), (3, 128, 0.0), (2, 32, 2.0), (1, 160, 1.0)])
def test_half_precision_decode_operands(N, M, spread):
    """The decode emission kernels (k_emis_dec for M <= 16, k_emis_ws<false> above) with half-precision operands (kind::f16
    MMAs, per-dimension power-of-two scaling; the default) against the 3xTF32 form of the same kernels and against the oracle (calc_gaus / calc_symbol_probab, R-FS:860-947, through the
    forward score R-FS:739-836).  `spread` stretches every feature dimension by its own factor 10^U(-spread, spread)
    (models transformed with it), so that the dimensions' magnitudes differ by up to six decades: the scaling has to bring
    each of them into the half's range on its own."""
    ms, x, off, labels = _synth(6, N, M, 12, seed=4100 + N * M, tmin=40, tmax=90)
    if spread > 0:
        g = 10.0 ** np.random.default_rng(17).uniform(-spread, spread, size=x.shape[1])
        x = x * g
        ms = api.ModelSet(ms.A, ms.c, ms.mu * g, ms.iv / g ** 2, ms.det * np.prod(g ** 2))
    want = np.array([[o.forward_score(_oracle_model(ms, v), x[off[u]:off[u + 1]]) for v in range(ms.V)] for u in range(len(labels))])
    got = {}
    for f16 in (1, 0):
        c = api.Context(0)
        c.set_option("dec_f16", f16)
        c.set_features(x, off)
        c.set_models(ms)
        got[f16] = c.forward_scores()
        assert (c.kernel_ms("dec_grid") > 0) == (M <= 16) and c.kernel_ms("tc_active") == 1 and c.kernel_ms("dec_f16_active") == f16
        lab, _ = c.rank(got[f16])
        assert (lab == labels).all()
        c.close()
        assert np.allclose(got[f16], want, rtol=RTOL, atol=0)
    e16, e32 = np.abs(got[1] / want - 1).max(), np.abs(got[0] / want - 1).max()
    assert e16 < 2e-6 and e16 < 4 * e32 + 1e-7, (e16, e32)     # as accurate as the TF32 split, not merely inside the bar


@pytest.mark.parametrize("M", [3, 5, 4])
def test_decode_in_many_batches_equals_one_batch(M):
    """hmmcu_forward_scores / hmmcu_viterbi_scores work in utterance batches (R-FS:283-390 is one loop over the test list);
    a batch starts at an arbitrary frame, so the interleaved log-emission layout (blocks of 8 frames) is addressed relative
    to the batch.  With a budget of a few KiB every utterance or two is a batch of its own: the scores must be the
    bits of the single-batch run, for the unpadded M = 3 / M = 5 image layouts and a padded one, and within 1e-4 of the
    oracle.  Also with the reference's underflow emulated (k_fwd_score reads the same layout)."""
    ms, x, off, labels = _synth(7, 5, M, 11, seed=77 + M, tmin=5, tmax=61)
    c = api.Context(0)
    c.set_features(x, off)
    c.set_models(ms)
    one = (c.forward_scores(), c.viterbi_scores(), c.forward_scores(emulate_underflow=True))
    c.set_option("dec_budget_kb", 16)   # 16 KiB / (4 B * 35 state columns) = 117 frames per batch
    many = (c.forward_scores(), c.viterbi_scores(), c.forward_scores(emulate_underflow=True))
    for a, b in zip(one, many):
        assert np.array_equal(a, b, equal_nan=True)
    want = np.array([[o.forward_score(_oracle_model(ms, v), x[off[u]:off[u + 1]]) for v in range(ms.V)] for u in range(len(labels))])
    fin = np.isfinite(want)
    assert fin.all() and np.allclose(many[0], want, rtol=RTOL, atol=0)
    lab, _ = c.rank(many[0])
    assert (lab == labels).all()
    c.close()


@pytest.mark.parametrize("dense", [False, True])
def test_forward_cell_scorer_against_the_oracle(dense):
    """k_fwd_cells32 (log-domain single-precision chain) against the oracle's calc_alpha + calc_probability
    (R-FS:739-836), for the reference's banded topology and for a dense A, on mismatched models (a state's mass falls
    by e^-100 per frame there: a linear single-precision chain loses the best path in such cells) and with an
    utterance shorter than the chain."""
    ms, x, off, labels = _synth(6, 5, 3, 12, seed=31, tmin=3, tmax=140)
    if dense:
        rng = np.random.default_rng(5)
        A = rng.random(ms.A.shape) + 0.05
        ms = api.ModelSet(A / A.sum(axis=2, keepdims=True), ms.c, ms.mu, ms.iv, ms.det)
    want = np.array([[o.forward_score(_oracle_model(ms, v), x[off[u]:off[u + 1]]) for v in range(ms.V)] for u in range(len(labels))])
    c = api.Context(0)
    c.set_features(x, off)
    c.set_models(ms)
    got = c.forward_scores()
    c.close()
    fin = np.isfinite(want)
    assert (np.isfinite(got) == fin).all()
    assert np.allclose(got[fin], want[fin], rtol=RTOL, atol=0)
    assert np.abs(got[fin] / want[fin] - 1).max() < 2e-6


@pytest.mark.parametrize("N,M", [(5, 1), (5, 3), (5, 16), (3, 6), (6, 2)])
def test_device_initial_models_are_bit_identical_to_the_host_builder(N, M):
    """hmmcu_init_models (creating_initial_model, T-FS:732-1317, for all words at once on the device) against
    hmmh_init_model, the host restatement that tests/test_host_cpu.py pins to the oracle: same IEEE operations in
    the same order, so every parameter must be equal bit for bit."""
    V, U = 3, 12
    ms, x, off, labels = _synth(V, N, max(M, 2), U, seed=4242 + N * M, tmin=40, tmax=90)
    c = api.Context(0)
    c.set_features(x, off)
    got = c.init_models(labels, V, N, M)
    c.close()
    for v in range(V):
        us = np.nonzero(labels == v)[0]
        xv = np.concatenate([x[off[u]:off[u + 1]] for u in us])
        offv = np.concatenate([[0], np.cumsum([off[u + 1] - off[u] for u in us])]).astype(np.int64)
        want = api.init_model(N, M, xv, offv)
        for name in ("A", "c", "mu", "iv", "det"):
            assert np.array_equal(getattr(got, name)[v], getattr(want, name)[0]), (v, name)


def test_forward_backward_kernels_agree():
    """k_fb_res (whole utterance resident in shared memory, the default) against k_fb (one chain per utterance, windows of
    64 frames): same statistics and log-likelihoods; ragged lengths including T = 3 < N; an utterance too long for the
    resident kernel's shared memory takes the windowed kernel on its own."""
    ms, x, off, labels = _synth(2, 5, 3, 10, seed=777, tmin=3, tmax=140)
    out = []
    for res in (0, 1):
        c = api.Context(0)
        c.set_option("res_fb", res)
        c.set_features(x, off)
        c.set_models(ms)
        out.append(c.estep(labels))
        c.close()
    st0, lp0 = out[0]
    fin, sf = np.isfinite(lp0), np.isfinite(st0)  # sum_logp is -inf for a word with an utterance shorter than its state chain
    for k, (st, lp) in enumerate(out[1:]):
        assert (np.isfinite(lp) == fin).all() and np.allclose(lp[fin], lp0[fin], rtol=1e-8), k
        assert (np.isfinite(st) == sf).all() and (st[~sf] == st0[~sf]).all(), k
        assert np.allclose(st[sf], st0[sf], rtol=2e-5, atol=1e-6 * np.abs(st0[sf]).max()), k
    # the resident kernel sums every model's utterances in a fixed order: two runs are bit-identical
    c = api.Context(0)
    c.set_features(x, off)
    c.set_models(ms)
    a = c.estep(labels)
    b = c.estep(labels)
    c.close()
    assert (a[0][sf] == b[0][sf]).all() and (a[1][fin] == b[1][fin]).all()
    # an utterance beyond a team's shared memory (2 N T words): the library falls back to k_fb by itself
    msl, xl, offl, labl = _synth(1, 5, 2, 2, seed=778, tmin=1500, tmax=1600)
    c = api.Context(0)
    c.set_features(xl, offl)
    c.set_models(msl)
    _, lpl = c.estep(labl)
    c.close()
    for u in range(2):
        want = o.forward_score(_oracle_model(msl, 0), xl[offl[u]:offl[u + 1]])
        assert abs(lpl[u] - want) <= RTOL * abs(want)


@pytest.mark.parametrize("N", [1, 2, 3, 4, 6, 7, 8])
def test_resident_forward_backward_other_state_counts(ctx, N):
    """k_fb_res for every supported number of states (odd row stride for even N), statistics against the oracle."""
    ms, x, off, labels = _synth(2, N, 2, 7, seed=880 + N, tmin=max(N, 2), tmax=150)
    ctx.set_features(x, off)
    ctx.set_models(ms)
    stats, lpu = ctx.estep(labels)
    for v in range(2):
        us = np.nonzero(labels == v)[0]
        xv = np.concatenate([x[off[u]:off[u + 1]] for u in us])
        offv = np.concatenate([[0], np.cumsum([off[u + 1] - off[u] for u in us])])
        st, lp = o.estep(_oracle_model(ms, v), xv, offv)
        sp = api.split_stats(stats[v], N, 2, ms.D)
        assert np.allclose(lpu[us], lp, rtol=RTOL)
        for name in ("num_trans", "den_trans", "den_mix", "S0"):
            want = getattr(st, name)
            assert np.allclose(sp[name], want, rtol=RTOL, atol=1e-6 * np.abs(want).max()), name


# ------------------------------------------------- resume from a model file (optional last argument) ----
def test_cli_resumes_from_an_initial_model(tmp_path, monkeypatch):
    """hmm_continuous_fs ... out.hmm initial.hmm (T-FS:216-222; the reference reads argv[argc] there and would crash,
    SURVEY section 5 'checkpoint / resume'): training continues from the model in the file.  The first model is trained
    on two utterances, the resumed run on all eight, so that it has several iterations of real work.  Expected values:
    the oracle's EM loop started from the same file -- equal iteration count, mean log-probability and parameters
    within 1e-4 (the test first checks that no stopping decision of that loop is within 5 % of the threshold)."""
    monkeypatch.chdir(tmp_path)
    N, M = 4, 2
    cen, sc = synth.make_centres(1, N, M, 39, seed=341)
    x, off = synth.make_utterances(cen, sc, [0] * 8, seed=342, tmin=50, tmax=80)
    files = []
    for u in range(len(off) - 1):
        files.append(str(tmp_path / ("u%d.bin" % u)))
        api.write_features(files[-1], x[off[u]:off[u + 1]])
    lst2, lst = str(tmp_path / "list2.txt"), str(tmp_path / "list.txt")
    write_list(lst2, files[:2])
    write_list(lst, files)
    exe = os.path.join(os.path.dirname(api.LIB_PATH), "bin", "hmm_continuous_fs")
    first, second = str(tmp_path / "first.hmm"), str(tmp_path / "second.hmm")
    subprocess.run([exe, "word", str(N), "1", str(M), lst2, "first.hmm"], check=True, stdout=subprocess.DEVNULL)
    subprocess.run([exe, "word", str(N), "1", str(M), lst, "second.hmm", "first.hmm"], check=True, stdout=subprocess.DEVNULL)
    mean2, its2 = r.parse_train_report(second[:-4] + ".txt")
    # the oracle's loop from the same start (T-FS:238-358), keeping the stopping rule's variations
    mo = r.read_model(first)
    old, its_o, variations = 1.0, 0, []
    while True:
        its_o += 1
        st, lp = o.estep(mo, x, off)
        probab = float(np.sum(lp))
        variations.append(abs((old - probab) / old))
        if not variations[-1] > 1e-3:
            break
        old = probab
        o.mstep(mo, st)
    mean_o = probab / (len(off) - 1)
    assert all(abs(v / 1e-3 - 1.0) > 0.05 for v in variations), variations
    assert its_o >= 3
    assert its2 == its_o and abs(mean2 - mean_o) <= RTOL * abs(mean_o)
    got = api.read_model(second)
    assert got.words == ["word"] and (got.N, got.M, got.D) == (N, M, 39)
    _assert_params_close(got, 0, mo)
    rep = open(second[:-4] + ".txt").read()
    assert "number of states: %d \n" % N in rep and "number of mixtures 1: %d \n" % M in rep


# ----------------------------------------------------- parity at the shapes BASELINE.json names ----
def test_c4_shape_scores_and_labels_match_oracle(ctx):
    """BASELINE configs[3] shape: a 1,000-word model set (N=5, M=3: 5,000 state columns, 63 emission images) scored
    against a handful of utterances.  Every one of the 1,000 forward scores per utterance within 1e-4 of the oracle's
    (R-FS:341-369), the label and the second candidate equal to the oracle's ranking (R-FS:968-995, 380-388), and the
    Viterbi score of every cell within 1e-4 of the oracle's."""
    V, N, M, U = 1000, 5, 3, 8
    cen, s = synth.make_centres(V, N, M, 39, seed=4000)
    labels = (np.arange(U) * 137 + 5) % V
    x, off = synth.make_utterances(cen, s, labels, seed=4001, tmin=40, tmax=70)
    ms = api.ModelSet.from_dict(synth.make_models(cen, s))
    ctx.set_features(x, off)
    ctx.set_models(ms)
    sc = ctx.forward_scores()
    vs = ctx.viterbi_scores()
    lab, sec = ctx.rank(sc)
    want = np.empty((U, V))
    wantv = np.empty((U, V))
    with np.errstate(all="ignore"):
        for v in range(V):
            mo = _oracle_model(ms, v)
            for u in range(U):
                xu = x[off[u]:off[u + 1]]
                want[u, v] = o.forward_score(mo, xu)
                if v % 50 == 0 or v == labels[u]:
                    b, _ = o.emissions(mo, xu, want_post=False)
                    wantv[u, v] = o.viterbi(mo, b)[0]
                else:
                    wantv[u, v] = np.nan
    fin = np.isfinite(want)
    assert fin.mean() > 0.5, "the test is meant to sit in the finite regime"
    assert (np.abs(sc - want)[fin] <= RTOL * np.abs(want[fin])).all()
    # cells where the reference's linear-domain arithmetic underflows: the log-domain score must be hopeless too
    assert (sc[~fin] < want[fin].min()).all() if (~fin).any() else True
    chk = np.isfinite(wantv)
    assert chk.sum() >= 20 * U and (np.abs(vs - wantv)[chk] <= RTOL * np.abs(wantv[chk])).all()
    for u in range(U):
        row = np.where(fin[u], want[u], -np.inf)   # (finite regime: no NaN barriers in this case)
        idx = o.rank(row)
        assert lab[u] == idx[0] == labels[u] and sec[u] == idx[1]


def test_c5_shape_forward_and_viterbi_scores_match_oracle(ctx):
    """BASELINE configs[4] shape: N=3 states of M=128 mixtures (one state per 128-column image group), 16 models."""
    V, N, M, U = 16, 3, 128, 8
    cen, s = synth.make_centres(V, N, M, 39, seed=5000)
    labels = (np.arange(U) * 3 + 1) % V
    x, off = synth.make_utterances(cen, s, labels, seed=5001, tmin=40, tmax=70)
    ms = api.ModelSet.from_dict(synth.make_models(cen, s))
    ctx.set_features(x, off)
    ctx.set_models(ms)
    sc = ctx.forward_scores()
    vs = ctx.viterbi_scores()
    vown, path = ctx.viterbi(labels)
    lab, _ = ctx.rank(sc)
    with np.errstate(all="ignore"):
        for u in range(U):
            xu = x[off[u]:off[u + 1]]
            for v in range(V):
                mo = _oracle_model(ms, v)
                want = o.forward_score(mo, xu)
                b, _ = o.emissions(mo, xu, want_post=False)
                wv, wp = o.viterbi(mo, b)
                if np.isfinite(want):
                    assert abs(sc[u, v] - want) <= RTOL * abs(want), (u, v)
                    assert abs(vs[u, v] - wv) <= RTOL * abs(wv), (u, v)
                if v == labels[u]:
                    assert np.isfinite(want)
                    assert (path[off[u]:off[u + 1]] == wp).all() and abs(vown[u] - wv) <= 1e-9 * abs(wv)
    assert (lab == labels).all()


def test_large_estep_default_dispatch_matches_oracle(ctx):
    """A 1,600-utterance E-step through the default dispatch (534 batches of at most 3 utterances for the 592 teams of
    the resident forward-backward kernel on 148 SMs, several CTAs' partial sums per accumulate image): the statistics of
    three of the 16 words against the oracle's E-step on those words' utterances (T-FS:244-321).  Full batches and
    several batches per team: tests/test_fb_res_batches.py."""
    V, N, M, U = 16, 5, 4, 1600
    cen, s = synth.make_centres(V, N, M, 39, seed=6000)
    labels = np.arange(U) % V
    x, off = synth.make_utterances(cen, s, labels, seed=6001, tmin=30, tmax=90)
    rng = np.random.default_rng(6002)
    ms = api.ModelSet.from_dict(synth.make_models(cen + 0.3 * s * rng.standard_normal(cen.shape), s))
    ctx.set_features(x, off)
    ctx.set_models(ms)
    stats, lpu = ctx.estep(labels)
    assert np.isfinite(lpu).all()
    for v in (0, 7, 15):
        us = np.nonzero(labels == v)[0]
        xv = np.concatenate([x[off[u]:off[u + 1]] for u in us])
        offv = np.concatenate([[0], np.cumsum([off[u + 1] - off[u] for u in us])])
        st, lp = o.estep(_oracle_model(ms, v), xv, offv)
        sp = api.split_stats(stats[v], N, M, ms.D)
        assert np.allclose(lpu[us], lp, rtol=RTOL)
        assert abs(sp["sum_logp"] - st.sum_logp) <= RTOL * abs(st.sum_logp) and sp["n_utt"] == len(us)
        for name in ("num_trans", "den_trans", "den_mix", "S0"):
            want = getattr(st, name)
            assert np.allclose(sp[name], want, rtol=RTOL, atol=1e-6 * np.abs(want).max()), name
        S0 = np.maximum(st.S0, 1e-300)[..., None]
        sd = np.sqrt(st.S2c / S0)
        assert (np.abs(sp["S1"] / S0 - st.S1 / S0) <= RTOL * np.maximum(np.abs(st.S1 / S0), sd)).all(), "S1"
        assert np.allclose(sp["S2c"] / S0, st.S2c / S0, rtol=RTOL), "S2c"
        # and through the M-step: the re-estimated parameters
        mo = _oracle_model(ms, v)
        o.mstep(mo, st)
        one = api.ModelSet(ms.A[v:v + 1].copy(), ms.c[v:v + 1].copy(), ms.mu[v:v + 1].copy(), ms.iv[v:v + 1].copy(), ms.det[v:v + 1].copy())
        got = api.mstep(one, stats[v:v + 1])
        _assert_params_close(got, 0, mo)


def test_viterbi_tiny_cases_against_brute_force():
    """Second pin for the Viterbi kernels (the reference has none, R-FS:10-11): every state sequence of tiny
    models enumerated on the host (tests/viterbi_pins.py), emissions from a numpy restatement of calc_gaus."""
    from viterbi_pins import brute_viterbi, np_log_emissions, np_viterbi
    rng = np.random.default_rng(4242)
    c = api.Context(0)
    for N, D, full in ((1, 2, False), (2, 3, False), (3, 2, False), (3, 4, True), (2, 2, True)):
        V, M, U = 3, 2, 9
        A = rng.uniform(0.1, 1.0, size=(V, N, N))
        if not full:
            A = np.triu(A) - np.triu(A, 2)
        A /= A.sum(axis=2, keepdims=True)
        cw = rng.uniform(0.2, 1.0, size=(V, N, M)); cw /= cw.sum(axis=2, keepdims=True)
        mu = rng.standard_normal((V, N, M, D))
        var = rng.uniform(0.5, 2.0, size=(V, N, M, D))
        ms = api.ModelSet(A, cw, mu, 1.0 / var, var.prod(axis=3))
        T = rng.integers(max(N, 1), 9, size=U)
        T[0] = 1 if N == 1 else N                       # shortest utterance that can reach the final state
        off = np.concatenate([[0], np.cumsum(T)]).astype(np.int64)
        x = rng.standard_normal((int(off[-1]), D))
        labels = (np.arange(U) % V).astype(np.int32)
        c.set_features(x, off)
        c.set_models(ms)
        score, path = c.viterbi(labels)
        allsc = c.viterbi_scores()
        for u in range(U):
            v = labels[u]
            lb = np_log_emissions(ms.c[v], ms.mu[v], ms.iv[v], ms.det[v], x[off[u]:off[u + 1]])
            sb, pb = brute_viterbi(ms.A[v], lb)
            sn, pn = np_viterbi(ms.A[v], lb)
            assert sb == sn and (pb == pn).all()
            assert (path[off[u]:off[u + 1]] == pb).all(), (N, D, full, u)
            assert abs(score[u] - sb) <= 1e-9 * abs(sb)
            for w in range(V):
                lw = np_log_emissions(ms.c[w], ms.mu[w], ms.iv[w], ms.det[w], x[off[u]:off[u + 1]])
                assert abs(allsc[u, w] - brute_viterbi(ms.A[w], lw)[0]) <= 1e-5 * abs(sb) + 1e-4
    # exact ties: identical states and equal transition entries -> the lowest predecessor (R-FS:984's strict compare)
    A = np.array([[[0.25, 0.25, 0.5], [0.0, 0.5, 0.5], [0.0, 0.0, 1.0]]])
    ms = api.ModelSet(A, np.ones((1, 3, 1)), np.zeros((1, 3, 1, 2)), np.ones((1, 3, 1, 2)), np.ones((1, 3, 1)))
    off = np.array([0, 3, 7, 13, 21], dtype=np.int64)
    x = np.tile(rng.standard_normal((1, 2)), (21, 1))     # the same frame everywhere: equal emissions in every state
    c.set_features(x, off)
    c.set_models(ms)
    score, path = c.viterbi(np.zeros(4, dtype=np.int32))
    for u in range(4):
        lb = np_log_emissions(ms.c[0], ms.mu[0], ms.iv[0], ms.det[0], x[off[u]:off[u + 1]])
        sb, pb = brute_viterbi(A[0], lb)
        assert (path[off[u]:off[u + 1]] == pb).all() and abs(score[u] - sb) <= 1e-9 * abs(sb)
    c.close()


def test_cli_job_file_runs_every_line_in_one_process(tmp_path, monkeypatch):
    """`hmm_continuous_fs @jobs.txt` (one ordinary argument list per line, one CUDA context for all of them) writes the same
    models and reports as one invocation per word."""
    monkeypatch.chdir(tmp_path)
    N, M, V = 5, 3, 3
    cen, sc = synth.make_centres(V, N, M, 39, seed=901)
    labels = np.repeat(np.arange(V), 5)
    x, off = synth.make_utterances(cen, sc, labels, seed=902, tmin=50, tmax=90)
    exe = os.path.join(os.path.dirname(api.LIB_PATH), "bin", "hmm_continuous_fs")
    jobs = []
    for v in range(V):
        files = []
        for u in np.nonzero(labels == v)[0]:
            files.append(str(tmp_path / ("w%d_u%d.bin" % (v, u))))
            api.write_features(files[-1], x[off[u]:off[u + 1]])
        lst = str(tmp_path / ("list%d.txt" % v))
        write_list(lst, files)
        subprocess.run([exe, "word%d" % v, str(N), "1", str(M), lst, "single%d.hmm" % v], check=True, stdout=subprocess.DEVNULL)
        jobs.append("word%d %d 1 %d %s batch%d.hmm" % (v, N, M, lst, v))
    jf = str(tmp_path / "jobs.txt")
    open(jf, "w").write("\n".join(jobs) + "\n\n")
    subprocess.run([exe, "@" + jf], check=True, stdout=subprocess.DEVNULL)
    for v in range(V):
        a, b = api.read_model(str(tmp_path / ("single%d.hmm" % v))), api.read_model(str(tmp_path / ("batch%d.hmm" % v)))
        assert a.words == b.words == ["word%d" % v]
        for name in ("A", "c", "mu", "iv", "det"):
            assert np.allclose(getattr(a, name), getattr(b, name), rtol=1e-9, atol=1e-300), (v, name)
        assert r.parse_train_report(str(tmp_path / ("single%d.txt" % v))) == r.parse_train_report(str(tmp_path / ("batch%d.txt" % v)))


def test_peer_allreduce_sums_two_co_resident_ranks_in_rank_order():
    """hmmcu_peer_allreduce (the all-reduce of the sufficient statistics through peer memory, SURVEY 8e) with two
    contexts of one process standing in for two ranks: both end with the same bytes, equal to rank 0's statistics +
    rank 1's (double addition in rank order), over five iterations (the two slot sets alternate, so each is reused).
    The two ranks' kernels spin on each other's tagged words; here they run on the two contexts' streams and are
    co-resident on one GPU (each grid is at most 128 blocks of 256 threads, so both fit at once), so each one's words
    land while the other waits."""
    ms, x, off, labels = _synth(3, 5, 4, 12, seed=1212)
    U = len(labels)
    halves = [(0, U // 2), (U // 2, U)]
    ctxs = []
    for r_, (u0, u1) in enumerate(halves):
        c = api.Context(0)
        c.set_features(x[off[u0]:off[u1]], off[u0:u1 + 1] - off[u0])
        c.set_models(ms)
        c.peer_export(2)
        ctxs.append(c)
    areas = [c.peer_area() for c in ctxs]
    for r_, c in enumerate(ctxs):
        c.peer_import_pointers(r_, 2, areas)
    for it in range(5):
        local = []
        for r_, (c, (u0, u1)) in enumerate(zip(ctxs, halves)):
            st, _ = c.estep(labels[u0:u1])
            local.append(st)
        for c in ctxs:
            c.peer_allreduce()
        got = [c.stats_download() for c in ctxs]
        assert not ctxs[0].peer_error() and not ctxs[1].peer_error()
        want = local[0] + local[1]
        assert np.array_equal(got[0], got[1]) and np.array_equal(got[0], want), it
        for c in ctxs:  # the M-step on the summed statistics: identical models on both ranks
            c.em_reset() if it == 0 else None
        outs = [c.mstep(threshold=-1.0) for c in ctxs]
        assert np.array_equal(outs[0][0], outs[1][0])
        m0, m1 = ctxs[0].get_models(ms.D), ctxs[1].get_models(ms.D)
        assert np.array_equal(m0.mu, m1.mu) and np.array_equal(m0.iv, m1.iv) and np.array_equal(m0.A, m1.A)
    # against one E-step over all utterances
    c = api.Context(0)
    c.set_features(x, off)
    c.set_models(ms)
    full, _ = c.estep(labels)
    c.close()
    first = None
    for c in ctxs:
        c.set_models(ms)
    local = [c.estep(labels[u0:u1])[0] for c, (u0, u1) in zip(ctxs, halves)]
    assert np.allclose(local[0] + local[1], full, rtol=1e-5, atol=1e-6 * np.abs(full).max())
    for c in ctxs:
        c.close()
