"""Function-level parity of the oracle restatement against the reference's own object code
(oracle/_ref/libref_*.so).  The tests that call it are skipped where oracle/_ref has not been built."""
import os
import tempfile

import numpy as np
import pytest

from oracle import oracle as o
from oracle import ref as r
from speech_recognition_hmm_continuous_b200 import synth

needs_ref = pytest.mark.skipif(not r.available("d39m16"), reason="oracle/_ref not built (oracle/build_ref.sh)")


def _case(M, seed, U=3):
    cen, s = synth.make_centres(2, 5, M, 39, seed=seed)
    x, off = synth.make_utterances(cen, s, [0] * U, seed=seed + 1, tmin=40, tmax=70)
    mods = synth.make_models(cen, s)
    m = o.Model(mods["A"][0], mods["c"][0], mods["mu"][0], mods["iv"][0], mods["det"][0])
    return m, x, off


@needs_ref
@pytest.mark.parametrize("M", [1, 3, 16])
def test_estep_functions_bit_exact(M):
    m, x, off = _case(M, 11 + M)
    rt = r.RefTrain("d39m16")
    acc = rt.new_acc()
    tot = 0.0
    for u in range(len(off) - 1):
        xu = x[off[u]:off[u + 1]]
        out = rt.utterance(m, xu, acc)
        tot += out["logp"]
        b, post = o.emissions(m, xu)
        al, sc = o.forward(m, b)
        be = o.backward(m, b, sc)
        assert (b == out["b"]).all() and (post == out["post"]).all()
        assert (al == out["alpha"]).all() and (sc == out["scale"]).all() and (be == out["beta"]).all()
        assert o.logprob(al, sc) == out["logp"]
        assert o.gauss(xu[0], m.mu[0, 0], m.iv[0, 0], m.det[0, 0]) == rt.calc_gaus(xu[0], m.mu[0, 0], m.iv[0, 0], m.det[0, 0])
    st, _ = o.estep(m, x, off)
    rs = rt.acc_to_stats(acc, m.N, m.M, m.D)
    for k in ("num_trans", "den_trans", "den_mix", "S0", "S1", "S2c"):
        assert (getattr(st, k) == getattr(rs, k)).all(), k
    assert st.sum_logp == tot
    m_ref = rt.mstep(m, acc)
    m_orc = o.mstep(m.copy(), st)
    for k in ("A", "c", "mu", "iv", "det"):
        assert (getattr(m_ref, k) == getattr(m_orc, k)).all(), k


def test_final_state_weighting():
    """SURVEY 0.3: sum_i gamma_t(i) is the same at every t and equals alpha^[T-1][N-1] (<= 1)."""
    m, x, off = _case(3, 40, U=1)
    b, _ = o.emissions(m, x)
    al, sc = o.forward(m, b)
    be = o.backward(m, b, sc)
    g = (al * be / sc[:, None]).sum(axis=1)
    assert np.allclose(g, al[-1, -1], rtol=1e-9)


@needs_ref
@pytest.mark.parametrize("M", [2, 3, 5, 16])
def test_init_builder_and_cli_training(M):
    """creating_initial_model through the reference's entry point, and the whole trainer CLI
    (init + EM loop + model file) against orc_init_model + orc_train."""
    m0, x, off = _case(M, 70 + M, U=5)
    tmp = tempfile.mkdtemp()
    files = []
    for u in range(len(off) - 1):
        f = os.path.join(tmp, "u%d.bin" % u)
        r.write_features(f, x[off[u]:off[u + 1]])
        files.append(f)
    lst = os.path.join(tmp, "list.txt")
    open(lst, "w").write("\n".join(files) + "\n")
    mi = r.RefTrain("d39m16").init_model(5, M, lst)
    mo = o.init_model(5, M, x, off)
    for k in ("A", "c", "mu", "iv", "det"):
        assert (getattr(mi, k) == getattr(mo, k)).all(), k
    r.run_train_cli("d39m16", "w", 5, M, lst, os.path.join(tmp, "m.hmm"))
    mean_r, it_r = r.parse_train_report(os.path.join(tmp, "m.txt"))
    it, mean = o.train(mo, x, off)
    mr = r.read_model(os.path.join(tmp, "m.hmm"))
    assert it == it_r and "%.6f" % mean == "%.6f" % mean_r
    for k in ("A", "c", "mu", "iv", "det"):
        assert (getattr(mr, k) == getattr(mo, k)).all(), k


@needs_ref
def test_forward_score_and_rank():
    m, x, off = _case(3, 90)
    rte = r.RefTest("d39m16")
    for u in range(len(off) - 1):
        xu = x[off[u]:off[u + 1]]
        assert rte.forward_score(m, xu) == o.forward_score(m, xu)
    rng = np.random.default_rng(0)
    for _ in range(20):
        sc = rng.standard_normal(12)
        sc[rng.random(12) < 0.2] = np.nan
        sc[rng.random(12) < 0.1] = -np.inf
        sc[3] = sc[7]
        assert (rte.rank(sc) == o.rank(sc)).all()
