"""The host half of MMI training, without a GPU: hmmh_mstep_ebw (the extended Baum-Welch update) against the numpy
restatement in mmi_oracle.py, on statistics formed by oracle.estep, and the MMI buffer summed over two gloo ranks."""
import os
import socket

import numpy as np
import pytest

from mmi_oracle import FLOOR, ebw, mmi_buffer, model
from oracle import oracle as o
from speech_recognition_hmm_continuous_b200 import api, synth

V, N, M, D, U = 3, 4, 3, 13, 12


def _data(seed=7100):
    cen, s = synth.make_centres(V, N, M, D, seed=seed)
    labels = np.arange(U) % V
    x, off = synth.make_utterances(cen, s, labels, seed=seed + 1, tmin=12, tmax=30)
    rng = np.random.default_rng(seed + 2)
    ms = api.ModelSet.from_dict(synth.make_models(cen + 0.5 * s * rng.standard_normal(cen.shape), s))
    return ms, x, off, labels


def _scores(ms, x, off):
    return np.array([[o.forward_score(model(ms, v), x[off[u]:off[u + 1]]) for v in range(ms.V)] for u in range(len(off) - 1)])


def _check(ms, num, den, E, tau):
    want, got = ms.copy(), ms.copy()
    branch = {}
    ebw(want, num, den, E, tau, branch)
    api.mstep_ebw(got, num, den, E, tau)
    for a, b in ((got.mu, want.mu), (got.iv, want.iv), (got.det, want.det)):
        assert np.allclose(a, b, rtol=1e-12, atol=0), np.abs(a - b).max()
    assert (got.iv > 0).all() and (1.0 / got.iv >= FLOOR).all() and (got.det > 0).all()
    assert np.array_equal(got.A, ms.A) and np.array_equal(got.c, ms.c)  # weights and transitions stay
    return branch, got


def test_ebw_takes_both_constants_and_matches_the_restatement():
    ms, x, off, labels = _data()
    buf = mmi_buffer(ms, x, off, labels, _scores(ms, x, off), kappa=0.05, H=3)
    num, den = buf[0], buf[1].copy()
    # word 0: a denominator 1.5 times the numerator's occupancy, on frames one standard deviation away from the numerator's
    # (the D_min branch in every Gaussian of the word); the other words keep the E S0_den branch
    G, o0 = N * M, N * N + 2 * N
    s0, s1 = num[0, o0:o0 + G], num[0, o0 + G:o0 + G + G * D].reshape(G, D)
    s2 = num[0, o0 + G + G * D:o0 + G + 2 * G * D].reshape(G, D)
    mu, dl = ms.mu[0].reshape(G, D), np.sqrt(1.0 / ms.iv[0].reshape(G, D))
    den[0, o0:o0 + G] = 1.5 * s0
    den[0, o0 + G:o0 + G + G * D] = (1.5 * (s1 + dl * s0[:, None])).ravel()
    den[0, o0 + G + G * D:o0 + G + 2 * G * D] = (1.5 * (s2 + 2 * dl * (s1 - mu * s0[:, None]) + dl ** 2 * s0[:, None])).ravel()
    for tau in (0.0, 100.0):
        branch, _ = _check(ms, num, den, E=2.0, tau=tau)
        if tau == 0.0:  # (I-smoothing lifts the numerator above the denominator again)
            assert all(branch[(0, k)] == "dmin" for k in range(G)) and all(branch[(v, k)] == "e" for v in (1, 2) for k in range(G)), branch


def test_ebw_leaves_a_gaussian_without_occupancy_unchanged():
    ms, x, off, labels = _data(7200)
    buf = mmi_buffer(ms, x, off, labels, _scores(ms, x, off), kappa=0.05, H=3)
    num, den = buf[0].copy(), buf[1].copy()
    G = N * M
    o0 = N * N + 2 * N
    k = 4  # Gaussian 4 of word 1: nothing in either block
    for blk in (num, den):
        blk[1, o0 + k] = 0.0
        blk[1, o0 + G + k * D:o0 + G + (k + 1) * D] = 0.0
        blk[1, o0 + G + G * D + k * D:o0 + G + G * D + (k + 1) * D] = 0.0
    branch, got = _check(ms, num, den, E=2.0, tau=100.0)
    assert branch[(1, k)] == "none"
    g = got.mu[1].reshape(G, D)[k], got.iv[1].reshape(G, D)[k], got.det[1].reshape(G)[k]
    assert np.array_equal(g[0], ms.mu[1].reshape(G, D)[k]) and np.array_equal(g[1], ms.iv[1].reshape(G, D)[k]) and g[2] == ms.det[1].reshape(G)[k]


def test_ebw_without_denominator_is_the_textbook_ml_update():
    """den = 0, tau = 0: mu' = S1 / S0 (hmmh_mstep's mean, bit for bit), var' = Q / S0 - mu'^2, the variance about the
    NEW mean (hmmh_mstep's is about the old one: S2c / S0)."""
    ms, x, off, labels = _data(7300)
    buf = mmi_buffer(ms, x, off, labels, _scores(ms, x, off), kappa=0.05, H=1)
    num, den = buf[0], np.zeros_like(buf[0])
    _, got = _check(ms, num, den, E=2.0, tau=0.0)
    ml = api.mstep(ms.copy(), num)
    G = N * M
    o0 = N * N + 2 * N
    for v in range(V):
        s0 = num[v, o0:o0 + G]
        s2c = num[v, o0 + G + G * D:o0 + G + 2 * G * D].reshape(G, D)
        occ = s0 > 0
        assert np.array_equal(got.mu[v].reshape(G, D)[occ], ml.mu[v].reshape(G, D)[occ])
        shift = got.mu[v].reshape(G, D) - ms.mu[v].reshape(G, D)
        want_var = np.maximum(s2c / np.maximum(s0, 1e-300)[:, None] - shift ** 2, FLOOR)
        assert np.allclose((1.0 / got.iv[v].reshape(G, D))[occ], want_var[occ], rtol=1e-9)


def test_ebw_refuses_bad_constants():
    ms, x, off, labels = _data()
    z = np.zeros((V, api.stats_size(N, M, D)))
    for E, tau in ((1.0, 0.0), (0.5, 0.0), (2.0, -1.0)):
        with pytest.raises(api.HmmCudaError):
            api.mstep_ebw(ms.copy(), z, z, E, tau)


# ------------------------------------------------------------------------------ two gloo ranks ----
def _worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    ms, x, off, labels = _data()
    u0, u1 = api.shard_utterances(off, rank, world)
    t = torch.from_numpy(mmi_buffer(ms, x, off, labels, _scores(ms, x, off), kappa=0.05, H=3, us=range(u0, u1)))
    dist.all_reduce(t)  # both blocks and the objective in one collective
    buf = t.numpy()
    api.mstep_ebw(ms, buf[0], buf[1], 2.0, 100.0)
    q.put((rank, buf.copy(), ms.mu.copy(), ms.iv.copy(), ms.det.copy()))
    dist.barrier()
    dist.destroy_process_group()


def test_two_gloo_ranks_reproduce_the_single_process_mmi_iteration():
    torch = pytest.importorskip("torch")
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=300) for _ in procs], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for a, b in zip(res[0][1:], res[1][1:]):
        assert np.array_equal(a, b)  # bit-identical ranks
    ms, x, off, labels = _data()
    buf = mmi_buffer(ms, x, off, labels, _scores(ms, x, off), kappa=0.05, H=3)
    assert np.allclose(res[0][1], buf, rtol=1e-12, atol=1e-9)
    api.mstep_ebw(ms, buf[0], buf[1], 2.0, 100.0)
    for a, b in zip(res[0][2:], (ms.mu, ms.iv, ms.det)):
        assert np.allclose(a, b, rtol=1e-9, atol=0)
