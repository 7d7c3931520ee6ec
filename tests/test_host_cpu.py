"""Host-side logic of the product library (no GPU needed): C-ABI surface, file formats, initial-model
builder, M-step -- each against the oracle restatement / the reference's formats."""
import os
import re
import struct
import tempfile

import numpy as np
import pytest

from oracle import oracle as o
from oracle import ref as r
from speech_recognition_hmm_continuous_b200 import api, synth
from cli_lists import write_list

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _oracle_model(ms, v=0):
    return o.Model(ms.A[v], ms.c[v], ms.mu[v], ms.iv[v], ms.det[v], ms.words[v])


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "hmm_cuda.h")).read()
    declared = sorted(set(re.findall(r"\b(hmmcu_\w+|hmmh_\w+)\s*\(", hdr)) - {"hmmh_allreduce_fn"})
    lib = api.load()
    assert len(declared) >= 30
    for name in declared:
        assert hasattr(lib, name), name
    assert sorted(set(api.EXPORTS)) == declared


def test_no_device_fails_loudly():
    lib = api.load()
    if lib.hmmcu_device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(api.HmmCudaError) as e:
        api.Context(0)
    assert "no CPU path" in str(e.value) or "failed" in str(e.value)


def _case(M, seed, U=4, N=5):
    cen, s = synth.make_centres(1, N, M, 39, seed=seed)
    return synth.make_utterances(cen, s, [0] * U, seed=seed + 1, tmin=50, tmax=90)


@pytest.mark.parametrize("M", [1, 2, 3, 16])
def test_init_model_bit_exact_with_oracle(M):
    x, off = _case(M, 300 + M)
    ms = api.init_model(5, M, x, off)
    mo = o.init_model(5, M, x, off)
    for name, a in (("A", ms.A), ("c", ms.c), ("mu", ms.mu), ("iv", ms.iv), ("det", ms.det)):
        assert (a[0] == getattr(mo, name)).all(), name


@pytest.mark.parametrize("M", [1, 3])
def test_mstep_bit_exact_with_oracle(M):
    x, off = _case(M, 400 + M)
    mo = o.init_model(5, M, x, off)
    st, _ = o.estep(mo, x, off)
    vec = np.concatenate([st.num_trans.ravel(), st.den_trans, st.den_mix, st.S0.ravel(), st.S1.ravel(), st.S2c.ravel(),
                          [st.sum_logp, st.n_utt]])
    assert len(vec) == api.stats_size(5, M, 39)
    ms = api.ModelSet(mo.A[None], mo.c[None], mo.mu[None], mo.iv[None], mo.det[None])
    # a state without occupancy keeps its parameters and has its inverse variance inverted again (reference quirk)
    vec2 = vec.copy()
    sp = api.split_stats(vec2, 5, M, 39)
    sp["den_mix"][2] = 0.0
    st.den_mix[2] = 0.0
    api.mstep(ms, vec2[None])
    o.mstep(mo, st)
    for name, a in (("A", ms.A), ("c", ms.c), ("mu", ms.mu), ("iv", ms.iv), ("det", ms.det)):
        assert (a[0] == getattr(mo, name)).all(), name


def test_model_file_format(tmp_path):
    x, off = _case(3, 77)
    mo = o.init_model(5, 3, x, off, "palavra")
    ms = api.ModelSet(mo.A[None], mo.c[None], mo.mu[None], mo.iv[None], mo.det[None], ["palavra"])
    p = str(tmp_path / "m.hmm")
    api.write_model(p, ms)
    # byte-identical with the layout the reference writes (python restatement pinned in test_oracle_vs_ref)
    q = str(tmp_path / "q.hmm")
    r.write_model(q, mo)
    assert open(p, "rb").read() == open(q, "rb").read()
    back = api.read_model(p)
    assert back.words == ["palavra"] and (back.mu == ms.mu).all() and (back.iv == ms.iv).all() and (back.A == ms.A).all()
    # the shipped fixtures were written by a 32-bit build: 4-byte length header (SURVEY 4.2)
    raw = open(p, "rb").read()
    p32 = str(tmp_path / "m32.hmm")
    open(p32, "wb").write(struct.pack("<I", 7) + raw[8:])
    b32 = api.read_model(p32)
    assert b32.words == ["palavra"] and (b32.det == ms.det).all()


@pytest.mark.skipif(not r.available("d39m16"), reason="oracle/_ref not built")
def test_reads_model_written_by_reference(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    x, off = _case(3, 78)
    files = []
    for u in range(len(off) - 1):
        f = str(tmp_path / ("u%d.bin" % u))
        api.write_features(f, x[off[u]:off[u + 1]])
        files.append(f)
    lst = str(tmp_path / "l.txt")
    write_list(lst, files)
    r.run_train_cli("d39m16", "abc", 5, 3, "l.txt", "m.hmm")
    a = api.read_model(str(tmp_path / "m.hmm"))
    b = r.read_model(str(tmp_path / "m.hmm"))
    assert a.words == ["abc"]
    for name, arr in (("A", a.A), ("c", a.c), ("mu", a.mu), ("iv", a.iv), ("det", a.det)):
        assert (arr[0] == getattr(b, name)).all()


def test_feature_file_format(golden_dir, tmp_path):
    f = os.path.join(golden_dir, "perfil", "mean_vc_186_f_03_ap_0225.perfil")
    x = api.read_features(f)
    assert x.shape == (151, 9) and (x == r.read_features(f)).all()
    p = str(tmp_path / "x.bin")
    api.write_features(p, x)
    assert open(p, "rb").read() == open(f, "rb").read()


def test_split_stats_layout():
    N, M, D = 3, 2, 4
    vec = np.arange(api.stats_size(N, M, D), dtype=np.float64)
    sp = api.split_stats(vec, N, M, D)
    assert sp["num_trans"][0, 0] == 0 and sp["den_trans"][0] == 9 and sp["den_mix"][0] == 12 and sp["S0"][0, 0] == 15
    assert sp["S1"][0, 0, 0] == 21 and sp["S2c"][0, 0, 0] == 45 and sp["sum_logp"] == 69 and sp["n_utt"] == 70


# ---- many-files reader (SURVEY 8f-2): the pipeline of hmmh_ingest driven into a memory sink ----
def _write_files(tmp_path, lens, D=7, seed=5):
    rng = np.random.default_rng(seed)
    paths, xs = [], []
    for i, T in enumerate(lens):
        x = rng.standard_normal((T, D))
        p = str(tmp_path / ("f%04d.bin" % i))
        api.write_features(p, x)
        paths.append(p)
        xs.append(x)
    return paths, xs


@pytest.mark.parametrize("threads,stage_frames", [(1, 0), (4, 0), (8, 64), (3, 1)])
def test_ingest_pipeline_matches_per_file_reader(tmp_path, threads, stage_frames):
    lens = [1, 17, 300, 250, 64, 2, 349, 33, 90, 128, 5, 77] * 3   # ragged, including one-frame utterances
    paths, xs = _write_files(tmp_path, lens)
    x, off, st, log = api.ingest_to_memory(paths, threads=threads, stage_frames=stage_frames)
    assert off.tolist() == np.concatenate([[0], np.cumsum(lens)]).tolist()
    assert np.array_equal(x, np.concatenate(xs))          # bit-exact and every frame delivered exactly once
    assert sum(n for _, n in log) == sum(lens) and st.bytes == 8 * 7 * sum(lens)
    if stage_frames:   # batches respect the staging size except for single longer utterances; consecutive and ordered
        assert all(n <= max(stage_frames, max(lens)) for _, n in log)
        assert [f for f, _ in log] == np.concatenate([[0], np.cumsum([n for _, n in log])[:-1]]).tolist()
        assert st.batches == len(log) > 1
    # the per-file reader sees the same frames
    for p, xr in zip(paths[:4], xs[:4]):
        assert np.array_equal(api.read_features(p), xr)


def test_ingest_scan_drops_a_trailing_partial_frame_and_reports_bad_files(tmp_path):
    paths, xs = _write_files(tmp_path, [10, 20, 30])
    with open(paths[1], "ab") as f:
        f.write(b"\0" * 13)                                 # a torn last frame (T-FS:536 reads until fread fails)
    off, D = api.scan_features(paths)
    assert D == 7 and off.tolist() == [0, 10, 30, 60]
    x, off2, _, _ = api.ingest_to_memory(paths, threads=2)
    assert np.array_equal(x, np.concatenate(xs))
    with pytest.raises(api.HmmCudaError, match="file 2"):
        api.ingest_to_memory(paths[:2] + [str(tmp_path / "missing.bin")])
    other = [str(tmp_path / "d9.bin")]
    api.write_features(other[0], np.zeros((5, 9)))
    with pytest.raises(api.HmmCudaError, match="file 3"):    # a file of another width
        api.ingest_to_memory(paths + other)
    empty = str(tmp_path / "empty.bin")
    with open(empty, "wb") as f:
        f.write(struct.pack("i", 7))
    with pytest.raises(api.HmmCudaError, match="file 1"):    # header only: no frames
        api.ingest_to_memory([paths[0], empty])


def test_read_list_tokens(tmp_path):
    import ctypes as C
    lib = api.load()
    lst = tmp_path / "list.txt"
    lst.write_text("a.bin  b.bin\n\n c.bin\t" + "x" * 120 + "\n")
    pp, n = C.POINTER(C.c_char_p)(), C.c_int()
    lib.hmmh_read_list.argtypes = [C.c_char_p, C.POINTER(C.POINTER(C.c_char_p)), C.POINTER(C.c_int)]
    assert lib.hmmh_read_list(str(lst).encode(), C.byref(pp), C.byref(n)) == 0
    toks = [pp[i].decode() for i in range(n.value)]
    # fscanf("%99s") semantics: a 120-character token arrives as 99 + 21 characters (T-FS:272, char[100])
    assert toks == ["a.bin", "b.bin", "c.bin", "x" * 99, "x" * 21]
    lib.hmmh_free_list.argtypes = [C.POINTER(C.c_char_p), C.c_int]
    lib.hmmh_free_list(pp, n.value)


# ---- bulk .hmm I/O (SURVEY 8f-3) ----
def _random_set(V, N, M, D, seed):
    rng = np.random.default_rng(seed)
    A = rng.random((V, N, N))
    return api.ModelSet(A, rng.random((V, N, M)), rng.standard_normal((V, N, M, D)), rng.random((V, N, M, D)) + 0.1,
                        rng.random((V, N, M)) + 1e-3, ["w%03d_%s" % (v, "x" * (v % 40)) for v in range(V)])


@pytest.mark.parametrize("threads", [1, 7])
def test_model_set_bulk_io_is_byte_identical_to_the_single_file_path(tmp_path, threads):
    V, N, M, D = 37, 5, 3, 39
    ms = _random_set(V, N, M, D, 77)
    one = [str(tmp_path / ("one%03d.hmm" % v)) for v in range(V)]
    bulk = [str(tmp_path / ("bulk%03d.hmm" % v)) for v in range(V)]
    for v in range(V):
        api.write_model(one[v], ms, v)
    api.write_model_set(bulk, ms, threads=threads)
    for a, b in zip(one, bulk):
        assert open(a, "rb").read() == open(b, "rb").read()
    back = api.read_model_set(one, threads=threads)
    assert back.words == ms.words
    for k in ("A", "c", "mu", "iv", "det"):
        assert np.array_equal(getattr(back, k), getattr(ms, k)), k
    single = api.read_model(one[5])
    assert np.array_equal(single.mu[0], back.mu[5]) and single.words[0] == back.words[5]


def test_model_set_reader_takes_32_bit_headers_and_reports_bad_files(tmp_path):
    ms = _random_set(4, 3, 2, 5, 3)
    paths = [str(tmp_path / ("m%d.hmm" % v)) for v in range(4)]
    api.write_model_set(paths, ms)
    raw = open(paths[2], "rb").read()                         # the shipped fixtures carry a 4-byte length (SURVEY 4.2)
    open(paths[2], "wb").write(raw[:4] + raw[8:])
    back = api.read_model_set(paths)
    assert np.array_equal(back.mu, ms.mu) and back.words == ms.words
    open(paths[3], "wb").write(open(paths[3], "rb").read()[:-8])   # truncated
    with pytest.raises(api.HmmCudaError, match=r"\(5\) at file 3"):
        api.read_model_set(paths)
    other = str(tmp_path / "other.hmm")
    api.write_model_set([other], _random_set(1, 3, 4, 5, 1))        # another mixture count
    with pytest.raises(api.HmmCudaError, match=r"\(1\) at file 1"):
        api.read_model_set([paths[0], other, paths[1]])
    with pytest.raises(api.HmmCudaError, match="at file 0"):
        api.read_model_set([str(tmp_path / "missing.hmm")])


def test_model_set_reader_reads_reference_written_files(tmp_path, monkeypatch):
    """Models written by the compiled reference trainer come back identical through the bulk reader."""
    if not r.available("d39m16"):
        pytest.skip("compiled reference not present")
    monkeypatch.chdir(tmp_path)
    paths = []
    for w in range(2):
        x, off = _case(3, 78 + w)
        files = []
        for u in range(len(off) - 1):
            f = str(tmp_path / ("w%du%d.bin" % (w, u)))
            api.write_features(f, x[off[u]:off[u + 1]])
            files.append(f)
        lst = str(tmp_path / ("l%d.txt" % w))
        write_list(lst, files)
        paths.append(str(tmp_path / ("m%d.hmm" % w)))
        r.run_train_cli("d39m16", "word%d" % w, 5, 3, os.path.basename(lst), os.path.basename(paths[-1]))
    back = api.read_model_set(paths)
    assert back.words == ["word0", "word1"]
    for w in range(2):
        b = r.read_model(paths[w])
        for name, arr in (("A", back.A), ("c", back.c), ("mu", back.mu), ("iv", back.iv), ("det", back.det)):
            assert (arr[w] == getattr(b, name)).all()


# ---- feature streams (param_number > 1): the P-stream .hmm file ----
def test_multi_stream_model_file_round_trip_and_reference_layout(tmp_path, golden_dir):
    g = np.load(os.path.join(golden_dir, "synth_p2.npz"))
    streams = [api.ModelSet(*[g["trained_s%d_%s" % (p, k)][:1] for k in ("A", "c", "mu", "iv", "det")], words=["word0"]) for p in range(2)]
    path = str(tmp_path / "p2.hmm")
    api.write_model_streams(path, streams)
    back = api.read_model_streams(path)
    assert len(back) == 2 and back[0].words == ["word0"] and (back[0].M, back[0].D, back[1].M, back[1].D) == (2, 6, 3, 4)
    for p in range(2):
        for k in ("A", "c", "mu", "iv", "det"):
            assert np.array_equal(getattr(back[p], k), getattr(streams[p], k)), (p, k)
    # the layout is the reference's (T-FS:2058-2144): its own parser restated in oracle/ref.py reads the file ...
    ref = r.read_model_streams(path)
    assert len(ref) == 2 and ref[0].word == "word0" and np.array_equal(ref[1].mu, streams[1].mu[0])
    # ... a single-stream reader refuses it, and a one-stream file written through the P-stream writer is the old format
    with pytest.raises(api.HmmCudaError):
        api.read_model(path)
    one, one_s = str(tmp_path / "a.hmm"), str(tmp_path / "b.hmm")
    api.write_model(one, streams[0])
    api.write_model_streams(one_s, streams[:1])
    assert open(one, "rb").read() == open(one_s, "rb").read()


def test_multi_stream_model_file_written_by_reference(tmp_path, golden_dir, monkeypatch):
    """The reference trainer run with two streams writes a file our reader takes (and vice versa: byte-identical rewrite)."""
    if not r.available("p2"):
        pytest.skip("compiled two-stream reference not present")
    import subprocess
    monkeypatch.chdir(tmp_path)
    g = np.load(os.path.join(golden_dir, "synth_p2.npz"))
    off, lists = g["off"], []
    for p in range(2):
        files = []
        for u in np.nonzero(g["train_labels"] == 0)[0]:
            files.append(str(tmp_path / ("s%d_%d.bin" % (p, u))))
            api.write_features(files[-1], g["x%d" % p][off[u]:off[u + 1]])
        lists.append(str(tmp_path / ("l%d.txt" % p)))
        write_list(lists[-1], files)
    hmm = str(tmp_path / "ref.hmm")
    subprocess.run([os.path.join(r.REF_DIR, "hmm_fs_p2"), "word0", str(int(g["N"])), "2", str(g["M"][0]), str(g["M"][1]), "l0.txt", "l1.txt", "ref.hmm"],
                   stdout=subprocess.DEVNULL, check=True)
    back = api.read_model_streams(hmm)
    for p in range(2):
        for k in ("A", "c", "mu", "iv", "det"):
            assert np.array_equal(getattr(back[p], k)[0], g["trained_s%d_%s" % (p, k)][0]), (p, k)
    again = str(tmp_path / "again.hmm")
    api.write_model_streams(again, back)
    assert open(again, "rb").read() == open(hmm, "rb").read()


# ---- drop-in programs: argument and file errors happen before any device work (reference: message on stdout, exit(1)) ----
def test_cli_usage_and_file_errors():
    import subprocess
    bindir = os.path.join(os.path.dirname(api.LIB_PATH), "bin")
    tr, te = os.path.join(bindir, "hmm_continuous_fs"), os.path.join(bindir, "recognition_continuous_fs")
    p = subprocess.run([tr, "w", "5"], stdout=subprocess.PIPE)
    assert p.returncode == 1 and p.stdout.decode().startswith("Usage: hmm_continuous_fs word states_number param_number")
    p = subprocess.run([te, "1"], stdout=subprocess.PIPE)
    assert p.returncode == 1 and p.stdout.decode().startswith("Usage: recognition_continuous_fs models_number")
    p = subprocess.run([tr, "w", "5", "1", "3", "/nonexistent/list.txt", "/tmp/o.hmm"], stdout=subprocess.PIPE)
    assert p.returncode == 1 and "file /nonexistent/list.txt not found" in p.stdout.decode()
    p = subprocess.run([tr, "w", "5", "2", "3", "3", "/nonexistent/a.txt", "/nonexistent/b.txt", "/tmp/o.hmm"], stdout=subprocess.PIPE)
    assert p.returncode == 1 and "file /nonexistent/a.txt not found" in p.stdout.decode()
    # the recogniser opens the model lists first, then the feature lists, then the words file (R-FS:203-266)
    p = subprocess.run([te, "1", "/nonexistent/m.txt", "1", "/nonexistent/f.txt", "/nonexistent/w.txt", "/tmp/r.txt"], stdout=subprocess.PIPE)
    assert p.returncode == 1 and "file /nonexistent/m.txt not found" in p.stdout.decode()
    p = subprocess.run([te, "2", "/nonexistent/m.txt", "1", "/nonexistent/f.txt", "/nonexistent/w.txt", "/tmp/r.txt"], stdout=subprocess.PIPE)
    assert p.returncode == 1 and "does not match the argument list" in p.stdout.decode()


def test_cli_refuses_models_beyond_the_state_limit_up_front(tmp_path, monkeypatch):
    """The kernels are built for HMMCU_MAX_STATES = 8 states per model (the reference allows 20 / 15, T-FS:41, R-FS:37).
    Both programs say so before reading any feature file or touching the device; .hmm files with more states are still
    read and written by the host-side file code (HMMH_MAX_FILE_STATES)."""
    import subprocess
    bindir = os.path.join(os.path.dirname(api.LIB_PATH), "bin")
    tr, te = os.path.join(bindir, "hmm_continuous_fs"), os.path.join(bindir, "recognition_continuous_fs")
    p = subprocess.run([tr, "w", "9", "1", "3", "/nonexistent/list.txt", "/tmp/o.hmm"], stdout=subprocess.PIPE)
    out = p.stdout.decode()
    assert p.returncode == 1 and "states_number 9 is beyond this build's limit of 8 states" in out and "not found" not in out
    # a 12-state model file: written and read back by the file code, refused by the recogniser with its name
    N, M, Dm = 12, 2, 5
    rng = np.random.default_rng(3)
    A = np.triu(np.ones((N, N))) - np.triu(np.ones((N, N)), 2)
    A /= A.sum(axis=1, keepdims=True)
    var = rng.uniform(0.5, 2.0, size=(1, N, M, Dm))
    ms = api.ModelSet(A[None], np.full((1, N, M), 0.5), rng.standard_normal((1, N, M, Dm)), 1.0 / var, var.prod(axis=3), words=["big"])
    hmm = str(tmp_path / "big.hmm")
    api.write_model(hmm, ms)
    back = api.read_model(hmm)
    assert back.N == N and np.array_equal(back.mu, ms.mu)
    ml = str(tmp_path / "models.txt")
    monkeypatch.chdir(tmp_path)
    write_list(ml, [hmm])
    fl, wl = str(tmp_path / "f.txt"), str(tmp_path / "w.txt")   # empty test set: the model check comes before any device work
    open(fl, "w").close()
    open(wl, "w").close()
    p = subprocess.run([te, "1", ml, "1", fl, wl, str(tmp_path / "r.txt")], stdout=subprocess.PIPE)
    out = p.stdout.decode()
    assert p.returncode == 1 and "has 12 states: beyond this build's limit of 8" in out
