"""Python mirror of the C ABI in include/hmm_cuda.h (ctypes over libhmmcu.so).

This is the host-side harness used by tests/ and bench.py; the product is the shared library.
There is NO fallback: if libhmmcu.so is missing or no sm_100 device is present, every entry point
raises.  Names follow the reference's functions they stand in for (see the header).
"""
import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libhmmcu.so")

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)
_lp = C.POINTER(C.c_int64)

EXPORTS = [
    "hmmcu_create", "hmmcu_destroy", "hmmcu_last_error", "hmmcu_device_count", "hmmcu_stream", "hmmcu_synchronize",
    "hmmcu_host_alloc", "hmmcu_host_free", "hmmcu_set_option", "hmmcu_set_features", "hmmcu_set_features_device", "hmmcu_set_models",
    "hmmcu_init_models", "hmmcu_emissions", "hmmcu_forward_scores", "hmmcu_rank", "hmmcu_stats_size", "hmmcu_estep", "hmmcu_estep_viterbi", "hmmcu_estep_mmi", "hmmcu_stats_device",
    "hmmcu_stats_download", "hmmcu_em_reset", "hmmcu_mstep", "hmmcu_mstep_ebw", "hmmcu_get_models", "hmmcu_viterbi", "hmmcu_viterbi_scores", "hmmcu_launch_count", "hmmcu_last_kernel_ms",
    "hmmcu_enable_timing", "hmmh_model_alloc", "hmmh_model_free", "hmmh_read_features", "hmmh_write_features",
    "hmmh_read_model", "hmmh_write_model", "hmmh_init_model", "hmmh_mstep", "hmmh_mstep_ebw", "hmmh_upload_models", "hmmh_train", "hmmh_train_viterbi", "hmmh_train_mmi",
    "hmmh_train_main", "hmmh_test_main",
    "hmmcu_features_begin", "hmmcu_features_append", "hmmcu_features_wait", "hmmcu_features_end", "hmmcu_staging", "hmmcu_link_streams", "hmmh_read_model_streams", "hmmh_write_model_streams", "hmmh_train_streams",
    "hmmh_model_set_alloc", "hmmh_model_set_free", "hmmh_read_model_set", "hmmh_write_model_set", "hmmh_upload_model_set",
    "hmmh_read_list", "hmmh_free_list", "hmmh_scan_features", "hmmh_ingest_to", "hmmh_ingest",
    "hmmcu_peer_export", "hmmcu_peer_import", "hmmcu_peer_area", "hmmcu_peer_import_pointers", "hmmcu_peer_allreduce",
    "hmmcu_peer_error",
]


class HmmCudaError(RuntimeError):
    pass


class _CModel(C.Structure):
    _fields_ = [("word", C.c_char * 64), ("N", C.c_int), ("M", C.c_int), ("D", C.c_int), ("A", _dp), ("c", _dp),
                ("mu", _dp), ("inv_var", _dp), ("det", _dp)]


class _CModelSet(C.Structure):  # hmmh_model_set
    _fields_ = [("V", C.c_int), ("N", C.c_int), ("M", C.c_int), ("D", C.c_int), ("word", C.POINTER(C.c_char * 64)), ("A", _dp), ("c", _dp),
                ("mu", _dp), ("inv_var", _dp), ("det", _dp)]


ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p)

_lib = None


class IngestStats(C.Structure):  # hmmh_ingest_stats
    _fields_ = [("scan_s", C.c_double), ("stage_s", C.c_double), ("read_s", C.c_double), ("total_s", C.c_double), ("bytes", C.c_int64),
                ("batches", C.c_int), ("threads", C.c_int)]


_SinkBegin = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_int64), C.c_int, C.c_int)
_SinkAppend = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_double), C.c_int64, C.c_int64, C.POINTER(C.c_int))
_SinkWait = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int)
_SinkEnd = C.CFUNCTYPE(C.c_int, C.c_void_p)


class _CSink(C.Structure):  # hmmh_sink
    _fields_ = [("user", C.c_void_p), ("begin", _SinkBegin), ("append", _SinkAppend), ("wait", _SinkWait), ("end", _SinkEnd),
                ("stage_alloc", C.c_void_p)]


def _libc_free(p):
    libc = C.CDLL(None)
    libc.free.argtypes = [C.c_void_p]
    libc.free(C.cast(p, C.c_void_p))


def load():
    """Loads libhmmcu.so (built in-tree by build.py).  Fails loudly when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise HmmCudaError("%s not found: build it with `python -m speech_recognition_hmm_continuous_b200.build` "
                           "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    lib.hmmcu_last_error.restype = C.c_char_p
    lib.hmmcu_last_error.argtypes = [C.c_void_p]
    lib.hmmcu_stream.restype = C.c_void_p
    lib.hmmcu_stream.argtypes = [C.c_void_p]
    lib.hmmcu_stats_size.restype = C.c_int64
    lib.hmmcu_launch_count.restype = C.c_int64
    lib.hmmcu_launch_count.argtypes = [C.c_void_p]
    lib.hmmcu_last_kernel_ms.restype = C.c_double
    lib.hmmcu_last_kernel_ms.argtypes = [C.c_void_p, C.c_char_p]
    lib.hmmcu_stats_device.restype = C.c_void_p
    lib.hmmcu_stats_device.argtypes = [C.c_void_p, _lp]
    lib.hmmcu_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    lib.hmmcu_destroy.argtypes = [C.c_void_p]
    lib.hmmcu_synchronize.argtypes = [C.c_void_p]
    lib.hmmcu_enable_timing.argtypes = [C.c_void_p, C.c_int]
    lib.hmmcu_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
    lib.hmmcu_set_features.argtypes = [C.c_void_p, C.c_void_p, _lp, C.c_int, C.c_int]
    lib.hmmcu_set_features_device.argtypes = [C.c_void_p, C.c_void_p, _lp, C.c_int, C.c_int]
    lib.hmmcu_set_models.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, _dp, _dp, _dp, _dp, _dp]
    lib.hmmcu_emissions.argtypes = [C.c_void_p, C.c_int, C.c_int, _dp, _dp]
    lib.hmmcu_init_models.argtypes = [C.c_void_p, _ip, C.c_int, C.c_int, C.c_int]
    lib.hmmcu_forward_scores.argtypes = [C.c_void_p, _dp, C.c_int]
    lib.hmmcu_viterbi_scores.argtypes = [C.c_void_p, _dp]
    lib.hmmcu_rank.argtypes = [C.c_void_p, _dp, C.c_int, C.c_int, C.c_double, _ip, _ip]
    lib.hmmcu_estep.argtypes = [C.c_void_p, _ip, _dp, _dp]
    lib.hmmcu_estep_viterbi.argtypes = [C.c_void_p, _ip, _dp, _dp, _ip]
    lib.hmmcu_estep_mmi.argtypes = [C.c_void_p, _ip, C.c_double, C.c_int, _dp]
    lib.hmmcu_mstep_ebw.argtypes = [C.c_void_p, C.c_double, C.c_double]
    lib.hmmcu_stats_download.argtypes = [C.c_void_p, _dp]
    lib.hmmcu_em_reset.argtypes = [C.c_void_p]
    lib.hmmcu_mstep.argtypes = [C.c_void_p, C.c_double, _dp, _dp, _ip]
    lib.hmmcu_get_models.argtypes = [C.c_void_p, _dp, _dp, _dp, _dp, _dp]
    lib.hmmcu_viterbi.argtypes = [C.c_void_p, _ip, _dp, _ip]
    lib.hmmcu_host_alloc.argtypes = [C.POINTER(C.c_void_p), C.c_uint64]
    lib.hmmcu_host_free.argtypes = [C.c_void_p]
    lib.hmmh_model_alloc.argtypes = [C.POINTER(_CModel), C.c_int, C.c_int, C.c_int]
    lib.hmmh_model_free.argtypes = [C.POINTER(_CModel)]
    lib.hmmh_read_model.argtypes = [C.c_char_p, C.POINTER(_CModel), C.c_int]
    lib.hmmh_write_model.argtypes = [C.c_char_p, C.POINTER(_CModel)]
    lib.hmmh_read_features.argtypes = [C.c_char_p, C.POINTER(_dp), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.hmmh_write_features.argtypes = [C.c_char_p, _dp, C.c_int, C.c_int]
    lib.hmmh_init_model.argtypes = [C.POINTER(_CModel), _dp, _lp, C.c_int]
    lib.hmmh_model_set_free.argtypes = [C.POINTER(_CModelSet)]
    lib.hmmh_read_model_set.argtypes = [C.POINTER(C.c_char_p), C.c_int, C.c_int, C.POINTER(_CModelSet), C.POINTER(C.c_int)]
    lib.hmmh_write_model_set.argtypes = [C.POINTER(C.c_char_p), C.POINTER(_CModelSet), C.c_int, C.POINTER(C.c_int)]
    lib.hmmh_upload_model_set.argtypes = [C.c_void_p, C.POINTER(_CModelSet)]
    lib.hmmcu_link_streams.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_int]
    lib.hmmcu_features_begin.argtypes = [C.c_void_p, _lp, C.c_int, C.c_int]
    lib.hmmcu_features_append.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.POINTER(C.c_int)]
    lib.hmmcu_features_wait.argtypes = [C.c_void_p, C.c_int]
    lib.hmmcu_features_end.argtypes = [C.c_void_p]
    lib.hmmh_scan_features.argtypes = [C.POINTER(C.c_char_p), C.c_int, C.c_int, C.POINTER(C.c_int), _lp, C.POINTER(C.c_int)]
    lib.hmmh_ingest_to.argtypes = [C.POINTER(_CSink), C.POINTER(C.c_char_p), C.c_int, C.c_int, C.c_int64, _lp, C.POINTER(C.c_int),
                                   C.POINTER(C.c_int), C.POINTER(IngestStats)]
    lib.hmmh_ingest.argtypes = [C.c_void_p, C.POINTER(C.c_char_p), C.c_int, C.c_int, _lp, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                C.POINTER(IngestStats)]
    lib.hmmh_mstep.argtypes = [C.POINTER(_CModel), _dp]
    lib.hmmh_mstep_ebw.argtypes = [C.POINTER(_CModel), _dp, _dp, C.c_double, C.c_double]
    lib.hmmh_train_mmi.argtypes = [C.c_void_p, C.POINTER(_CModel), C.c_int, _ip, C.c_int, C.c_double, C.c_int, C.c_double, C.c_double,
                                   C.c_int, _dp, C.c_void_p, C.c_void_p]
    lib.hmmh_upload_models.argtypes = [C.c_void_p, C.POINTER(_CModel), C.c_int]
    for f in ("hmmh_train", "hmmh_train_viterbi"):
        getattr(lib, f).argtypes = [C.c_void_p, C.POINTER(_CModel), C.c_int, _ip, C.c_int, _dp, C.POINTER(C.c_int), C.c_int,
                                    C.c_void_p, C.c_void_p]
    lib.hmmcu_peer_export.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    lib.hmmcu_peer_import.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_char_p]
    lib.hmmcu_peer_area.restype = C.c_void_p
    lib.hmmcu_peer_area.argtypes = [C.c_void_p]
    lib.hmmcu_peer_import_pointers.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
    for f in ("hmmcu_peer_allreduce", "hmmcu_peer_error"):
        getattr(lib, f).argtypes = [C.c_void_p]
    _lib = lib
    return lib


def _d(a):
    return a.ctypes.data_as(_dp)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def stats_size(N, M, D):
    return N * N + 2 * N + N * M + 2 * N * M * D + 2


def split_stats(vec, N, M, D):
    """One model's statistics vector -> dict of arrays (layout of hmmcu_stats_size)."""
    vec = np.asarray(vec)
    o = 0
    out = {}
    for name, shape in (("num_trans", (N, N)), ("den_trans", (N,)), ("den_mix", (N,)), ("S0", (N, M)),
                        ("S1", (N, M, D)), ("S2c", (N, M, D))):
        n = int(np.prod(shape))
        out[name] = vec[o:o + n].reshape(shape)
        o += n
    out["sum_logp"] = float(vec[o])
    out["n_utt"] = float(vec[o + 1])
    return out


class ModelSet:
    """V models of one topology, stacked float64 arrays in the reference's semantics."""

    def __init__(self, A, c, mu, iv, det, words=None):
        self.A, self.c, self.mu, self.iv, self.det = _f64(A), _f64(c), _f64(mu), _f64(iv), _f64(det)
        self.V, self.N, self.M, self.D = self.mu.shape
        assert self.A.shape == (self.V, self.N, self.N) and self.c.shape == (self.V, self.N, self.M)
        assert self.iv.shape == self.mu.shape and self.det.shape == (self.V, self.N, self.M)
        self.words = list(words) if words is not None else ["word%d" % v for v in range(self.V)]

    @classmethod
    def from_dict(cls, d, words=None):
        return cls(d["A"], d["c"], d["mu"], d["iv"], d["det"], words)

    def copy(self):
        return ModelSet(self.A.copy(), self.c.copy(), self.mu.copy(), self.iv.copy(), self.det.copy(), self.words)

    def _cmodels(self):
        arr = (_CModel * self.V)()
        for v in range(self.V):
            m = arr[v]
            m.word = self.words[v].encode()[:63]
            m.N, m.M, m.D = self.N, self.M, self.D
            m.A, m.c, m.mu, m.inv_var, m.det = _d(self.A[v]), _d(self.c[v]), _d(self.mu[v]), _d(self.iv[v]), _d(self.det[v])
        return arr


def _allreduce_hook(allreduce):
    """allreduce(dev_ptr, n_doubles, stream_ptr) -> None as an hmmh_allreduce_fn (None stays None)."""
    if allreduce is None:
        return None

    def _cb(user, dev, n, stream):
        allreduce(dev, n, stream)
        return 0
    return ALLREDUCE_FN(_cb)


class Context:
    """One device context (hmmcu_create).  Raises HmmCudaError when no B200 is present."""

    def __init__(self, device=0, timing=False):
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.hmmcu_create(int(device), C.byref(h))
        if rc != 0:
            raise HmmCudaError("hmmcu_create(%d) failed (%d): %s" % (device, rc, self.lib.hmmcu_last_error(None).decode()))
        self.h = h
        self.U = self.V = 0
        self._keep = None
        if timing:
            self.lib.hmmcu_enable_timing(self.h, 1)

    def enable_timing(self, on=True):
        """Per-kernel device timers (kernel_ms); turns the CUDA-graph replay of the EM iteration off."""
        self.lib.hmmcu_enable_timing(self.h, 1 if on else 0)

    def close(self):
        if getattr(self, "h", None):
            self.lib.hmmcu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc, what):
        if rc != 0:
            raise HmmCudaError("%s failed (%d): %s" % (what, rc, self.lib.hmmcu_last_error(self.h).decode()))

    # ---- inputs ----
    def set_features(self, x, off):
        x = _f64(x)
        off = np.ascontiguousarray(off, dtype=np.int64)
        self.U, self.D, self.F = len(off) - 1, x.shape[1], int(off[-1])
        self.off = off
        self._ck(self.lib.hmmcu_set_features(self.h, x.ctypes.data, off.ctypes.data_as(_lp), self.U, self.D), "hmmcu_set_features")

    def set_features_ptr(self, host_ptr, off, D):
        """x given as a raw host pointer (e.g. pinned memory)."""
        off = np.ascontiguousarray(off, dtype=np.int64)
        self.U, self.D, self.F = len(off) - 1, D, int(off[-1])
        self.off = off
        self._ck(self.lib.hmmcu_set_features(self.h, host_ptr, off.ctypes.data_as(_lp), self.U, D), "hmmcu_set_features")

    def set_features_device(self, dev_ptr, off, D):
        off = np.ascontiguousarray(off, dtype=np.int64)
        self.U, self.D, self.F = len(off) - 1, D, int(off[-1])
        self.off = off
        self._ck(self.lib.hmmcu_set_features_device(self.h, dev_ptr, off.ctypes.data_as(_lp), self.U, D), "hmmcu_set_features_device")

    def ingest(self, paths, threads=0):
        """Feature files -> HBM through the many-files reader (hmmh_ingest); returns (off, D, IngestStats)."""
        U = len(paths)
        arr = (C.c_char_p * U)(*[os.fsencode(p) for p in paths])
        off = np.zeros(U + 1, dtype=np.int64)
        D, bad, st = C.c_int(), C.c_int(-1), IngestStats()
        rc = self.lib.hmmh_ingest(self.h, arr, U, threads, off.ctypes.data_as(_lp), C.byref(D), C.byref(bad), C.byref(st))
        if rc == 5:
            raise HmmCudaError("hmmh_ingest: cannot read %s" % (paths[bad.value] if bad.value >= 0 else "?"))
        self._ck(rc, "hmmh_ingest")
        self.U, self.D, self.F, self.off = U, D.value, int(off[-1]), off
        return off, D.value, st

    def features_stream(self, off, D, chunks):
        """hmmcu_features_begin / append / end over (first_frame, ndarray) pairs -- the streaming form of set_features."""
        off = np.ascontiguousarray(off, dtype=np.int64)
        self.U, self.D, self.F, self.off = len(off) - 1, D, int(off[-1]), off
        self._ck(self.lib.hmmcu_features_begin(self.h, off.ctypes.data_as(_lp), self.U, D), "hmmcu_features_begin")
        keep = []
        for f0, xc in chunks:
            xc = _f64(xc)
            keep.append(xc)  # pageable sources are staged by the runtime before the call returns; kept anyway
            t = C.c_int()
            self._ck(self.lib.hmmcu_features_append(self.h, xc.ctypes.data, int(f0), xc.shape[0], C.byref(t)), "hmmcu_features_append")
            self._ck(self.lib.hmmcu_features_wait(self.h, t.value), "hmmcu_features_wait")
        self._ck(self.lib.hmmcu_features_end(self.h), "hmmcu_features_end")

    def link_streams(self, others):
        """Make this context the primary of a multi-stream model; `others` = the contexts of the further streams."""
        arr = (C.c_void_p * max(1, len(others)))(*[c.h for c in others])
        self._ck(self.lib.hmmcu_link_streams(self.h, arr, len(others)), "hmmcu_link_streams")
        self._linked = list(others)

    def set_models(self, ms):
        self.V, self.N, self.M = ms.V, ms.N, ms.M
        self._ck(self.lib.hmmcu_set_models(self.h, ms.V, ms.N, ms.M, ms.D, _d(ms.A), _d(ms.c), _d(ms.mu), _d(ms.iv), _d(ms.det)),
                 "hmmcu_set_models")

    def init_models(self, utt2model, V, N, M):
        """hmmcu_init_models: the reference's initial-model builder for V words on the device -> ModelSet."""
        u2m = np.ascontiguousarray(utt2model, dtype=np.int32)
        self._ck(self.lib.hmmcu_init_models(self.h, u2m.ctypes.data_as(_ip), int(V), int(N), int(M)), "hmmcu_init_models")
        self.V, self.N, self.M = int(V), int(N), int(M)
        return self.get_models(self.D)

    # ---- compute ----
    def emissions(self, u, v):
        T = int(self.off[u + 1] - self.off[u])
        logb = np.zeros((T, self.N))
        post = np.zeros((T, self.N, self.M))
        self._ck(self.lib.hmmcu_emissions(self.h, u, v, _d(logb), _d(post)), "hmmcu_emissions")
        return logb, post

    def forward_scores(self, emulate_underflow=False):
        out = np.zeros((self.U, self.V))
        self._ck(self.lib.hmmcu_forward_scores(self.h, _d(out), int(emulate_underflow)), "hmmcu_forward_scores")
        return out

    def viterbi_scores(self):
        out = np.zeros((self.U, self.V))
        self._ck(self.lib.hmmcu_viterbi_scores(self.h, _d(out)), "hmmcu_viterbi_scores")
        return out

    def rank(self, logp, weight=1.0):
        logp = _f64(logp)
        U, V = logp.shape
        label = np.zeros(U, dtype=np.int32)
        second = np.zeros(U, dtype=np.int32)
        self._ck(self.lib.hmmcu_rank(self.h, _d(logp), U, V, float(weight), label.ctypes.data_as(_ip), second.ctypes.data_as(_ip)),
                 "hmmcu_rank")
        return label, second

    def estep(self, utt2model, download=True, want_logp=True):
        u2m = np.ascontiguousarray(utt2model, dtype=np.int32)
        ss = stats_size(self.N, self.M, self.D)
        stats = np.zeros((self.V, ss)) if download else None
        lpu = np.zeros(self.U) if want_logp else None
        self._ck(self.lib.hmmcu_estep(self.h, u2m.ctypes.data_as(_ip), _d(stats) if download else None,
                                      _d(lpu) if want_logp else None), "hmmcu_estep")
        return stats, lpu

    def estep_viterbi(self, utt2model, download=True, want_logp=True, want_path=False):
        """hmmcu_estep_viterbi: the E-step of Viterbi training -> (stats, Viterbi score per utterance, path[F] or None)."""
        u2m = np.ascontiguousarray(utt2model, dtype=np.int32)
        ss = stats_size(self.N, self.M, self.D)
        stats = np.zeros((self.V, ss)) if download else None
        lpu = np.zeros(self.U) if want_logp else None
        path = np.zeros(self.F, dtype=np.int32) if want_path else None
        self._ck(self.lib.hmmcu_estep_viterbi(self.h, u2m.ctypes.data_as(_ip), _d(stats) if download else None,
                                              _d(lpu) if want_logp else None,
                                              path.ctypes.data_as(_ip) if want_path else None), "hmmcu_estep_viterbi")
        return stats, lpu, path

    def estep_mmi(self, label, kappa, max_hyp, download=True):
        """hmmcu_estep_mmi: the MMI E-step -> stats[2][V][stats_size] (numerator, denominator) or None."""
        lab = np.ascontiguousarray(label, dtype=np.int32)
        stats = np.zeros((2, self.V, stats_size(self.N, self.M, self.D))) if download else None
        self._ck(self.lib.hmmcu_estep_mmi(self.h, lab.ctypes.data_as(_ip), float(kappa), int(max_hyp), _d(stats) if download else None),
                 "hmmcu_estep_mmi")
        return stats

    def stats_device(self):
        n = C.c_int64(0)
        p = self.lib.hmmcu_stats_device(self.h, C.byref(n))
        return p, n.value

    def stats_download(self):
        """[V][stats_size], or [2][V][stats_size] after estep_mmi."""
        ss = stats_size(self.N, self.M, self.D)
        stats = np.zeros((self.V, ss)) if self.stats_device()[1] <= self.V * ss else np.zeros((2, self.V, ss))
        self._ck(self.lib.hmmcu_stats_download(self.h, _d(stats)), "hmmcu_stats_download")
        return stats

    def em_reset(self):
        self._ck(self.lib.hmmcu_em_reset(self.h), "hmmcu_em_reset")

    def mstep(self, threshold=1e-3):
        """Device M-step + stopping rule on the model set held by the context -> (sum_logp, n_utt, updated)."""
        lp, nu = np.zeros(self.V), np.zeros(self.V)
        upd = np.zeros(self.V, dtype=np.int32)
        self._ck(self.lib.hmmcu_mstep(self.h, float(threshold), _d(lp), _d(nu), upd.ctypes.data_as(_ip)), "hmmcu_mstep")
        return lp, nu, upd

    def mstep_ebw(self, E=2.0, tau=100.0):
        """hmmcu_mstep_ebw: the extended Baum-Welch update of the means and variances on the device, after estep_mmi."""
        self._ck(self.lib.hmmcu_mstep_ebw(self.h, float(E), float(tau)), "hmmcu_mstep_ebw")

    def get_models(self, D):
        ms = ModelSet(np.zeros((self.V, self.N, self.N)), np.zeros((self.V, self.N, self.M)), np.zeros((self.V, self.N, self.M, D)),
                      np.zeros((self.V, self.N, self.M, D)), np.zeros((self.V, self.N, self.M)))
        self._ck(self.lib.hmmcu_get_models(self.h, _d(ms.A), _d(ms.c), _d(ms.mu), _d(ms.iv), _d(ms.det)), "hmmcu_get_models")
        return ms

    def viterbi(self, utt2model):
        u2m = np.ascontiguousarray(utt2model, dtype=np.int32)
        score = np.zeros(self.U)
        path = np.zeros(self.F, dtype=np.int32)
        self._ck(self.lib.hmmcu_viterbi(self.h, u2m.ctypes.data_as(_ip), _d(score), path.ctypes.data_as(_ip)), "hmmcu_viterbi")
        return score, path

    def train(self, ms, utt2model, max_iter=0, allreduce=None):
        """hmmh_train: the reference's EM loop for all V words at once (in place on `ms`).
        allreduce(dev_ptr, n_doubles, stream_ptr) -> None sums the device buffer across ranks."""
        return self._train(self.lib.hmmh_train, "hmmh_train", ms, utt2model, max_iter, allreduce)

    def train_viterbi(self, ms, utt2model, max_iter=0, allreduce=None):
        """hmmh_train_viterbi: the same loop with the Viterbi E-step (estep_viterbi), in place on `ms`."""
        return self._train(self.lib.hmmh_train_viterbi, "hmmh_train_viterbi", ms, utt2model, max_iter, allreduce)

    def train_mmi(self, ms, label, kappa, max_hyp, E=2.0, tau=100.0, iterations=4, allreduce=None):
        """hmmh_train_mmi: `iterations` MMI iterations (estep_mmi, the all-reduce, mstep_ebw) in place on `ms`
        -> objective[iterations] (-log P(label | O) per utterance of the models entering each iteration)."""
        lab = np.ascontiguousarray(label, dtype=np.int32)
        cm = ms._cmodels()
        obj = np.zeros(max(int(iterations), 1))
        cb = _allreduce_hook(allreduce)
        self.V, self.N, self.M = ms.V, ms.N, ms.M
        self._ck(self.lib.hmmh_train_mmi(self.h, cm, ms.V, lab.ctypes.data_as(_ip), len(lab), float(kappa), int(max_hyp), float(E),
                                         float(tau), int(iterations), _d(obj), C.cast(cb, C.c_void_p) if cb else None, None),
                 "hmmh_train_mmi")
        return obj[:int(iterations)]

    def _train(self, fn, what, ms, utt2model, max_iter, allreduce):
        u2m = np.ascontiguousarray(utt2model, dtype=np.int32)
        cm = ms._cmodels()
        mean = np.zeros(ms.V)
        its = np.zeros(ms.V, dtype=np.int32)
        cb = _allreduce_hook(allreduce)
        self.V, self.N, self.M = ms.V, ms.N, ms.M
        self._ck(fn(self.h, cm, ms.V, u2m.ctypes.data_as(_ip), len(u2m), _d(mean), its.ctypes.data_as(C.POINTER(C.c_int)),
                    int(max_iter), C.cast(cb, C.c_void_p) if cb else None, None), what)
        return its, mean

    # ---- statistics summed over the ranks through peer memory (NVLink), no library collective ----
    def peer_export(self, world):
        """-> the 64-byte CUDA IPC handle of this rank's receive area (exchange it with all ranks, then peer_import)."""
        h = C.create_string_buffer(64)
        self._ck(self.lib.hmmcu_peer_export(self.h, int(world), h), "hmmcu_peer_export")
        return h.raw

    def peer_import(self, rank, world, handles):
        buf = b"".join(handles)
        assert len(buf) == 64 * world
        self._ck(self.lib.hmmcu_peer_import(self.h, int(rank), int(world), buf), "hmmcu_peer_import")

    def peer_area(self):
        return self.lib.hmmcu_peer_area(self.h)

    def peer_import_pointers(self, rank, world, areas):
        arr = (C.c_void_p * world)(*[C.c_void_p(a) for a in areas])
        self._ck(self.lib.hmmcu_peer_import_pointers(self.h, int(rank), int(world), arr), "hmmcu_peer_import_pointers")

    def peer_allreduce(self):
        self._ck(self.lib.hmmcu_peer_allreduce(self.h), "hmmcu_peer_allreduce")

    def peer_error(self):
        return bool(self.lib.hmmcu_peer_error(self.h))

    def set_option(self, key, value):
        self._ck(self.lib.hmmcu_set_option(self.h, key.encode(), int(value)), "hmmcu_set_option")

    # ---- instrumentation ----
    def stream(self):
        return self.lib.hmmcu_stream(self.h)

    def synchronize(self):
        self._ck(self.lib.hmmcu_synchronize(self.h), "hmmcu_synchronize")

    def launch_count(self):
        return int(self.lib.hmmcu_launch_count(self.h))

    def kernel_ms(self, name):
        return float(self.lib.hmmcu_last_kernel_ms(self.h, name.encode()))


# ---------------------------------------------------------------- host-side helpers (no GPU) ----
def mstep(ms, stats):
    """hmmh_mstep on every model of the set, in place.  stats[V][stats_size]."""
    lib = load()
    stats = _f64(stats)
    cm = ms._cmodels()
    for v in range(ms.V):
        rc = lib.hmmh_mstep(C.byref(cm[v]), _d(stats[v]))
        if rc:
            raise HmmCudaError("hmmh_mstep failed (%d)" % rc)
    return ms


def mstep_ebw(ms, num, den, E=2.0, tau=100.0):
    """hmmh_mstep_ebw on every model of the set, in place: num, den = blocks 0 and 1 ([V][stats_size]) of estep_mmi."""
    lib = load()
    num, den = _f64(num), _f64(den)
    cm = ms._cmodels()
    for v in range(ms.V):
        rc = lib.hmmh_mstep_ebw(C.byref(cm[v]), _d(num[v]), _d(den[v]), float(E), float(tau))
        if rc:
            raise HmmCudaError("hmmh_mstep_ebw failed (%d)" % rc)
    return ms


def init_model(N, M, x, off, word="w"):
    """hmmh_init_model (creating_initial_model, T-FS:732) -> ModelSet with V = 1."""
    lib = load()
    x = _f64(x)
    off = np.ascontiguousarray(off, dtype=np.int64)
    D = x.shape[1]
    ms = ModelSet(np.zeros((1, N, N)), np.zeros((1, N, M)), np.zeros((1, N, M, D)), np.zeros((1, N, M, D)), np.zeros((1, N, M)), [word])
    cm = ms._cmodels()
    rc = lib.hmmh_init_model(C.byref(cm[0]), _d(x), off.ctypes.data_as(_lp), len(off) - 1)
    if rc:
        raise HmmCudaError("hmmh_init_model failed (%d)" % rc)
    return ms


def read_model(path, len_bytes=0):
    lib = load()
    m = _CModel()
    rc = lib.hmmh_read_model(path.encode(), C.byref(m), len_bytes)
    if rc:
        raise HmmCudaError("hmmh_read_model(%s) failed (%d)" % (path, rc))
    N, M, D = m.N, m.M, m.D
    g = N * M
    ms = ModelSet(np.ctypeslib.as_array(m.A, (1, N, N)).copy(), np.ctypeslib.as_array(m.c, (1, N, M)).copy(),
                  np.ctypeslib.as_array(m.mu, (1, N, M, D)).copy(), np.ctypeslib.as_array(m.inv_var, (1, N, M, D)).copy(),
                  np.ctypeslib.as_array(m.det, (1, N, M)).copy(), [m.word.decode()])
    lib.hmmh_model_free(C.byref(m))
    return ms


def write_model(path, ms, v=0):
    lib = load()
    cm = ms._cmodels()
    rc = lib.hmmh_write_model(path.encode(), C.byref(cm[v]))
    if rc:
        raise HmmCudaError("hmmh_write_model(%s) failed (%d)" % (path, rc))


def read_model_streams(path, len_bytes=0, max_streams=6):
    """A .hmm file with P >= 1 feature streams -> [ModelSet (V = 1) per stream] (hmmh_read_model_streams)."""
    lib = load()
    lib.hmmh_read_model_streams.argtypes = [C.c_char_p, C.POINTER(_CModel), C.c_int, C.POINTER(C.c_int), C.c_int]
    arr = (_CModel * max_streams)()
    P = C.c_int()
    rc = lib.hmmh_read_model_streams(os.fsencode(path), arr, max_streams, C.byref(P), len_bytes)
    if rc:
        raise HmmCudaError("hmmh_read_model_streams(%s) failed (%d)" % (path, rc))
    out = []
    for p in range(P.value):
        m = arr[p]
        N, M, D = m.N, m.M, m.D
        out.append(ModelSet(np.ctypeslib.as_array(m.A, (1, N, N)).copy(), np.ctypeslib.as_array(m.c, (1, N, M)).copy(),
                            np.ctypeslib.as_array(m.mu, (1, N, M, D)).copy(), np.ctypeslib.as_array(m.inv_var, (1, N, M, D)).copy(),
                            np.ctypeslib.as_array(m.det, (1, N, M)).copy(), [m.word.decode()]))
        lib.hmmh_model_free(C.byref(arr[p]))
    return out


def write_model_streams(path, streams, v=0):
    """[ModelSet per stream] (word v of each) -> one .hmm file with len(streams) feature streams."""
    lib = load()
    lib.hmmh_write_model_streams.argtypes = [C.c_char_p, C.POINTER(_CModel), C.c_int]
    arr = (_CModel * len(streams))()
    keep = [ms._cmodels() for ms in streams]
    for p, cm in enumerate(keep):
        C.memmove(C.byref(arr[p]), C.byref(cm[v]), C.sizeof(_CModel))
    rc = lib.hmmh_write_model_streams(os.fsencode(path), arr, len(streams))
    if rc:
        raise HmmCudaError("hmmh_write_model_streams(%s) failed (%d)" % (path, rc))


def read_model_set(paths, threads=0):
    """V .hmm files of one topology -> ModelSet through the bulk reader (hmmh_read_model_set)."""
    lib = load()
    V = len(paths)
    arr = (C.c_char_p * V)(*[os.fsencode(p) for p in paths])
    cs, bad = _CModelSet(), C.c_int(-1)
    rc = lib.hmmh_read_model_set(arr, V, threads, C.byref(cs), C.byref(bad))
    if rc:
        raise HmmCudaError("hmmh_read_model_set failed (%d) at file %d" % (rc, bad.value))
    N, M, D = cs.N, cs.M, cs.D
    ms = ModelSet(np.ctypeslib.as_array(cs.A, (V, N, N)).copy(), np.ctypeslib.as_array(cs.c, (V, N, M)).copy(),
                  np.ctypeslib.as_array(cs.mu, (V, N, M, D)).copy(), np.ctypeslib.as_array(cs.inv_var, (V, N, M, D)).copy(),
                  np.ctypeslib.as_array(cs.det, (V, N, M)).copy(), [cs.word[v].value.decode() for v in range(V)])
    lib.hmmh_model_set_free(C.byref(cs))
    return ms


def write_model_set(paths, ms, threads=0):
    """ModelSet -> one .hmm file per word (hmmh_write_model_set), the bytes hmmh_write_model produces."""
    lib = load()
    assert len(paths) == ms.V
    arr = (C.c_char_p * ms.V)(*[os.fsencode(p) for p in paths])
    words = ((C.c_char * 64) * ms.V)()
    for v in range(ms.V):
        words[v].value = ms.words[v].encode()[:63]
    cs = _CModelSet(ms.V, ms.N, ms.M, ms.D, C.cast(words, C.POINTER(C.c_char * 64)), _d(ms.A), _d(ms.c), _d(ms.mu), _d(ms.iv), _d(ms.det))
    bad = C.c_int(-1)
    rc = lib.hmmh_write_model_set(arr, C.byref(cs), threads, C.byref(bad))
    if rc:
        raise HmmCudaError("hmmh_write_model_set failed (%d) at file %d" % (rc, bad.value))


def read_features(path):
    lib = load()
    p = _dp()
    T = C.c_int()
    D = C.c_int()
    rc = lib.hmmh_read_features(path.encode(), C.byref(p), C.byref(T), C.byref(D))
    if rc:
        raise HmmCudaError("hmmh_read_features(%s) failed (%d)" % (path, rc))
    x = np.ctypeslib.as_array(p, (T.value, D.value)).copy() if T.value > 0 else np.zeros((0, D.value))
    _libc_free(p)
    return x


def scan_features(paths, threads=0):
    """Frame offsets and D of a list of feature files from their sizes (hmmh_scan_features)."""
    lib = load()
    U = len(paths)
    arr = (C.c_char_p * U)(*[os.fsencode(p) for p in paths])
    off = np.zeros(U + 1, dtype=np.int64)
    D, bad = C.c_int(), C.c_int(-1)
    rc = lib.hmmh_scan_features(arr, U, threads, C.byref(D), off.ctypes.data_as(_lp), C.byref(bad))
    if rc:
        raise HmmCudaError("hmmh_scan_features failed (%d) at file %d" % (rc, bad.value))
    return off, D.value


def ingest_to_memory(paths, threads=0, stage_frames=0):
    """The ingest pipeline of hmmh_ingest into a numpy array instead of the device (host logic tests):
    returns (x[F][D], off, IngestStats)."""
    lib = load()
    U = len(paths)
    arr = (C.c_char_p * U)(*[os.fsencode(p) for p in paths])
    off = np.zeros(U + 1, dtype=np.int64)
    box = {"x": None, "log": []}

    def begin(user, foff, u, d):
        box["x"] = np.full((int(foff[u]), d), np.nan)
        return 0

    def append(user, xp, f0, n, ticket):
        d = box["x"].shape[1]
        box["x"][f0:f0 + n] = np.ctypeslib.as_array(xp, (n, d))
        box["log"].append((int(f0), int(n)))
        ticket[0] = len(box["log"]) % 16
        return 0

    sink = _CSink(None, _SinkBegin(begin), _SinkAppend(append), _SinkWait(lambda user, t: 0), _SinkEnd(lambda user: 0), None)
    D, bad, st = C.c_int(), C.c_int(-1), IngestStats()
    rc = lib.hmmh_ingest_to(C.byref(sink), arr, U, threads, stage_frames, off.ctypes.data_as(_lp), C.byref(D), C.byref(bad), C.byref(st))
    if rc:
        raise HmmCudaError("hmmh_ingest_to failed (%d) at file %d" % (rc, bad.value))
    return box["x"], off, st, box["log"]


def write_features(path, x):
    lib = load()
    x = _f64(x)
    rc = lib.hmmh_write_features(path.encode(), _d(x), x.shape[0], x.shape[1])
    if rc:
        raise HmmCudaError("hmmh_write_features(%s) failed (%d)" % (path, rc))


class NcclAllReduce:
    """ncclAllReduce(sum, double) in place on the context's own stream, straight through the NCCL C API (the
    library torch ships): what INTEGRATION.md shows a C caller doing between hmmcu_estep and hmmcu_mstep.
    Going through torch.distributed instead puts the collective on torch's internal NCCL stream behind two
    event hand-offs, which costs more than the 0.5 MB all-reduce itself.  The unique id travels through the
    already initialised torch.distributed group."""

    class _Uid(C.Structure):
        _fields_ = [("internal", C.c_byte * 128)]

    def __init__(self, rank, world):
        import glob
        import torch
        import torch.distributed as dist
        cands = glob.glob(os.path.join(os.path.dirname(torch.__file__), "..", "nvidia", "nccl", "lib", "libnccl.so*"))
        self.lib = C.CDLL(cands[0] if cands else "libnccl.so.2")
        self.lib.ncclGetUniqueId.argtypes = [C.POINTER(self._Uid)]
        self.lib.ncclCommInitRank.argtypes = [C.POINTER(C.c_void_p), C.c_int, self._Uid, C.c_int]
        self.lib.ncclAllReduce.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        self.lib.ncclCommDestroy.argtypes = [C.c_void_p]
        uid = self._Uid()
        if rank == 0 and self.lib.ncclGetUniqueId(C.byref(uid)) != 0:
            raise HmmCudaError("ncclGetUniqueId failed")
        box = [bytes(uid.internal)]
        dist.broadcast_object_list(box, src=0)
        C.memmove(C.byref(uid), box[0], 128)
        self.comm = C.c_void_p()
        rc = self.lib.ncclCommInitRank(C.byref(self.comm), int(world), uid, int(rank))
        if rc != 0:
            raise HmmCudaError("ncclCommInitRank failed (%d)" % rc)

    def __call__(self, dev_ptr, n_doubles, stream_ptr):
        rc = self.lib.ncclAllReduce(C.c_void_p(dev_ptr), C.c_void_p(dev_ptr), int(n_doubles), 8, 0, self.comm, C.c_void_p(stream_ptr))  # ncclDouble, ncclSum
        if rc != 0:
            raise HmmCudaError("ncclAllReduce failed (%d)" % rc)

    def close(self):
        if getattr(self, "comm", None):
            self.lib.ncclCommDestroy(self.comm)
            self.comm = None


def shard_utterances(off, rank, world):
    """Utterances [u0, u1) of rank `rank` out of `world`: contiguous, balanced by frame count (SURVEY 8e: the
    utterances are partitioned across the GPUs by contiguous frame count; every rank keeps the full model set and
    the sufficient statistics are summed with one all-reduce per EM iteration)."""
    off = np.asarray(off, dtype=np.int64)
    U, F = len(off) - 1, int(off[-1])
    cuts = [int(np.searchsorted(off, (k * F + world - 1) // world, side="left")) for k in range(world + 1)]
    cuts[0], cuts[-1] = 0, U
    cuts = np.maximum.accumulate(np.minimum(cuts, U))
    return int(cuts[rank]), int(cuts[rank + 1])


def stack_models(sets):
    """Concatenates single-topology ModelSets along V."""
    return ModelSet(np.concatenate([s.A for s in sets]), np.concatenate([s.c for s in sets]), np.concatenate([s.mu for s in sets]),
                    np.concatenate([s.iv for s in sets]), np.concatenate([s.det for s in sets]), sum([s.words for s in sets], []))
