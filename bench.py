#!/usr/bin/env python
"""bench.py -- frames/s of one Baum-Welch EM iteration (and of decode) on B200, next to the
reference's own CPU implementation.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
  torchrun ... bench.py --gpus N ...        (one rank per GPU; utterances sharded, one all-reduce of the
                                             sufficient statistics per EM iteration)

A "step" is one EM iteration over the rank's utterances -- the loop body of the reference trainer's
main() (T-FS:238-358) through the C ABI: hmmcu_estep (emissions, forward-backward, accumulators),
the all-reduce of the statistics, hmmcu_mstep (device M-step + the stopping rule; its 3V+1 doubles
are read back every step).  The stopping threshold is set to -1 so that every word is re-estimated
in every step and the work per step stays the full workload.  `value` times it with the features
resident in HBM; `e2e` additionally re-uploads the double-precision features from pinned host
memory every step (hmmcu_set_features), i.e. what the drop-in trainer pays on its first iteration.

The headline workload is BASELINE.json configs[1] ("c2"): 5-state left-to-right HMMs, 16 mixtures/state,
39-dim frames, 10 words, 1,000 utterances of ~300 frames PER GPU (weak scaling).  The same JSON line carries,
under `configs`, the other configurations BASELINE.json names at their full size:
  c3  Baum-Welch over 100,000 utterances (30 M frames), STRONG scaling: the corpus is the same for every N and is
      cut into N contiguous shards; per-kernel times and the event-timed all-reduce are listed
  c4  forward and Viterbi scores of 100,000 utterances against a 1,000-word model set, utterances sharded over the N GPUs
  c5  3-state, 128-mixture models: 1,000 utterances against all 2,000 models
and, at N > 1, `multi_gpu_parity`: rank 0 recomputes every rank's E-step and compares the all-reduced statistics.
"""
import argparse
import json
import os
import sys
import tempfile
import threading
import time

import numpy as np

# NCCL prints its version banner on stdout at NCCL_DEBUG=VERSION (some images export that); stdout carries the one JSON line
if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
    os.environ["NCCL_DEBUG"] = "WARN"

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: V words, N states, M mixtures, U utterances per GPU, description
    "c2": dict(V=10, N=5, M=16, U=1000, desc="BASELINE configs[1]: N=5 M=16 D=39, 10 words, 1000 utterances (~300 frames) per GPU"),
    "c1": dict(V=10, N=5, M=3, U=220, desc="BASELINE configs[0]: N=5 M=3 D=39, 10 words, 22 utterances per word"),
    "c3": dict(V=10, N=5, M=16, U=12500, desc="BASELINE configs[2] shard: N=5 M=16 D=39, 10 words, 12,500 utterances (100k over 8 GPUs) per GPU"),
}
D = 39
K_AUG = 2 * D + 1  # [x, x^2, 1]
C3_UTTS, C4_UTTS, C4_WORDS, C5_UTTS, C5_MODELS = 100000, 100000, 1000, 1000, 2000
GEN_BLOCK = 12500  # utterances per device-generator block: the corpus is identical however it is sharded over 1/2/4/8 ranks


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return dict(hbm_gbs=j["hbm_gbs"], bf16_tflops=j["bf16_tflops"], bf16_sustained=j.get("bf16_tflops_sustained"), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_sustained=1400.0, source="fallback")


def traffic_table():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` captures."""
    for name in ("r2_traffic.json", "r1_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            return json.load(open(p)), name
    return {}, None


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU during the timed region (pynvml, 20 ms)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._halt = index, [], set(), None, threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown if hasattr(nv, "nvmlClocksEventReasonHwSlowdown") else 0x8,
                 "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.02)

    def stop(self):
        self._halt.set()
        if self.is_alive():
            self.join(timeout=1.0)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": float(self.max_mhz) if self.max_mhz else None, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def make_workload(w, rank, seed=1234):
    from speech_recognition_hmm_continuous_b200 import synth
    cen, s = synth.make_centres(w["V"], w["N"], w["M"], D, seed=seed)
    labels = (np.arange(w["U"]) % w["V"]).astype(np.int32)
    x, off = synth.make_utterances(cen, s, labels, seed=seed + 1000 * rank)
    # initial models: the generating centres perturbed, so that EM has real work to do
    rng = np.random.default_rng(seed + 7)
    mods = synth.make_models(cen + 0.3 * s * rng.standard_normal(cen.shape), s)
    return x, off, labels, mods


def workload_config(name, world):
    """The `config` object of the JSON line: a function of the workload and N only, so that both arms print the same."""
    w = WORKLOADS[name]
    frames = 0
    for r in range(world):  # the utterance lengths of every rank's shard (same generator as make_workload, lengths only)
        rng = np.random.default_rng(1234 + 1000 * r + 1)
        frames += int(rng.integers(250, 351, size=w["U"]).sum())
    return {"workload": name + ": " + w["desc"], "words": w["V"], "states": w["N"], "mixtures": w["M"], "dim": D,
            "utterances": w["U"] * world, "frames": frames, "n_gpus": world,
            "l2": "flushed between timed iterations (256 MiB write)"}


def gen_corpus_device(torch, dev, cen, s, labels_all, u0, u1, seed, block=None):
    """Utterances [u0, u1) of a synthetic corpus of len(labels_all) utterances, generated on the device (SURVEY 8d's
    generator: left-to-right walk with +-20 % jitter, T ~ U{250..350}, a random mixture centre + N(0, s^2) noise).
    The corpus does not depend on how it is sharded: lengths and state cuts come from one host generator over the
    whole corpus, mixtures and noise from a device generator seeded per block of GEN_BLOCK utterances (u0 and u1 must be
    multiples of GEN_BLOCK or the ends).  -> (x float64 [F][D] on the device, off int64 [u1-u0+1], labels int32)"""
    V, N, M, _ = cen.shape
    Uall = len(labels_all)
    GEN_BLOCK = block or globals()["GEN_BLOCK"]
    rng = np.random.default_rng(seed)
    T = rng.integers(250, 351, size=Uall)
    wj = 1.0 + 0.4 * (rng.random((Uall, N)) - 0.5)
    cuts = np.floor(np.cumsum(wj, axis=1) / wj.sum(axis=1, keepdims=True) * T[:, None]).astype(np.int64)
    cuts[:, -1] = T
    seg = np.diff(np.concatenate([np.zeros((Uall, 1), dtype=np.int64), cuts], axis=1), axis=1)
    assert u0 % GEN_BLOCK == 0 and (u1 % GEN_BLOCK == 0 or u1 == Uall)
    cen_d = torch.from_numpy(np.ascontiguousarray(cen)).to(dev)
    s_d = torch.from_numpy(np.ascontiguousarray(s)).to(dev)
    F = int(T[u0:u1].sum())
    x = torch.empty((F, cen.shape[3]), dtype=torch.float64, device=dev)
    f0 = 0
    for b0 in range(u0, u1, GEN_BLOCK):
        b1 = min(b0 + GEN_BLOCK, u1)
        Tb = T[b0:b1]
        Fb = int(Tb.sum())
        word = torch.from_numpy(np.repeat(labels_all[b0:b1].astype(np.int64), Tb)).to(dev)
        state = torch.from_numpy(np.repeat(np.tile(np.arange(N, dtype=np.int64), b1 - b0), seg[b0:b1].ravel())).to(dev)
        g = torch.Generator(device=dev)
        g.manual_seed(seed * 1000003 + b0 // GEN_BLOCK)
        mix = torch.randint(0, M, (Fb,), generator=g, device=dev)
        noise = torch.randn((Fb, cen.shape[3]), dtype=torch.float64, generator=g, device=dev)
        x[f0:f0 + Fb] = cen_d[word, state, mix] + s_d * noise
        f0 += Fb
        del word, state, mix, noise
    off = np.concatenate([[0], np.cumsum(T[u0:u1])]).astype(np.int64)
    return x, off, labels_all[u0:u1].astype(np.int32)


def rel_groups(a, b, N, M):
    """max over the statistics groups (num_trans, den_trans, den_mix, S0, S1, S2c, sum_logP) of max|a-b| / max|b|."""
    from speech_recognition_hmm_continuous_b200 import api
    worst = 0.0
    for v in range(a.shape[0]):
        sa, sb = api.split_stats(a[v], N, M, D), api.split_stats(b[v], N, M, D)
        for k in ("num_trans", "den_trans", "den_mix", "S0", "S1", "S2c", "sum_logp"):
            x, y = np.asarray(sa[k], dtype=np.float64), np.asarray(sb[k], dtype=np.float64)
            den = np.abs(y).max()
            if den > 0 and np.isfinite(den):
                worst = max(worst, float(np.abs(x - y).max() / den))
    return worst


# ================================================================================ our arm ====
def run_ours(args):
    import torch
    import torch.distributed as dist
    from speech_recognition_hmm_continuous_b200 import api, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = None
    if not args.no_affinity:
        # keep this rank (and therefore the first touch of its host buffers, pinned staging included) on the CPUs
        # of the NUMA node its GPU hangs off: with eight ranks uploading at once, remote-node pinned memory halves
        # the host-to-device rate
        try:
            import pynvml
            pynvml.nvmlInit()
            pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
            numa = sorted(os.sched_getaffinity(0))
            numa = "%d cpus [%d..%d]" % (len(numa), numa[0], numa[-1])
        except Exception as e:  # noqa: BLE001
            numa = "unavailable: %s" % e
    w = WORKLOADS[args.workload]
    x, off, labels, mods = make_workload(w, rank)
    F = int(off[-1])
    N, M, V, U = w["N"], w["M"], w["V"], w["U"]
    G = N * M
    pk = peaks()
    tf32_peak = tf32_peak_tflops(dev)

    ctx = api.Context(local, timing=False)
    if args.upload_chunks:
        ctx.set_option("upload_chunks", args.upload_chunks)
    for kv in args.set:  # library A/B switches (hmmcu_set_option), experiments only
        k, v = kv.split("=")
        ctx.set_option(k, int(v))
    ext = torch.cuda.ExternalStream(ctx.stream(), device=local)
    ms = api.ModelSet.from_dict(mods)

    class _Alias:  # device statistics buffer as a torch tensor (no copy) for the NCCL all-reduce
        def __init__(self, ptr, n):
            self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 3}

    def allreduce_torch(dev_ptr, n, stream_ptr):
        t = torch.as_tensor(_Alias(dev_ptr, n), device=dev)
        with torch.cuda.stream(torch.cuda.ExternalStream(stream_ptr, device=local)):
            dist.all_reduce(t)

    ar = allreduce_torch if world > 1 else None
    ar_kind = ["torch.distributed (nccl)"]
    if world > 1 and not args.torch_allreduce:
        try:  # the collective on the context's own stream through the NCCL C API
            ar = api.NcclAllReduce(rank, world)
            ar_kind[0] = "ncclAllReduce on the context's stream"
        except Exception as e:  # noqa: BLE001
            print("direct NCCL unavailable (%s); using torch.distributed" % e, file=sys.stderr)

    def setup_allreduce(c):
        """The sum of the statistics over the ranks for context c (after its set_models): the library's own kernel pair over
        peer memory (NVLink, CUDA IPC handles exchanged through the process group) unless --nccl-allreduce; else NCCL."""
        c._ar = None
        if world == 1:
            return
        c._ar = ar
        if args.nccl_allreduce or args.torch_allreduce:
            return
        ok = 1
        try:
            hs = [None] * world
            dist.all_gather_object(hs, c.peer_export(world))
            c.peer_import(rank, world, hs)
        except Exception as e:  # noqa: BLE001
            print("peer all-reduce unavailable on rank %d (%s); using NCCL" % (rank, e), file=sys.stderr)
            ok = 0
        t = torch.tensor([ok], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)   # all ranks or none
        if int(t.item()) == 1:
            c._ar = lambda p, n, s: c.peer_allreduce()
            ar_kind[0] = "hmmcu_peer_allreduce: one kernel over NVLink peer memory, tagged 8-byte words, no fence and no flags (no library collective)"
    # pinned host copy of the features (e2e leg) and a device-resident copy (value leg)
    xpin = torch.from_numpy(x).pin_memory()
    xdev = xpin.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()

    def make_iteration(c, lab, ar_events=None):
        st = torch.cuda.ExternalStream(c.stream(), device=local)

        def em_iteration():
            c.estep(lab, download=False, want_logp=False)
            if c._ar is not None:
                p, n = c.stats_device()
                if ar_events is not None:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(st)
                    c._ar(p, n, c.stream())
                    e1.record(st)
                    ar_events.append((e0, e1))
                else:
                    c._ar(p, n, c.stream())
            return c.mstep(threshold=-1.0)  # reads sum_logp / n_utt / updated back: the step's result
        return em_iteration

    def timed(c, fn, steps, warmup, kernel_names=(), last=None):
        st = torch.cuda.ExternalStream(c.stream(), device=local)
        for _ in range(warmup):
            fn()
        c.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        l0 = c.launch_count()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        align = torch.zeros(1, device=dev)
        kms = {k: [] for k in kernel_names}
        wall0 = time.perf_counter()
        for i in range(steps):
            flush.fill_(i & 0xFF)  # L2 flush between timed iterations (256 MiB > 126 MB L2), outside the event pair
            torch.cuda.synchronize()
            if world > 1:
                # The flush and the host-side synchronisation above end at a different moment on every rank; without a common
                # start the first rank's step would be charged the wait for the last rank's FLUSH in the step's all-reduce.  A
                # one-element collective on the step's stream releases all ranks together; the start event follows it.
                with torch.cuda.stream(st):
                    dist.all_reduce(align)
            ev[i][0].record(st)
            out = fn()
            ev[i][1].record(st)
            c.synchronize()
            for k in kernel_names:
                kms[k].append(c.kernel_ms(k))
        torch.cuda.synchronize()
        wall = time.perf_counter() - wall0
        if last is not None:  # what the last timed step returned
            last.append(out)
        if world > 1:
            dist.barrier()
        total_ms = sum(a.elapsed_time(b) for a, b in ev)
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), c.launch_count() - l0, {k: float(np.mean(v)) for k, v in kms.items()}, wall

    def kernel_pass(c, lab, steps):
        """Per-kernel device times: a second, shorter pass with the library's event timers on (they record events
        between the kernels, which turns the CUDA-graph replay of the iteration off -- so not the pass `value` uses),
        and the all-reduce between two events on the same stream."""
        are = []
        c.enable_timing(True)
        _, _, kms, _ = timed(c, make_iteration(c, lab, are), steps, 3, ("emis", "fwdbwd", "accum", "mstep"))
        c.enable_timing(False)
        c.synchronize()
        ar_ms = float(np.mean([a.elapsed_time(b) for a, b in are[3:]])) if len(are) > 3 else None
        if ar_ms is not None:
            t = torch.tensor([ar_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ar_ms = float(t.item())
        return kms, ar_ms

    ctx.set_features_device(xdev.data_ptr(), off, D)
    ctx.set_models(ms)
    ctx.em_reset()
    setup_allreduce(ctx)
    step_resident = make_iteration(ctx, labels)

    def step_e2e():
        ctx.set_features_ptr(xpin.data_ptr(), off, D)
        step_resident()

    sampler = ClockSampler(local)
    sampler.start()
    last_step = []
    tot_ms, launches, _, wall = timed(ctx, step_resident, args.steps, args.warmup, last=last_step)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:   # before the passes below re-estimate the models further
        dump_outputs(args.dump_outputs, last_step[0], ctx.get_models(D))
    kms, ar_ms = kernel_pass(ctx, labels, max(3, min(args.steps, 20)))
    ar_alone_ms = None
    if world > 1 and ctx._ar is not None:
        # the collective by itself: all ranks released together (one-element collective), nothing in front of it -- what is left
        # of allreduce_ms above this is the wait for the slowest rank's E-step
        st_ = torch.cuda.ExternalStream(ctx.stream(), device=local)
        al_ = torch.zeros(1, device=dev)
        evs = []
        p_, n_ = ctx.stats_device()
        for _ in range(13):
            torch.cuda.synchronize()
            with torch.cuda.stream(st_):
                dist.all_reduce(al_)
                torch.cuda._sleep(200000)  # ~0.1 ms of device time: the host gets ahead, so its launch latency is not in the interval
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st_)
            ctx._ar(p_, n_, ctx.stream())
            e1.record(st_)
            evs.append((e0, e1))
        torch.cuda.synchronize()
        t_ = torch.tensor([float(np.mean([a_.elapsed_time(b_) for a_, b_ in evs[3:]]))], dtype=torch.float64, device=dev)
        dist.all_reduce(t_, op=dist.ReduceOp.MAX)
        ar_alone_ms = float(t_.item())
    e2e_steps = max(3, min(args.steps, 50))
    e2e_ms, _, _, _ = timed(ctx, step_e2e, e2e_steps, max(3, min(args.warmup, 5)))

    # ---- multi-GPU parity: the all-reduced statistics against the double-precision sum of every rank's E-step, recomputed
    # on rank 0 (same kernels, same shards), and against ONE E-step over the union of all shards ----
    parity = None
    if world > 1:
        ctx.set_features_device(xdev.data_ptr(), off, D)
        ctx.set_models(ms)
        ctx.estep(labels, download=False, want_logp=False)
        p, n = ctx.stats_device()
        ctx._ar(p, n, ctx.stream())
        ctx.synchronize()
        reduced = ctx.stats_download()
        if rank == 0:
            total, xs, offs, labs = None, [], [], []
            c2 = api.Context(local)
            for r in range(world):
                xr, offr, labr, _ = make_workload(w, r)
                c2.set_features(xr, offr)
                c2.set_models(ms)
                str_, _ = c2.estep(labr)
                total = str_.copy() if total is None else total + str_
                xs.append(xr); offs.append(offr); labs.append(labr)
            offu = np.concatenate([[0]] + [o[1:] + sum(int(q[-1]) for q in offs[:k]) for k, o in enumerate(offs)]).astype(np.int64)
            c2.set_features(np.concatenate(xs), offu)
            c2.set_models(ms)
            union, _ = c2.estep(np.concatenate(labs))
            c2.close()
            ss = api.stats_size(N, M, D)
            parity = {"max_rel_stats": rel_groups(reduced, total, N, M),
                      "max_rel_logp": float(np.abs(reduced[:, ss - 2] - total[:, ss - 2]).max() / np.abs(total[:, ss - 2]).max()),
                      "n_utt_equal": bool((reduced[:, ss - 1] == total[:, ss - 1]).all()),
                      "tolerance": 1e-9,
                      "what": "all-reduced statistics (fp64 payload) vs the fp64 sum of every rank's E-step recomputed on rank 0",
                      "max_rel_stats_vs_union_estep": rel_groups(reduced, union, N, M),
                      "union_tolerance": 1e-4,
                      "union_what": "the same statistics vs ONE E-step over the union of all shards (T-FS:244-321: accumulators zeroed once, every utterance added); "
                                    "differs by the single-precision partial sums inside the accumulate kernel, which follow the shard boundaries"}
            parity["ok"] = bool(parity["max_rel_stats"] <= 1e-9 and parity["max_rel_logp"] <= 1e-9 and parity["n_utt_equal"]
                                and parity["max_rel_stats_vs_union_estep"] <= 1e-4)
        flag = torch.tensor([1 if (parity is None or parity["ok"]) else 0], device=dev)
        dist.broadcast(flag, src=0)
        if int(flag.item()) == 0:
            if rank == 0:
                print("multi_gpu_parity FAILED: %s" % json.dumps(parity), file=sys.stderr)
            sys.exit(3)

    # ---- decode legs on the headline workload (forward scoring of every utterance against all V models + ranking; Viterbi) ----
    ctx.set_features_device(xdev.data_ptr(), off, D)
    ctx.set_models(ms)
    ctx.enable_timing(True)  # per-kernel timers for the decode legs (no graph replay involved there)
    dec = {}
    for name, fn in (("forward", lambda: ctx.rank(ctx.forward_scores())), ("viterbi", lambda: ctx.viterbi(labels))):
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 5
        ctx.synchronize()
        e0.record(ext)
        for _ in range(reps):
            fn()
        e1.record(ext)
        ctx.synchronize()
        ms_dec = e0.elapsed_time(e1) / reps
        t = torch.tensor([ms_dec], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        kn = ("emis", "score") if name == "forward" else ("logb64", "viterbi")
        dec[name] = {"frames_per_s": F * world / (float(t.item()) * 1e-3), "ms": float(t.item()),
                     "kernel_ms": {k: ctx.kernel_ms(k) for k in kn},
                     "frame_model_pairs_per_s": (F * V * world / (float(t.item()) * 1e-3)) if name == "forward" else None}
    ctx.enable_timing(False)

    # initial-model builder (creating_initial_model, T-FS:732-1317): all words on the device vs the host builder
    # (single-threaded C, one word after the other) -- what the drop-in trainer pays before its first EM iteration
    init = None
    if world == 1 and not args.no_init:
        ctx.set_features_device(xdev.data_ptr(), off, D)
        ctx.init_models(labels, V, N, M)
        ctx.synchronize()
        t0 = time.perf_counter()
        reps = 3
        for _ in range(reps):
            ctx.init_models(labels, V, N, M)
        dev_ms = (time.perf_counter() - t0) / reps * 1e3
        us0 = np.nonzero(labels == 0)[0]
        x0 = np.concatenate([x[off[u]:off[u + 1]] for u in us0])
        off0 = np.concatenate([[0], np.cumsum([off[u + 1] - off[u] for u in us0])]).astype(np.int64)
        t0 = time.perf_counter()
        api.init_model(N, M, x0, off0)
        host_ms_word = (time.perf_counter() - t0) * 1e3
        init = {"device_ms_all_words": dev_ms, "host_ms_one_word": host_ms_word, "host_ms_all_words_extrapolated": host_ms_word * V,
                "note": "wall clock incl. the read-back of the models; results are bit-identical (tests)"}
        ctx.set_models(ms)
    # ingest (SURVEY 8f-2): the workload's utterances as feature files -> HBM.  Serial = one read per file, concatenate,
    # hmmcu_set_features (what a straightforward host does; the reference itself issues one fread per FRAME and re-reads
    # every file twice per iteration).  Pipelined = hmmh_ingest: reader pool -> pinned staging -> async copies.
    ingest = None
    if world == 1 and not args.no_ingest:
        import shutil
        base = "/dev/shm" if os.path.isdir("/dev/shm") else None
        tmpd = tempfile.mkdtemp(prefix="hmmcu_ingest_", dir=base)
        try:
            paths = []
            for u in range(U):
                pth = os.path.join(tmpd, "u%06d.bin" % u)
                api.write_features(pth, x[off[u]:off[u + 1]])
                paths.append(pth)

            def serial():
                xs = [api.read_features(pth) for pth in paths]
                xo = np.concatenate(xs)
                oo = np.concatenate([[0], np.cumsum([len(a) for a in xs])]).astype(np.int64)
                ctx.set_features(xo, oo)
                ctx.synchronize()

            def piped():
                st = ctx.ingest(paths)[2]
                ctx.synchronize()
                return st
            serial(); piped()
            t0 = time.perf_counter(); serial(); ser_ms = (time.perf_counter() - t0) * 1e3
            best, st = None, None
            for _ in range(3):
                t0 = time.perf_counter(); st = piped(); dt = (time.perf_counter() - t0) * 1e3
                best = dt if best is None else min(best, dt)
            ingest = {"files": U, "bytes": int(x.nbytes), "where": base or "tmp", "serial_ms": ser_ms, "pipelined_ms": best,
                      "pipelined_gb_per_s": x.nbytes / (best * 1e-3) / 1e9, "threads": int(st.threads), "batches": int(st.batches),
                      "scan_ms": st.scan_s * 1e3, "stage_ms": st.stage_s * 1e3, "read_ms": st.read_s * 1e3,
                      "note": "files in the page cache / tmpfs; wall clock through the Python binding, best of 3"}
        finally:
            shutil.rmtree(tmpd, ignore_errors=True)

    ms_step = tot_ms / args.steps
    value = F * world / (ms_step * 1e-3)
    traffic, traffic_src = traffic_table()
    rooflines = training_rooflines(kms, F, N, M, V, pk, tf32_peak, traffic.get(args.workload, {}), acc_h=ctx.kernel_ms("acc_h_active") > 0)
    for leg, kn, per_pair in (("forward", "score", 4.0 * N), ("viterbi", "viterbi", None)):
        kt = dec[leg]["kernel_ms"].get(kn)
        if per_pair and kt and kt > 0:
            ach = per_pair * V * F / (kt * 1e-3) / 1e9
            rooflines["decode_" + kn] = {"kernel": "k_fwd_cells32", "bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s",
                                         "frac": ach / pk["hbm_gbs"], "ms": kt, "algorithmic_bytes": per_pair * V * F, "traffic": None}
    dom = max(kms, key=lambda k: kms[k])
    roofline = dict(rooflines[dom])
    roofline.update({"peak_source": pk["source"], "kernel_ms": kms, "traffic_source": traffic_src,
                     "all_kernels": "see `rooflines`: one entry per kernel of the step, each against its own bound"})
    cfg = workload_config(args.workload, world)
    out = {
        "metric": "frames/sec per Baum-Welch EM iteration", "value": value, "unit": "frames/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
        "details": {"frames_this_rank": F, "utterances_per_gpu": U, "cpu_affinity": numa,
                    "parallelism": ("utterances sharded, the statistics summed over the ranks once per iteration (%s)" % ar_kind[0]) if world > 1 else "single GPU"},
        "e2e": {"value": F * world / (e2e_ms / e2e_steps * 1e-3), "unit": "frames/s", "ms_per_step": e2e_ms / e2e_steps,
                "h2d_bytes_per_step": int(x.nbytes + off.nbytes),
                "d2h_bytes_per_step": int(8 * (3 * V + 1))},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "rooflines": rooflines, "allreduce_ms": ar_ms, "allreduce_alone_ms": ar_alone_ms,
        "multi_gpu_parity": parity, "decode": dec, "init_model": init, "ingest": ingest,
        "wall_s_timed_region": wall, "tf32_peak_tflops": tf32_peak,
        "tf32_peak_note": "library TF32 GEMM 8192^3 measured in this run (same protocol as MEASURED_PEAKS.json); 3xTF32 issues 3 MMAs per algorithmic MMA",
    }
    ctx.close()
    del xdev, xpin
    torch.cuda.empty_cache()
    if not args.no_configs:
        tools = dict(torch=torch, dist=dist, api=api, synth=synth, dev=dev, local=local, rank=rank, world=world, setup_allreduce=setup_allreduce, pk=pk,
                     tf32_peak=tf32_peak, make_iteration=make_iteration, timed=timed, kernel_pass=kernel_pass, traffic=traffic)
        out["configs"] = {"c3": run_c3(tools, args), "c4": run_c4(tools, args), "c5": run_c5(tools, args)}
    if rank == 0:
        if world == 1 and not args.no_cpu:
            out["cpu_baseline"] = cpu_baseline(w, budget_s=args.cpu_seconds)
        if world == 1 and not args.no_cli:
            out["c1_cli"] = c1_cli_wall_clock()
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, step_result, models):
    """What the last timed EM iteration hands its caller, one float64 array per DIR/<name>.npy: the M-step's per-word
    results (sum of the utterance log-likelihoods, utterance count, re-estimated flag) and the re-estimated model set.
    The workload is generated from fixed seeds, so two builds run with the same arguments can be compared file by file."""
    os.makedirs(out_dir, exist_ok=True)
    lp, nu, upd = step_result
    arrays = {"sum_logp": lp, "n_utt": nu, "updated": upd,
              "A": models.A, "c": models.c, "mu": models.mu, "inv_var": models.iv, "det": models.det}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def training_rooflines(kms, F, N, M, V, pk, tf32_peak, traffic, acc_h=False):
    """One entry per kernel of the EM iteration, each against the bound that really limits it (DESIGN.md section 5).
    F = frames of one launch on this rank."""
    from speech_recognition_hmm_continuous_b200 import api
    G = N * M
    out = {}

    def tensor(name, kernel, flops, ms, hbm_bytes, f16=False):
        if not ms or ms <= 0:
            return
        ach = flops / (ms * 1e-3) / 1e12
        peak = (pk.get("bf16_sustained") or pk.get("bf16_tflops")) if f16 else tf32_peak
        out[name] = {"kernel": kernel, "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                     "peak_what": "fp16 / bf16 dense, sustained (MEASURED_PEAKS.json)" if f16 else "TF32 dense, library GEMM measured in this run",
                     ("issued_3xf16" if f16 else "issued_3xtf32"): {"achieved": 3 * ach, "frac": 3 * ach / peak}, "ms": ms, "algorithmic_flops": flops,
                     "hbm_view": {"algorithmic_bytes": hbm_bytes, "gbs": hbm_bytes / (ms * 1e-3) / 1e9, "frac": hbm_bytes / (ms * 1e-3) / 1e9 / pk["hbm_gbs"]},
                     "traffic": traffic.get(name)}

    def hbm(name, kernel, nbytes, ms, extra=None):
        if not ms or ms <= 0:
            return
        ach = nbytes / (ms * 1e-3) / 1e9
        out[name] = {"kernel": kernel, "bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"], "ms": ms,
                     "algorithmic_bytes": nbytes, "traffic": traffic.get(name)}
        if extra:
            out[name].update(extra)

    # emissions: 2 K G flops per frame; moves x (4 D) in and logb (4 N) out
    tensor("emis", "k_emis_ws", 2.0 * K_AUG * G * F, kms.get("emis"), F * (4.0 * D + 4.0 * N))
    # forward-backward: SURVEY 8d counts 16 N + 4 bytes per frame (read b, write alpha; read b, read alpha; c_t); k_fb_res keeps
    # alpha / beta in shared memory and moves 8 N (logb in, gamma out)
    hbm("fwdbwd", "k_fb_res", F * (16.0 * N + 4.0), kms.get("fwdbwd"), {"bytes_the_kernel_moves": F * 8.0 * N})
    # accumulate: two chained contractions (posteriors recomputed, then S += w Xaug): 4 K G flops per frame
    # (k_accum_h: half-precision operands; it reads its frames as packed tiles, 2 x 2 x 3 DP bytes per frame, instead of 4 D)
    if acc_h:
        # HBM is the nearer ceiling (ncu at the C3 shard: DRAM 63 % of its peak, tensor pipe 64 % active): per frame the kernel reads its
        # tile (3 column blocks x DP x hi / lo halves = 12 DP = 480 bytes) and gamma, logb (8 N); SURVEY 8d counts 496 bytes per frame
        tensor("accum", "k_accum_h", 4.0 * K_AUG * G * F, kms.get("accum"), F * (12.0 * (K_AUG // 2 + 1) + 8.0 * N), f16=True)
        a = out.get("accum")
        if a:
            tv = {k: a[k] for k in ("achieved", "peak", "unit", "frac", "peak_what", "issued_3xf16", "algorithmic_flops")}
            hv = a["hbm_view"]
            out["accum"] = {"kernel": "k_accum_h", "bound": "hbm", "achieved": hv["gbs"], "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": hv["frac"],
                            "ms": a["ms"], "algorithmic_bytes": hv["algorithmic_bytes"], "survey_8d_bytes": F * 496.0, "traffic": a["traffic"],
                            "tensor_view": tv}
    else:
        tensor("accum", "k_accum_ws", 4.0 * K_AUG * G * F, kms.get("accum"), F * (4.0 * D + 8.0 * N))
    hbm("mstep", "k_mstep_ctl+k_mstep_apply+packers", 8.0 * V * api.stats_size(N, M, D), kms.get("mstep"),
        {"note": "a few hundred KB: launch / dependency latency, not bandwidth"})
    return out


def tf32_peak_tflops(device):
    """Dense TF32 throughput of this GPU by the protocol of MEASURED_PEAKS.json (library GEMM 8192^3,
    best of 10, CUDA events): the denominator of the tensor-pipe roofline.  Measurement only."""
    import torch
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        a = torch.randn(8192, 8192, device=device)
        b = torch.randn(8192, 8192, device=device)
        best = 1e9
        for _ in range(3):
            torch.matmul(a, b)
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return 2.0 * 8192 ** 3 / (best * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


# ============================================================= the other BASELINE configurations ====
def _shard(total, rank, world, block=None):
    """Contiguous shard of `total` utterances in whole generator blocks (the corpus is the same for every world size)."""
    GEN_BLOCK = block or globals()["GEN_BLOCK"]
    blocks = (total + GEN_BLOCK - 1) // GEN_BLOCK
    b0, b1 = blocks * rank // world, blocks * (rank + 1) // world
    return min(b0 * GEN_BLOCK, total), min(b1 * GEN_BLOCK, total)


def run_c3(t, args):
    """BASELINE configs[2]: Baum-Welch over 100,000 utterances (10 words, N=5, M=16), STRONG scaling over the ranks."""
    torch, dist, api, synth, dev, world, rank = t["torch"], t["dist"], t["api"], t["synth"], t["dev"], t["world"], t["rank"]
    V, N, M = 10, 5, 16
    U = args.c3_utts
    cen, s = synth.make_centres(V, N, M, D, seed=1234)
    labels_all = (np.arange(U) % V).astype(np.int32)
    u0, u1 = _shard(U, rank, world)
    x, off, lab = gen_corpus_device(torch, dev, cen, s, labels_all, u0, u1, seed=3003)
    rng = np.random.default_rng(1241)
    ms = api.ModelSet.from_dict(synth.make_models(cen + 0.3 * s * rng.standard_normal(cen.shape), s))
    F = int(off[-1])
    c = api.Context(t["local"])
    c.set_features_device(x.data_ptr(), off, D)
    c.set_models(ms)
    c.em_reset()
    t["setup_allreduce"](c)
    steps = max(3, min(args.steps, 10))
    tot_ms, launches, _, _ = t["timed"](c, t["make_iteration"](c, lab), steps, 3)
    kms, ar_ms = t["kernel_pass"](c, lab, 5)
    ft = torch.tensor([float(F)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ft)
    Ftot = float(ft.item())
    ms_step = tot_ms / steps
    out = {"workload": "BASELINE configs[2]: Baum-Welch EM over %d utterances (10 words, N=5, M=16, D=39), %d contiguous shards" % (U, world),
           "scaling": "strong", "utterances_total": U, "frames_total": int(Ftot), "frames_this_rank": F, "n_gpus": world,
           "ms_per_step": ms_step, "frames_per_s": Ftot / (ms_step * 1e-3), "steps": steps, "kernel_ms": kms, "allreduce_ms": ar_ms,
           "gpu_launches": int(launches),
           "rooflines": training_rooflines(kms, F, N, M, V, t["pk"], t["tf32_peak"], t["traffic"].get("c3", {}), acc_h=c.kernel_ms("acc_h_active") > 0),
           "l2": "flushed between timed iterations; the shard's features alone exceed the L2"}
    c.close()
    del x
    torch.cuda.empty_cache()
    return out


def _decode_emis_roofline(c, t, flops, em_ms, name):
    """Emission contraction of a decode leg against the tensor-pipe rate of its operand type: the library TF32 GEMM
    measured in this run for the 3xTF32 kernels, MEASURED_PEAKS.json's sustained bf16 / fp16 rate for the half-precision
    form of k_emis_dec (three kind::f16 MMAs per algorithmic one)."""
    dec = c.kernel_ms("dec_grid") > 0
    f16 = c.kernel_ms("dec_f16_active") > 0
    peak = (t["pk"]["bf16_sustained"] or t["pk"]["bf16_tflops"]) if f16 else t["tf32_peak"]
    ach = flops / (em_ms * 1e-3) / 1e12
    return {"kernel": ("k_emis_dec" if dec else "k_emis_ws<decode>") + ("<f16>" if f16 else ""), "bound": "tensor", "achieved": ach, "peak": peak,
            "peak_what": "fp16 / bf16 dense, sustained (MEASURED_PEAKS.json)" if f16 else "TF32 dense, library GEMM measured in this run",
            "unit": "TFLOP/s", "frac": ach / peak, ("issued_3xf16" if f16 else "issued_3xtf32"): {"achieved": 3 * ach, "frac": 3 * ach / peak},
            "algorithmic_flops": flops, "traffic": t["traffic"].get(name, {}).get("emis")}


def _decode_config(t, args, name, desc, V, N, M, U, seed):
    """Forward and Viterbi scores of the rank's shard of U utterances against all V models (R-FS:341-369)."""
    torch, dist, api, synth, dev, world, rank = t["torch"], t["dist"], t["api"], t["synth"], t["dev"], t["world"], t["rank"]
    cen, s = synth.make_centres(V, N, M, D, seed=seed)
    labels_all = (np.arange(U) % V).astype(np.int32)
    block = GEN_BLOCK if U >= 8 * GEN_BLOCK else max(1, U // 8)   # at least eight generator blocks: every rank of 8 gets a shard
    u0, u1 = _shard(U, rank, world, block)
    x, off, lab = gen_corpus_device(torch, dev, cen, s, labels_all, u0, u1, seed=seed + 1, block=block)
    F = int(off[-1])
    c = api.Context(t["local"], timing=True)
    c.set_features_device(x.data_ptr(), off, D)
    c.set_models(api.ModelSet.from_dict(synth.make_models(cen, s)))
    ft = torch.tensor([float(F)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ft)
    Ftot = float(ft.item())
    res = {"workload": desc, "utterances_total": U, "frames_total": int(Ftot), "frames_this_rank": F, "models": V, "n_gpus": world,
           "gaussians_per_frame": V * N * M, "scaling": "strong"}
    flops = 2.0 * K_AUG * V * N * M * F          # algorithmic; the 3xTF32 scheme issues three times as many
    top1 = None
    for leg, fn in (("forward", c.forward_scores), ("viterbi", c.viterbi_scores)):
        fn()
        em, sc, wl = [], [], []
        for _ in range(2):
            t0 = time.perf_counter()
            sco = fn()
            wl.append((time.perf_counter() - t0) * 1e3)
            em.append(c.kernel_ms("emis_total"))
            sc.append(c.kernel_ms("score_total" if leg == "forward" else "viterbi_total"))
        em_ms, sc_ms, wall_ms = float(np.median(em)), float(np.median(sc)), float(np.median(wl))
        mx = torch.tensor([em_ms + sc_ms, wall_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dev_ms, wall_max = float(mx[0].item()), float(mx[1].item())
        sbytes = 4.0 * N * V * F + (N * V * F if leg == "viterbi" else 0.0)   # SURVEY 8d: 4N (+N) bytes per (frame, model)
        res[leg] = {
            "emis_ms": em_ms, "score_ms": sc_ms, "device_ms_max_over_ranks": dev_ms, "api_wall_ms_max_over_ranks": wall_max,
            "frames_per_s": Ftot / (dev_ms * 1e-3), "frame_model_pairs_per_s": Ftot * V / (dev_ms * 1e-3),
            "frames_per_s_through_api": Ftot / (wall_max * 1e-3),
            "rooflines": {
                "emis": _decode_emis_roofline(c, t, flops, em_ms, name),
                "score": {"kernel": "k_fwd_cells32" if leg == "forward" else "k_vit_cells", "bound": "hbm", "achieved": sbytes / (sc_ms * 1e-3) / 1e9,
                          "peak": t["pk"]["hbm_gbs"], "unit": "GB/s", "frac": sbytes / (sc_ms * 1e-3) / 1e9 / t["pk"]["hbm_gbs"],
                          "algorithmic_bytes": sbytes, "traffic": t["traffic"].get(name, {}).get("score" if leg == "forward" else "viterbi")}},
        }
        if leg == "forward":
            labg, _ = c.rank(sco)
            top1 = float(np.mean(labg == lab))
        del sco
    res["top1_matches_generating_word"] = top1
    c.close()
    del x
    torch.cuda.empty_cache()
    return res


def run_c4(t, args):
    return _decode_config(t, args, "c4", "BASELINE configs[3]: %d utterances against a %d-word model set (N=5, M=3), utterances sharded over the GPUs"
                          % (args.c4_utts, C4_WORDS), C4_WORDS, 5, 3, args.c4_utts, seed=4004)


def run_c5(t, args):
    return _decode_config(t, args, "c5", "BASELINE configs[4]: N=3, M=128, all %d models, %d utterances sharded over the GPUs" % (args.c5_models, C5_UTTS),
                          args.c5_models, 3, 128, C5_UTTS, seed=5005)


# ========================================================================== reference arm ====
def _ref_tag(M):
    return "d39m16" if M <= 16 else "d39m128"


def _write_word_files(tmp, x, off, labels, word, tag):
    """Feature files + list file of the utterances of one word; returns (list path, frames)."""
    from oracle import ref as r
    us = np.nonzero(labels == word)[0]
    files = []
    for u in us:
        f = os.path.join(tmp, "%s_w%d_u%d.bin" % (tag, word, u))
        r.write_features(f, x[off[u]:off[u + 1]])
        files.append(f)
    lst = os.path.join(tmp, "%s_list_w%d.txt" % (tag, word))
    open(lst, "w").write("\n".join(files) + "\n")
    return lst, int(sum(off[u + 1] - off[u] for u in us))


def _ref_iterations(tag, N, M, lst, out_hmm, need):
    """EM-iteration durations of the reference trainer on one word's list: the trainer is run (to its own convergence) as
    often as it takes to collect `need` iterations."""
    from oracle import ref as r
    d = []
    while len(d) < need:
        d += r.run_train_cli_timed(tag, "w", N, M, lst, out_hmm, stack_unlimited=(M > 16))
    return d[:need]


def reference_em(w, world, steps, warmup, cores):
    """The reference trainer on the FULL workload: one process per word model and rank shard (as the reference is used: one
    invocation per word), `cores` of them at a time.  Every job runs its EM loop until it has done warmup + steps
    iterations; the step time of the job set is the slowest worker's time for its jobs' `steps` timed iterations."""
    import concurrent.futures as cf
    tag = _ref_tag(w["M"])
    base = "/dev/shm" if os.path.isdir("/dev/shm") else None
    tmp = tempfile.mkdtemp(prefix="hmmref_", dir=base)
    jobs = []
    for rk in range(world):
        x, off, labels, _ = make_workload(w, rk)
        for word in range(w["V"]):
            lst, frames = _write_word_files(tmp, x, off, labels, word, "r%d" % rk)
            jobs.append((lst, frames, os.path.join(tmp, "r%d_w%d.hmm" % (rk, word))))
    workers = max(1, min(cores, len(jobs)))
    shares = [jobs[k::workers] for k in range(workers)]

    def work(share):
        tsum, fsum = 0.0, 0
        for lst, frames, hmm in share:
            d = _ref_iterations(tag, w["N"], w["M"], lst, hmm, warmup + steps)
            tsum += sum(d[warmup:])
            fsum += frames
        return tsum, fsum
    t0 = time.perf_counter()
    with cf.ThreadPoolExecutor(workers) as ex:
        res = list(ex.map(work, shares))
    wall = time.perf_counter() - t0
    import shutil
    shutil.rmtree(tmp, ignore_errors=True)
    t_steps = max(r[0] for r in res)
    frames = sum(r[1] for r in res)
    return {"frames": frames, "seconds_for_steps": t_steps, "workers": workers, "jobs": len(jobs), "wall_s": wall}


def cpu_baseline(w, budget_s=15.0):
    """The reference trainer (oracle/_ref, gcc -O2, single-threaded by construction) on ONE host core: all utterances of one
    word of the workload, EM iterations timed inside the run (initial-model builder excluded, BASELINE.md section 4)."""
    from oracle import ref as r
    tag = _ref_tag(w["M"])
    if not r.available(tag):
        return {"value": None, "unit": "frames/s", "cores": 1, "kind": "reference", "sample": "oracle/_ref missing"}
    tmp = tempfile.mkdtemp(prefix="hmmref1_")
    x, off, labels, _ = make_workload(w, 0)
    lst, frames = _write_word_files(tmp, x, off, labels, 0, "b")
    d = []
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < budget_s and len(d) < 200:
        d += r.run_train_cli_timed(tag, "w", w["N"], w["M"], lst, os.path.join(tmp, "m.hmm"), stack_unlimited=(w["M"] > 16))
    import shutil
    shutil.rmtree(tmp, ignore_errors=True)
    use = d[1:] if len(d) > 1 else d
    return {"value": frames / float(np.median(use)), "unit": "frames/s", "cores": 1, "kind": "reference",
            "sample": "the %d utterances (%d frames) of one word of the workload, %d EM iterations of the reference trainer binary (oracle/_ref/hmm_fs_%s), "
                      "each timed inside its run (median), initial-model builder excluded" % (int((labels == 0).sum()), frames, len(use), tag),
            "host_cores_available": os.cpu_count()}


def c1_cli_wall_clock():
    """BASELINE configs[0] end to end through the drop-in programs and through the reference's own: 10 words, N=5, M=3,
    20 training + 2 test utterances per word (SURVEY 8d); `train` = the ten trainer invocations one after the other,
    `test` = one recogniser invocation over the 20 test utterances.  Wall clock of the processes, files on tmpfs."""
    import shutil
    import subprocess
    from oracle import ref as r
    from speech_recognition_hmm_continuous_b200 import api, synth
    V, N, M = 10, 5, 3
    base = "/dev/shm" if os.path.isdir("/dev/shm") else None
    tmp = tempfile.mkdtemp(prefix="hmmc1_", dir=base)
    try:
        cen, s = synth.make_centres(V, N, M, D, seed=1234)
        lab_tr = np.repeat(np.arange(V), 20)
        lab_te = np.repeat(np.arange(V), 2)
        xtr, otr = synth.make_utterances(cen, s, lab_tr, seed=1234)
        xte, ote = synth.make_utterances(cen, s, lab_te, seed=4321)
        lists = []
        for v in range(V):
            files = []
            for u in np.nonzero(lab_tr == v)[0]:
                f = os.path.join(tmp, "tr_w%d_u%d.bin" % (v, u))
                api.write_features(f, xtr[otr[u]:otr[u + 1]])
                files.append(f)
            lists.append(os.path.join(tmp, "train_w%d.txt" % v))
            open(lists[-1], "w").write("\n".join(files) + "\n")
        tfiles = []
        for u in range(len(lab_te)):
            f = os.path.join(tmp, "te_u%d.bin" % u)
            api.write_features(f, xte[ote[u]:ote[u + 1]])
            tfiles.append(f)
        flist, wlist = os.path.join(tmp, "test_feats.txt"), os.path.join(tmp, "test_words.txt")
        open(flist, "w").write("\n".join(tfiles) + "\n")
        open(wlist, "w").write("\n".join("word%d" % v for v in lab_te) + "\n")
        bindir = os.path.join(os.path.dirname(api.LIB_PATH), "bin")
        arms = {"ours": (os.path.join(bindir, "hmm_continuous_fs"), os.path.join(bindir, "recognition_continuous_fs")),
                "reference": (os.path.join(r.REF_DIR, "hmm_fs_d39m16"), os.path.join(r.REF_DIR, "rec_fs_d39m16"))}
        out = {"workload": "BASELINE configs[0]: 10 words, N=5, M=3, D=39, 20 training + 2 test utterances per word, full CLI train -> test"}
        arms["ours_one_process"] = arms["ours"]   # the trainer's job-file mode: all ten words in one process, one CUDA context
        for arm, (tr, te) in arms.items():
            if not (os.path.exists(tr) and os.path.exists(te)):
                out[arm] = {"unavailable": "program missing"}
                continue
            d = os.path.join(tmp, arm)
            os.makedirs(d)
            t0 = time.perf_counter()
            if arm == "ours_one_process":
                jf = os.path.join(d, "jobs.txt")
                open(jf, "w").write("".join("word%d %d 1 %d %s %s\n" % (v, N, M, lists[v], os.path.join(d, "w%d.hmm" % v)) for v in range(V)))
                subprocess.run([tr, "@" + jf], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            else:
                for v in range(V):
                    subprocess.run([tr, "word%d" % v, str(N), "1", str(M), lists[v], os.path.join(d, "w%d.hmm" % v)], check=True,
                                   stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            t_train = time.perf_counter() - t0
            mlist = os.path.join(d, "models.txt")
            open(mlist, "w").write("\n".join(os.path.join(d, "w%d.hmm" % v) for v in range(V)) + "\n")
            t0 = time.perf_counter()
            subprocess.run([te, "1", mlist, "1", flist, wlist, os.path.join(d, "result.txt")], check=True, stdout=subprocess.DEVNULL,
                           stderr=subprocess.DEVNULL)
            t_test = time.perf_counter() - t0
            acc = None
            for line in open(os.path.join(d, "result.txt"), errors="replace"):
                if "otal" in line and "%" in line:
                    acc = line.strip()
            out[arm] = {"train_s": t_train, "test_s": t_test, "total_s": t_train + t_test, "last_total_line": acc}
        try:  # where one drop-in invocation spends its wall clock (HMMCU_TRACE, train_main.c)
            tr = arms["ours"][0]
            pr = subprocess.run([tr, "word0", str(N), "1", str(M), lists[0], os.path.join(tmp, "trace.hmm")], stdout=subprocess.DEVNULL,
                                stderr=subprocess.PIPE, env=dict(os.environ, HMMCU_TRACE="1"))
            out["one_invocation_trace"] = [ln.strip() for ln in pr.stderr.decode(errors="replace").splitlines() if ln.startswith("[hmmcu]")]
            t0 = time.perf_counter()
            subprocess.run([tr], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)   # usage text only: the cost of loading the program
            out["program_load_s"] = time.perf_counter() - t0
            jf = os.path.join(tmp, "ours_one_process", "jobs.txt")
            if os.path.exists(jf):
                pr = subprocess.run([tr, "@" + jf], stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, env=dict(os.environ, HMMCU_TRACE="1"))
                out["job_file_trace"] = [ln.strip() for ln in pr.stderr.decode(errors="replace").splitlines() if ln.startswith("[hmmcu]")][:24]
            d1 = os.path.join(tmp, "ours_one_process")
            pr = subprocess.run([arms["ours"][1], "1", os.path.join(d1, "models.txt"), "1", flist, wlist, os.path.join(tmp, "trace_result.txt")],
                                stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, env=dict(os.environ, HMMCU_TRACE="1"))
            out["recogniser_trace"] = [ln.strip() for ln in pr.stderr.decode(errors="replace").splitlines() if ln.startswith("[hmmcu]")]
        except Exception as e:  # noqa: BLE001
            out["one_invocation_trace"] = "unavailable: %s" % e
        if "total_s" in out.get("ours", {}) and "total_s" in out.get("reference", {}):
            out["speedup_total"] = out["reference"]["total_s"] / out["ours"]["total_s"]
            if "total_s" in out.get("ours_one_process", {}):
                out["speedup_total_one_process"] = out["reference"]["total_s"] / out["ours_one_process"]["total_s"]
            out["note"] = ("each drop-in invocation creates its own CUDA context (0.25 s beside a process that already holds one, 1-3 s on "
                           "an otherwise idle GPU of this pool; see the traces); at this size that start-up is most of the wall clock of "
                           "the drop-in programs, the work itself (ingest, initial model, EM loop) is a few ms per word")
        return out
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    from oracle import ref as r
    w = WORKLOADS[args.workload]
    tag = _ref_tag(w["M"])
    if not r.available(tag):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/hmm_fs_%s not built (oracle/build_ref.sh needs /root/reference)" % tag}))
        return
    cores = os.cpu_count() or 1
    res = reference_em(w, world, args.steps, args.warmup, cores)
    ms_step = res["seconds_for_steps"] / args.steps * 1e3
    value = res["frames"] / (ms_step * 1e-3)
    sample = ("the full workload: %d trainer processes (one per word model and GPU shard, %d utterances each), %d at a time on %d host cores; "
              "every process runs %d + %d EM iterations (re-running the trainer until it has), each timed inside its run; initial-model builder excluded"
              % (res["jobs"], w["U"] // w["V"], res["workers"], cores, args.warmup, args.steps))
    print(json.dumps({
        "impl": "reference", "metric": "frames/sec per Baum-Welch EM iteration", "value": value, "unit": "frames/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.workload, world),
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": res["workers"], "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": res["wall_s"],
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-configs", action="store_true", help="skip the full-size c3 / c4 / c5 legs")
    ap.add_argument("--no-ingest", action="store_true", help="skip the feature-file ingest leg")
    ap.add_argument("--no-init", action="store_true", help="skip the initial-model leg")
    ap.add_argument("--no-cli", action="store_true", help="skip the C1 drop-in CLI wall-clock leg")
    ap.add_argument("--no-affinity", action="store_true", help="do not bind the rank to its GPU's NUMA-local CPUs")
    ap.add_argument("--torch-allreduce", action="store_true", help="all-reduce through torch.distributed instead of the NCCL C API")
    ap.add_argument("--nccl-allreduce", action="store_true", help="ncclAllReduce instead of the library's peer-memory kernels")
    ap.add_argument("--upload-chunks", type=int, default=0, help="override the library's upload chunk count (experiments)")
    ap.add_argument("--set", action="append", default=[], metavar="KEY=INT", help="hmmcu_set_option switches (experiments)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--c3-utts", type=int, default=C3_UTTS)
    ap.add_argument("--c4-utts", type=int, default=C4_UTTS)
    ap.add_argument("--c5-models", type=int, default=C5_MODELS)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed EM iteration computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
