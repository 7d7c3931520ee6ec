"""Time one MMI iteration (hmmcu_estep_mmi + hmmcu_mstep_ebw) against one Baum-Welch iteration (hmmcu_estep +
hmmcu_mstep) in one process, at the bench's C2 shape (10 words, N = 5, M = 16, 1,000 utterances) and at the same corpus
shape with 100 words:

   python scripts/mmi_step.py [--steps 20] [--runs 5] [--max-hyp 4] [--out DIR]

The context is built as bench.py builds it (features resident in HBM; Baum-Welch with threshold -1, so that every word
is re-estimated every iteration).  kappa is set from the forward scores so that the median utterance's best competitor
sits 3 nats below its label (a soft, many-round setting).  Runs of --steps iterations alternate between the two kinds;
each run's time is a host clock around the run, which ends in a synchronising read-back.  Then, with the per-kernel
timers on (no graphs), the stages of the MMI iteration: scoring ("mmi_score"), posteriors ("mmi_post"), numerator E-step
("mmi_num"), the denominator rounds ("mmi_den", and how many), the EBW M-step ("mstep"), medians of 5 iterations.  The
card's name and power limit are read in the same process.  One JSON line per shape goes to stdout (and to
DIR/mmi_step.json with --out)."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def power_limit_w():
    try:
        import pynvml
        pynvml.nvmlInit()
        return pynvml.nvmlDeviceGetPowerManagementLimit(pynvml.nvmlDeviceGetHandleByIndex(0)) / 1000.0
    except Exception:
        return None


def kappa_for(S, labels, spread=3.0):
    gaps = [abs(S[u, labels[u]] - np.max(np.delete(S[u], labels[u]))) for u in range(len(labels)) if np.isfinite(S[u, labels[u]])]
    return spread / max(float(np.median(gaps)), 1e-9)


def run_shape(name, w, args, api, bench, torch):
    x, off, labels, mods = bench.make_workload(w, 0)
    xdev = torch.from_numpy(x).to(torch.device("cuda", 0))
    ctx = api.Context(0)
    ctx.set_features_device(xdev.data_ptr(), off, bench.D)
    ms = api.ModelSet.from_dict(mods)
    ctx.set_models(ms)
    kappa = kappa_for(ctx.forward_scores(), labels)

    def bw():
        ctx.estep(labels, download=False, want_logp=False)
        return ctx.mstep(threshold=-1.0)

    def mmi():
        ctx.estep_mmi(labels, kappa, args.max_hyp, download=False)
        ctx.mstep_ebw(2.0, 100.0)

    # every run starts from the same models, so that the hypotheses do not drift with the iterations
    def reset():
        ctx.set_models(ms)
        ctx.em_reset()

    kinds = {"baum_welch": bw, "mmi": mmi}
    for fn in kinds.values():
        reset()
        for _ in range(3):
            fn()
    t = {k: [] for k in kinds}
    for _ in range(args.runs):
        for k, fn in kinds.items():
            reset()
            ctx.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                fn()
            t[k].append((time.perf_counter() - t0) * 1e3 / args.steps)
    ctx.enable_timing(True)
    stages = {k: [] for k in ("mmi_score", "mmi_post", "mmi_num", "mmi_den", "mmi_rounds", "mstep")}
    reset()
    for _ in range(5):
        mmi()
        for k in stages:
            stages[k].append(ctx.kernel_ms(k))
    ctx.enable_timing(False)
    ctx.close()
    res = {"shape": name, "desc": w["desc"], "kappa": kappa, "max_hyp": args.max_hyp, "E": 2.0, "tau": 100.0,
           "steps_per_run": args.steps, "runs": args.runs}
    for k, v in t.items():
        res[k + "_ms_per_iteration"] = {"median": float(np.median(v)), "min": float(min(v)), "max": float(max(v))}
    for k, v in stages.items():
        res[k if k == "mmi_rounds" else k + "_ms"] = float(np.median(v))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--max-hyp", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import bench
    from speech_recognition_hmm_continuous_b200 import api

    c2 = bench.WORKLOADS["c2"]
    shapes = {"c2": c2, "v100": dict(c2, V=100, desc="C2 with 100 words: N=5 M=16 D=39, 1000 utterances")}
    props = torch.cuda.get_device_properties(0)
    lines = []
    for name, w in shapes.items():
        res = run_shape(name, w, args, api, bench, torch)
        res.update({"device": props.name, "power_limit_w": power_limit_w()})
        lines.append(json.dumps(res))
        print(lines[-1], flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "mmi_step.json"), "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
