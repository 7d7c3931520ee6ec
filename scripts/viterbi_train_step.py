"""Time one Viterbi-training EM iteration (hmmcu_estep_viterbi + hmmcu_mstep) against one Baum-Welch iteration
(hmmcu_estep + hmmcu_mstep) at the bench's workload (C2 by default), in one process:

   python scripts/viterbi_train_step.py [--workload c2] [--steps 200] [--runs 5] [--out DIR]

The context is built as bench.py builds it (features resident in HBM, threshold -1 so that every word is re-estimated
every iteration).  Runs of --steps graph-replayed iterations alternate between the two kinds on one context; each run's
time is a host clock around the run, which ends in the M-step's read-back.  Reported: the median and range of the
per-iteration time over --runs runs of each kind, then, in a separate pass with the per-kernel timers on (no graphs),
the device time of the alignment kernel ("align") and of the forward-backward it replaces ("fwdbwd"), medians of 20
iterations.  The card's name and power limit are read in the same process.  One JSON line goes to stdout (and to
DIR/viterbi_train_step.json with --out)."""
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c2")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import bench
    from speech_recognition_hmm_continuous_b200 import api

    w = bench.WORKLOADS[args.workload]
    x, off, labels, mods = bench.make_workload(w, 0)
    dev = torch.device("cuda", 0)
    xdev = torch.from_numpy(x).to(dev)
    ctx = api.Context(0)
    ctx.set_features_device(xdev.data_ptr(), off, bench.D)
    ctx.set_models(api.ModelSet.from_dict(mods))
    ctx.em_reset()

    def bw():
        ctx.estep(labels, download=False, want_logp=False)
        return ctx.mstep(threshold=-1.0)

    def vit():
        ctx.estep_viterbi(labels, download=False, want_logp=False)
        return ctx.mstep(threshold=-1.0)

    kinds = {"baum_welch": bw, "viterbi": vit}
    for fn in kinds.values():  # the third call of each launch sequence captures its graph; later ones replay it
        for _ in range(10):
            fn()
    ms = {k: [] for k in kinds}
    for _ in range(args.runs):
        for k, fn in kinds.items():
            ctx.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                fn()
            ms[k].append((time.perf_counter() - t0) * 1e3 / args.steps)
    ctx.enable_timing(True)
    kern = {"align": [], "fwdbwd": []}
    for _ in range(20):
        vit()
        kern["align"].append(ctx.kernel_ms("align"))
        bw()
        kern["fwdbwd"].append(ctx.kernel_ms("fwdbwd"))
    ctx.enable_timing(False)
    ctx.close()
    props = torch.cuda.get_device_properties(0)
    res = {"device": props.name, "power_limit_w": power_limit_w(), "workload": args.workload, "desc": w["desc"],
           "steps_per_run": args.steps, "runs": args.runs}
    for k, v in ms.items():
        res[k + "_ms_per_step"] = {"median": float(np.median(v)), "min": float(min(v)), "max": float(max(v))}
    for k, v in kern.items():
        res[k + "_kernel_ms"] = float(np.median(v))
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "viterbi_train_step.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
