"""Device timeline of graph-replayed EM iterations at the bench's workload (C2 by default):

   python scripts/step_timeline.py [--workload c2] [--iters 5] [--warmup 5] [--out DIR]

Builds the context as bench.py does (features resident in HBM, threshold -1 so that every word is re-estimated),
replays a few warm EM iterations under torch.profiler with CUDA activities, each after the bench's 256 MiB L2 flush,
and prints for every kernel, memset and copy of an iteration its stream, start (us after the iteration's first
event), duration and the gap before it: the start minus the latest end of any earlier event of the iteration (negative
when it overlaps the previous one, e.g. under programmatic dependent launch).  The per-iteration table and a summary
(median over the iterations) go to DIR/timeline.txt, the chrome trace to DIR/step_timeline.pt.trace.json."""
import argparse
import json
import os
import re
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def short_name(name):
    m = re.search(r"(k_\w+)(<[^()]*>)?", name)
    return (m.group(1) + (m.group(2) or "")) if m else name[:40]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c2")
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default="step_timeline_out")
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    import bench
    from speech_recognition_hmm_continuous_b200 import api

    w = bench.WORKLOADS[args.workload]
    x, off, labels, mods = bench.make_workload(w, 0)
    dev = torch.device("cuda", 0)
    xdev = torch.from_numpy(x).to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ctx = api.Context(0, timing=False)
    ctx.set_features_device(xdev.data_ptr(), off, bench.D)
    ctx.set_models(api.ModelSet.from_dict(mods))
    ctx.em_reset()

    def em_iteration():
        ctx.estep(labels, download=False, want_logp=False)
        return ctx.mstep(threshold=-1.0)

    for _ in range(args.warmup):  # the third call of each launch sequence captures its graph; later ones replay it
        em_iteration()
    ctx.synchronize()
    torch.cuda.synchronize()
    os.makedirs(args.out, exist_ok=True)
    trace = os.path.join(args.out, "step_timeline.pt.trace.json")
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(args.iters):
            flush.fill_(i & 0xFF)
            torch.cuda.synchronize()
            em_iteration()
            ctx.synchronize()
    prof.export_chrome_trace(trace)
    ev = [e for e in json.load(open(trace))["traceEvents"]
          if e.get("ph") == "X" and e.get("cat") in ("kernel", "gpu_memset", "gpu_memcpy")]
    ev.sort(key=lambda e: e["ts"])
    # iterations: the library's events between two of the flush kernels
    iters, cur = [], None
    for e in ev:
        if e["cat"] == "kernel" and "hmmk::" not in e["name"] and "k_" not in e["name"]:
            if cur:
                iters.append(cur)
            cur = []
        elif cur is not None:
            cur.append(e)
    if cur:
        iters.append(cur)
    lines = []
    props = torch.cuda.get_device_properties(0)
    lines.append("device: %s (%d SMs); workload %s: %s" % (props.name, props.multi_processor_count, args.workload, w["desc"]))
    rows = {}
    spans = []
    for k, it in enumerate(iters):
        t0 = it[0]["ts"]
        end = t0
        lines.append("")
        lines.append("iteration %d" % k)
        lines.append("%-34s %6s %9s %9s %9s" % ("event", "stream", "start_us", "dur_us", "gap_us"))
        seen = {}
        for e in it:
            nm = short_name(e["name"]) if e["cat"] == "kernel" else e["cat"]
            gap = e["ts"] - end
            lines.append("%-34s %6s %9.2f %9.2f %9.2f" % (nm, e["args"].get("stream", "?"), e["ts"] - t0, e["dur"], gap))
            n = seen.get(nm, 0)
            seen[nm] = n + 1
            rows.setdefault((nm, n), []).append((e["ts"] - t0, e["dur"], gap))
            end = max(end, e["ts"] + e["dur"])
        spans.append(end - t0)
        lines.append("span (first start to last end): %.2f us" % (end - t0))
    lines.append("")
    lines.append("median over %d iterations" % len(iters))
    lines.append("%-34s %9s %9s %9s" % ("event", "start_us", "dur_us", "gap_us"))
    order = sorted(rows, key=lambda r: np.median([v[0] for v in rows[r]]))
    gaps = 0.0
    for r in order:
        a = np.array(rows[r])
        med = np.median(a, axis=0)
        gaps += max(med[2], 0.0)
        lines.append("%-34s %9.2f %9.2f %9.2f" % (r[0], med[0], med[1], med[2]))
    lines.append("iteration span: median %.2f us (min %.2f, max %.2f); sum of positive median gaps %.2f us"
                 % (np.median(spans), min(spans), max(spans), gaps))
    text = "\n".join(lines)
    with open(os.path.join(args.out, "timeline.txt"), "w") as f:
        f.write(text + "\n")
    print(text)
    ctx.close()


if __name__ == "__main__":
    main()
